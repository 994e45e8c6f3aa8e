"""Per-call times for repeated identical shots (looks for sporadic slow calls) + a torch-only control."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from full_waveform_inversion_b200 import acoustic as ac

def timed(fn, reps):
    out = []
    for i in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(); fn(); e1.record()
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        out.append((e0.elapsed_time(e1), (t1 - t0) * 1e3))
    return out

def show(tag, out):
    print(tag, "gpu ms:", " ".join("%.1f" % a for a, _ in out))
    print("   host call ms:", " ".join("%.1f" % b for _, b in out), flush=True)

def run(shape, nt, reps):
    prop = ac.Propagator(shape, 10.0, 5e-4, nabs=20)
    prop.set_model(torch.full(shape, 2500.0, device="cuda"))
    mid = tuple(s // 2 for s in shape)
    rec = [(4,) * (len(shape) - 1) + (x,) for x in range(0, shape[-1], 4)]
    prop.set_geometry([mid], rec)
    wav = torch.from_numpy(ac.ricker(nt, 5e-4, 15.0)).cuda()
    obs = torch.zeros((nt, prop.nrec), device="cuda")
    prop.gradient(wav, obs, want_misfit=False); prop.forward(wav); torch.cuda.synchronize()
    show("%s nt %d gradient" % (shape, nt), timed(lambda: prop.gradient(wav, obs, want_misfit=False), reps))
    show("%s nt %d forward " % (shape, nt), timed(lambda: prop.forward(wav), reps))
    prop.close()

# control: a torch CUDA graph of 2000 small kernels on 12 MB buffers (same launch count / footprint as a 2-D shot)
a = torch.zeros(3_000_000, device="cuda"); b = torch.ones(3_000_000, device="cuda")
s = torch.cuda.Stream()
with torch.cuda.stream(s):
    for _ in range(3): a.add_(b)
torch.cuda.current_stream().wait_stream(s)
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    for _ in range(2000): a.add_(b)
g.replay(); torch.cuda.synchronize()
show("control: torch graph, 2000 x add_ on 12 MB", timed(g.replay, 16))

run((1000, 3000), 1000, 16)
run((256, 256, 256), 60, 16)
show("control again", timed(g.replay, 16))
