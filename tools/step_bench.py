"""Per-step timing of the 2-D step kernels (forward only, no snapshots) for several grid sizes and kernel
variants: fits t = a + b * points to separate the fixed per-launch cost from the streaming rate."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from full_waveform_inversion_b200 import acoustic as ac

def time_forward(nz, nx, nt, **kw):
    prop = ac.Propagator2D((nz, nx), 10.0, 7e-4, nabs=40, **kw)
    prop.set_model(torch.full((nz, nx), 2500.0, device="cuda"))
    prop.set_geometry([(4, nx // 2)], [(4, x) for x in range(0, nx, 4)])
    wav = torch.from_numpy(ac.ricker(nt, 7e-4, 10.0)).cuda()
    prop.forward(wav); prop.forward(wav)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); prop.forward(wav); e1.record(); torch.cuda.synchronize()
    prop.close()
    return e0.elapsed_time(e1) * 1e3 / nt     # us per step

variants = [("tile", (28, 4)), ("tile", (32, 4)), ("tile", (56, 8))]
if len(sys.argv) > 1:
    variants = []
    for a in sys.argv[1:]:
        k, v = a.split(":")
        vals = tuple(int(x) for x in v.split(","))
        variants.append((k, vals[0] if k == "tb2" else vals))
for kind, cfg in variants:
  for graphs in ((True,) if kind == 'tb2' else (True, False)):
    pts, ts = [], []
    print("graphs =", graphs)
    for nz in (125, 500, 1000, 2000, 4000):
        t = time_forward(nz, 3000, 1500, graphs=graphs, **{kind: cfg})
        pts.append(nz * 3000); ts.append(t)
        print("%s %s  %5d x 3000: %7.2f us/step  %6.1f Gpt/s" % (kind, cfg, nz, t, nz * 3000 / t / 1e3), flush=True)
    b, a = np.polyfit(pts[:4], ts[:4], 1)
    print("   fit: t = %.2f us + points / (%.1f Gpt/s)" % (a, 1e-3 / b), flush=True)
