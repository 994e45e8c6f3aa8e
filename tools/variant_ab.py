"""Tuning aid: times the bench workload's forward and gradient and prints SHA-256 digests of the traces and the gradient,
so two builds (two checkouts, run one after the other) can be compared for bit-identity.
  python tools/variant_ab.py [nt]"""
import sys, os, hashlib
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from full_waveform_inversion_b200 import _lib
from full_waveform_inversion_b200 import acoustic as ac

class A: grid = "1000x3000"; nt = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
w = bench.workload(A)
dev = torch.device("cuda", 0)
prop = ac.Propagator2D((w["nz"], w["nx"]), w["h"], w["dt"], nabs=w["nabs"], alpha=w["alpha"])
v = torch.from_numpy(w["v"]).to(dev)
prop.set_model(v * 1.02); prop.set_geometry(*w["shots"][0])
wav = torch.from_numpy(w["wav"]).to(dev)
obs = prop.forward(wav).clone()
prop.set_model(v)
grad = torch.zeros((w["nz"], w["nx"]), device=dev)
tr = prop.forward(wav).clone()
prop.gradient(wav, obs, grad=grad, want_misfit=False)
torch.cuda.synchronize()
print("lib", _lib.LIB_PATH)
print("traces", hashlib.sha256(tr.cpu().numpy().tobytes()).hexdigest()[:16], "gradient", hashlib.sha256(grad.cpu().numpy().tobytes()).hexdigest()[:16])
for name, fn in (("forward", lambda: prop.forward(wav)), ("gradient", lambda: prop.gradient(wav, obs, grad=grad, want_misfit=False))):
    ts = []
    for rep in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3 / (2 * A.nt))
    print("%s us per time step: %s" % (name, " ".join("%.2f" % t for t in ts)), flush=True)
