"""Diagnostic: ms per shot-gradient for consecutive steps of the bench workload (looking for warm-up drift)."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from full_waveform_inversion_b200 import acoustic as ac

class A: grid = "1000x3000"; nt = int(sys.argv[1]) if len(sys.argv) > 1 else 5000
w = bench.workload(A)
dev = torch.device("cuda", 0)
prop = ac.Propagator2D((w["nz"], w["nx"]), w["h"], w["dt"], nabs=w["nabs"], alpha=w["alpha"])
v = torch.from_numpy(w["v"]).to(dev)
prop.set_model(v * 1.02); prop.set_geometry(*w["shots"][0])
wav = torch.from_numpy(w["wav"]).to(dev)
obs = prop.forward(wav).clone()
prop.set_model(v)
grad = torch.zeros((w["nz"], w["nx"]), device=dev)
ts = []
t_start = time.perf_counter()
for i in range(12):
    prop.set_geometry(*w["shots"][i % 64])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); prop.gradient(wav, obs, grad=grad, want_misfit=False); e1.record(); torch.cuda.synchronize()
    ts.append(e0.elapsed_time(e1))
    if i == 7:
        time.sleep(1.0)            # an idle gap, like the one between the bench's timed regions
print(" ".join("%.1f" % t for t in ts))
# back-to-back without per-step synchronisation (what the bench's device-timed region does)
torch.cuda.synchronize()
for rep in range(3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(8):
        prop.set_geometry(*w["shots"][i % 64])
        prop.gradient(wav, obs, grad=grad, want_misfit=False)
    e1.record(); torch.cuda.synchronize()
    print("8 shots back-to-back: %.1f ms/shot" % (e0.elapsed_time(e1) / 8))
