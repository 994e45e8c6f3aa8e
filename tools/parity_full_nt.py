"""Track B parity at the FULL bench workload (1000 x 3000, 3000 receivers, nt = 5000) against the float64 self-oracle
(checkpointed on the CPU side: segments of 100 steps).  Takes a few minutes of host time, so it is a tool run once per
round, not a test; the output goes to profiles/.   python tools/parity_full_nt.py [nt] [grid]

Besides the global rel-L2 it prints the region/window table of oracle/fd_check.py: rel-L2 per receiver group (near /
far from the source) x 1000-step window and per gradient region (sponge strips, last tile row / column, interior), next
to the float32 port's on the same selection and the selection's share of the float64 norm - the global norms are
dominated by the strong early arrivals next to the source."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from full_waveform_inversion_b200 import acoustic as ac
from oracle import fd_check as fc, fd_oracle as fo, fd_oracle_c as foc

nt = int(sys.argv[1]) if len(sys.argv) > 1 else 5000
nz, nx = (int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "1000x3000").split("x"))
rel = fc.rel_l2
v = fo.layered_model((nz, nx), 1500.0, 4500.0, 6).astype(np.float32)
h, nabs = 10.0, 40
dt = fo.stable_dt(4500.0, h, 2)
wav = fo.ricker(nt, dt, 10.0).astype(np.float32)
src, rec = [(4, nx // 3)], [(4, x) for x in range(nx)]
prop = ac.Propagator2D((nz, nx), h, dt, nabs=nabs)
prop.set_model(torch.from_numpy(v) * 1.02)
prop.set_geometry(src, rec)
obs = prop.forward(wav).clone()
prop.set_model(v)
J, g, tr = prop.gradient(wav, obs, want_traces=True)
g, tr, obs_h = g.cpu().numpy(), tr.cpu().numpy(), obs.cpu().numpy()
prop.close()
t0 = time.perf_counter()
J64, g64, tr64 = foc.misfit_and_gradient(v, h, dt, src, rec, wav, obs_h, nabs=nabs, dtype=np.float64, seg=100)
t64 = time.perf_counter() - t0
t0 = time.perf_counter()
J32, g32, tr32 = foc.misfit_and_gradient(v, h, dt, src, rec, wav, obs_h, nabs=nabs, dtype=np.float32, seg=100)
t32 = time.perf_counter() - t0
d = fc.Decomp.for_plan((nz, nx), torch.cuda.get_device_properties(0).multi_processor_count, nabs)
print("grid %dx%d nt=%d, %d receivers, default CUDA path (%s, PDL + graphs) on %s vs float64 self-oracle (%d host threads, %.0f s; float32 port %.0f s)"
      % (nz, nx, nt, len(rec), d, torch.cuda.get_device_name(0), foc.num_threads(), t64, t32))
print("  GPU      : traces rel-L2 %.3e   gradient rel-L2 %.3e   misfit rel %.3e" % (rel(tr, tr64), rel(g, g64), abs(J - J64) / J64))
print("  CPU fp32 : traces rel-L2 %.3e   gradient rel-L2 %.3e   misfit rel %.3e   (the specification's own fp32 noise at this size)" % (rel(tr32, tr64), rel(g32, g64), abs(J32 - J64) / J64))
sx = src[0][1]
xs = np.array([x for _, x in rec])
groups = {"receivers |x - xs| <= 600": np.nonzero(np.abs(xs - sx) <= 600)[0], "receivers |x - xs| > 600": np.nonzero(np.abs(xs - sx) > 600)[0]}
windows = [(k, min(nt, k + 1000)) for k in range(0, nt, 1000)]
rows = fc.region_table(tr, tr32, tr64, fc.trace_selections(groups, nt, windows))
masks = d.masks()
masks["lower half z >= %d" % (nz // 2)] = np.broadcast_to((np.arange(nz) >= nz // 2)[:, None], (nz, nx))
rows += fc.region_table(g, g32, g64, {"gradient " + k: m for k, m in masks.items()})
print(fc.format_table("  per selection (a share of 0 means the float64 oracle is exactly zero there: nothing is checked)", rows))
print("  north_star tolerances: traces <= 1e-5, gradient <= 1e-4 ->", "HELD" if rel(tr, tr64) <= 1e-5 and rel(g, g64) <= 1e-4 else "NOT HELD")
