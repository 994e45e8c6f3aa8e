"""Forward and gradient time per step for the 2-D kernel variants over grid sizes (picks the auto-selection thresholds).
  python tools/variant_bench.py [nz ...]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from full_waveform_inversion_b200 import acoustic as ac

def bench(nz, nx, nt, **kw):
    prop = ac.Propagator2D((nz, nx), 10.0, 7e-4, nabs=40, **kw)
    prop.set_model(torch.full((nz, nx), 2500.0, device="cuda"))
    prop.set_geometry([(4, nx // 2)], [(4, x) for x in range(0, nx, 2)])
    wav = torch.from_numpy(ac.ricker(nt, 7e-4, 10.0)).cuda()
    obs = torch.zeros((nt, prop.nrec), device="cuda")
    out = []
    for fn in (lambda: prop.forward(wav), lambda: prop.gradient(wav, obs, want_misfit=False)):
        fn(); fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); fn(); e1.record(); torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) * 1e3 / (2 * nt))
    prop.close()
    return out          # us per forward step, us per gradient time step (forward+adjoint pair)

sizes = [int(a) for a in sys.argv[1:]] or [250, 500, 750, 1000, 1500, 2000, 3000, 4000, 6000]
for nz in sizes:
    nt = max(200, min(1000, int(2.4e9 / (nz * 3000 * 4) / 3)))       # keep the snapshots under ~2.4 GB... scaled below
    nt = min(nt, 600)
    row = []
    for name, kw in (("auto", {}), ("tile", {"tile": (32, 4)}), ("tb2:24", {"tb2": 24}), ("tb2:32", {"tb2": 32})):
        f, g = bench(nz, 3000, nt, **kw)
        row.append("%s fwd %6.2f grad %6.2f" % (name, f, g))
    print("%5d x 3000 nt %d | " % (nz, nt) + " | ".join(row), flush=True)
