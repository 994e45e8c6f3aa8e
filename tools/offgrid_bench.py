#!/usr/bin/env python
"""Cost of off-grid sources and receivers (spec B7): the same calls with the points on the grid and shifted off it, in one
process.

    python tools/offgrid_bench.py [--nt 5000] [--grid 1000x3000] [--reps 5] [--nt3 200] [--grid3 512] [--no-profile]

2-D: bench.py's layered model and the middle shot of its 64-shot geometry (one source at z = 4, a receiver at z = 4 in every
column but the last), and the same shot with every point shifted by (+0.5, +0.5) cells: 8 x 8 taps per point, 8 x 3000
receiver cells.
Per-shot forward, gradient, Born and Gauss-Newton.  3-D: ms per step launch of a forward over --nt3 steps on a --grid3
cube with bench.py's config-4 geometry (source at (8, n/2, n/2), receivers at z = 6 every 8 cells in y and x), on the grid
and with every point shifted by (+0.5, +0.5, +0.5).  One plan per setting, both warmed up (two calls each) before timing;
the timed calls alternate on / off grid, `--reps` of each, timed with CUDA events; the median and the spread are printed.
Then, unless --no-profile, one forward and one gradient shot of each 2-D setting under torch.profiler: device time per
kernel.  The card's name and power limit are printed in the same run."""
from __future__ import annotations

import argparse
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(ROOT))

import numpy as np  # noqa: E402
from born_bench import card_info  # noqa: E402
from free_surface_bench import alternate, fmt  # noqa: E402


def report(name, res, per=1.0, unit="ms"):
    on, off = np.median(res["on"]) / per, np.median(res["off"]) / per
    print("  %-13s on grid %9.3f %s   off grid %9.3f %s   off / on %.4f   (on %s | off %s)"
          % (name, on, unit, off, unit, off / on, fmt(res["on"]), fmt(res["off"])))


def kernel_times(fn):
    """{kernel name: (launches, device ms)} of one call of fn."""
    import warnings
    import torch
    from torch.profiler import ProfilerActivity, profile
    warnings.filterwarnings("ignore", message=".*Profiler clears events.*")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            out[e.key] = (e.count, t / 1000.0)
    return out


def print_kernels(name, times):
    print("  %s:" % name)
    for k, (n, ms) in sorted(times.items(), key=lambda kv: -kv[1][1])[:8]:
        print("    %9.3f ms  %6d x  %s" % (ms, n, k[:110]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nt", type=int, default=5000)
    ap.add_argument("--grid", default="1000x3000")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--nt3", type=int, default=200)
    ap.add_argument("--grid3", type=int, default=512)
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args()
    import torch
    from full_waveform_inversion_b200 import acoustic as ac
    from oracle import fd_oracle as fo

    name, q = card_info()
    print("card: %s | nvidia-smi name, power limit, max SM clock: %s" % (name, q))
    nz, nx = (int(x) for x in args.grid.lower().split("x"))
    nt, h = args.nt, 10.0
    v = torch.from_numpy(fo.layered_model((nz, nx), 1500.0, 4500.0, 6).astype(np.float32)).cuda()     # bench.py's workload
    dt = fo.stable_dt(4500.0, h, 2)
    wav = torch.from_numpy(fo.ricker(nt, dt, 10.0).astype(np.float32)).cuda()
    sx = int(np.linspace(60, nx - 61, 64).astype(int)[32])
    src, rec = np.array([(4, sx)]), np.array([(4, x) for x in range(nx - 1)])
    geoms = {"on": (src, rec), "off": (src + 0.5, rec + 0.5)}
    zz, xx = np.meshgrid(np.arange(nz), np.arange(nx), indexing="ij")
    dv = sum(np.exp(-((zz - z0) ** 2 + (xx - x0) ** 2) / (2.0 * 20.0 ** 2)) for z0, x0 in ((200, sx), (450, sx - 400), (700, sx + 300)))
    dv = torch.from_numpy(dv.astype(np.float32)).cuda()
    print("2-D workload: %dx%d, nt = %d, one shot: source at (4, %d), %d receivers at z = 4, x = 0 .. %d; off grid every "
          "point + (0.5, 0.5); default plan, %d alternating reps" % (nz, nx, nt, sx, nx - 1, nx - 2, args.reps))

    plans, bufs = {}, {}
    for k, (s, r) in geoms.items():
        p = ac.Propagator((nz, nx), h, dt, nabs=40)
        p.set_model(v)
        p.set_geometry(s, r)
        p.reserve(nt, gradient=True)
        plans[k] = p
        bufs[k] = dict(obs=torch.zeros((nt, len(r)), dtype=torch.float32, device="cuda"),
                       grad=torch.zeros((nz, nx), dtype=torch.float32, device="cuda"),
                       out=torch.empty((nt, len(r)), dtype=torch.float32, device="cuda"))
    calls = {
        "forward": {k: (lambda k=k: plans[k].forward(wav, out=bufs[k]["out"])) for k in plans},
        "gradient": {k: (lambda k=k: plans[k].gradient(wav, bufs[k]["obs"], grad=bufs[k]["grad"], want_misfit=False)) for k in plans},
        "born": {k: (lambda k=k: plans[k].born(wav, dv, out=bufs[k]["out"])) for k in plans},
        "gauss_newton": {k: (lambda k=k: plans[k].gauss_newton(wav, dv, hv=bufs[k]["grad"])) for k in plans},
    }
    print("\nper shot:")
    for op, c in calls.items():
        report(op, alternate(c, args.reps))
    launches = {k: p.launch_count() for k, p in plans.items()}
    print("  launches so far: on grid %d, off grid %d" % (launches["on"], launches["off"]))
    if not args.no_profile:
        print("\ndevice time per kernel, one shot (torch.profiler; a separate run from the timings above):")
        for op in ("forward", "gradient"):
            for k in plans:
                print_kernels("%s, %s grid" % (op, k), kernel_times(calls[op][k]))
    for p in plans.values():
        p.close()
    del plans, bufs
    torch.cuda.empty_cache()

    n3, nt3 = args.grid3, args.nt3
    shape = (n3, n3, n3)
    dt3 = fo.stable_dt(4500.0, h, 3)
    v3 = torch.from_numpy(np.linspace(1500.0, 4500.0, n3, dtype=np.float32)).cuda()[:, None, None].expand(shape).contiguous()
    w3 = torch.from_numpy(fo.ricker(nt3, dt3, 8.0).astype(np.float32)).cuda()
    src3 = np.array([(8, n3 // 2, n3 // 2)])
    rec3 = np.array([(6, y, x) for y in range(16, n3 - 16, 8) for x in range(16, n3 - 16, 8)])
    geoms3 = {"on": (src3, rec3), "off": (src3 + 0.5, rec3 + 0.5)}
    print("\n3-D workload: %d^3, forward over nt = %d steps, config-4 geometry (%d receivers at z = 6), off grid every point "
          "+ (0.5, 0.5, 0.5); time per step launch:" % (n3, nt3, len(rec3)))
    plans = {}
    for k, (s, r) in geoms3.items():
        p = ac.Propagator(shape, h, dt3, nabs=24)
        p.set_model(v3)
        p.set_geometry(s, r)
        p.reserve(nt3, gradient=False)
        plans[k] = p
    out3 = {k: torch.empty((nt3, len(rec3)), dtype=torch.float32, device="cuda") for k in plans}
    report("forward step", alternate({k: (lambda k=k: plans[k].forward(w3, out=out3[k])) for k in plans}, args.reps),
           per=nt3 / 1000.0, unit="us")
    for p in plans.values():
        p.close()


if __name__ == "__main__":
    main()
