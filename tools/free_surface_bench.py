#!/usr/bin/env python
"""Cost of the free-surface top boundary (spec B6): the same calls with the surface off and on, in one process.

    python tools/free_surface_bench.py [--nt 5000] [--grid 1000x3000] [--reps 5] [--nt3 200] [--grid3 512]

2-D: bench.py's layered model and the middle shot of its 64-shot geometry (one source at z = 4, a receiver in every
column at z = 4), per-shot forward, gradient, Born and Gauss-Newton.  3-D: ms per step launch of a forward over --nt3
steps on a --grid3 cube.  One plan per setting, both built and warmed up (two calls each) before timing; the timed calls
alternate off / on, `--reps` of each, timed with CUDA events; the median and the spread are printed.  The card's name
and power limit are printed in the same run."""
from __future__ import annotations

import argparse
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(ROOT))

import numpy as np  # noqa: E402
from born_bench import card_info  # noqa: E402


def event_ms(fn):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def alternate(calls, reps, warmup=2):
    """calls: {setting: fn}.  Warm-up of every setting, then `reps` rounds that time each setting once, in turn."""
    import torch
    for fn in calls.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    out = {k: [] for k in calls}
    for _ in range(reps):
        for k, fn in calls.items():
            out[k].append(event_ms(fn))
    return {k: np.array(v) for k, v in out.items()}


def fmt(ms):
    return "%8.2f ms (min %.2f, max %.2f)" % (np.median(ms), ms.min(), ms.max())


def report(name, res, per=1.0, unit="ms"):
    off, on = np.median(res["off"]) / per, np.median(res["on"]) / per
    print("  %-13s off %9.3f %s   on %9.3f %s   on / off %.4f   (off %s | on %s)"
          % (name, off, unit, on, unit, on / off, fmt(res["off"]), fmt(res["on"])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nt", type=int, default=5000)
    ap.add_argument("--grid", default="1000x3000")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--nt3", type=int, default=200)
    ap.add_argument("--grid3", type=int, default=512)
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
    src, rec = [(4, sx)], [(4, x) for x in range(nx)]
    zz, xx = np.meshgrid(np.arange(nz), np.arange(nx), indexing="ij")
    dv = sum(np.exp(-((zz - z0) ** 2 + (xx - x0) ** 2) / (2.0 * 20.0 ** 2)) for z0, x0 in ((200, sx), (450, sx - 400), (700, sx + 300)))
    dv = torch.from_numpy(dv.astype(np.float32)).cuda()
    print("2-D workload: %dx%d, nt = %d, one shot (source at (4, %d), %d receivers at z = 4), default plan, %d alternating reps"
          % (nz, nx, nt, sx, nx, args.reps))

    plans, bufs = {}, {}
    for k, fs in (("off", False), ("on", True)):
        p = ac.Propagator((nz, nx), h, dt, nabs=40, free_surface=fs)
        p.set_model(v)
        p.set_geometry(src, rec)
        p.reserve(nt, gradient=True)
        plans[k] = p
        bufs[k] = dict(obs=torch.zeros((nt, nx), dtype=torch.float32, device="cuda"),
                       grad=torch.zeros((nz, nx), dtype=torch.float32, device="cuda"),
                       out=torch.empty((nt, nx), dtype=torch.float32, device="cuda"))
    print("\nper shot:")
    report("forward", alternate({k: (lambda k=k: plans[k].forward(wav, out=bufs[k]["out"])) for k in plans}, args.reps))
    report("gradient", alternate({k: (lambda k=k: plans[k].gradient(wav, bufs[k]["obs"], grad=bufs[k]["grad"], want_misfit=False))
                                  for k in plans}, args.reps))
    report("born", alternate({k: (lambda k=k: plans[k].born(wav, dv, out=bufs[k]["out"])) for k in plans}, args.reps))
    report("gauss_newton", alternate({k: (lambda k=k: plans[k].gauss_newton(wav, dv, hv=bufs[k]["grad"])) for k in plans},
                                     args.reps))
    launches = {k: p.launch_count() for k, p in plans.items()}
    print("  step-kernel launches so far: off %d, on %d" % (launches["off"], launches["on"]))
    for p in plans.values():
        p.close()
    del plans, bufs
    torch.cuda.empty_cache()

    n3, nt3 = args.grid3, args.nt3
    shape = (n3, n3, n3)
    dt3 = fo.stable_dt(4500.0, h, 3)
    v3 = torch.from_numpy(fo.layered_model(shape, 1500.0, 4500.0, 6).astype(np.float32)).cuda()
    w3 = torch.from_numpy(fo.ricker(nt3, dt3, 10.0).astype(np.float32)).cuda()
    src3, rec3 = [(4, n3 // 2, n3 // 2)], [(4, n3 // 2, x) for x in range(n3)]
    print("\n3-D workload: %d^3, forward over nt = %d steps, source at (4, %d, %d), %d receivers at z = 4; time per step launch:"
          % (n3, nt3, n3 // 2, n3 // 2, n3))
    plans = {}
    for k, fs in (("off", False), ("on", True)):
        p = ac.Propagator(shape, h, dt3, nabs=20, free_surface=fs)
        p.set_model(v3)
        p.set_geometry(src3, rec3)
        p.reserve(nt3, gradient=False)
        plans[k] = p
    out3 = {k: torch.empty((nt3, n3), dtype=torch.float32, device="cuda") for k in plans}
    report("forward step", alternate({k: (lambda k=k: plans[k].forward(w3, out=out3[k])) for k in plans}, args.reps),
           per=nt3 / 1000.0, unit="us")
    for p in plans.values():
        p.close()


if __name__ == "__main__":
    main()
