#!/usr/bin/env python
"""Per-shot time of Born modelling and Gauss-Newton products next to forward and gradient, in bench.py's workload.

    python tools/born_bench.py [--nt 5000] [--grid 1000x3000] [--reps 5] [--segments 1,2,8,32,128,5000] [--kw tb2=24]

One Propagator, bench.py's layered model and the middle shot of its 64-shot geometry (one source, a receiver in every
column).  Each call is timed with CUDA events after two warm-up calls, `--reps` times; the median and the spread
(min - max) are printed.  Born is also timed at each segment length S in `--segments`, forced through the memory limit
(S = min(nt, kBornSeg, planes the limit holds), so values above the library's kBornSeg are clamped to it); its results
must not change with S, which is checked bit for bit.  The card's name and power limit are printed in the same run."""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def card_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the timing does not depend on it, the label does
        q = "nvidia-smi unavailable (%s)" % e
    return name, q


def timed(fn, reps, warmup=2):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return np.array(out)


def fmt(ms):
    return "%8.2f ms  (min %.2f, max %.2f, spread %.1f %%)" % (np.median(ms), ms.min(), ms.max(), 100.0 * (ms.max() - ms.min()) / np.median(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nt", type=int, default=5000)
    ap.add_argument("--grid", default="1000x3000")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--segments", default="1,2,8,32,128,5000")
    ap.add_argument("--kw", default="", help="plan option, e.g. tb2=24 or tile=32,4")
    args = ap.parse_args()
    import torch
    from full_waveform_inversion_b200 import acoustic as ac
    from oracle import fd_oracle as fo

    nz, nx = (int(x) for x in args.grid.lower().split("x"))
    nt, h = args.nt, 10.0
    v = fo.layered_model((nz, nx), 1500.0, 4500.0, 6).astype(np.float32)        # bench.py's workload
    dt = fo.stable_dt(4500.0, h, 2)
    wav = fo.ricker(nt, dt, 10.0).astype(np.float32)
    sx = np.linspace(60, nx - 61, 64).astype(int)[32]
    src, rec = [(4, int(sx))], [(4, x) for x in range(nx)]
    # perturbation: smooth blobs below the source, 1 m/s peak
    zz, xx = np.meshgrid(np.arange(nz), np.arange(nx), indexing="ij")
    dv = sum(np.exp(-((zz - z0) ** 2 + (xx - x0) ** 2) / (2.0 * 20.0 ** 2)) for z0, x0 in ((200, sx), (450, sx - 400), (700, sx + 300)))
    dv = torch.from_numpy(dv.astype(np.float32)).cuda()

    kw = {}
    if args.kw:
        k, val = args.kw.split("=")
        kw[k] = tuple(int(t) for t in val.split(",")) if "," in val else int(val)
    name, q = card_info()
    print("card: %s | nvidia-smi name, power limit, max SM clock: %s" % (name, q))
    print("workload: %dx%d, nt = %d, one shot (source at x = %d, %d receivers), plan options %s, %d reps after 2 warm-up calls"
          % (nz, nx, nt, sx, nx, kw or "default", args.reps))

    prop = ac.Propagator((nz, nx), h, dt, nabs=40, **kw)
    prop.set_model(torch.from_numpy(v).cuda())
    prop.set_geometry(src, rec)
    wav_d = torch.from_numpy(wav).cuda()
    obs = torch.zeros((nt, nx), dtype=torch.float32, device="cuda")
    grad = torch.zeros((nz, nx), dtype=torch.float32, device="cuda")
    out = torch.empty((nt, nx), dtype=torch.float32, device="cuda")
    prop.reserve(nt, gradient=True)

    pts = nz * nx
    res = {}
    res["forward"] = timed(lambda: prop.forward(wav_d, out=out), args.reps)
    res["gradient"] = timed(lambda: prop.gradient(wav_d, obs, grad=grad, want_misfit=False), args.reps)
    res["born"] = timed(lambda: prop.born(wav_d, dv, out=out), args.reps)
    res["gauss_newton"] = timed(lambda: prop.gauss_newton(wav_d, dv, hv=grad), args.reps)
    print("\nper shot (default storage: every snapshot of the gradient / Gauss-Newton in HBM, Born with the library's segment):")
    for k, ms in res.items():
        print("  %-13s %s   %.2f us/step" % (k, fmt(ms), 1e3 * np.median(ms) / nt))
    print("  born / gradient = %.3f, born / forward = %.3f, gauss_newton / gradient = %.3f"
          % (np.median(res["born"]) / np.median(res["gradient"]), np.median(res["born"]) / np.median(res["forward"]),
             np.median(res["gauss_newton"]) / np.median(res["gradient"])))
    # algorithmic HBM traffic per time step (B/pt): forward 16, FWD_SAVE 20, Born scattered step 24 (u_{n-1}, m in;
    # u_{n+1} out; w_n, dm in), adjoint with deferred imaging 17 + 29 per pair
    print("  algorithmic traffic, bytes per grid point per time step: forward 16, gradient 20 + 23 = 43, born 20 + 24 = 44,"
          " gauss_newton 20 + 24 + 23 = 67")

    ref = prop.born(wav_d, dv)[0].cpu().numpy()
    plane = nz * ((nx + 31) // 32 * 32) * 4
    print("\nborn per shot by segment length S (snapshot planes between the background and the scattered sweep):")
    for s in [int(t) for t in args.segments.split(",")]:
        prop.set_memory_limit(s * plane)
        ms = timed(lambda: prop.born(wav_d, dv, out=out), args.reps)
        same = np.array_equal(out.cpu().numpy(), ref)
        print("  S = %5d (limit %6.1f MB)  %s   bit-identical to the default: %s" % (s, s * plane / 2 ** 20, fmt(ms), same))
    prop.set_memory_limit(0)
    prop.close()


if __name__ == "__main__":
    main()
