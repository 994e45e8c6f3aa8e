#!/usr/bin/env python
"""bench.py - the driver's benchmark contract.

Headline (BASELINE.json): stencil Gpt-updates/s per GPU and FWI-gradient shots/s on config[1]
"2D acoustic synthetic layered model 1000x3000 grid, 8th-order space, 5k time steps, 64 shots, one FWI gradient".

One STEP = one shot's FWI gradient: 5000 forward leapfrog steps (source injection + receiver sampling fused,
forward field w_n streamed to HBM) + residual + 5000 adjoint steps with the imaging condition fused.  Weak
scaling: every rank runs its own shots (BASELINE config 3's shot-parallel layout) and the timed region ends with
the NCCL all-reduce of the gradient.  `value` counts wavefield point-updates (2 * nt * nz * nx per shot).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--nt 5000] [--grid 1000x3000] [--dump-outputs DIR]

`--dump-outputs DIR` writes what the timed steps computed, the FWI gradient summed over their shots, as DIR/gradient.npy
(float32), so that two builds can be compared output for output; the inputs depend only on the arguments.

Extra objects in the same JSON line:
  track_a        the reference-pinned Monte-Carlo source inversion (BASELINE configs 1 and 5), with its own reference
                 arm: oracle/ref_loop_port.py, the timing port of the reference's per-sample loop (bit-identical samples
                 and within ~10 % of the live reference's speed, tools/ref_port_fidelity.py), 1 process and nproc processes
  configs        config 3 (2301 x 751, 256 shots sharded over the ranks: one full gradient + all-reduce + one line-search
                 evaluation, STRONG scaling) and config 4 (512^3 single shot, checkpointed gradient over z slabs with the
                 fused NVLink halo push); present for every N so that the scaling can be read off the per-N lines
`--impl reference`: the reference repository has no propagator (SURVEY 0), so the CPU arm of the headline is the
self-oracle's C port (oracle/fd_oracle_c.c, POSIX threads over all host cores); each step is a real shot gradient over a
bounded number of time steps of the same grid.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nt", type=int, default=5000)
    ap.add_argument("--grid", default="1000x3000")
    ap.add_argument("--tile", default="")
    ap.add_argument("--tb2", type=int, default=0)
    ap.add_argument("--no-track-a", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--cpu-sample-nt", type=int, default=600)
    ap.add_argument("--settle-idle", type=float, default=8.0,
                    help="seconds of idle between the warm-up and the settle steps (0 = none): a burst of memory traffic - e.g. the "
                         "driver clearing the 60 GB snapshot buffer when it is first allocated - leaves the L2 / fabric side of the "
                         "GPU ~5 %% slower for a few seconds (SM clocks and throttle reasons unchanged); see DESIGN 5")
    ap.add_argument("--force-dist", action="store_true", help="diagnostic: initialise NCCL even with one rank")
    ap.add_argument("--no-graphs", action="store_true", help="diagnostic: individual launches instead of CUDA-graph replay of the time loops")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the gradient of the timed steps to DIR/gradient.npy (a fixed sample of it above %d MB)" % (DUMP_LIMIT >> 20))
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm")
    return args


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy.  Arrays over their share of DUMP_LIMIT are replaced by the same seeded
    sample of their elements on every run (flat, in index order)."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT // len(arrays)
    for name, a in arrays.items():
        if a.nbytes > share:
            a = a.reshape(-1)[np.unique(np.random.default_rng(0).integers(0, a.size, share // a.itemsize))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload(args):
    from oracle import fd_oracle as fo
    nz, nx = (int(x) for x in args.grid.lower().split("x"))
    h = 10.0
    v = fo.layered_model((nz, nx), 1500.0, 4500.0, 6).astype(np.float32)
    dt = fo.stable_dt(4500.0, h, 2)
    nt = args.nt
    wav = fo.ricker(nt, dt, 10.0).astype(np.float32)
    n_shots = 64
    sx = np.linspace(60, nx - 61, n_shots).astype(int)
    shots = [([(4, int(s))], [(4, x) for x in range(nx)]) for s in sx]
    return dict(nz=nz, nx=nx, h=h, dt=dt, nt=nt, v=v, wav=wav, shots=shots, nabs=40, alpha=0.3)


def workload_label(w):
    return ("BASELINE config[1]: 2D acoustic layered %dx%d, 8th-order space, %d time steps, one shot's FWI gradient per step "
            "(64-shot survey geometry, %d receivers/shot)" % (w["nz"], w["nx"], w["nt"], w["nx"]))


class ClockSampler:
    """Samples nvidia-smi SM clocks and throttle reasons while the timed region runs."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": min(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------------------------------- CPU arm (Track B)
def cpu_shot_gradient(w, nt_sample):
    """One REAL shot gradient of the self-oracle's C port (float32, all host cores) on the full grid with the bench
    geometry, over `nt_sample` time steps: forward with every w_n held, residual, adjoint with imaging.
    -> (seconds, useful point-updates, cores, description)"""
    from oracle import fd_oracle_c as foc
    src, rec = w["shots"][len(w["shots"]) // 2]
    wav = np.ascontiguousarray(w["wav"][:nt_sample])
    obs = np.zeros((nt_sample, len(rec)), dtype=np.float32)
    t = foc.time_gradient(w["v"], w["h"], w["dt"], src, rec, wav, obs, w["nabs"], w["alpha"], seg=0)
    return t, 2.0 * nt_sample * w["nz"] * w["nx"], foc.num_threads(), \
        "oracle/fd_oracle_c.c float32 (pthreads): one shot gradient over %d of the %d time steps on the full %dx%d grid, %d receivers, every w_n held (%.1f GB)" \
        % (nt_sample, w["nt"], w["nz"], w["nx"], len(rec), nt_sample * w["nz"] * w["nx"] * 4 / 1e9)


def run_reference(args):
    """Reference arm: every step is a real shot gradient on the host over a bounded number of time steps; ms_per_step
    is the measured time of such a step (nothing extrapolated), value the rate it achieved."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = workload(args)
    nt_s = min(args.cpu_sample_nt, w["nt"])
    times = []
    for i in range(args.warmup + args.steps):
        t, updates, cores, sample = cpu_shot_gradient(w, nt_s)
        if i >= args.warmup:
            times.append(t)
    t_med = float(np.median(times))
    rate = updates / t_med
    per_shot = 2.0 * w["nt"] * w["nz"] * w["nx"]
    line = {
        "impl": "reference", "metric": "stencil_gpt_updates_per_s", "value": rate / 1e9, "unit": "Gpt-updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_med * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "shots_per_s": rate / per_shot, "ms_per_full_shot_at_this_rate": per_shot / rate * 1e3,
        "step_ms_min_med_max": [min(times) * 1e3, t_med * 1e3, max(times) * 1e3],
        "config": {"workload": workload_label(w), "grid": [w["nz"], w["nx"]], "nt": w["nt"],
                   "cpu_step": "each step is a bounded sample of the workload: a real shot gradient over %d of the %d time steps" % (nt_s, w["nt"])},
        "cpu_baseline": {"value": rate / 1e9, "unit": "Gpt-updates/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "the reference repository has no propagator (SURVEY 0); this is the self-oracle's C port"},
        "e2e": {"value": rate / 1e9, "unit": "Gpt-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------- Track A
def _ev_time(torch, dev, fn, reps):
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for r in range(reps):
        fn(r)
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps * 1e-3


def track_a_numbers(device, dist=None, cpu=True):
    """The reference-pinned Monte-Carlo path (BASELINE configs 1 and 5) with its own reference arm."""
    import torch
    from full_waveform_inversion_b200 import full_waveform_inversion as fw
    from oracle import mc_oracle as orc
    K, C, T = 21, 9, 512
    d, G, _ = orc.synthetic_inputs(K=K, C=C, T=T, seed=0)
    amp = float(np.linalg.norm(orc.perform_inversion(d, G)))
    prob = fw.SourceInversion(d, G, device=device)
    out = {"workload": "MC source inversion K=21 C=9 T=512, VR per-trace, type single_force_crack_no_coupling (FWI:46-71 defaults)"}
    flops = (2 * C + 3) * K * T
    world = dist.get_world_size() if dist else 1
    rank = dist.get_rank() if dist else 0
    dev = torch.device("cuda", device)
    # ---- N GPUs: contiguous sample ranges per rank (FWI:833-834 order), one all-reduce of sum L (FWI:847)
    if dist:
        N = 8_000_000
        tot = torch.zeros(1, dtype=torch.float64, device=dev)

        def shard(r):
            _, _, L, _ = prob.sample_eval_dev(6, 1 + r, rank * N, N, amp, 0, 0, reduce=False)
            tot.copy_(L.sum(dtype=torch.float64))          # sum L of this rank's shard, on the device
            dist.all_reduce(tot)                            # p_data over all ranks (FWI:847), stream-ordered: no host sync
        shard(0)
        dist.barrier()
        dt_ = _ev_time(torch, dev, shard, 4)
        t = torch.tensor([dt_], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out["multi_gpu"] = {"samples_per_s": world * N / float(t[0]), "samples_per_rank": N, "n_gpus": world, "scaling": "weak",
                            "ms_per_batch": float(t[0]) * 1e3,
                            "collective": "one NCCL all-reduce of sum L (float64 scalar) per batch"}
        prob.close()
        return out
    NO_TENSOR = 32          # FWI_FLAG_NO_TENSOR: the CUDA-core fp32 kernels (the tensor-core path is the default for N >= 256)
    for N in (10_000, 4_000_000):
        for _ in range(3):
            prob.sample_eval_dev(6, 1, 0, N, amp, 0, 0)
        dt_ = _ev_time(torch, dev, lambda r: prob.sample_eval_dev(6, 1 + r, 0, N, amp, 0, 0, reduce=False), 5)
        dt_c = _ev_time(torch, dev, lambda r: prob.sample_eval_dev(6, 1 + r, 0, N, amp, 0, NO_TENSOR, reduce=False), 5)
        out["N=%d" % N] = {"samples_per_s": N / dt_, "ms": dt_ * 1e3, "path": "tcgen05 3xTF32 + TMEM epilogue (default)",
                           "tf32_tflops_issued": N * 2 * 32 * K * T / dt_ / 1e12,
                           "cuda_core_fp32": {"samples_per_s": N / dt_c, "ms": dt_c * 1e3, "fp32_tflops_direct": N * flops / dt_c / 1e12}}
    # the other metric families on the tensor cores vs the CUDA cores (N = 4e6, device-resident, sampler included)
    fam = {}
    for name, metric, fl in (("VR_normalised_flattened", 0, 3), ("PCC_per_trace", 2, 0), ("PCC_normalised_flattened", 2, 3), ("gau_per_trace", 4, 0),
                             ("CC_shift_per_trace", 3, 0), ("CC_shift_normalised_flattened", 3, 3)):
        N = 4_000_000
        prob.sample_eval_dev(6, 1, 0, N, amp, metric, fl, reduce=False)
        prob.sample_eval_dev(6, 1, 0, N, amp, metric, fl | NO_TENSOR, reduce=False)
        t1 = _ev_time(torch, dev, lambda r: prob.sample_eval_dev(6, 1 + r, 0, N, amp, metric, fl, reduce=False), 3)
        t2 = _ev_time(torch, dev, lambda r: prob.sample_eval_dev(6, 1 + r, 0, N, amp, metric, fl | NO_TENSOR, reduce=False), 3)
        fam[name] = {"tensor_core_samples_per_s": N / t1, "cuda_core_samples_per_s": N / t2}
    out["metric_families_N=4000000"] = fam
    # Gram-matrix mode: a different algorithm (2 K C^2 fp64 flop per sample, un-normalised metrics only) - own line
    N = 4_000_000
    prob.sample_eval_dev(6, 1, 0, N, amp, 0, 8, reduce=False)
    dt_ = _ev_time(torch, dev, lambda r: prob.sample_eval_dev(6, 1 + r, 0, N, amp, 0, 8, reduce=False), 5)
    out["gram_mode_N=%d" % N] = {"samples_per_s": N / dt_, "ms": dt_ * 1e3, "fp64_gflops_gram": N * 2 * K * (C * (C + 1) // 2 + C) / dt_ / 1e9,
                                 "note": "different algorithm (quadratic forms, no traces); not comparable to the direct flop count"}
    # config 1 through the drop-in entry point, host arrays in / host arrays out (sampler + eval + reduce + normalise + D2H)
    fw.perform_monte_carlo_sampled_waveform_inversion(d, G, 10_000, amp, "single_force_crack_no_coupling", "VR", False, False)
    t0 = time.perf_counter()
    for r in range(5):
        fw.perform_monte_carlo_sampled_waveform_inversion(d, G, 10_000, amp, "single_force_crack_no_coupling", "VR", False, False, seed=r)
    out["cfg1_e2e_samples_per_s"] = 5 * 10_000 / (time.perf_counter() - t0)
    # host-buffer e2e of config 5: 10k caller-supplied source vectors, float64 in / float64 out
    Ms = np.random.default_rng(0).standard_normal((10_000, C)) * amp
    prob.similarity(Ms, "VR", False, False)
    t0 = time.perf_counter()
    for _ in range(5):
        prob.similarity(Ms, "VR", False, False)
    out["cfg5_e2e_likelihood_evals_per_s"] = 5 * 10_000 / (time.perf_counter() - t0)
    # roofline of the direct formulation (SURVEY 8d): achieved FP32 rate over the FMA peak measured on this GPU
    import ctypes
    from full_waveform_inversion_b200 import _lib
    peak = ctypes.c_double(0.0)
    _lib.check(_lib.require_gpu().fwi_diag_fp32_peak(device, ctypes.byref(peak)))
    ach = out["N=4000000"]["cuda_core_fp32"]["fp32_tflops_direct"]
    out["roofline_cuda_core_fp32"] = {"bound": "fp32 fma", "achieved": ach, "peak": peak.value, "unit": "TFLOP/s", "frac": ach / peak.value,
                                      "peak_source": "measured: register-only FMA kernel (fwi_diag_fp32_peak)",
                                      "algorithmic_flop_per_sample": flops}
    bf16 = None
    try:
        bf16 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
    except Exception:
        pass
    tf32_peak = (bf16 / 2.0) if bf16 else 1125.0
    issued = out["N=4000000"]["tf32_tflops_issued"]
    out["roofline"] = {"bound": "tensor", "achieved": issued, "peak": tf32_peak, "unit": "TFLOP/s", "frac": issued / tf32_peak,
                       "peak_source": ("half of MEASURED_PEAKS.json bf16_tflops (TF32 runs at half the bf16 rate)" if bf16 else "nominal 1125 TFLOP/s dense TF32"),
                       "issued_flop_per_sample": 2 * 32 * K * T,
                       "note": "flops ISSUED to the tensor cores: the 3 x TF32 split pads the 10-term contraction to K = 32; in units of the "
                               "direct algorithm ((2C+3) K T = %d flop per sample) the default path delivers %.1f TFLOP/s-equivalent" % (flops, out["N=4000000"]["samples_per_s"] * flops / 1e12)}
    # trace-length sweep of config 1 (SURVEY 8d: T in {128, 512, 2048})
    gpu_T = {512: out["N=4000000"]["samples_per_s"]}
    for T2 in (128, 2048):
        d2, G2, _ = orc.synthetic_inputs(K=K, C=C, T=T2, seed=0)
        pr2 = fw.SourceInversion(d2, G2, device=device)
        N2 = 4_000_000 if T2 == 128 else 1_000_000
        pr2.sample_eval_dev(6, 1, 0, N2, amp, 0, 0, reduce=False)
        dt_ = _ev_time(torch, dev, lambda r: pr2.sample_eval_dev(6, 1 + r, 0, N2, amp, 0, 0, reduce=False), 3)
        if T2 <= 1536:
            out["T=%d_N=%d" % (T2, N2)] = {"samples_per_s": N2 / dt_, "tf32_tflops_issued": N2 * 2 * 32 * K * T2 / dt_ / 1e12, "path": "tensor cores"}
        else:       # B'' of one trace (T x 128 B) no longer fits in shared memory: the CUDA-core kernels take over
            out["T=%d_N=%d" % (T2, N2)] = {"samples_per_s": N2 / dt_, "fp32_tflops_direct": N2 * (2 * C + 3) * K * T2 / dt_ / 1e12, "path": "CUDA cores (T > 1536)"}
        gpu_T[T2] = N2 / dt_
        pr2.close()
    prob.close()
    if not cpu:
        return out
    # ---- reference arm of Track A: the reference's per-sample loop (timing port, see the module docstring), 1 process
    # (the reference default, FWI:65) and one process per host core (its scaling mechanism, FWI:824-827)
    from oracle import ref_loop_port as rp
    ncpu = os.cpu_count() or 1
    ref = {"kind": "port: oracle/ref_loop_port.py - same call sequence as FWI:448-510, 253-264, 664-668 (bit-identical samples; "
                   "892 vs 855 samples/s for the live reference in the build container, tools/ref_port_fidelity.py)",
           "sample": "1500 samples per process (the reference default is 10^4; the rate does not depend on N)", "cores": ncpu}
    for T2 in (128, 512, 2048):
        d2, G2, _ = orc.synthetic_inputs(K=K, C=C, T=T2, seed=0)
        ref["T=%d" % T2] = {"samples_per_s_1proc": rp.samples_per_second(d2, G2, amp, 1500, 1),
                            "samples_per_s_%dproc" % ncpu: rp.samples_per_second(d2, G2, amp, 1500, ncpu)}
    out["reference_arm"] = ref
    r512 = ref["T=512"]
    out["vs_reference"] = {
        "N=1e4_device_resident_vs_1proc": out["N=10000"]["samples_per_s"] / r512["samples_per_s_1proc"],
        "N=1e4_host_to_host_cfg1_vs_1proc": out["cfg1_e2e_samples_per_s"] / r512["samples_per_s_1proc"],
        "N=1e4_host_to_host_cfg5_vs_1proc": out["cfg5_e2e_likelihood_evals_per_s"] / r512["samples_per_s_1proc"],
        "N=4e6_device_resident_vs_1proc": out["N=4000000"]["samples_per_s"] / r512["samples_per_s_1proc"],
        "N=4e6_device_resident_vs_%dproc" % ncpu: out["N=4000000"]["samples_per_s"] / r512["samples_per_s_%dproc" % ncpu],
        "by_T_vs_%dproc" % ncpu: {"T=%d" % t: gpu_T[t] / ref["T=%d" % t]["samples_per_s_%dproc" % ncpu] for t in (128, 512, 2048)},
    }
    # the vectorised NumPy restatement: the "fair CPU" line of BASELINE.md (not the reference's own speed)
    t0 = time.perf_counter()
    orc.similarity_batch_fast_vr(d, G, Ms[:2000])
    out["cpu_numpy_vectorised_oracle_samples_per_s_1core"] = 2000 / (time.perf_counter() - t0)
    return out


# --------------------------------------------------------------------------------------------------- Track B extras
def track_b_extras(device):
    """Secondary Track B numbers: forward-only stepping rates (no snapshots) in 2-D and 3-D, incl. the temporally
    blocked kernel on a grid that does not fit L2 (where it beats the 16 B/pt HBM roofline)."""
    import torch
    from full_waveform_inversion_b200 import acoustic as ac
    out = {}

    def rate(shape, nt, **kw):
        prop = ac.Propagator(shape, 10.0, 5e-4, nabs=20, device=device, **kw)
        prop.set_model(torch.full(shape, 2500.0, device=torch.device("cuda", device)))
        mid = tuple(n // 2 for n in shape)
        prop.set_geometry([mid], [mid])
        wav = torch.from_numpy(ac.ricker(nt, 5e-4, 15.0)).to(torch.device("cuda", device))
        prop.forward(wav)
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        prop.forward(wav)
        e1.record()
        torch.cuda.synchronize(device)
        prop.close()
        return float(np.prod(shape)) * nt / (e0.elapsed_time(e1) * 1e-3) / 1e9

    out["forward_2d_1000x3000_gpt_s"] = rate((1000, 3000), 2000)
    out["forward_2d_4000x3000_tile_gpt_s"] = rate((4000, 3000), 600, tile=(32, 4))
    out["forward_2d_4000x3000_gpt_s"] = rate((4000, 3000), 600)          # default for this size: two steps per pass
    out["forward_2d_500x3000_gpt_s"] = rate((500, 3000), 2000)
    out["forward_3d_384_gpt_s"] = rate((384, 384, 384), 40)
    out["forward_3d_512_gpt_s"] = rate((512, 512, 512), 30)
    out["note"] = "forward stepping only (fused injection/sampling, no snapshots); 16 B/pt roofline at the measured HBM peak = 404 Gpt/s"
    return out


# --------------------------------------------------------------------------------------------------- configs 3 and 4
def config3_strong(device, dist):
    """BASELINE config 3: Marmousi-sized 2301 x 751 grid (nz = 751, nx = 2301), 256 shots sharded round-robin over the
    ranks, ONE FWI iteration = gradient of every shot + NCCL all-reduce + one line-search evaluation (forward of every shot +
    misfit all-reduce).  STRONG scaling: the total work is fixed.  3000 time steps per shot (0.89 s of record at h = 4 m)."""
    import torch
    from full_waveform_inversion_b200 import acoustic as ac
    from oracle import fd_oracle as fo
    world = dist.get_world_size() if dist else 1
    rank = dist.get_rank() if dist else 0
    dev = torch.device("cuda", device)
    nz, nx, nt, nshots, h = 751, 2301, 3000, 256, 4.0
    v_true = torch.from_numpy(fo.layered_model((nz, nx), 1500.0, 4500.0, 8).astype(np.float32)).to(dev)
    v0 = torch.from_numpy(np.linspace(1500.0, 4500.0, nz, dtype=np.float32)[:, None].repeat(nx, 1)).to(dev)
    dt = fo.stable_dt(4500.0, h, 2)
    wav = torch.from_numpy(fo.ricker(nt, dt, 12.0).astype(np.float32)).to(dev)
    sx = np.linspace(20, nx - 21, nshots).astype(int)
    rec = [(3, x) for x in range(0, nx, 2)]
    ids = ac.shard_shots(nshots, world, rank)
    shots = [([(3, int(sx[i]))], rec) for i in ids]
    prop = ac.Propagator2D((nz, nx), h, dt, nabs=40, device=device)
    prop.set_model(v_true)
    obs = []
    for s, r in shots:                                   # observed data of this rank's shots (untimed set-up)
        prop.set_geometry(s, r)
        obs.append(prop.forward(wav).clone())

    def iteration():
        J, g = ac.gradient(v0, h, dt, shots, wav, obs, propagator=prop, shot_ids=ids)       # sharded + ONE all-reduce
        step = 0.01 * ac.absmax(v0) / max(ac.absmax(g), 1e-30)
        trial = ac.model_update(v0.clone(), g, step, 1500.0, 4500.0)
        prop.set_model(trial)
        Jt = 0.0
        for (s, r), o in zip(shots, obs):
            prop.set_geometry(s, r)
            Jt += ac.misfit(prop.forward(wav), o)
        if dist:
            t = torch.tensor([Jt], dtype=torch.float64, device=dev)
            dist.all_reduce(t)
            Jt = float(t[0])
        return J, Jt

    iteration()                                          # warm-up: graph capture, snapshot buffers
    torch.cuda.synchronize(dev)
    if dist:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    J, Jt = iteration()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    prop.close()
    sec = float(ms[0]) * 1e-3
    updates = nshots * 3.0 * nt * nz * nx               # gradient: 2 nt steps, line search: nt steps, per shot
    return {"workload": "BASELINE config[2]: 2301x751 (nz=751, nx=2301, h=4 m), 256 shots, nt=%d, one FWI iteration = all gradients + all-reduce + one line-search evaluation" % nt,
            "scaling": "strong", "n_gpus": world, "shots_total": nshots, "shots_per_rank_max": len(ids),
            "s_per_iteration": sec, "s_per_20_iterations_at_this_rate": 20 * sec, "shots_per_s_gradient_plus_linesearch": nshots / sec,
            "gpt_updates_per_s": updates / sec / 1e9, "misfit": J, "misfit_trial": Jt,
            "collectives_per_iteration": "1 all-reduce of the %0.1f MB fp32 gradient + misfit, 1 all-reduce of the trial misfit" % (nz * nx * 4 / 1e6)}


def config4_slab(device, dist, nt=500):
    """BASELINE config 4: 3-D 512^3, one shot, forward + adjoint with CHECKPOINTED forward field; on N > 1 ranks the grid is
    split into z slabs and the step kernel pushes its boundary planes into the neighbours' ghost planes over NVLink.
    Useful point-updates = 2 nt 512^3 (the checkpointed recompute adds another nt 512^3 that is not counted)."""
    import torch
    from full_waveform_inversion_b200 import acoustic as ac
    from oracle import fd_oracle as fo
    world = dist.get_world_size() if dist else 1
    dev = torch.device("cuda", device)
    n, h = 512, 10.0
    shape = (n, n, n)
    dt = fo.stable_dt(4500.0, h, 3)
    wav = torch.from_numpy(fo.ricker(nt, dt, 8.0).astype(np.float32)).to(dev)
    src = [(8, n // 2, n // 2)]
    rec = [(6, y, x) for y in range(16, n - 16, 8) for x in range(16, n - 16, 8)]
    prof = np.linspace(1500.0, 4500.0, n, dtype=np.float32)
    if world > 1:
        slab = ac.SlabPropagator(shape, h, dt, nabs=24, device=device)
        lo, hi = slab.local_range
        slab.prop.set_memory_limit(80 * (hi - lo) * n * n * 4)           # 80 planes-worth per rank < nt snapshots -> checkpointing
        v_loc = torch.from_numpy(prof[lo:hi]).to(dev)[:, None, None].expand(hi - lo, n, n).contiguous()
        slab.set_model(v_loc, local=True)                               # per-rank upload: nobody holds the global model
        slab.set_geometry(src, rec)
        obs = torch.zeros((nt, len(rec)), dtype=torch.float32, device=dev)
        run = lambda: slab.gradient(wav, obs, gather=False)
        closer, nloc = slab, slab.n_own
    else:
        prop = ac.Propagator(shape, h, dt, nabs=24, device=device, memory_limit=80 * n * n * n * 4)
        prop.set_model(torch.from_numpy(prof).to(dev)[:, None, None].expand(n, n, n).contiguous())
        prop.set_geometry(src, rec)
        obs = torch.zeros((nt, len(rec)), dtype=torch.float32, device=dev)
        run = lambda: prop.gradient(wav, obs, want_misfit=False)
        closer, nloc = prop, n
    run()                                                 # graph capture, buffers
    torch.cuda.synchronize(dev)
    if dist:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    closer.close()
    sec = float(ms[0]) * 1e-3
    seg = int(np.ceil(np.sqrt(2.0 * nt)))
    return {"workload": "BASELINE config[3]: 3D 512^3 single shot, nt=%d, forward + adjoint, checkpointed (segments of %d steps, per rank), %s"
                        % (nt, seg, "z slabs with the fused NVLink halo push (no collective per step)" if world > 1 else "single GPU"),
            "scaling": "strong", "n_gpus": world, "planes_per_rank": nloc, "s_per_gradient": sec,
            "us_per_useful_step": sec / (2 * nt) * 1e6, "us_per_launch": sec / (3 * nt) * 1e6,
            "gpt_updates_per_s_useful": 2.0 * nt * n ** 3 / sec / 1e9, "gpt_updates_per_s_incl_recompute": 3.0 * nt * n ** 3 / sec / 1e9,
            "halo_bytes_per_step_per_interior_rank": 2 * 4 * n * n * 4 if world > 1 else 0}


# --------------------------------------------------------------------------------------------------- B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from full_waveform_inversion_b200 import acoustic as ac

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 or args.force_dist:
        if world == 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("MASTER_PORT", "29533")
            dist.init_process_group("nccl", device_id=dev, rank=0, world_size=1)
            dist.all_reduce(torch.zeros(1, device=dev))         # force communicator creation
        else:
            dist.init_process_group("nccl", device_id=dev)
    D = dist if world > 1 else None

    w = workload(args)
    nz, nx, nt = w["nz"], w["nx"], w["nt"]
    tile = tuple(int(x) for x in args.tile.split(",")) if args.tile else None
    prop = ac.Propagator2D((nz, nx), w["h"], w["dt"], nabs=w["nabs"], alpha=w["alpha"], device=local, tile=tile, tb2=(args.tb2 or None), graphs=not args.no_graphs)
    v_dev = torch.from_numpy(w["v"]).to(dev)
    wav_dev = torch.from_numpy(w["wav"]).to(dev)
    nrun = args.warmup + args.steps

    # this rank's shots (round-robin over the 64-shot survey) and THEIR observed data: synthetics of a perturbed model,
    # kept on the device for the device-resident timing and in pinned host memory for the end-to-end timing
    my_shots = [w["shots"][(rank + i * world) % len(w["shots"])] for i in range(nrun)]
    prop.set_model(v_dev * 1.02)
    obs_dev, obs_host = [], []
    for s, r in my_shots:
        prop.set_geometry(s, r)
        o = prop.forward(wav_dev).clone()
        obs_dev.append(o)
        obs_host.append(o.cpu().pin_memory())
    prop.set_model(v_dev)
    wav_host = torch.from_numpy(w["wav"]).pin_memory()
    grad = torch.zeros((nz, nx), dtype=torch.float32, device=dev)
    grad_host = torch.empty((nz, nx), dtype=torch.float32).pin_memory()

    # Rank barrier of the timed regions: the GPU is drained first, then the ranks meet on the CPU (gloo).  An NCCL barrier is a
    # collective KERNEL, and NCCL kernels issued while the GPUs are busy are among the triggers of the slow state (DESIGN 5).
    cpu_group = None
    if world > 1 and os.environ.get("FWI_BENCH_NCCL_BARRIER") != "1":
        try:
            cpu_group = dist.new_group(backend="gloo")
        except Exception as exc:                                   # no usable interface for gloo: fall back to NCCL
            print("bench: gloo barrier group unavailable (%r), using NCCL barriers" % (exc,), file=sys.stderr)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            if cpu_group is not None:
                dist.barrier(group=cpu_group)
            else:
                dist.barrier()
                torch.cuda.synchronize(dev)

    def one_step(i, host_io):
        src, rec = my_shots[i]
        prop.set_geometry(src, rec)
        if host_io:
            o = obs_host[i].to(dev, non_blocking=True)
            wv = wav_host.to(dev, non_blocking=True)
            J, _, _ = prop.gradient(wv, o, grad=grad, want_misfit=True)        # D2H read of the misfit (synchronises)
            grad_host.copy_(grad, non_blocking=True)                           # D2H of the accumulated gradient
            return J
        prop.gradient(wav_dev, obs_dev[i], grad=grad, want_misfit=False)
        return None

    # ---- device-resident timing (value) ------------------------------------------------------------------
    for i in range(args.warmup):
        one_step(i, False)
    if world > 1:
        dist.all_reduce(grad)           # warm-up of the collective too: NCCL sets its connections up on first use (~0.4 s)
    barrier()
    # settle: the first second after the 60 GB snapshot buffer is created runs ~20 % slow (first-touch of fresh
    # HBM pages); keep stepping (untimed) until two consecutive steps agree within 2 %, at most 12 extra steps.
    def timed_step(k):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        one_step(k % max(1, args.warmup), False)
        s1.record()
        torch.cuda.synchronize(dev)
        return s0.elapsed_time(s1)

    # A burst of memory traffic (the driver clearing the freshly allocated 60 GB snapshot buffer, a large memset or copy, even
    # a short FMA-only kernel) leaves the L2 / fabric side of the GPU ~5 % slower for the next seconds - SM clock, memory clock
    # and throttle reasons unchanged, FP32 rate unchanged, L2-resident copy 6.35 instead of 6.65 TB/s; the workload itself
    # never enters that state (profiles/r2_slow_state_probe.txt, DESIGN 5).  Everything that allocates has run by now (the
    # warm-up steps), so idle once and let it pass (measured: 3 s are not enough, 5 - 6 s are); the step time on either side of
    # the pause goes into the JSON line.
    if os.environ.get("FWI_BENCH_TRIGGER_GB"):       # diagnostic: provoke the slow state on purpose
        burst = torch.empty(int(float(os.environ["FWI_BENCH_TRIGGER_GB"]) * 1024**3), dtype=torch.uint8, device=dev)
        burst.fill_(1)
        torch.cuda.synchronize(dev)
        del burst
    ms_before_idle = timed_step(0)
    if args.settle_idle > 0:
        time.sleep(args.settle_idle)
        barrier()
    prev = None
    cur_ms = ms_before_idle
    for k in range(12):
        cur_ms = timed_step(k)
        if os.environ.get("FWI_BENCH_VERBOSE") == "1":
            print("settle step %d: %.2f ms" % (k, cur_ms), file=sys.stderr, flush=True)
        if prev is not None and abs(cur_ms - prev) <= 0.02 * prev:
            break
        prev = cur_ms
    grad.zero_()
    barrier()
    sampler = ClockSampler(local) if rank == 0 and os.environ.get("FWI_BENCH_NO_SAMPLER") != "1" else None     # (diagnostic switch)
    if sampler:
        sampler.start()
    l0 = prop.launch_count()
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    e1 = torch.cuda.Event(enable_timing=True)
    marks[0].record()
    sync_each = os.environ.get("FWI_BENCH_SYNC") == "1"        # diagnostic: drain the GPU after every shot
    for k, i in enumerate(range(args.warmup, nrun)):
        one_step(i, False)
        marks[k + 1].record()                       # per-shot marks (no synchronisation: the CPU keeps enqueueing)
        if sync_each:
            torch.cuda.synchronize(dev)
    if world > 1:
        dist.all_reduce(grad)                       # one FWI gradient = sum over every rank's shots
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"gradient": grad.cpu().numpy()})
    ms = marks[0].elapsed_time(e1)
    shot_ms = [marks[k].elapsed_time(marks[k + 1]) for k in range(args.steps)]
    launches = prop.launch_count() - l0
    clocks = sampler.stop() if sampler else None

    # ---- end-to-end through the public API with host buffers (e2e) ------------------------------------------
    grad.zero_()
    one_step(0, True)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    J_last = None
    for i in range(args.warmup, nrun):
        J_last = one_step(i, True)
    if world > 1:
        dist.all_reduce(grad)
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)

    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device=dev)
    stats = torch.tensor([min(shot_ms), float(np.median(shot_ms)), max(shot_ms)], dtype=torch.float64, device=dev)
    all_stats = [stats]
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        all_stats = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(all_stats, stats)
    ms, ms_e2e = float(t[0]), float(t[1])
    prop.close()

    per_shot = 2.0 * nt * nz * nx
    total_updates = per_shot * args.steps * world
    value = total_updates / (ms * 1e-3) / 1e9
    e2e = total_updates / (ms_e2e * 1e-3) / 1e9

    line = None
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        avg_launch_s = (ms * 1e-3) / max(1, launches)
        achieved = 16.0 * nz * nx / avg_launch_s / 1e9
        line = {
            "metric": "stencil_gpt_updates_per_s", "value": value, "unit": "Gpt-updates/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "shots_per_s": args.steps * world / (ms * 1e-3),
            "config": {"workload": workload_label(w) + ", forward field w_n held in HBM",
                       "grid": [nz, nx], "nt": nt, "shots_per_rank": args.steps, "parallelism": "shot-parallel x%d, NCCL gradient all-reduce" % world,
                       "l2": "inputs larger than L2: %.1f GB of forward-field snapshots stream through HBM per step; the 12 MB wavefields are L2-resident within a shot by design" % (nt * nz * prop_px(nx) * 4 / 1e9),
                       "parity": "vs self-oracle oracle/fd_oracle.py (float64 C port at this grid size: tests/test_fd_scale_gpu.py) - the reference has no propagator (SURVEY 0)"},
            "gpu_launches": int(launches),
            "per_rank_shot_ms_min_med_max": [[float(x) for x in s.cpu()] for s in all_stats],
            "e2e": {"value": e2e, "unit": "Gpt-updates/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int(obs_host[0].numel() * 4 + wav_host.numel() * 4),
                    "d2h_bytes_per_step": int(8 + grad_host.numel() * 4),
                    "misfit_last_step": J_last,
                    "note": "each step copies that shot's own observed traces and the wavelet from pinned host memory, reads the misfit back and copies the accumulated gradient to pinned host memory"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": 12.2e6 if (nz, nx) == (1000, 3000) else None, "peak_source": peak_src,
                         "traffic_note": "dram read+write per adjoint launch from ncu --set full --cache-control none (profiles/): the snapshot stream; the 3 x 12 MB wavefields are served by L2, so this grid is L2-bound, not HBM-bound - the HBM-bound cases are in track_b_extras / configs",
                         "kernel": "fd2d_step_kernel (forward-save, propagate-only and deferred-imaging adjoint variants, averaged)",
                         "algorithmic_bytes_per_launch": 16 * nz * nx,
                         "avg_launch_us": avg_launch_s * 1e6,
                         "note": "16 B per point-update (SURVEY 8d) over the mean step-kernel time incl. launch gaps; the snapshot stream adds 4 B/pt of real HBM traffic per step on top"},
            "clocks": clocks,
            "settle": {"idle_s": args.settle_idle, "ms_per_step_before_idle": ms_before_idle, "ms_per_step_after_idle": cur_ms,
                       "note": "untimed: one step, an idle pause, then steps until two agree within 2 % (rank 0's values); a burst of "
                               "memory traffic at start-up leaves the GPU's L2 side ~5 % slower for a few seconds (DESIGN 5)"},
        }
        if not args.no_cpu_baseline and world == 1:
            tsec, updates, cores, sample = cpu_shot_gradient(w, min(args.cpu_sample_nt, nt))
            line["cpu_baseline"] = {"value": updates / tsec / 1e9, "unit": "Gpt-updates/s", "cores": cores, "kind": "port", "sample": sample}
    # secondary objects: never allowed to take the headline down
    if not args.no_track_a:
        try:
            ta = track_a_numbers(local, D, cpu=(world == 1))
            if line is not None:
                line["track_a"] = ta
        except Exception as exc:
            if line is not None:
                line["track_a"] = {"error": repr(exc)}
    if not args.no_extras and world == 1:
        try:
            line["track_b_extras"] = track_b_extras(local)
        except Exception as exc:
            line["track_b_extras"] = {"error": repr(exc)}
    if not args.no_configs:
        cfgs = {}
        for name, fn in (("config3_strong_256_shots", config3_strong), ("config4_slab_512cubed", config4_slab)):
            try:
                cfgs[name] = fn(local, D)
            except Exception as exc:
                cfgs[name] = {"error": repr(exc)}
                torch.cuda.synchronize(dev)
        if line is not None:
            line["configs"] = cfgs
    if line is not None:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def prop_px(nx):
    return (nx + 31) // 32 * 32


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
