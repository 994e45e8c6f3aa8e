"""Tensor-core likelihood path (csrc/mc_umma.cu) vs the float64 oracle and the fp32 CUDA-core kernels, every metric x mode
it covers; then rates.   python tools/umma_check.py [N_bench] [--quick]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from full_waveform_inversion_b200 import full_waveform_inversion as fw
from oracle import mc_oracle as orc
TENSOR, NO_TENSOR = 16, 32

def check(K, C, T, N, seed=0):
    d, G, _ = orc.synthetic_inputs(K=K, C=C, T=T, seed=seed)
    amp = float(np.linalg.norm(orc.perform_inversion(d, G)))
    Ms = np.random.default_rng(seed + 1).standard_normal((N, C))
    Ms = Ms / np.linalg.norm(Ms, axis=1, keepdims=True) * amp
    Ms[0] = orc.perform_inversion(d, G)[:, 0]                      # the best-fitting source: SSE << sum d^2 (cancellation case)
    M_dev = torch.tensor(Ms.T.copy(), dtype=torch.float32, device="cuda")
    prob = fw.SourceInversion(d, G)
    worst = 0.0
    for metric in ("VR", "PCC", "CC", "CC-shift", "gau"):
        if metric == "gau" and T < 60:
            continue
        for norm in (False, True):
            for simul in (False, True):
                want = orc.similarity_batch(d, G, Ms[:64], metric, norm, simul)
                fl = (1 if norm else 0) | (2 if simul else 0)
                a = prob.eval_dev(M_dev, fw.METRICS.index(metric), fl | TENSOR).cpu().numpy()
                b = prob.eval_dev(M_dev, fw.METRICS.index(metric), fl | NO_TENSOR).cpu().numpy()
                e_tc, e_cc, e_ab = np.abs(a[:64] - want).max(), np.abs(b[:64] - want).max(), np.abs(a - b).max()
                worst = max(worst, e_tc)
                flag = "" if e_tc <= 1e-6 else "   <-- above 1e-6"
                print("K=%d C=%d T=%d N=%d %-4s norm=%d simul=%d: tensor-core |sim - oracle| %.2e, CUDA-core %.2e, tensor vs CUDA-core (all N) %.2e%s"
                      % (K, C, T, N, metric, norm, simul, e_tc, e_cc, e_ab, flag), flush=True)
    prob.close()
    return worst

quick = "--quick" in sys.argv
sys.argv = [x for x in sys.argv if x != "--quick"]
ok = True
for cfg in ((21, 9, 512, 1000), (4, 3, 320, 77)) if quick else ((21, 9, 512, 1000), (5, 6, 128, 300), (4, 3, 320, 77), (21, 9, 1024, 260), (7, 9, 72, 129), (3, 9, 1536, 40), (33, 9, 61, 300)):
    ok &= check(*cfg) <= 1e-6
print("UMMA_CHECK_OK" if ok else "UMMA_CHECK_FAILED", flush=True)
N = int(sys.argv[1]) if len(sys.argv) > 1 else 4_000_000
d, G, _ = orc.synthetic_inputs(K=21, C=9, T=512, seed=0)
amp = float(np.linalg.norm(orc.perform_inversion(d, G)))
prob = fw.SourceInversion(d, G)
for n in ((N,) if quick else (10_000, N)):
    MTs, _, _, _ = prob.sample_eval_dev(6, 1, 0, n, amp, 0, 0, reduce=False)
    for metric, fl in (("VR", 0), ("VR", 2), ("VR", 1), ("VR", 3), ("PCC", 0), ("PCC", 3), ("gau", 0),
                       ("CC-shift", 0), ("CC-shift", 2), ("CC-shift", 3)):
        out = []
        for name, extra in (("tensor", TENSOR), ("cuda-core", NO_TENSOR)):
            fn = lambda: prob.eval_dev(MTs, fw.METRICS.index(metric), fl | extra, want_likelihood=True)
            fn(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                fn()
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 3
            out.append("%s %.3f ms = %.1f M samples/s" % (name, ms, n / ms / 1e3))
        print("N=%d %-4s norm=%d simul=%d: %s" % (n, metric, fl & 1, (fl >> 1) & 1, " | ".join(out)), flush=True)
