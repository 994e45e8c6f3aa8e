// Track A on the 5th-generation tensor cores: the [N x C] . [C x K.T] contraction of the Monte-Carlo likelihood path
// (forward_model FWI:253-264 + variance_reduction FWI:512-520 per trace, FWI:664-668) as tcgen05.mma kind::tf32 with an
// error-compensated 3 x TF32 split, accumulators in TMEM, the misfit folded in the TMEM epilogue.
//
// Formulation.  For a trace k the residual of every sample n at every time t is ONE matrix product:
//     r[n, t] = sum_c M[n, c] G[k, c, t] - d[k, t]  =  A''[n, :] . B''[k][t, :]
// with 32-wide rows (four tcgen05 K-steps of 8):
//     A''[n] = [ M_hi (9) | M_hi (9) | M_lo (9) | -1 | -1 | 0 0 0 ]        hi = tf32(x), lo = tf32(x - hi)
//     B''[t] = [ G_hi (9) | G_lo (9) | G_hi (9) | d_hi | d_lo | 0 0 0 ]
// i.e. hi.hi + hi.lo + lo.hi (the lo.lo term is below fp32 rounding), accumulated in fp32 by the tensor core.  The
// epilogue reads the 128 x 256 accumulator tile from TMEM (one sample per thread, tcgen05.ld 32x32b.x32, double
// buffered) and folds the statistics of the (sample, trace) pair:
//   MODE_SSE      (un-normalised VR / gau, FWI:512-520, 578-582): sum_t r^2;
//   MODE_MOM      (CC == PCC, FWI:534-546, 568-576): B'' holds the CENTRED rows G' = G - mean_t G and the -1 columns of
//                 A'' are 0, so the accumulator is the centred synthetic s' and the fold is sum_t s'^2; the cross moment
//                 sum_t d' s' = M . (G' d') and the mean M . gbar are 9-term dot products with float64 constants;
//   MODE_MOM_MAX  (normalised modes, FWI:597-599): additionally max / min of s' (max |s| = max(|max + mu|, |min + mu|)).
//   CC-shift     (FWI:548-566): every shift rolls data and synthetic together, so the metric is PCC on the 4x linearly
//                 interpolated traces (np.interp, right edge clamped).  The interpolated synthetic is LINEAR in the
//                 accumulator's s'[t], so nothing is interpolated on the device: with S2 = sum_t s'[t]^2 and the lag-one
//                 product P = sum_t s'[t] s'[t+1] (adjacent TMEM columns, i.e. adjacent registers of the epilogue thread)
//                     sum_i s'_i^2 = 2.75 S2 + 1.25 P + 2.125 s'[T-1]^2 - 0.875 s'[0]^2
//                 and every first-order term (mean and cross moment of the interpolated rows, s'[0], s'[T-1]) is a 9-term
//                 dot product with float64 constants built at upload.  The flattened modes interpolate ACROSS trace
//                 boundaries (FWI:612): the three points after each internal boundary are patched from the neighbouring
//                 traces' last / first (normalised) values - inside a CTA from a carried value, across trace groups in
//                 the finishing kernel.
// The per-trace combination (float64, same expressions as mc_eval_kernel) runs in the same thread.
//
// Work split.  B'' of a few traces (6 tiles of 256 x 32 fp32 = 192 KB) stays RESIDENT in shared memory; a CTA walks over
// 128-sample groups, TMA-loading only the 16 KB A'' tile per group (2 stages).  Trace groups are separate CTAs that write
// partial sums part[g][n]; a small kernel adds them, divides by K and applies L = exp(-(1 - s)/2) (FWI:774).
// Per group and tile: 4 MMAs (128 x 256 x 8) into one of two TMEM accumulators (2 x 256 columns), committed to an
// mbarrier the four epilogue warps wait on; they hand the accumulator back through a second mbarrier.
//
// Warp roles (320 threads): warps 0-7 epilogue (two pipelines x four TMEM lane quarters), warp 8 TMA producer, warp 9 MMA issuer.
#include "fd_common.cuh"
#include "mc_common.cuh"
#include <vector>
#include <cstring>
#include <cmath>
#include <algorithm>

namespace fwi {

constexpr int kUK = 32;                 // padded K (floats per operand row = one 128-byte swizzle row)
constexpr int kUM = 128;                // samples per MMA tile (TMEM lanes)
constexpr int kUN = 256;                // time samples per resident B'' tile (one TMA box)
constexpr int kUPipes = 2;              // independent pipelines per CTA (sample groups in flight).  2 x 256 columns: 5.7 ms for N = 4e6 (VR);
                                        // 4 x 128: 9.2 ms - the single MMA-issuing lane pays ~0.45 us per accumulator use whatever its size
constexpr int kUNacc = 512 / kUPipes;   // time samples per accumulator use (MMA N; every pipeline owns that many TMEM columns)
constexpr int kUCst = 52;               // float64 constants per resident trace in shared memory: gbar[9] | gdc[9] (CC-shift: the interpolated
                                        // cross moment) | CC-shift: dgb[9], G'[.,0][9], G'[.,T-1][9] | TraceConst (7) at 45
constexpr int kUTilesMax = (227 * 1024 - kUPipes * 16384 - 256) / (kUN * 128 + kUCst * 8);     // resident B'' tiles (+ a trace's constants each)
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr) {
    // K-major, 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart (SBO), LBO unused (1), descriptor version 1
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// one lane of a converged warp (the tcgen05 instructions take uniform-register operands: with the WHOLE warp running the issuer
// loop and only the instruction itself under this predicate, the descriptors stay in uniform registers; a loop under
// `if (lane == 0)` makes the compiler wrap every tcgen05.mma in an elect / R2UR.BROADCAST / branch sequence of ~16 instructions)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xFFFFFFFF;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// the same wait, tied to the registers of the load it completes (keeps the compiler from using them earlier)
__device__ __forceinline__ void tmem_ld_wait_dep(float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                   "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]),
                   "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]),
                   "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :: "memory");
}

// float64 reciprocal / reciprocal square root from the fp32 SFU seed + two Newton steps (FMA only): the fp64 divide and
// sqrt sequences were the largest part of the per-trace combination
// (seeds: MUFU.RCP64H / MUFU.RSQ64H work on the double's own exponent, so products of small amplitudes such as
// s2 * ssd ~ 1e-44 that leave the fp32 range are handled; three Newton steps whatever the seed's accuracy)
__device__ __forceinline__ double rcp64(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return fma(r, fma(-x, r, 1.0), r);
}
__device__ __forceinline__ double rsqrt64(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    y = y * fma(-0.5 * x, y * y, 1.5);
    y = y * fma(-0.5 * x, y * y, 1.5);
    return y * fma(-0.5 * x, y * y, 1.5);
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {      // FMNMX3: one instruction for two comparisons
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}
__device__ __forceinline__ float fmin3(float a, float b, float c) {
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

__host__ __device__ inline float tf32_round(float x) {          // round to nearest-even onto the 10-bit tf32 mantissa
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0x7F800000u) return x;
    u += 0x00000FFFu + ((u >> 13) & 1u);
    u &= 0xFFFFE000u;
    float r;
    memcpy(&r, &u, 4);
    return r;
}

struct UmmaEvalArgs {
    int64_t N;                  // samples
    int n_groups;               // 128-sample groups = ceil(N / 128)
    int tiles_per_trace;        // ceil(T / 256): resident B'' tiles (TMA boxes) per trace
    int chunks_per_trace;       // ceil(T / 128): accumulator stages per trace
    int n_last;                 // MMA N of a trace's last chunk (multiple of 16, <= 128)
    int traces_per_cta;         // resident traces per CTA
    int ctas_full, ctas_last;   // CTAs working on a trace group with traces_per_cta traces / on the last (possibly smaller) group
    int K, C, T;
    int metric, flags, debug;      // debug (FWI_UMMA_DEBUG): 1 = no MMAs issued, 2 = no TMEM loads / folds (timing experiments)
    uint32_t idesc_full, idesc_last;      // instruction descriptors of a full chunk / of the last chunk of a trace
    const TraceConst* tc;       // [K]
    const double* gbar;         // [K][C] mean_t G
    const double* gdc;          // [K][C] sum_t (d - mean d) G
    const double* shc;          // CC-shift: [K][4][C] = mean_i G_i - mean_t G | sum_i (d_i - mean d_i) G_i | G'[.,0] | G'[.,T-1]   (_i: 4x interpolated)
    const float* M;             // the samples, (rows, N)
    int64_t ldm;
    double* part;               // [n_trace_groups][npart][N] partial sums of the per-trace combination
    int npart;                  // 3 sums (+ the group's first and last normalised synthetic value for the flattened CC-shift patch: 5)
};

// grid = (ctas_per_trace_group, n_trace_groups); block = (4 * pipelines + 2) warps.
// Several pipelines per CTA, each with its own sample group in flight, its own A'' stage, its own TMEM accumulator (512 /
// pipelines columns) and its own four epilogue warps; the MMA issuer goes round robin over them.  Measured on B200: the MMA <-> epilogue
// handshake of one accumulator costs ~0.3 us per use and the epilogue's serial work (TMEM load latency, per-trace
// combination) does not overlap with its own pipeline's MMAs, so two independent pipelines on the same resident B'' tiles
// is what keeps the tensor core and the epilogue warps busy at the same time.
constexpr int kUThreads = (4 * kUPipes + 2) * 32;        // 4 epilogue warps per pipeline + TMA producer + MMA issuer
template <int MODE, bool SH>
__global__ void __launch_bounds__(kUThreads, 1) mc_umma_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                                                               UmmaEvalArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    float* b_smem = reinterpret_cast<float*>(smem);                                    // [tiles][256][32] swizzled
    float* a_smem = reinterpret_cast<float*>(smem + (size_t)kUTilesMax * kUN * kUK * 4); // [pipeline][128][32] swizzled
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)kUTilesMax * kUN * kUK * 4 + (size_t)kUPipes * kUM * kUK * 4);
    uint64_t* b_full = bars;                       // 1
    uint64_t* a_full = bars + 1;                   // [pipes]
    uint64_t* a_empty = a_full + kUPipes;          // [pipes]
    uint64_t* t_full = a_empty + kUPipes;          // [pipes]
    uint64_t* t_empty = t_full + kUPipes;          // [pipes]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + kUPipes);
    double* cst = reinterpret_cast<double*>(reinterpret_cast<uint8_t*>(bars) + 256);     // [resident traces][kUCst]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tg = blockIdx.y;                                       // trace group
    // CTAs are shared out in proportion to the traces a group holds (the last group may hold fewer)
    const int ncta = (tg == (int)gridDim.y - 1) ? a.ctas_last : a.ctas_full;
    if ((int)blockIdx.x >= ncta) return;
    const int k0 = tg * a.traces_per_cta, k1 = min(a.K, k0 + a.traces_per_cta);
    const int ntiles = (k1 - k0) * a.tiles_per_trace;                // resident tiles of this CTA
    const int nchunks = (k1 - k0) * a.chunks_per_trace;              // accumulator uses per sample group
    constexpr int kProd = 4 * kUPipes, kMma = 4 * kUPipes + 1;       // warp indices of the two single-lane roles

    if (threadIdx.x == 0) {
        mbar_init(b_full, 1);
        for (int s = 0; s < kUPipes; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
        for (int s = 0; s < kUPipes; ++s) { mbar_init(&t_full[s], 1); mbar_init(&t_empty[s], 4); }
        fence_mbar_init();
        fence_proxy_async();
    }
    // The resident traces' constants go to shared memory once: the per-trace fold reads up to 52 of them per thread, and as
    // (L1-missing) global loads they cost ~2000 cycles per trace on the epilogue's critical path.
    for (int i = threadIdx.x; i < (k1 - k0) * kUCst; i += blockDim.x) {
        const int k = k0 + i / kUCst, j = i % kUCst;
        double v = 0.0;
        if (j < 9) { if (j < a.C) v = a.gbar[k * a.C + j]; }
        else if (j < 18) { if (j - 9 < a.C) v = SH ? a.shc[(size_t)k * 4 * a.C + a.C + (j - 9)] : a.gdc[k * a.C + (j - 9)]; }
        else if (j < 45) {
            const int w = (j - 18) / 9, c = (j - 18) % 9;                  // dgb, G'[.,0], G'[.,T-1]
            if (SH && c < a.C) v = a.shc[(size_t)k * 4 * a.C + (w == 0 ? 0 : w + 1) * a.C + c];
        } else v = reinterpret_cast<const double*>(a.tc + k)[j - 45];
        cst[i] = v;
    }
    if (warp == kMma) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == kProd) {
        // ------------------------------------------------ TMA producer: resident B'' tiles once, then the A'' tile of every group
        if (lane == 0) {
            mbar_expect_tx(b_full, (uint32_t)ntiles * kUN * kUK * 4);
            for (int j = 0; j < ntiles; ++j) {
                const int k = k0 + j / a.tiles_per_trace, tt = j % a.tiles_per_trace;
                tma_load_2d(b_smem + (size_t)j * kUN * kUK, &tm_b, 0, (k * a.tiles_per_trace + tt) * kUN, b_full);
            }
            int i = 0;
            for (int g = blockIdx.x; g < a.n_groups; g += ncta, ++i) {
                const int p = i % kUPipes, use = i / kUPipes;          // pipeline, and how often its A'' stage has been used
                if (use >= 1) mbar_wait(&a_empty[p], (use - 1) & 1);
                mbar_expect_tx(&a_full[p], kUM * kUK * 4);
                tma_load_2d(a_smem + (size_t)p * kUM * kUK, &tm_a, 0, g * kUM, &a_full[p]);
            }
        }
    } else if (warp >= kMma) {                                      // kMma is the last warp
        // ------------------------------------------------ MMA issuer (one elected lane), round robin over the pipelines.
        // The lane's own instructions sit on every accumulator's critical path (release -> MMAs -> commit), and a lone thread
        // issues a dependent instruction every 4-10 cycles: everything the MMAs need (descriptors, instruction word, TMEM
        // address) is therefore advanced incrementally AFTER the commit and ready in registers before the wait - no divisions,
        // no descriptor assembly between the wait and the four tcgen05.mma.
        {                                                       // all 32 lanes run the loop (uniform control flow and values)
            mbar_wait(b_full, 0);
            tc_fence_after();
            constexpr uint64_t kDescHi = ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
            const uint64_t b_desc0 = kDescHi | (uint64_t)((smem_u32(b_smem) >> 4) & 0x3FFF);
            const uint32_t trace_step = (uint32_t)a.tiles_per_trace * kUN * (kUK * 4 / 16);      // descriptor address units (16 B) per trace
            const int cpt = a.chunks_per_trace;
            int grp[kUPipes], chunk[kUPipes], ci[kUPipes];
            uint32_t use_a[kUPipes], use_t[kUPipes], b_tr[kUPipes], b_off[kUPipes];
            uint64_t a_desc[kUPipes];
#pragma unroll
            for (int p = 0; p < kUPipes; ++p) {
                grp[p] = blockIdx.x + p * ncta;
                chunk[p] = 0; ci[p] = 0; use_a[p] = 0; use_t[p] = 0; b_tr[p] = 0; b_off[p] = 0;
                a_desc[p] = kDescHi | (uint64_t)((smem_u32(a_smem + (size_t)p * kUM * kUK) >> 4) & 0x3FFF);
            }
            bool busy = true;
            while (busy) {
                busy = false;
#pragma unroll
                for (int p = 0; p < kUPipes; ++p) {
                    if (grp[p] >= a.n_groups) continue;
                    busy = true;
                    const uint32_t tm = tmem_base + p * kUNacc;                  // this pipeline's accumulator
                    const uint64_t ad = a_desc[p], bd = b_desc0 + b_off[p];
                    const uint32_t idesc = (ci[p] == cpt - 1) ? a.idesc_last : a.idesc_full;
                    if (chunk[p] == 0) mbar_wait(&a_full[p], use_a[p] & 1);
                    if (use_t[p] >= 1) mbar_wait(&t_empty[p], (use_t[p] - 1) & 1);
                    tc_fence_after();
                    const bool last_chunk = chunk[p] + 1 == nchunks;
                    if (elect_one()) {
                        if (!(a.debug & 1)) {                                   // a K-step of 8 floats advances the start address by 32 B
                            umma_tf32(tm, ad, bd, idesc, 0);
                            umma_tf32(tm, ad + 2, bd + 2, idesc, 1);
                            umma_tf32(tm, ad + 4, bd + 4, idesc, 1);
                            umma_tf32(tm, ad + 6, bd + 6, idesc, 1);
                        }
                        umma_commit(&t_full[p]);                    // accumulator ready for this pipeline's epilogue warps
                        if (last_chunk) umma_commit(&a_empty[p]);   // all MMAs reading this A'' tile have completed
                    }
                    __syncwarp();
                    ++use_t[p];
                    if (++ci[p] == cpt) { ci[p] = 0; b_tr[p] += trace_step; b_off[p] = b_tr[p]; }
                    else b_off[p] += kUNacc * (kUK * 4 / 16);
                    if (++chunk[p] == nchunks) {
                        chunk[p] = 0; ci[p] = 0; b_tr[p] = 0; b_off[p] = 0; ++use_a[p];
                        grp[p] += kUPipes * ncta;
                    }
                }
            }
        }
    } else {
        // ------------------------------------------------ epilogue warps: pipeline p = warp / 4, TMEM lane quarter = warp % 4,
        //                                                  one sample per thread
        const int p = warp >> 2, wq = warp & 3;
        const bool simul = a.flags & FWI_FLAG_SIMULTANEOUS;
        const bool vr_like = a.metric == FWI_METRIC_VR || a.metric == FWI_METRIC_GAU;
        const double Tn = (double)a.T;
        int use_t = 0;
        for (int g = blockIdx.x + p * ncta; g < a.n_groups; g += kUPipes * ncta) {
            const int64_t n = (int64_t)g * kUM + wq * 32 + lane;
            const bool live = n < a.N;
            double coef[9];
            if (MODE != MODE_SSE) {
#pragma unroll
                for (int c = 0; c < 9; ++c) coef[c] = (live && c < a.C) ? (double)a.M[(size_t)c * a.ldm + n] : 0.0;
            }
            double q0 = 0.0, q1 = 0.0, q2 = 0.0;
            double grp_first = 0.0, carry_s = 0.0, carry_d = 0.0;     // flattened CC-shift: boundary values (see the header)
            for (int k = k0; k < k1; ++k) {
                float s0 = 0.f, s1 = 0.f, s2a = 0.f, s3 = 0.f, vmax = -3.0e38f, vmin = 3.0e38f;
                float p0 = 0.f, p1 = 0.f, prev = 0.f;                 // CC-shift: lag-one products, last column of the previous piece
                // the trace's constants and the first-order terms (9-term dot products with float64 constants) do not need the
                // accumulator: they are issued here, so that their loads and fp64 chains overlap the wait for this trace's first MMAs
                const double* ck = cst + (k - k0) * kUCst;
                const TraceConst tc = *reinterpret_cast<const TraceConst*>(ck + 45);
                double mud = 0.0, sd = 0.0, dlt = 0.0, f = 0.0, l = 0.0;
                if (MODE != MODE_SSE) {
#pragma unroll
                    for (int c = 0; c < 9; ++c) {                     // (components past C hold 0 in both factors)
                        mud = fma(coef[c], ck[c], mud);
                        sd = fma(coef[c], ck[9 + c], sd);
                        if (SH) { dlt = fma(coef[c], ck[18 + c], dlt); f = fma(coef[c], ck[27 + c], f); l = fma(coef[c], ck[36 + c], l); }
                    }
                }
                for (int ci = 0; ci < a.chunks_per_trace; ++ci, ++use_t) {
                    mbar_wait(&t_full[p], use_t & 1);
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + p * kUNacc + ((uint32_t)(wq * 32) << 16);
                    // columns the MMA of this chunk wrote (those past T hold 0: B'' is zero-padded); a multiple of 16
                    const int ncol = (ci == a.chunks_per_trace - 1) ? a.n_last : kUNacc;
                    // one 32-column piece of the accumulator (a trace's last piece may hold 16 columns: `half`)
                    auto fold = [&](const float (&v)[32], const bool half) {
#pragma unroll
                        for (int i = 0; i < 32; i += 4) {
                            if (i < 16 || !half) {
                                s0 = fmaf(v[i], v[i], s0); s1 = fmaf(v[i + 1], v[i + 1], s1);
                                s2a = fmaf(v[i + 2], v[i + 2], s2a); s3 = fmaf(v[i + 3], v[i + 3], s3);
                                if (MODE == MODE_MOM_MAX) {
                                    vmax = fmax3(vmax, v[i], v[i + 1]); vmin = fmin3(vmin, v[i], v[i + 1]);
                                    vmax = fmax3(vmax, v[i + 2], v[i + 3]); vmin = fmin3(vmin, v[i + 2], v[i + 3]);
                                }
                                if (SH) {
                                    // s'[t] s'[t+1]: columns past T hold 0, so the products past the trace's end vanish
                                    p0 = fmaf(i == 0 ? prev : v[i - 1], v[i], p0); p1 = fmaf(v[i], v[i + 1], p1);
                                    p0 = fmaf(v[i + 1], v[i + 2], p0); p1 = fmaf(v[i + 2], v[i + 3], p1);
                                }
                            }
                        }
                        if (SH) prev = v[31];                           // (a 16-column piece is a trace's last: prev is reset)
                    };
                    auto release = [&]() {                              // accumulator drained by this warp
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&t_empty[p]);
                    };
                    if (a.debug & 2) {
                        release();
                    } else if (ncol == kUNacc) {
                        // full chunk, unrolled: the next piece's tcgen05.ld is in flight while the current piece is folded, and the
                        // accumulator goes back to the MMA issuer as soon as its last piece is in registers
                        float va[32], vb[32];
                        tmem_ld32(taddr, va);
#pragma unroll 4
                        for (int i = 0; i < kUNacc / 32; i += 2) {
                            tmem_ld_wait_dep(va);
                            tmem_ld32(taddr + (i + 1) * 32, vb);
                            fold(va, false);
                            tmem_ld_wait_dep(vb);
                            if (i + 2 < kUNacc / 32) tmem_ld32(taddr + (i + 2) * 32, va); else release();
                            fold(vb, false);
                        }
                    } else {
                        for (int c0 = 0; c0 < ncol; c0 += 32) {
                            float v[32];
                            tmem_ld32(taddr + c0, v);
                            tmem_ld_wait_dep(v);
                            fold(v, ncol - c0 < 32);
                        }
                        release();
                    }
                }
                // ---- combine trace k (float64; the expressions of mc_eval_kernel's fold)
                const double s2 = (double)((s0 + s1) + (s2a + s3));
                if (MODE == MODE_SSE) {
                    const double sse = s2, dd = tc.sumd2;
                    q1 += sse; q2 += dd;
                    if (a.metric == FWI_METRIC_VR) q0 += fmax(0.0, fma(-sse, rcp64(dd), 1.0));     // FWI:515-519
                    else q0 += exp(-sse / (2.0 * tc.sigma * tc.sigma));                         // FWI:581
                } else if (SH) {
                    // ---- CC-shift: moments of the 4x interpolated trace from S2, P and five dot products
                    const double Tv = 4.0 * Tn, P = (double)(p0 + p1);
                    const double ssq = fma(2.75, s2, fma(1.25, P, fma(2.125 * l, l, -0.875 * f * f))) - Tv * dlt * dlt;   // sum_i (s_i - mean_i s)^2
                    const double mui = mud + dlt;                                               // mean of the interpolated synthetic
                    if (!simul) {
                        const double pcc = sd * rsqrt64(ssq * tc.ssd);                          // FWI:572-573 on the interpolated rows
                        q0 += (pcc < 0.0) ? 0.0 : pcc;
                    } else {
                        double aa = 1.0, bb = 1.0;
                        if (MODE == MODE_MOM_MAX) {
                            aa = rcp64(fmax(fabs((double)vmax + mud), fabs((double)vmin + mud)));
                            bb = rcp64(tc.maxd);
                        }
                        double A1 = aa * Tv * mui, A2 = aa * aa * (ssq + Tv * mui * mui), A3 = aa * bb * (sd + Tv * tc.mean_d * mui);
                        const double first = (f + mud) * aa;
                        if (k > k0) {                                                           // np.interp across the boundary (FWI:612, 554-555)
                            const double dl = first - carry_s, dd = tc.d_first * bb - carry_d;
                            A1 += 1.5 * dl;
                            A2 += 3.0 * carry_s * dl + 0.875 * dl * dl;
                            A3 += 1.5 * (carry_d * dl + carry_s * dd) + 0.875 * dd * dl;
                        } else grp_first = first;
                        carry_s = (l + mud) * aa;
                        carry_d = tc.d_last * bb;
                        q0 += A1; q1 += A2; q2 += A3;
                    }
                } else {
                    double aa = 1.0, bb = 1.0;
                    if (MODE == MODE_MOM_MAX) {
                        aa = rcp64(fmax(fabs((double)vmax + mud), fabs((double)vmin + mud)));     // FWI:598-599
                        bb = rcp64(tc.maxd);
                    }
                    if (vr_like) {
                        const double Sss = (s2 + Tn * mud * mud) * aa * aa;
                        const double Sds = (sd + Tn * tc.mean_d * mud) * aa * bb;
                        const double dd = tc.sumd2 * bb * bb;
                        const double sse = dd - 2.0 * Sds + Sss;
                        const double sig = tc.sigma * bb;
                        q1 += sse; q2 += dd;
                        if (a.metric == FWI_METRIC_VR) q0 += fmax(0.0, fma(-sse, rcp64(dd), 1.0));
                        else q0 += exp(-sse / (2.0 * sig * sig));
                    } else if (!simul) {
                        const double pcc = sd * rsqrt64(s2 * tc.ssd);                           // FWI:572-573
                        q0 += (pcc < 0.0) ? 0.0 : pcc;                                          // FWI:574-575
                    } else {
                        q0 += aa * Tn * mud;
                        q1 += aa * aa * (s2 + Tn * mud * mud);
                        q2 += aa * bb * (sd + Tn * tc.mean_d * mud);
                    }
                }
            }
            if (live) {
                double* o = a.part + (size_t)tg * a.npart * a.N + n;
                o[0] = q0; o[a.N] = q1; o[2 * a.N] = q2;
                if (SH && a.npart == 5) { o[3 * a.N] = grp_first; o[4 * a.N] = carry_s; }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMma) tmem_dealloc(tmem_base, 512);
}

// A''[n][32] from the sampler's (rows, N) layout; `with_d`: the two -1 columns that subtract d (MODE_SSE)
__global__ void mc_umma_pack_kernel(const float* __restrict__ M, int64_t ldm, int C, int64_t N, int64_t Npad, int with_d, float* __restrict__ A) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= Npad) return;
    float row[kUK];
#pragma unroll
    for (int i = 0; i < kUK; ++i) row[i] = 0.f;
    if (n < N) {
#pragma unroll
        for (int c = 0; c < 9; ++c) {
            if (c < C) {
                const float x = M[(size_t)c * ldm + n];
                const float hi = tf32_round(x), lo = tf32_round(x - hi);
                row[c] = hi; row[C + c] = hi; row[2 * C + c] = lo;
            }
        }
        if (with_d) { row[3 * C] = -1.f; row[3 * C + 1] = -1.f; }
    }
    float4* dst = reinterpret_cast<float4*>(A + (size_t)n * kUK);
#pragma unroll
    for (int i = 0; i < kUK / 4; ++i) dst[i] = make_float4(row[4 * i], row[4 * i + 1], row[4 * i + 2], row[4 * i + 3]);
}

// adds the trace groups' partial sums and applies the final expressions of mc_eval_kernel (FWI:601-632, 682, 774)
// `tc` / `traces_per_cta`: flattened CC-shift only - the boundary patch between the last trace of a group and the first of the next
__global__ void mc_umma_finish_kernel(const double* __restrict__ part, int npart, int ngroups, int64_t N, int K, int metric, int flags, FlatConst fc,
                                      const TraceConst* __restrict__ tc, int traces_per_cta, float* __restrict__ sim, float* __restrict__ like) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const bool norm = flags & FWI_FLAG_NORMALISED, simul = flags & FWI_FLAG_SIMULTANEOUS;
    double q0 = 0.0, q1 = 0.0, q2 = 0.0;
    for (int g = 0; g < ngroups; ++g) {
        const double* o = part + (size_t)g * npart * N + n;
        q0 += o[0]; q1 += o[N]; q2 += o[2 * N];
        if (npart == 5 && g > 0) {
            const int kb = g * traces_per_cta;                                   // first trace of this group
            const double bl = norm ? 1.0 / tc[kb - 1].maxd : 1.0, bf = norm ? 1.0 / tc[kb].maxd : 1.0;
            const double cs = (o - (size_t)npart * N)[4 * N], cd = tc[kb - 1].d_last * bl;   // the previous group's last values
            const double dl = o[3 * N] - cs, dd = tc[kb].d_first * bf - cd;
            q0 += 1.5 * dl;
            q1 += 3.0 * cs * dl + 0.875 * dl * dl;
            q2 += 1.5 * (cd * dl + cs * dd) + 0.875 * dd * dl;
        }
    }
    const bool vr_like = metric == FWI_METRIC_VR || metric == FWI_METRIC_GAU;
    double result;
    if (vr_like) {
        if (simul) {
            if (metric == FWI_METRIC_VR) result = fmax(0.0, 1.0 - q1 / q2);
            else { const double sg = fc.sigma[norm ? 1 : 0]; result = exp(-q1 / (2.0 * sg * sg)); }
        } else {
            result = q0 / K;                                                               // FWI:682
            if (metric == FWI_METRIC_GAU && (flags & FWI_FLAG_STRICT_REF)) result = 0.0;   // quirk q1
        }
    } else if (!simul) {
        result = q0 / K;
    } else {
        const int ni = norm ? 1 : 0;
        const double nn = fc.n, D1 = fc.D1[ni], D2 = fc.D2[ni];
        const double cov = q2 - q0 * D1 / nn, vs = q1 - q0 * q0 / nn, vd = D2 - D1 * D1 / nn;
        const double pcc = cov / sqrt(vs * vd);
        result = (pcc < 0.0) ? 0.0 : pcc;
    }
    sim[n] = (float)result;
    if (like) like[n] = (float)exp(-(1.0 - result) * 0.5);                                 // FWI:774
}

typedef CUresult (*EncodeTiledFn2)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int encode_rows32_sw128(CUtensorMap* out, void* base, uint64_t rows, uint32_t box_rows) {
    static EncodeTiledFn2 fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        FWI_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        if (!p || q != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled not available from the driver"); return FWI_ECUDA; }
        fn = (EncodeTiledFn2)p;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)kUK, rows};
    const cuuint64_t strides[1] = {(cuuint64_t)kUK * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)kUK, box_rows}, es[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (swizzle 128B) failed with CUresult %d", (int)r); return FWI_ECUDA; }
    return FWI_OK;
}

// Device-resident state of the tensor-core path for one (G, d).
struct UmmaPath {
    int device = 0, K = 0, C = 0, T = 0, tiles_per_trace = 0, traces_per_cta = 0, n_tgroups = 0, sms = 148;
    float* B_raw = nullptr;      // [K][tiles_per_trace * 256][32]: G and d (MODE_SSE)
    float* B_cen = nullptr;      // same with centred G and no d (moment modes)
    double* gbar = nullptr;      // [K][C]
    double* gdc = nullptr;       // [K][C]
    const TraceConst* tc = nullptr;   // owned by the Monte-Carlo context
    FlatConst fc{};
    // CC-shift: constants of the 4x interpolated rows (per trace clamped; the flattened array runs across the boundaries)
    double* shc = nullptr;            // [K][4][C], see UmmaEvalArgs
    TraceConst* tc_hr = nullptr;      // [K]
    FlatConst fc_hr{};
    float* A = nullptr; size_t A_rows = 0;
    double* part = nullptr; size_t part_cap = 0;
    CUtensorMap tm_raw, tm_cen;
};

constexpr int kUSmem = kUTilesMax * kUN * kUK * 4 + kUPipes * kUM * kUK * 4 + 256 + kUTilesMax * kUCst * 8;
static_assert(kUSmem <= 227 * 1024, "shared memory budget");
static_assert(sizeof(TraceConst) == 7 * sizeof(double), "TraceConst is copied to shared memory as 7 doubles");

int umma_build(UmmaPath** out, int device, const double* G, const double* d, int K, int C, int T, const TraceConst* tc_dev,
               const FlatConst& fc) {
    *out = nullptr;
    const int tpt = (T + kUN - 1) / kUN;
    if (3 * C + 2 > kUK || C > 9 || tpt > kUTilesMax || K < 1 || T < 1) return FWI_OK;      // shape not covered: CUDA-core kernels only
    auto* u = new UmmaPath();
    u->device = device; u->K = K; u->C = C; u->T = T; u->tiles_per_trace = tpt; u->tc = tc_dev; u->fc = fc;
    u->traces_per_cta = std::max(1, kUTilesMax / tpt);
    u->n_tgroups = (K + u->traces_per_cta - 1) / u->traces_per_cta;
    cudaDeviceGetAttribute(&u->sms, cudaDevAttrMultiProcessorCount, device);
    const size_t rows = (size_t)K * tpt * kUN;
    std::vector<float> Br(rows * kUK, 0.f), Bc(rows * kUK, 0.f);
    std::vector<double> gbar((size_t)K * C), gdc((size_t)K * C);
    for (int k = 0; k < K; ++k) {
        double md = 0.0;
        for (int t = 0; t < T; ++t) md += d[(size_t)k * T + t];
        md /= T;
        for (int c = 0; c < C; ++c) {
            const double* g = G + ((size_t)k * C + c) * T;
            double gs = 0.0, gd = 0.0;
            for (int t = 0; t < T; ++t) { gs += g[t]; gd += (d[(size_t)k * T + t] - md) * g[t]; }
            gbar[(size_t)k * C + c] = gs / T;
            gdc[(size_t)k * C + c] = gd;
        }
        for (int t = 0; t < T; ++t) {
            float* rr = &Br[((size_t)k * tpt * kUN + t) * kUK];
            float* rc = &Bc[((size_t)k * tpt * kUN + t) * kUK];
            for (int c = 0; c < C; ++c) {
                const double gv = G[((size_t)k * C + c) * T + t];
                float x = (float)gv, hi = tf32_round(x), lo = tf32_round(x - hi);
                rr[c] = hi; rr[C + c] = lo; rr[2 * C + c] = hi;
                x = (float)(gv - gbar[(size_t)k * C + c]); hi = tf32_round(x); lo = tf32_round(x - hi);
                rc[c] = hi; rc[C + c] = lo; rc[2 * C + c] = hi;
            }
            const float dv = (float)d[(size_t)k * T + t];
            const float dhi = tf32_round(dv), dlo = tf32_round(dv - dhi);
            rr[3 * C] = dhi; rr[3 * C + 1] = dlo;
        }
    }
    // CC-shift (FWI:548-566): float64 constants of the 4x linearly interpolated rows.  x_i[4t + j] = x[t] + (x[t+1] - x[t]) j/4,
    // the right edge clamps (np.interp); the flattened array (FWI:612) runs into the next trace's first sample instead.
    const int Tv = 4 * T;
    std::vector<double> shc((size_t)K * 4 * C);
    std::vector<TraceConst> tch(K);
    {
        std::vector<double> di(Tv), gi(Tv);
        auto interp_clamped = [&](const double* x, std::vector<double>& out) {
            for (int t = 0; t < T; ++t)
                for (int j = 0; j < 4; ++j) out[4 * t + j] = (t + 1 < T) ? x[t] + (x[t + 1] - x[t]) * (0.25 * j) : x[t];
        };
        for (int k = 0; k < K; ++k) {
            const double* dk = d + (size_t)k * T;
            interp_clamped(dk, di);
            TraceConst& q = tch[k];
            double sum = 0.0, sum2 = 0.0, ssd = 0.0, mx = 0.0;
            for (int i = 0; i < Tv; ++i) { sum += di[i]; sum2 += di[i] * di[i]; }
            q.mean_d = sum / Tv; q.sumd2 = sum2;
            for (int i = 0; i < Tv; ++i) ssd += (di[i] - q.mean_d) * (di[i] - q.mean_d);
            for (int t = 0; t < T; ++t) mx = std::max(mx, std::fabs(dk[t]));
            q.ssd = ssd; q.maxd = mx; q.sigma = NAN; q.d_first = dk[0]; q.d_last = dk[T - 1];
            for (int c = 0; c < C; ++c) {
                const double* gk = G + ((size_t)k * C + c) * T;
                interp_clamped(gk, gi);
                double gs = 0.0, gd = 0.0;
                for (int i = 0; i < Tv; ++i) { gs += gi[i]; gd += (di[i] - q.mean_d) * gi[i]; }
                double* sc = &shc[(size_t)k * 4 * C];
                sc[c] = gs / Tv - gbar[(size_t)k * C + c];
                sc[C + c] = gd;
                sc[2 * C + c] = gk[0] - gbar[(size_t)k * C + c];
                sc[3 * C + c] = gk[T - 1] - gbar[(size_t)k * C + c];
            }
        }
        u->fc_hr = FlatConst{};
        u->fc_hr.n = (double)K * Tv;
        const size_t nf = (size_t)K * T;
        for (int norm = 0; norm < 2; ++norm) {
            auto at = [&](size_t i) { return d[i] / (norm ? tch[i / T].maxd : 1.0); };     // normalised BEFORE the interpolation (FWI:598, 612)
            double s1 = 0.0, s2 = 0.0;
            for (size_t i = 0; i < nf; ++i)
                for (int j = 0; j < 4; ++j) {
                    const double x = (i + 1 < nf) ? at(i) + (at(i + 1) - at(i)) * (0.25 * j) : at(i);
                    s1 += x; s2 += x * x;
                }
            u->fc_hr.D1[norm] = s1; u->fc_hr.D2[norm] = s2; u->fc_hr.sigma[norm] = NAN;
        }
    }
    DeviceGuard g(device);
    auto fail = [&](int rc) { umma_free(u); return rc; };
    if (cudaMalloc(&u->B_raw, Br.size() * sizeof(float)) != cudaSuccess || cudaMalloc(&u->B_cen, Bc.size() * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&u->gbar, gbar.size() * sizeof(double)) != cudaSuccess || cudaMalloc(&u->gdc, gdc.size() * sizeof(double)) != cudaSuccess ||
        cudaMalloc(&u->shc, shc.size() * sizeof(double)) != cudaSuccess || cudaMalloc(&u->tc_hr, tch.size() * sizeof(TraceConst)) != cudaSuccess) {
        cudaGetLastError(); set_error("umma_build: out of device memory"); return fail(FWI_ENOMEM);
    }
    cudaMemcpy(u->shc, shc.data(), shc.size() * sizeof(double), cudaMemcpyHostToDevice);
    cudaMemcpy(u->tc_hr, tch.data(), tch.size() * sizeof(TraceConst), cudaMemcpyHostToDevice);
    cudaMemcpy(u->B_raw, Br.data(), Br.size() * sizeof(float), cudaMemcpyHostToDevice);
    cudaMemcpy(u->B_cen, Bc.data(), Bc.size() * sizeof(float), cudaMemcpyHostToDevice);
    cudaMemcpy(u->gbar, gbar.data(), gbar.size() * sizeof(double), cudaMemcpyHostToDevice);
    cudaMemcpy(u->gdc, gdc.data(), gdc.size() * sizeof(double), cudaMemcpyHostToDevice);
    int rc = encode_rows32_sw128(&u->tm_raw, u->B_raw, rows, kUN);
    if (!rc) rc = encode_rows32_sw128(&u->tm_cen, u->B_cen, rows, kUN);
    if (rc) return fail(rc);
    if (cudaFuncSetAttribute(mc_umma_kernel<MODE_SSE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUSmem) != cudaSuccess ||
        cudaFuncSetAttribute(mc_umma_kernel<MODE_MOM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUSmem) != cudaSuccess ||
        cudaFuncSetAttribute(mc_umma_kernel<MODE_MOM_MAX, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUSmem) != cudaSuccess ||
        cudaFuncSetAttribute(mc_umma_kernel<MODE_MOM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUSmem) != cudaSuccess ||
        cudaFuncSetAttribute(mc_umma_kernel<MODE_MOM_MAX, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUSmem) != cudaSuccess) {
        cudaGetLastError(); return fail(FWI_OK);          // no tensor-core path on this device: CUDA-core kernels only
    }
    *out = u;
    return FWI_OK;
}

void umma_free(UmmaPath* u) {
    if (!u) return;
    DeviceGuard g(u->device);
    if (u->B_raw) cudaFree(u->B_raw);
    if (u->B_cen) cudaFree(u->B_cen);
    if (u->gbar) cudaFree(u->gbar);
    if (u->gdc) cudaFree(u->gdc);
    if (u->shc) cudaFree(u->shc);
    if (u->tc_hr) cudaFree(u->tc_hr);
    if (u->A) cudaFree(u->A);
    if (u->part) cudaFree(u->part);
    delete u;
}

bool umma_supports(const UmmaPath* u, int metric, int flags) {
    if (!u) return false;
    if (flags & FWI_FLAG_GRAM) return false;                                         // the Gram algorithm stays on the CUDA cores
    if (metric == FWI_METRIC_CC_SHIFT && u->T < 2) return false;
    if (metric == FWI_METRIC_GAU && u->T < 60) return false;
    return true;
}

int umma_eval(UmmaPath* u, const float* M_dev, int64_t ldm, int64_t N, int metric, int flags, float* sim_dev, float* like_dev, cudaStream_t st) {
    if (N == 0) return FWI_OK;
    DeviceGuard g(u->device);
    const bool norm = flags & FWI_FLAG_NORMALISED, simul = flags & FWI_FLAG_SIMULTANEOUS;
    int mode;
    if (metric == FWI_METRIC_VR || metric == FWI_METRIC_GAU) mode = norm ? MODE_MOM_MAX : MODE_SSE;
    else mode = (simul && norm) ? MODE_MOM_MAX : MODE_MOM;
    const bool shift = metric == FWI_METRIC_CC_SHIFT;
    const int npart = (shift && simul) ? 5 : 3;
    const int64_t ngroups = (N + kUM - 1) / kUM, Npad = ngroups * kUM;
    if (u->A_rows < (size_t)Npad) {
        if (u->A) cudaFree(u->A);
        u->A = nullptr; u->A_rows = 0;
        FWI_CUDA(cudaMalloc(&u->A, (size_t)Npad * kUK * sizeof(float)));
        u->A_rows = (size_t)Npad;
    }
    if (u->part_cap < (size_t)u->n_tgroups * npart * N) {
        if (u->part) cudaFree(u->part);
        u->part = nullptr; u->part_cap = 0;
        FWI_CUDA(cudaMalloc(&u->part, (size_t)u->n_tgroups * npart * N * sizeof(double)));
        u->part_cap = (size_t)u->n_tgroups * npart * N;
    }
    CUtensorMap tm_a;
    int rc = encode_rows32_sw128(&tm_a, u->A, (uint64_t)Npad, kUM);
    if (rc) return rc;
    mc_umma_pack_kernel<<<(unsigned)((Npad + 127) / 128), 128, 0, st>>>(M_dev, ldm, u->C, N, Npad, mode == MODE_SSE ? 1 : 0, u->A);
    FWI_CUDA(cudaGetLastError());
    // CTAs per trace group in proportion to its traces (K = 21, two resident traces: 10 groups x 14 CTAs + 1 group x 7 = 147)
    const int last_traces = u->K - (u->n_tgroups - 1) * u->traces_per_cta;
    const int ctas_full = (int)std::min<int64_t>(ngroups, std::max(1, u->sms * u->traces_per_cta / u->K));
    const int ctas_last = (int)std::min<int64_t>(ngroups, std::max(1, u->sms * last_traces / u->K));
    UmmaEvalArgs a{};
    a.N = N; a.n_groups = (int)ngroups; a.tiles_per_trace = u->tiles_per_trace; a.traces_per_cta = u->traces_per_cta;
    a.ctas_full = ctas_full; a.ctas_last = ctas_last;
    a.K = u->K; a.C = u->C; a.T = u->T; a.metric = metric; a.flags = flags;
    { const char* e = getenv("FWI_UMMA_DEBUG"); a.debug = e ? atoi(e) : 0; }
    a.chunks_per_trace = (u->T + kUNacc - 1) / kUNacc;
    a.n_last = ((u->T - (a.chunks_per_trace - 1) * kUNacc) + 15) & ~15;                     // MMA N of a trace's last chunk (multiple of 16)
    auto idesc = [](int n) { return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kUM >> 4) << 24); };
    a.idesc_full = idesc(kUNacc); a.idesc_last = idesc(a.n_last);
    a.tc = shift ? u->tc_hr : u->tc; a.gbar = u->gbar; a.gdc = u->gdc; a.shc = u->shc; a.M = M_dev; a.ldm = ldm; a.part = u->part; a.npart = npart;
    const dim3 grid(std::max(ctas_full, ctas_last), u->n_tgroups);
    if (mode == MODE_SSE) mc_umma_kernel<MODE_SSE, false><<<grid, kUThreads, kUSmem, st>>>(tm_a, u->tm_raw, a);
    else if (mode == MODE_MOM && !shift) mc_umma_kernel<MODE_MOM, false><<<grid, kUThreads, kUSmem, st>>>(tm_a, u->tm_cen, a);
    else if (mode == MODE_MOM) mc_umma_kernel<MODE_MOM, true><<<grid, kUThreads, kUSmem, st>>>(tm_a, u->tm_cen, a);
    else if (!shift) mc_umma_kernel<MODE_MOM_MAX, false><<<grid, kUThreads, kUSmem, st>>>(tm_a, u->tm_cen, a);
    else mc_umma_kernel<MODE_MOM_MAX, true><<<grid, kUThreads, kUSmem, st>>>(tm_a, u->tm_cen, a);
    FWI_CUDA(cudaGetLastError());
    mc_umma_finish_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(u->part, npart, u->n_tgroups, N, u->K, metric, flags, shift ? u->fc_hr : u->fc,
                                                                        u->tc_hr, u->traces_per_cta, sim_dev, like_dev);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

}  // namespace fwi
