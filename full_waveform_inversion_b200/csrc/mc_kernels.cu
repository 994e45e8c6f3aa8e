// Track A: batched Monte-Carlo source-inversion hot path for sm_100a.
//
//   sample -> forward model -> misfit -> likelihood            (FWI:713-774)
//
// A lane owns S source samples whose coefficient vectors live in registers; a warp walks the traces and streams each
// trace's prepared rows [t][G_0..G_{CC-1}, d, d'] with warp-uniform 16-byte loads (one LDG.128 feeds four FMAs of
// every lane), so the K*T*C contraction needs no cross-thread reduction at all.  After each trace the lane folds that
// trace's statistics into running per-sample sums in float64 (warp-private shared memory), so the footprint does not
// depend on K.  Big batches: every warp (pair) owns its own samples; small, latency-bound batches: the warps of a CTA
// share one sample group and split the traces.
// The path is FP32-FMA bound (G is ~0.4 MB and L2/L1 resident; ~40-80 B of HBM traffic per sample).
#include "common.cuh"
#include "mc_common.cuh"
#include <climits>
#include <cmath>
#include <cstring>
#include <vector>
#include <algorithm>

namespace fwi {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

struct EvalParams {
    const float* rows;
    const float* gbar;
    const TraceConst* tc;
    FlatConst fc;
    const int* phase;
    const float* M;
    int64_t ldm;
    const float* frac;
    int nfrac;
    int64_t N;
    int K, Tv, metric, flags, boundary_fix;
    int ks;                  // warps of a CTA that share one sample group and split the traces between them (1 = none)
    float* sim;
    float* like;
};

__host__ __device__ constexpr int row_width(int CC) { return (CC + 2 + 3) & ~3; }
__host__ __device__ constexpr int nstat(int mode) { return mode == MODE_SSE ? 1 : (mode == MODE_MOM ? 3 : 4); }

template <int C, int NM>
__device__ __forceinline__ void make_coef(float (&coef)[C * NM], const float (&m)[C], float f) {
    if (NM == 1) {
#pragma unroll
        for (int c = 0; c < C; ++c) coef[c] = m[c];
    } else {
#pragma unroll
        for (int c = 0; c < C; ++c) {
            coef[c] = m[c] * (1.0f - f);     // synth = (1-f) G0.M + f G1.M   (FWI:727, FWI:731)
            coef[C + c] = m[c] * f;
        }
    }
}

// ---------------------------------------------------------------------------------------------
constexpr int kMcAcc = 5;      // running sums per sample: 3 accumulators + the two boundary-patch carries of flattened CC-shift

template <int C, int NM, int S, int MODE>
__global__ void __launch_bounds__(S * NM >= 8 ? 128 : 256, 3) mc_eval_kernel(EvalParams p) {
    constexpr int CC = C * NM;
    constexpr int RW = row_width(CC);
    constexpr int RW4 = RW / 4;
    constexpr int SPW = 32 * S;               // samples per warp
    constexpr int CHUNK = 64;
    extern __shared__ double fold_smem[];     // [warps][kMcAcc][SPW] float64, private to each warp (no block-level sync)

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nwarps = blockDim.x >> 5;
    // Large batches: every warp owns its own SPW samples and walks all K traces (ks = 1, no block-level sync at all).
    // Small batches are latency-bound, so ks warps share one sample group and take every ks-th trace each.
    const int kw = warp % p.ks;
    const int64_t base = ((int64_t)blockIdx.x * (nwarps / p.ks) + warp / p.ks) * SPW;
    const bool active = base < p.N;           // warp-uniform
    double* acc = fold_smem + (size_t)warp * kMcAcc * SPW + lane;          // acc[j * SPW + s * 32]
#pragma unroll
    for (int j = 0; j < kMcAcc; ++j)
#pragma unroll
        for (int s = 0; s < S; ++s) acc[j * SPW + s * 32] = 0.0;

    float m[S][C];
    float fr[S][3];
#pragma unroll
    for (int s = 0; s < S; ++s) {
        int64_t n = base + s * 32 + lane;
        if (n >= p.N) n = p.N - 1;            // tail lanes recompute the last sample, never stored
#pragma unroll
        for (int c = 0; c < C; ++c) m[s][c] = __ldg(p.M + (int64_t)c * p.ldm + n);
#pragma unroll
        for (int j = 0; j < 3; ++j) fr[s][j] = 0.f;
        if (NM == 2) {
            for (int j = 0; j < p.nfrac; ++j) fr[s][j] = __ldg(p.frac + (int64_t)j * p.ldm + n);
        }
    }

    for (int k = active ? kw : p.K; k < p.K; k += p.ks) {
        float coef[S][CC];
        float mu[S];
        const int ph = (NM == 2 && p.nfrac == 3 && p.phase) ? p.phase[k] : 0;
#pragma unroll
        for (int s = 0; s < S; ++s) {
            make_coef<C, NM>(coef[s], m[s], fr[s][ph]);
            float a = 0.f;
            if (MODE != MODE_SSE) {
#pragma unroll
                for (int c = 0; c < CC; ++c) a = fmaf(__ldg(p.gbar + k * CC + c), coef[s][c], a);
            }
            mu[s] = a;
        }
        double t0[S], t1[S];
        float vmax[S], vmin[S];
#pragma unroll
        for (int s = 0; s < S; ++s) { t0[s] = 0.0; t1[s] = 0.0; vmax[s] = -INFINITY; vmin[s] = INFINITY; }

        const float4* rp = reinterpret_cast<const float4*>(p.rows) + (size_t)k * p.Tv * RW4;
        for (int tb = 0; tb < p.Tv; tb += CHUNK) {
            const int te = min(p.Tv, tb + CHUNK);
            float a0[S], a1[S];
#pragma unroll
            for (int s = 0; s < S; ++s) { a0[s] = 0.f; a1[s] = 0.f; }
            // two time samples per iteration: 2*S independent FMA chains per lane keep the fp32 pipe fed
            auto finish = [&](const float (&r)[RW], const float (&v)[S]) {
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    if (MODE == MODE_SSE) {
                        const float e = r[CC] - v[s];              // raw d - raw synth (FWI:515)
                        a0[s] = fmaf(e, e, a0[s]);
                    } else {
                        a0[s] = fmaf(v[s], v[s], a0[s]);           // sum s'^2
                        a1[s] = fmaf(r[CC + 1], v[s], a1[s]);      // sum d' s'
                        if (MODE == MODE_MOM_MAX) { vmax[s] = fmaxf(vmax[s], v[s]); vmin[s] = fminf(vmin[s], v[s]); }
                    }
                }
            };
            int t = tb;
#pragma unroll 2
            for (; t + 1 < te; t += 2) {
                float r0[RW], r1[RW];
#pragma unroll
                for (int q = 0; q < RW4; ++q) {
                    const float4 u = __ldg(rp + (size_t)t * RW4 + q), w = __ldg(rp + (size_t)(t + 1) * RW4 + q);
                    r0[4 * q] = u.x; r0[4 * q + 1] = u.y; r0[4 * q + 2] = u.z; r0[4 * q + 3] = u.w;
                    r1[4 * q] = w.x; r1[4 * q + 1] = w.y; r1[4 * q + 2] = w.z; r1[4 * q + 3] = w.w;
                }
                float v0[S], v1[S];
#pragma unroll
                for (int s = 0; s < S; ++s) { v0[s] = (MODE == MODE_SSE) ? 0.f : -mu[s]; v1[s] = v0[s]; }
#pragma unroll
                for (int c = 0; c < CC; ++c) {
#pragma unroll
                    for (int s = 0; s < S; ++s) { v0[s] = fmaf(r0[c], coef[s][c], v0[s]); v1[s] = fmaf(r1[c], coef[s][c], v1[s]); }
                }
                finish(r0, v0);
                finish(r1, v1);
            }
            for (; t < te; ++t) {
                float r[RW];
#pragma unroll
                for (int q = 0; q < RW4; ++q) {
                    const float4 u = __ldg(rp + (size_t)t * RW4 + q);
                    r[4 * q] = u.x; r[4 * q + 1] = u.y; r[4 * q + 2] = u.z; r[4 * q + 3] = u.w;
                }
                float v[S];
#pragma unroll
                for (int s = 0; s < S; ++s) v[s] = (MODE == MODE_SSE) ? 0.f : -mu[s];
#pragma unroll
                for (int c = 0; c < CC; ++c) {
#pragma unroll
                    for (int s = 0; s < S; ++s) v[s] = fmaf(r[c], coef[s][c], v[s]);
                }
                finish(r, v);
            }
#pragma unroll
            for (int s = 0; s < S; ++s) { t0[s] += (double)a0[s]; t1[s] += (double)a1[s]; }
        }

        // ---- fold trace k into the running per-sample sums (float64: the expressions cancel), each lane its own samples
        const TraceConst tc = p.tc[k];
        const bool simul = p.flags & FWI_FLAG_SIMULTANEOUS;
        const bool vr_like = p.metric == FWI_METRIC_VR || p.metric == FWI_METRIC_GAU;
        const double Tn = (double)p.Tv;
        // CC-shift, normalised, flattened: np.interp runs across trace boundaries on the already-normalised flattened
        // arrays (FWI:612, FWI:554-555); the rows hold the per-trace clamped interpolation, so the 3 points after each
        // internal boundary are patched from the first / last synthetic value of the neighbouring traces.
        const bool patch = MODE == MODE_MOM_MAX && !vr_like && simul && p.boundary_fix;
        const float* rf = p.rows + (size_t)k * p.Tv * RW;
        const float* rl = rf + (size_t)(p.Tv - 1) * RW;
#pragma unroll
        for (int s = 0; s < S; ++s) {
            double* q = acc + s * 32;
            const double s2 = t0[s], sd = t1[s], mud = (double)mu[s];
            double a = 1.0, b = 1.0;
            if (MODE == MODE_MOM_MAX) {
                a = 1.0 / fmax(fabs((double)vmax[s] + mud), fabs((double)vmin[s] + mud));      // FWI:598-599
                b = 1.0 / tc.maxd;
            }
            if (vr_like) {
                double sse, dd, sig = tc.sigma;
                if (MODE == MODE_SSE) {
                    sse = s2;
                    dd = tc.sumd2;
                } else {
                    const double Sss = (s2 + Tn * mud * mud) * a * a;
                    const double Sds = (sd + Tn * tc.mean_d * mud) * a * b;
                    dd = tc.sumd2 * b * b;
                    sse = dd - 2.0 * Sds + Sss;
                    sig = tc.sigma * b;
                }
                q[SPW] += sse;
                q[2 * SPW] += dd;
                if (p.metric == FWI_METRIC_VR) q[0] += fmax(0.0, 1.0 - sse / dd);      // FWI:515-519
                else q[0] += exp(-sse / (2.0 * sig * sig));                             // FWI:581
            } else if (!simul) {
                const double pcc = sd / sqrt(s2 * tc.ssd);                              // FWI:572-573
                q[0] += (pcc < 0.0) ? 0.0 : pcc;                                        // FWI:574-575
            } else {
                double A1 = a * Tn * mud, A2 = a * a * (s2 + Tn * mud * mud), A3 = a * b * (sd + Tn * tc.mean_d * mud);
                if (patch) {
                    double first = 0.0, last = 0.0;
#pragma unroll
                    for (int c = 0; c < CC; ++c) { first += (double)__ldg(rf + c) * coef[s][c]; last += (double)__ldg(rl + c) * coef[s][c]; }
                    if (k > 0) {
                        const double c_ = q[3 * SPW], cd = q[4 * SPW];
                        const double dl = first * a - c_, dd = tc.d_first * b - cd;
                        A1 += 1.5 * dl;
                        A2 += 3.0 * c_ * dl + 0.875 * dl * dl;
                        A3 += 1.5 * (cd * dl + c_ * dd) + 0.875 * dd * dl;
                    }
                    q[3 * SPW] = last * a;
                    q[4 * SPW] = tc.d_last * b;
                }
                q[0] += A1; q[SPW] += A2; q[2 * SPW] += A3;
            }
        }
    }

    // ---- similarity and likelihood of this lane's samples (the first warp of a group adds its partners' sums first)
    if (p.ks > 1) {
        __syncthreads();
        if (kw == 0) {
            for (int w = 1; w < p.ks; ++w) {
                const double* o = acc + (size_t)w * kMcAcc * SPW;
#pragma unroll
                for (int j = 0; j < 3; ++j)
#pragma unroll
                    for (int s = 0; s < S; ++s) acc[j * SPW + s * 32] += o[j * SPW + s * 32];
            }
        }
    }
    if (!active || kw != 0) return;
    const bool norm = p.flags & FWI_FLAG_NORMALISED;
    const bool simul = p.flags & FWI_FLAG_SIMULTANEOUS;
    const bool vr_like = p.metric == FWI_METRIC_VR || p.metric == FWI_METRIC_GAU;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const int64_t n = base + s * 32 + lane;
        if (n >= p.N) continue;
        const double* q = acc + s * 32;
        double result;
        if (vr_like) {
            if (simul) {
                if (p.metric == FWI_METRIC_VR) result = fmax(0.0, 1.0 - q[SPW] / q[2 * SPW]);
                else { const double sg = p.fc.sigma[norm ? 1 : 0]; result = exp(-q[SPW] / (2.0 * sg * sg)); }
            } else {
                result = q[0] / p.K;                                                   // FWI:682
                if (p.metric == FWI_METRIC_GAU && (p.flags & FWI_FLAG_STRICT_REF)) result = 0.0;   // quirk q1
            }
        } else if (!simul) {
            result = q[0] / p.K;
        } else {
            const int ni = norm ? 1 : 0;
            const double A1 = q[0], A2 = q[SPW], A3 = q[2 * SPW];
            const double nn = p.fc.n, D1 = p.fc.D1[ni], D2 = p.fc.D2[ni];
            const double cov = A3 - A1 * D1 / nn, vs = A2 - A1 * A1 / nn, vd = D2 - D1 * D1 / nn;
            const double pcc = cov / sqrt(vs * vd);
            result = (pcc < 0.0) ? 0.0 : pcc;
        }
        p.sim[n] = (float)result;
        if (p.like) p.like[n] = (float)exp(-(1.0 - result) * 0.5);                   // FWI:774
    }
}

// --------------------------------------------------------------------------------------------- Gram-matrix mode
// For the un-normalised metrics the misfit of a sample is a quadratic form in M (SURVEY 7 "algebraic shortcut"):
//   sum_t s^2 = M^T A_k M,  sum_t d s = b_k^T M,  mean_t s = gbar_k^T M     with A_k = G_k G_k^T (C x C) per trace,
// so a sample costs O(K C^2) instead of O(K C T) flops.  It is a DIFFERENT ALGORITHM from the reference's
// (no synthetic trace is ever formed, so per-trace max-abs normalisation is impossible) and is reported as its
// own mode.  float64 throughout: the forms cancel (SSE = dd - 2 b.M + M.A.M), and 2 K C^2 ~ 3.4 kflop per sample is
// cheap even on the fp64 pipe.  Per trace: [A raw (C(C+1)/2), b raw (C), A centred, b centred, gbar (C)] doubles.
template <int C>
__global__ void __launch_bounds__(128) mc_gram_kernel(const double* __restrict__ gram, EvalParams p) {
    constexpr int NS = C * (C + 1) / 2;
    constexpr int PT = 2 * NS + 3 * C;
    extern __shared__ double sg[];
    for (int i = threadIdx.x; i < p.K * PT; i += blockDim.x) sg[i] = gram[i];
    __syncthreads();
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= p.N) return;
    double m[C];
#pragma unroll
    for (int c = 0; c < C; ++c) m[c] = (double)__ldg(p.M + (int64_t)c * p.ldm + n);
    const bool simul = p.flags & FWI_FLAG_SIMULTANEOUS;
    const bool pcc_like = !(p.metric == FWI_METRIC_VR || p.metric == FWI_METRIC_GAU);
    const double Tn = (double)p.Tv;
    double acc = 0.0, tot_sse = 0.0, tot_dd = 0.0, A1 = 0.0, A2 = 0.0, A3 = 0.0;
    for (int k = 0; k < p.K; ++k) {
        const double* g = sg + (size_t)k * PT + (pcc_like ? NS + C : 0);
        double quad = 0.0, lin = 0.0;
        int e = 0;
#pragma unroll
        for (int i = 0; i < C; ++i) {
            double row = 0.5 * g[e++] * m[i];                    // diagonal once, off-diagonals twice
#pragma unroll
            for (int j = i + 1; j < C; ++j) row = fma(g[e++], m[j], row);
            quad = fma(2.0 * m[i], row, quad);
        }
#pragma unroll
        for (int c = 0; c < C; ++c) lin = fma(g[NS + c], m[c], lin);
        const TraceConst tc = p.tc[k];
        if (!pcc_like) {
            const double sse = fmax(0.0, tc.sumd2 - 2.0 * lin + quad);
            tot_sse += sse;
            tot_dd += tc.sumd2;
            if (p.metric == FWI_METRIC_VR) acc += fmax(0.0, 1.0 - sse / tc.sumd2);
            else acc += exp(-sse / (2.0 * tc.sigma * tc.sigma));
        } else {
            double mu = 0.0;
            const double* gb = sg + (size_t)k * PT + 2 * NS + 2 * C;
#pragma unroll
            for (int c = 0; c < C; ++c) mu = fma(gb[c], m[c], mu);
            const double pcc = lin / sqrt(quad * tc.ssd);
            acc += (pcc < 0.0) ? 0.0 : pcc;
            A1 += Tn * mu;
            A2 += quad + Tn * mu * mu;
            A3 += lin + Tn * tc.mean_d * mu;
        }
    }
    double result;
    if (!pcc_like) {
        if (simul) result = (p.metric == FWI_METRIC_VR) ? fmax(0.0, 1.0 - tot_sse / tot_dd) : exp(-tot_sse / (2.0 * p.fc.sigma[0] * p.fc.sigma[0]));
        else { result = acc / p.K; if (p.metric == FWI_METRIC_GAU && (p.flags & FWI_FLAG_STRICT_REF)) result = 0.0; }
    } else if (!simul) {
        result = acc / p.K;
    } else {
        const double nn = p.fc.n, D1 = p.fc.D1[0], D2 = p.fc.D2[0];
        const double pcc = (A3 - A1 * D1 / nn) / sqrt((A2 - A1 * A1 / nn) * (D2 - D1 * D1 / nn));
        result = (pcc < 0.0) ? 0.0 : pcc;
    }
    p.sim[n] = (float)result;
    if (p.like) p.like[n] = (float)exp(-(1.0 - result) * 0.5);
}

// --------------------------------------------------------------------------------------------- forward traces
template <int C, int NM>
__global__ void mc_forward_kernel(const float* __restrict__ rows, const int* __restrict__ phase,
                                  const float* __restrict__ M, int64_t ldm, int n_comp,
                                  const float* __restrict__ frac, int nfrac, int64_t N, int K, int T,
                                  float* __restrict__ out) {
    constexpr int CC = C * NM;
    constexpr int RW = row_width(CC);
    const int64_t kt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (kt >= (int64_t)K * T) return;
    const int k = (int)(kt / T);
    float r[RW];
    const float4* rp = reinterpret_cast<const float4*>(rows) + kt * (RW / 4);
#pragma unroll
    for (int q = 0; q < RW / 4; ++q) {
        float4 v = __ldg(rp + q);
        r[4 * q] = v.x; r[4 * q + 1] = v.y; r[4 * q + 2] = v.z; r[4 * q + 3] = v.w;
    }
    const int ph = (NM == 2 && nfrac == 3 && phase) ? phase[k] : 0;
    for (int64_t n = blockIdx.y; n < N; n += gridDim.y) {
        float f = 0.f;
        if (NM == 2 && frac) f = __ldg(frac + (int64_t)ph * ldm + n);
        float v = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            if (c < n_comp) {                                                          // FWI:262
                const float mc = __ldg(M + (int64_t)c * ldm + n);
                if (NM == 1) v = fmaf(r[c], mc, v);
                else { v = fmaf(r[c], mc * (1.0f - f), v); v = fmaf(r[C + c], mc * f, v); }
            }
        }
        out[n * (int64_t)K * T + kt] = v;
    }
}

// --------------------------------------------------------------------------------------------- samplers
struct Philox {
    uint32_t c[4], k[2];
    __device__ __forceinline__ void round_() {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k[0], n2 = hi0 ^ c[3] ^ k[1];
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k[0] += 0x9E3779B9u; k[1] += 0xBB67AE85u;
    }
    __device__ __forceinline__ void run() {
#pragma unroll
        for (int i = 0; i < 10; ++i) round_();
    }
};

__device__ __forceinline__ void philox4(uint64_t seed, uint64_t index, uint32_t block, uint32_t out[4]) {
    Philox p;
    p.c[0] = (uint32_t)index; p.c[1] = (uint32_t)(index >> 32); p.c[2] = block; p.c[3] = 0x46574921u;
    p.k[0] = (uint32_t)seed; p.k[1] = (uint32_t)(seed >> 32);
    p.run();
    out[0] = p.c[0]; out[1] = p.c[1]; out[2] = p.c[2]; out[3] = p.c[3];
}
__device__ __forceinline__ float u01(uint32_t x) { return ((x >> 8) + 0.5f) * (1.0f / 16777216.0f); }   // (0,1)

__device__ __forceinline__ void unit3(const float* a, float* o) {
    const float inv = rsqrtf(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    // one Newton step on the reciprocal root keeps the norm within 1 ulp
    const float n2 = a[0] * a[0] + a[1] * a[1] + a[2] * a[2];
    const float r = inv * (1.5f - 0.5f * n2 * inv * inv);
    o[0] = a[0] * r; o[1] = a[1] * r; o[2] = a[2] * r;
}

// R = Rz(phi) Ry(theta) from cos/sin (FWI:228-229)
__device__ __forceinline__ void make_rot(float ct, float st, float cp, float sp, float R[3][3]) {
    R[0][0] = cp * ct; R[0][1] = -sp; R[0][2] = cp * st;
    R[1][0] = sp * ct; R[1][1] = cp;  R[1][2] = sp * st;
    R[2][0] = -st;     R[2][1] = 0.f; R[2][2] = ct;
}
// B = R A R^T for symmetric A, returned as the 6-vector of FWI:206-208
__device__ __forceinline__ void rot_sym6(const float R[3][3], const float A[3][3], float o[6]) {
    float RA[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) RA[i][j] = R[i][0] * A[0][j] + R[i][1] * A[1][j] + R[i][2] * A[2][j];
    float B[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) B[i][j] = RA[i][0] * R[j][0] + RA[i][1] * R[j][1] + RA[i][2] * R[j][2];
    const float sq2 = 1.41421356237309515f;
    o[0] = B[0][0]; o[1] = B[1][1]; o[2] = B[2][2]; o[3] = sq2 * B[0][1]; o[4] = sq2 * B[0][2]; o[5] = sq2 * B[1][2];
}
__device__ __forceinline__ void unit6(float* v) {
    float n2 = 0.f;
#pragma unroll
    for (int i = 0; i < 6; ++i) n2 = fmaf(v[i], v[i], n2);
    const float r = 1.0f / sqrtf(n2);
#pragma unroll
    for (int i = 0; i < 6; ++i) v[i] *= r;
}
// theta = atan2(sqrt(x^2+y^2), z), phi = atan2(y, x) of a unit vector (FWI:308-309): only the
// cosines and sines are ever used, and those are algebraic in (x,y,z).
__device__ __forceinline__ void rot_from_vec_atan2(const float* a, float R[3][3]) {
    float u[3];
    unit3(a, u);
    const float rho = sqrtf(u[0] * u[0] + u[1] * u[1]);
    make_rot(u[2], rho, u[0] / rho, u[1] / rho, R);
}
// theta = arccos(z), phi = arccos(x / sin(theta)) (FWI:497-498): phi in [0, pi] so sin(phi) >= 0.
__device__ __forceinline__ void rot_from_vec_acos(const float* a, float R[3][3]) {
    float u[3];
    unit3(a, u);
    const float rho = sqrtf(u[0] * u[0] + u[1] * u[1]);
    make_rot(u[2], rho, u[0] / rho, fabsf(u[1]) / rho, R);
}
// crack tensor on the lune perimeter (FWI:395-423): diag entries
__device__ __forceinline__ void crack_diag(float u, float r1, float r2, float dg[3]) {
    const float a = (r1 <= 0.5f) ? 0.f : 0.866025403784438597f;   // sin(phi_lune): 0 or sin(pi/3)
    const float b = sinpif(0.5f * u);                             // sin(theta_lune)
    const float h = 1.0f / sqrtf(a * a + b * b);
    float ca = fabsf(b) * h, sa = copysignf(a, b) * h;            // alpha = arctan(a/b)
    if (r2 > 0.25f && r2 <= 0.5f) { ca = -ca; sa = -sa; }                         // + pi
    else if (r2 > 0.5f && r2 <= 0.75f) { const float t = ca; ca = -sa; sa = t; }  // + pi/2
    else if (r2 > 0.75f && r2 <= 1.0f) { const float t = ca; ca = sa; sa = -t; }  // + 3pi/2
    const float sq2 = 1.41421356237309515f;
    const float sc = 1.0f / (sqrtf(4.f * sa * sa + ca * ca) * 1.73205080756887729f);
    dg[0] = sc * (ca - sq2 * sa); dg[1] = dg[0]; dg[2] = sc * (ca + 2.f * sq2 * sa);
}

// raw draws (reference consumption order) -> tensor rows; returns amp-frac (or -1)
__device__ float transform_draws(int type, const float* q, float amp, float* out) {
    const float DC0[3][3] = {{0.f, 0.f, 1.f}, {0.f, 0.f, 0.f}, {1.f, 0.f, 0.f}};   // FWI:299
    float R[3][3];
    float frac = -1.f;
    switch (type) {
        case FWI_TYPE_FULL_MT: {
#pragma unroll
            for (int i = 0; i < 6; ++i) out[i] = q[i];
            unit6(out);
        } break;
        case FWI_TYPE_SINGLE_FORCE: unit3(q, out); break;
        case FWI_TYPE_DC: {
            rot_from_vec_atan2(q, R);
            rot_sym6(R, DC0, out);
            unit6(out);
        } break;
        case FWI_TYPE_DC_SF_COUPLE: {
            rot_from_vec_atan2(q, R);
            rot_sym6(R, DC0, out);
            unit6(out);
            frac = q[3];
#pragma unroll
            for (int i = 0; i < 6; ++i) out[i] *= frac;
            // force = R [1,0,0] = first column of R, NED -> END swaps the first two (FWI:359)
            out[6] = R[1][0] * (1.f - frac); out[7] = R[0][0] * (1.f - frac); out[8] = R[2][0] * (1.f - frac);
        } break;
        case FWI_TYPE_DC_SF_NO_COUPLING: {
            rot_from_vec_atan2(q, R);
            rot_sym6(R, DC0, out);
            unit6(out);
            frac = q[6];
#pragma unroll
            for (int i = 0; i < 6; ++i) out[i] *= frac;
            unit3(q + 3, out + 6);
            out[6] *= (1.f - frac); out[7] *= (1.f - frac); out[8] *= (1.f - frac);
        } break;
        case FWI_TYPE_DC_CRACK_COUPLE: {
            float dg[3];
            crack_diag(q[0], q[1], q[2], dg);
            frac = q[3];
            float A[3][3] = {{(1.f - frac) * dg[0], 0.f, frac}, {0.f, (1.f - frac) * dg[1], 0.f}, {frac, 0.f, (1.f - frac) * dg[2]}};
            rot_from_vec_atan2(q + 4, R);
            rot_sym6(R, A, out);
            unit6(out);
        } break;
        case FWI_TYPE_SF_CRACK_NO_COUPLING: {
            float sf[3];
            unit3(q, sf);
            float dg[3];
            crack_diag(q[3], q[4], q[5], dg);
            const float A[3][3] = {{dg[0], 0.f, 0.f}, {0.f, dg[1], 0.f}, {0.f, 0.f, dg[2]}};
            rot_from_vec_acos(q + 6, R);
            rot_sym6(R, A, out);                      // not re-normalised (FWI:501-503)
            frac = q[9];                              // fraction of the force (FWI:505-507)
#pragma unroll
            for (int i = 0; i < 6; ++i) out[i] *= (1.f - frac);
            out[6] = sf[0] * frac; out[7] = sf[1] * frac; out[8] = sf[2] * frac;
        } break;
    }
    const int nc = (type == FWI_TYPE_SINGLE_FORCE) ? 3 : ((type == FWI_TYPE_FULL_MT || type == FWI_TYPE_DC || type == FWI_TYPE_DC_CRACK_COUPLE) ? 6 : 9);
    for (int i = 0; i < nc; ++i) out[i] *= amp;
    return frac;
}

__host__ __device__ inline int type_components(int t) {
    return (t == FWI_TYPE_SINGLE_FORCE) ? 3 : ((t == FWI_TYPE_FULL_MT || t == FWI_TYPE_DC || t == FWI_TYPE_DC_CRACK_COUPLE) ? 6 : 9);
}
__host__ __device__ inline int type_draws(int t) {
    const int nd[7] = {6, 3, 3, 4, 7, 7, 10};
    return nd[t];
}
__host__ __device__ inline bool type_combined(int t) { return t >= FWI_TYPE_DC_SF_COUPLE; }

__global__ void mc_transform_kernel(int type, const float* __restrict__ draws, int64_t ldn, int64_t N, float amp,
                                    float* __restrict__ out, int64_t ldo) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float q[10], o[9];
    const int nd = type_draws(type);
    for (int j = 0; j < nd; ++j) q[j] = draws[(int64_t)j * ldn + n];
    const float frac = transform_draws(type, q, amp, o);
    const int nc = type_components(type);
    for (int c = 0; c < nc; ++c) out[(int64_t)c * ldo + n] = o[c];
    if (type_combined(type)) out[(int64_t)nc * ldo + n] = frac;
}

// draw pattern per type: 'n' normal, 'u' U(-1,1), 'r' U[0,1)   (oracle/mc_oracle.py DRAW_PATTERN)
__device__ __constant__ char c_patterns[7][11] = {"nnnnnn", "nnn", "nnn", "nnnr", "nnnnnnr", "urrrnnn", "nnnurrnnnr"};

__global__ void mc_sample_kernel(int type, uint64_t seed, int64_t first, int64_t N, float amp, int nfrac,
                                 float* __restrict__ out, int64_t ldo) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const uint64_t gidx = (uint64_t)(first + n);
    uint32_t w[16];
    philox4(seed, gidx, 0, w);
    philox4(seed, gidx, 1, w + 4);
    philox4(seed, gidx, 2, w + 8);
    philox4(seed, gidx, 3, w + 12);
    // six normals from three Box-Muller pairs, then four uniforms, then three media fractions
    float nrm[6];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const float r = sqrtf(-2.f * logf(u01(w[2 * j])));
        float s, c;
        sincospif(2.f * u01(w[2 * j + 1]), &s, &c);
        nrm[2 * j] = r * c; nrm[2 * j + 1] = r * s;
    }
    float q[10], o[9];
    int in = 0, iu = 6;
    const int nd = type_draws(type);
    for (int j = 0; j < nd; ++j) {
        const char ch = c_patterns[type][j];
        if (ch == 'n') q[j] = nrm[in++];
        else if (ch == 'u') q[j] = 2.f * u01(w[iu++]) - 1.f;
        else q[j] = u01(w[iu++]);
    }
    const float frac = transform_draws(type, q, amp, o);
    const int nc = type_components(type);
    for (int c = 0; c < nc; ++c) out[(int64_t)c * ldo + n] = o[c];
    int row = nc;
    if (type_combined(type)) out[(int64_t)(row++) * ldo + n] = frac;
    for (int j = 0; j < nfrac; ++j) out[(int64_t)(row++) * ldo + n] = u01(w[10 + j]);     // FWI:719-721, FWI:730
}

// --------------------------------------------------------------------------------------------- reductions
__global__ void mc_reduce_kernel(const float* __restrict__ L, int64_t N, double* __restrict__ psum,
                                 float* __restrict__ pmax, long long* __restrict__ parg) {
    __shared__ double ssum[32];
    __shared__ float smax[32];
    __shared__ long long sarg[32];
    double s = 0.0;
    float mx = -INFINITY;
    long long am = -1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const float v = L[i];
        s += (double)v;
        if (v > mx) { mx = v; am = i; }
    }
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        const float omx = __shfl_xor_sync(0xffffffffu, mx, o);
        const long long oam = __shfl_xor_sync(0xffffffffu, am, o);
        if (omx > mx || (omx == mx && oam >= 0 && (am < 0 || oam < am))) { mx = omx; am = oam; }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { ssum[warp] = s; smax[warp] = mx; sarg[warp] = am; }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int nw = blockDim.x >> 5;
        for (int w = 1; w < nw; ++w) {
            s += ssum[w];
            if (smax[w] > mx || (smax[w] == mx && sarg[w] >= 0 && (am < 0 || sarg[w] < am))) { mx = smax[w]; am = sarg[w]; }
        }
        psum[blockIdx.x] = s; pmax[blockIdx.x] = mx; parg[blockIdx.x] = am;
    }
}

__global__ void mc_normalise_kernel(const float* __restrict__ L, int64_t N, double scale, float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) out[i] = (float)((double)L[i] * scale);
}


// --------------------------------------------------------------------------------------------- input preparation (f2)
// Green's-function conditioning of load_input_data / get_overall_real_and_green_func_data (FWI:92-111, FWI:178-196):
// integer time shift (np.roll along t) with the wrapped head zeroed, optional per-trace phase-window cut, unit
// scaling.  float64 in, float64 out, the two scale factors applied one after the other exactly like the
// reference's `*(10**3)` then `*(10**7)`, so the result is bit-identical to NumPy's.
__global__ void mc_prepare_kernel(const double* __restrict__ raw, int K, int C, int T, int NM, const int* __restrict__ shift,
                                  int zero_head, const int* __restrict__ cut_start, int Tout, double scale1, double scale2,
                                  double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t total = (int64_t)K * C * Tout * NM;
    if (i >= total) return;
    const int med = (int)(i % NM);
    const int64_t j = i / NM;
    const int t_out = (int)(j % Tout);
    const int c = (int)((j / Tout) % C);
    const int k = (int)(j / ((int64_t)Tout * C));
    const int t = t_out + (cut_start ? cut_start[k] : 0);          // index in the shifted, uncut trace (FWI:108-109)
    double v = 0.0;
    if (t >= 0 && t < T) {
        const int sh = shift ? shift[k] : 0;
        if (sh == INT_MIN) v = 0.0;                                 // fewer shifts than traces: FWI:95-96 fills only the given ones
        else {
            int src = (t - sh) % T;                                 // np.roll(x, sh)[t] = x[(t - sh) mod T]   (FWI:97)
            if (src < 0) src += T;
            v = raw[(((int64_t)k * C + c) * T + src) * NM + med];
            // FWI:98-99 zeroes the slice [0:sh]; for a negative shift that slice is everything but the last |sh| samples
            if (shift && zero_head && t < (sh >= 0 ? sh : max(0, T + sh))) v = 0.0;
        }
    }
    if (scale1 != 1.0) v *= scale1;
    if (scale2 != 1.0) v *= scale2;
    out[i] = v;
}


// --------------------------------------------------------------------------------------------- posterior reductions (f4)
// The consumer's per-sample Python loops (plot_full_waveform_inversion.py, cited PLOT:<line>) as histogram kernels.
// float64 throughout so that bin assignment matches NumPy's; block-private shared histograms, one flush per block.
__device__ __forceinline__ int nearest_label(double v, double first, double step, int n) {
    // index of the label closest to v in arange(first, ..., step) (find_nearest, PLOT:84-86; ties -> lower index)
    if (!(v == v)) return 0;                                   // NaN: argmin of all-NaN is 0
    double q = (v - first) / step;
    int i = (int)floor(q + 0.5);
    if (q + 0.5 == (double)i && i > 0) {                        // exact tie: argmin keeps the first (lower) label
        const double dl = fabs(first + (i - 1) * step - v), dh = fabs(first + i * step - v);
        if (dl <= dh) i -= 1;
    }
    return min(max(i, 0), n - 1);
}

// mode 0: theta-phi 5-degree histogram of force vectors weighted by MTp (PLOT:522-555, single_force branch)
// mode 1: percentage histograms of the amp-frac row, f and 1-f, 101 one-percent bins (PLOT:943-960)
// mode 2: lune delta-gamma counts of 6-vectors from the eigenvalues of the 3x3 tensor (PLOT:1011-1059)
__global__ void mc_hist_kernel(int mode, const float* __restrict__ MTs, int64_t ldn, const float* __restrict__ MTp,
                               const long long* __restrict__ idx, int64_t n, int row0, double* __restrict__ hist, int nbins) {
    extern __shared__ double sh[];
    for (int i = threadIdx.x; i < nbins; i += blockDim.x) sh[i] = 0.0;
    __syncthreads();
    const double PI = 3.14159265358979323846;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = idx ? idx[t] : t;
        if (mode == 0) {
            // x, y, z in NED from the (E, N, D)-ordered force: x = F[1], y = F[0], z = -F[2]  (PLOT:528-530)
            const double x = MTs[(int64_t)(row0 + 1) * ldn + j], y = MTs[(int64_t)row0 * ldn + j], z = -(double)MTs[(int64_t)(row0 + 2) * ldn + j];
            const double r = sqrt(x * x + y * y + z * z);
            const double theta = acos(z / r);                                   // PLOT:478
            double phi;
            if (y == 0.0) phi = (x >= 0.0) ? 0.0 : PI;                          // PLOT:480-484
            else {
                const double a = acos(x / (r * sin(theta)));
                phi = (y > 0.0) ? a : 2.0 * PI - a;                             // PLOT:485-488
            }
            const int it = nearest_label(theta, PI / 360.0, 5.0 * PI / 180.0, 36);     // PLOT:524
            const int ip = nearest_label(phi, PI / 720.0, 5.0 * PI / 180.0, 72);       // PLOT:525
            atomicAdd(&sh[it * 72 + ip], (double)MTp[j]);
        } else if (mode == 1) {
            const double p = MTp[j];
            if (p != 0.0) {                                                     // PLOT:951
                const double f = MTs[(int64_t)row0 * ldn + j];
                atomicAdd(&sh[nearest_label(f * 100.0, 0.0, 1.0, 101)], p);                // PLOT:957-958
                atomicAdd(&sh[101 + nearest_label((1.0 - f) * 100.0, 0.0, 1.0, 101)], p);  // PLOT:960-961
            }
        } else {
            double m[6];
            for (int c = 0; c < 6; ++c) m[c] = MTs[(int64_t)(row0 + c) * ldn + j];
            const double s2 = 0.70710678118654752440;
            const double a11 = m[0], a22 = m[1], a33 = m[2], a12 = m[3] * s2, a13 = m[4] * s2, a23 = m[5] * s2;   // PLOT:93-97
            // eigenvalues of a symmetric 3x3 (trigonometric form), l1 >= l2 >= l3
            const double q = (a11 + a22 + a33) / 3.0;
            const double p1 = a12 * a12 + a13 * a13 + a23 * a23;
            const double p2 = (a11 - q) * (a11 - q) + (a22 - q) * (a22 - q) + (a33 - q) * (a33 - q) + 2.0 * p1;
            double l1, l2, l3;
            if (p2 <= 0.0) { l1 = l2 = l3 = q; }
            else {
                const double pp = sqrt(p2 / 6.0);
                const double b11 = (a11 - q) / pp, b22 = (a22 - q) / pp, b33 = (a33 - q) / pp, b12 = a12 / pp, b13 = a13 / pp, b23 = a23 / pp;
                double rr = 0.5 * (b11 * (b22 * b33 - b23 * b23) - b12 * (b12 * b33 - b23 * b13) + b13 * (b12 * b23 - b22 * b13));
                rr = fmin(1.0, fmax(-1.0, rr));
                const double ph = acos(rr) / 3.0;
                l1 = q + 2.0 * pp * cos(ph);
                l3 = q + 2.0 * pp * cos(ph + 2.0 * PI / 3.0);
                l2 = 3.0 * q - l1 - l3;
            }
            const double gamma = atan((-l1 + 2.0 * l2 - l3) / (sqrt(3.0) * (l1 - l3)));                       // PLOT:1026
            const double beta = acos((l1 + l2 + l3) / (sqrt(3.0) * sqrt(l1 * l1 + l2 * l2 + l3 * l3)));        // PLOT:1027
            const double delta = PI / 2.0 - beta;                                                              // PLOT:1028
            const double bs = PI / 120.0;
            const int id = nearest_label(delta, -PI / 2.0, bs, 122), ig = nearest_label(gamma, -PI / 6.0, bs, 41);   // PLOT:1041-1042, 1056-1057
            atomicAdd(&sh[id * 41 + ig], 1.0);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nbins; i += blockDim.x) if (sh[i] != 0.0) atomicAdd(&hist[i], sh[i]);
}


// --------------------------------------------------------------------------------------------- least squares (a15)
// perform_inversion (FWI:242-250): min || A m - d ||, A = stacked (K*T) x C Green's functions.  Normal equations in
// float64: one pass accumulates A^T A (upper triangle) and A^T d, a single thread then solves the C x C system by
// Cholesky.  C <= 9 and the Green's functions are far from rank deficient, so this agrees with LAPACK's gelsd to
// ~1e-12; a non-positive pivot (rank-deficient input) is reported instead of returning garbage.
template <int C>
__global__ void mc_normal_eq_kernel(const double* __restrict__ G, const double* __restrict__ d, int K, int T, double* __restrict__ acc) {
    constexpr int NS = C * (C + 1) / 2;
    double a[NS + C];
#pragma unroll
    for (int i = 0; i < NS + C; ++i) a[i] = 0.0;
    const int64_t rows = (int64_t)K * T;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(r / T), t = (int)(r % T);
        double g[C];
#pragma unroll
        for (int c = 0; c < C; ++c) g[c] = G[((int64_t)k * C + c) * T + t];
        const double dv = d[r];
        int e = 0;
#pragma unroll
        for (int i = 0; i < C; ++i)
#pragma unroll
            for (int j = i; j < C; ++j) a[e++] += g[i] * g[j];
#pragma unroll
        for (int c = 0; c < C; ++c) a[NS + c] += g[c] * dv;
    }
#pragma unroll
    for (int i = 0; i < NS + C; ++i) {
        double v = a[i];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) atomicAdd(acc + i, v);
    }
}

template <int C>
__global__ void mc_cholesky_kernel(const double* __restrict__ acc, double* __restrict__ m_out, int* __restrict__ status) {
    constexpr int NS = C * (C + 1) / 2;
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double A[C][C], b[C];
    int e = 0;
    for (int i = 0; i < C; ++i)
        for (int j = i; j < C; ++j) { A[i][j] = acc[e]; A[j][i] = acc[e]; ++e; }
    for (int c = 0; c < C; ++c) b[c] = acc[NS + c];
    *status = 0;
    for (int j = 0; j < C; ++j) {                       // A = L L^T, L stored in the lower triangle
        double s = A[j][j];
        for (int k = 0; k < j; ++k) s -= A[j][k] * A[j][k];
        if (!(s > 0.0)) { *status = 1; return; }
        const double l = sqrt(s);
        A[j][j] = l;
        for (int i = j + 1; i < C; ++i) {
            double t = A[i][j];
            for (int k = 0; k < j; ++k) t -= A[i][k] * A[j][k];
            A[i][j] = t / l;
        }
    }
    for (int i = 0; i < C; ++i) {                       // L y = b
        double t = b[i];
        for (int k = 0; k < i; ++k) t -= A[i][k] * b[k];
        b[i] = t / A[i][i];
    }
    for (int i = C - 1; i >= 0; --i) {                  // L^T m = y
        double t = b[i];
        for (int k = i + 1; k < C; ++k) t -= A[k][i] * b[k];
        b[i] = t / A[i][i];
    }
    for (int c = 0; c < C; ++c) m_out[c] = b[c];
}

// --------------------------------------------------------------------------------------------- FP32 peak probe
// SURVEY 8(d): the Monte-Carlo path is bound by FP32 FMA throughput, which MEASURED_PEAKS.json does not hold.  Eight
// independent FMA chains per thread, no memory traffic; the result is stored so the chains cannot be removed.
__global__ void __launch_bounds__(256) fp32_fma_probe_kernel(float* out, int iters, float seed) {
    float a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = seed + (float)(threadIdx.x + i);
    const float b = 1.0000001f, c = 1e-7f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = fmaf(a[i], b, c);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += a[i];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace fwi

// =============================================================================================== host side
using namespace fwi;

struct RowSet {
    float* rows = nullptr;
    float* gbar = nullptr;
    TraceConst* tc = nullptr;
    FlatConst fc{};
    int Tv = 0;
    bool built = false;
    double* gram = nullptr;     // per-trace Gram blocks for the Gram mode (built with the row set, n_media == 1 only)
};

struct fwi_mc_ctx {
    int device = 0, K = 0, C = 0, T = 0, NM = 1, CC = 0, RW = 0;
    std::vector<double> G, d;     // host copies (reference layout) for the lazily built CC-shift rows
    std::vector<int> phase;
    int* phase_dev = nullptr;
    RowSet base, hr, hrflat;
    // scratch
    float* stage_M = nullptr; float* stage_sim = nullptr; float* stage_frac = nullptr; int64_t stage_cap = 0;
    double* dstage = nullptr; int64_t dstage_bytes = 0;
    int sm_count = 148;
    bool uploaded = false;
    UmmaPath* umma = nullptr;     // tensor-core evaluation path (mc_umma.cu), built at upload when the shapes allow it
};

static void free_rowset(RowSet& r) {
    if (r.rows) cudaFree(r.rows);
    if (r.gbar) cudaFree(r.gbar);
    if (r.tc) cudaFree(r.tc);
    if (r.gram) cudaFree(r.gram);
    r = RowSet{};
}

// data(k, t) accessors on the host copies
static inline double G_at(const fwi_mc_ctx* c, int k, int comp, int t, int med) {
    return c->G[(((size_t)k * c->C + comp) * c->T + t) * c->NM + med];
}

// Build one prepared row set.  variant 0: base (Tv = T); 1: 4x linear interpolation clamped per trace
// (np.interp on each trace, FWI:554-555); 2: 4x interpolation of the flattened array (runs into the
// next trace's first sample; only the very last trace clamps).
static int build_rowset(fwi_mc_ctx* c, RowSet& rs, int variant) {
    const int K = c->K, C = c->C, T = c->T, NM = c->NM, CC = c->CC, RW = c->RW;
    const int Tv = (variant == 0) ? T : 4 * T;
    std::vector<float> rows((size_t)K * Tv * RW, 0.f);
    std::vector<float> gbar((size_t)K * CC, 0.f);
    std::vector<TraceConst> tc(K);
    std::vector<double> dv((size_t)K * Tv);
    auto interp = [&](auto&& val, int k, int tv) -> double {   // val(k, t) on the original grid
        if (variant == 0) return val(k, tv);
        const int i = tv >> 2, j = tv & 3;
        const double a = val(k, i);
        if (j == 0) return a;
        double b;
        if (i + 1 < T) b = val(k, i + 1);
        else if (variant == 2 && k + 1 < K) b = val(k + 1, 0);
        else return a;                                          // right edge clamps
        return a + (b - a) * (0.25 * j);
    };
    for (int k = 0; k < K; ++k) {
        auto dval = [&](int kk, int t) { return c->d[(size_t)kk * T + t]; };
        double sum = 0.0, sum2 = 0.0;
        for (int tv = 0; tv < Tv; ++tv) {
            const double x = interp(dval, k, tv);
            dv[(size_t)k * Tv + tv] = x;
            sum += x; sum2 += x * x;
        }
        TraceConst& q = tc[k];
        q.mean_d = sum / Tv;
        q.sumd2 = sum2;
        double ssd = 0.0, mx = 0.0;
        for (int tv = 0; tv < Tv; ++tv) { const double e = dv[(size_t)k * Tv + tv] - q.mean_d; ssd += e * e; }
        for (int t = 0; t < T; ++t) mx = std::max(mx, std::fabs(c->d[(size_t)k * T + t]));
        q.ssd = ssd; q.maxd = mx;
        q.sigma = NAN;
        if (Tv >= 60) { double s = 0.0; for (int tv = Tv - 60; tv < Tv - 10; ++tv) s += std::fabs(dv[(size_t)k * Tv + tv]); q.sigma = s / 50.0; }
        q.d_first = dv[(size_t)k * Tv]; q.d_last = dv[(size_t)k * Tv + Tv - 1];
        for (int med = 0; med < NM; ++med)
            for (int comp = 0; comp < C; ++comp) {
                auto gval = [&](int kk, int t) { return G_at(c, kk, comp, t, med); };
                double gs = 0.0;
                for (int tv = 0; tv < Tv; ++tv) {
                    const double x = interp(gval, k, tv);
                    rows[((size_t)k * Tv + tv) * RW + med * C + comp] = (float)x;
                    gs += (double)(float)x;
                }
                gbar[(size_t)k * CC + med * C + comp] = (float)(gs / Tv);
            }
        for (int tv = 0; tv < Tv; ++tv) {
            rows[((size_t)k * Tv + tv) * RW + CC] = (float)dv[(size_t)k * Tv + tv];
            rows[((size_t)k * Tv + tv) * RW + CC + 1] = (float)(dv[(size_t)k * Tv + tv] - q.mean_d);
        }
    }
    // Gram blocks (float64, from the float64 Green's functions of this variant): A raw, b raw, A centred, b centred, gbar
    std::vector<double> gram;
    if (NM == 1) {
        const int NS = C * (C + 1) / 2, PT = 2 * NS + 3 * C;
        gram.assign((size_t)K * PT, 0.0);
        std::vector<double> gv((size_t)C * Tv);
        for (int k = 0; k < K; ++k) {
            for (int comp = 0; comp < C; ++comp) {
                auto gval = [&](int kk, int t) { return G_at(c, kk, comp, t, 0); };
                for (int tv = 0; tv < Tv; ++tv) gv[(size_t)comp * Tv + tv] = interp(gval, k, tv);
            }
            double* g = gram.data() + (size_t)k * PT;
            std::vector<double> gb(C, 0.0);
            for (int comp = 0; comp < C; ++comp) { double s_ = 0.0; for (int tv = 0; tv < Tv; ++tv) s_ += gv[(size_t)comp * Tv + tv]; gb[comp] = s_ / Tv; }
            int e = 0;
            for (int i = 0; i < C; ++i)
                for (int j = i; j < C; ++j) {
                    double raw = 0.0, cen = 0.0;
                    for (int tv = 0; tv < Tv; ++tv) {
                        const double a_ = gv[(size_t)i * Tv + tv], b_ = gv[(size_t)j * Tv + tv];
                        raw += a_ * b_;
                        cen += (a_ - gb[i]) * (b_ - gb[j]);
                    }
                    g[e] = raw; g[NS + C + e] = cen; ++e;
                }
            for (int comp = 0; comp < C; ++comp) {
                double raw = 0.0, cen = 0.0;
                for (int tv = 0; tv < Tv; ++tv) {
                    const double dd_ = dv[(size_t)k * Tv + tv], gg_ = gv[(size_t)comp * Tv + tv];
                    raw += dd_ * gg_;
                    cen += (dd_ - tc[k].mean_d) * (gg_ - gb[comp]);
                }
                g[NS + comp] = raw; g[2 * NS + C + comp] = cen; g[2 * NS + 2 * C + comp] = gb[comp];
            }
        }
    }
    // flattened constants (raw and normalised)
    FlatConst fc{};
    fc.n = (double)K * Tv;
    for (int norm = 0; norm < 2; ++norm) {
        // the normalised flattened array is built from the normalised ORIGINAL traces and then (for the
        // CC-shift variants) interpolated, exactly as FWI:598 followed by FWI:554 does.
        std::vector<double> flat((size_t)K * Tv);
        for (int k = 0; k < K; ++k) {
            auto dn = [&](int kk, int t) { return c->d[(size_t)kk * T + t] / (norm ? tc[kk].maxd : 1.0); };
            for (int tv = 0; tv < Tv; ++tv) flat[(size_t)k * Tv + tv] = interp(dn, k, tv);
        }
        double s1 = 0.0, s2 = 0.0;
        for (double x : flat) { s1 += x; s2 += x * x; }
        fc.D1[norm] = s1; fc.D2[norm] = s2;
        fc.sigma[norm] = NAN;
        if (flat.size() >= 60) { double s = 0.0; for (size_t i = flat.size() - 60; i < flat.size() - 10; ++i) s += std::fabs(flat[i]); fc.sigma[norm] = s / 50.0; }
    }
    FWI_CUDA(cudaMalloc(&rs.rows, rows.size() * sizeof(float)));
    FWI_CUDA(cudaMalloc(&rs.gbar, gbar.size() * sizeof(float)));
    FWI_CUDA(cudaMalloc(&rs.tc, tc.size() * sizeof(TraceConst)));
    FWI_CUDA(cudaMemcpy(rs.rows, rows.data(), rows.size() * sizeof(float), cudaMemcpyHostToDevice));
    FWI_CUDA(cudaMemcpy(rs.gbar, gbar.data(), gbar.size() * sizeof(float), cudaMemcpyHostToDevice));
    FWI_CUDA(cudaMemcpy(rs.tc, tc.data(), tc.size() * sizeof(TraceConst), cudaMemcpyHostToDevice));
    if (!gram.empty()) {
        FWI_CUDA(cudaMalloc(&rs.gram, gram.size() * sizeof(double)));
        FWI_CUDA(cudaMemcpy(rs.gram, gram.data(), gram.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    rs.fc = fc; rs.Tv = Tv; rs.built = true;
    return FWI_OK;
}

template <int C, int NM, int S, int MODE>
static int launch_eval_t(const EvalParams& p, int nwarps, cudaStream_t st) {
    constexpr int SPW = 32 * S;
    const size_t smem = (size_t)nwarps * kMcAcc * SPW * sizeof(double);
    auto kern = mc_eval_kernel<C, NM, S, MODE>;
    if (smem > 48 * 1024) FWI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t blocks = ceil_div(p.N, (int64_t)SPW * (nwarps / p.ks));
    kern<<<(unsigned)blocks, nwarps * 32, smem, st>>>(p);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}
template <int C, int NM, int MODE>
static int launch_eval_s(const EvalParams& p, int S, int nwarps, cudaStream_t st) {
    // "wide" kernels for big batches: 8 samples per lane (4 for two media: the coefficient vector is twice as long).
    // Every warp-uniform row load (the load/store unit moves 128 B per float and warp whatever the address pattern)
    // then feeds twice the FMAs - the direct kernel is LSU-bound at 4 samples per lane.  168 registers, 128 threads.
    if (S == 8) return launch_eval_t<C, NM, (NM == 1 ? 8 : 4), MODE>(p, std::min(nwarps, 4), st);
    if (S == 4) return launch_eval_t<C, NM, (NM == 1 ? 4 : 2), MODE>(p, nwarps, st);
    if (S == 2) return launch_eval_t<C, NM, (NM == 1 ? 2 : 1), MODE>(p, nwarps, st);
    return launch_eval_t<C, NM, 1, MODE>(p, nwarps, st);
}
template <int C, int NM>
static int launch_eval_m(const EvalParams& p, int mode, int S, int nwarps, cudaStream_t st) {
    if (mode == MODE_SSE) return launch_eval_s<C, NM, MODE_SSE>(p, S, nwarps, st);
    if (mode == MODE_MOM) return launch_eval_s<C, NM, MODE_MOM>(p, S, nwarps, st);
    return launch_eval_s<C, NM, MODE_MOM_MAX>(p, S, nwarps, st);
}

static int pick_warps(int K) {
    // warps per CTA so that ceil(K/nw)*nw wastes the least; ties -> more warps
    int best = 4; double best_w = 1e9;
    for (int nw = 4; nw <= 8; ++nw) {
        const double waste = (double)(((K + nw - 1) / nw) * nw) / K;
        if (waste <= best_w + 1e-12) { best_w = waste; best = nw; }
    }
    return std::min(best, std::max(1, K));
}

extern "C" {

const char* fwi_last_error(void) { return g_err; }
int fwi_version(void) { return 100; }
int fwi_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int fwi_mc_type_components(int t) { return (t < 0 || t > 6) ? FWI_EINVAL : type_components(t); }
int fwi_mc_type_draws(int t) { return (t < 0 || t > 6) ? FWI_EINVAL : type_draws(t); }
int fwi_mc_type_rows(int t) { return (t < 0 || t > 6) ? FWI_EINVAL : type_components(t) + (type_combined(t) ? 1 : 0); }

int fwi_mc_create(int device, int K, int C, int T, int n_media, fwi_mc_ctx** out) {
    FWI_REQUIRE(out != nullptr, "fwi_mc_create: out is NULL");
    FWI_REQUIRE(K >= 1 && T >= 1, "fwi_mc_create: K and T must be >= 1 (got K=%d T=%d)", K, T);
    FWI_REQUIRE(C == 3 || C == 6 || C == 9, "fwi_mc_create: C must be 3, 6 or 9 (got %d)", C);
    FWI_REQUIRE(n_media == 1 || n_media == 2, "fwi_mc_create: n_media must be 1 or 2 (got %d)", n_media);
    int ndev = 0;
    FWI_CUDA(cudaGetDeviceCount(&ndev));
    FWI_REQUIRE(device >= 0 && device < ndev, "fwi_mc_create: device %d out of range (%d visible)", device, ndev);
    DeviceGuard g(device);
    auto* c = new fwi_mc_ctx();
    c->device = device; c->K = K; c->C = C; c->T = T; c->NM = n_media; c->CC = C * n_media; c->RW = row_width(c->CC);
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    *out = c;
    return FWI_OK;
}

int fwi_mc_destroy(fwi_mc_ctx* c) {
    if (!c) return FWI_OK;
    DeviceGuard g(c->device);
    umma_free(c->umma); c->umma = nullptr;
    free_rowset(c->base); free_rowset(c->hr); free_rowset(c->hrflat);
    if (c->phase_dev) cudaFree(c->phase_dev);
    if (c->stage_M) cudaFree(c->stage_M);
    if (c->stage_sim) cudaFree(c->stage_sim);
    if (c->stage_frac) cudaFree(c->stage_frac);
    if (c->dstage) cudaFree(c->dstage);
    delete c;
    return FWI_OK;
}

int fwi_mc_upload(fwi_mc_ctx* c, const double* G, const double* d, const int* phase) {
    FWI_REQUIRE(c && G && d, "fwi_mc_upload: NULL argument");
    DeviceGuard g(c->device);
    const size_t nG = (size_t)c->K * c->C * c->T * c->NM, nd = (size_t)c->K * c->T;
    c->G.assign(G, G + nG);
    c->d.assign(d, d + nd);
    free_rowset(c->base); free_rowset(c->hr); free_rowset(c->hrflat);
    if (c->phase_dev) { cudaFree(c->phase_dev); c->phase_dev = nullptr; }
    c->phase.clear();
    if (phase) {
        for (int k = 0; k < c->K; ++k) FWI_REQUIRE(phase[k] >= 0 && phase[k] <= 2, "fwi_mc_upload: phase_index[%d]=%d not in {0,1,2}", k, phase[k]);
        c->phase.assign(phase, phase + c->K);
        FWI_CUDA(cudaMalloc(&c->phase_dev, c->K * sizeof(int)));
        FWI_CUDA(cudaMemcpy(c->phase_dev, phase, c->K * sizeof(int), cudaMemcpyHostToDevice));
    }
    for (int k = 0; k < c->K; ++k) {
        double mx = 0.0;
        for (int t = 0; t < c->T; ++t) mx = std::max(mx, std::fabs(d[(size_t)k * c->T + t]));
        FWI_REQUIRE(std::isfinite(mx), "fwi_mc_upload: non-finite value in data trace %d", k);
    }
    umma_free(c->umma); c->umma = nullptr;
    int rc = build_rowset(c, c->base, 0);
    if (rc) return rc;
    if (c->NM == 1) {       // operands of the tensor-core path (one medium; two-media batches stay on the CUDA-core kernels)
        rc = umma_build(&c->umma, c->device, c->G.data(), c->d.data(), c->K, c->C, c->T, c->base.tc, c->base.fc);
        if (rc) return rc;
    }
    c->uploaded = true;
    return FWI_OK;
}

static int check_media(const fwi_mc_ctx* c, const float* frac, int nfrac, const char* who) {
    if (c->NM == 1) { FWI_REQUIRE(frac == nullptr && nfrac == 0, "%s: media fractions given but the context has one medium", who); }
    else {
        FWI_REQUIRE(frac != nullptr && (nfrac == 1 || nfrac == 3), "%s: two-media context needs media_frac with nfrac 1 or 3 (got %d)", who, nfrac);
        FWI_REQUIRE(nfrac == 1 || c->phase_dev, "%s: nfrac=3 needs phase_index at upload", who);
    }
    return FWI_OK;
}

int fwi_mc_forward(fwi_mc_ctx* c, const float* M, int64_t ldm, int n_comp, const float* frac, int nfrac,
                   int64_t N, float* traces, void* stream) {
    FWI_REQUIRE(c && c->uploaded, "fwi_mc_forward: context has no data (call fwi_mc_upload)");
    if (N == 0) return FWI_OK;                       // empty batch: nothing to do (pointers may be NULL)
    FWI_REQUIRE(M && traces && N >= 0 && ldm >= N, "fwi_mc_forward: bad M / traces / N / ldm");
    FWI_REQUIRE(n_comp >= 0 && n_comp <= c->C, "fwi_mc_forward: n_comp=%d exceeds C=%d", n_comp, c->C);
    int rc = check_media(c, frac, nfrac, "fwi_mc_forward");
    if (rc) return rc;
    if (N == 0) return FWI_OK;
    DeviceGuard g(c->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t KT = (int64_t)c->K * c->T;
    dim3 grid((unsigned)ceil_div(KT, 128), (unsigned)std::min<int64_t>(N, 4096));
#define FWD(CV, NMV) mc_forward_kernel<CV, NMV><<<grid, 128, 0, st>>>(c->base.rows, c->phase_dev, M, ldm, n_comp, frac, nfrac, N, c->K, c->T, traces)
    if (c->NM == 1) { if (c->C == 3) FWD(3, 1); else if (c->C == 6) FWD(6, 1); else FWD(9, 1); }
    else { if (c->C == 3) FWD(3, 2); else if (c->C == 6) FWD(6, 2); else FWD(9, 2); }
#undef FWD
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

int fwi_mc_eval(fwi_mc_ctx* c, const float* M, int64_t ldm, const float* frac, int nfrac, int64_t N, int metric,
                int flags, float* sim, float* like, void* stream) {
    FWI_REQUIRE(c && c->uploaded, "fwi_mc_eval: context has no data (call fwi_mc_upload)");
    if (N == 0) return FWI_OK;                       // empty batch: nothing to do (pointers may be NULL)
    FWI_REQUIRE(M && sim && N >= 0 && ldm >= N, "fwi_mc_eval: bad M / similarity / N / ldm");
    FWI_REQUIRE(metric >= 0 && metric <= 4, "fwi_mc_eval: unknown metric %d", metric);
    int rc = check_media(c, frac, nfrac, "fwi_mc_eval");
    if (rc) return rc;
    if (N == 0) return FWI_OK;
    DeviceGuard g(c->device);
    const bool norm = flags & FWI_FLAG_NORMALISED, simul = flags & FWI_FLAG_SIMULTANEOUS;
    if (metric == FWI_METRIC_GAU) {
        const int tv = simul ? c->K * c->T : c->T;
        FWI_REQUIRE(tv >= 60, "fwi_mc_eval: 'gau' needs at least 60 samples for its noise window (FWI:580), got %d", tv);
    }
    // Tensor-core path (tcgen05, 3 x TF32 split, TMEM epilogue; mc_umma.cu): every metric and mode, one medium.  Default for
    // batches of 256 samples and more; FWI_FLAG_TENSOR requires it, FWI_FLAG_NO_TENSOR / FWI_MC_TENSOR=0 keep the CUDA-core kernels.
    {
        const char* e = getenv("FWI_MC_TENSOR");
        const bool env_off = e && e[0] == '0';
        const bool can = c->umma && c->NM == 1 && nfrac == 0 && umma_supports(c->umma, metric, flags);
        FWI_REQUIRE(!(flags & FWI_FLAG_TENSOR) || can, "fwi_mc_eval: FWI_FLAG_TENSOR but the tensor-core path does not cover this case (two media, Gram mode, T > 1536 or C > 9)");
        if (can && !(flags & FWI_FLAG_NO_TENSOR) && ((flags & FWI_FLAG_TENSOR) || (!env_off && N >= 256)))
            return umma_eval(c->umma, M, ldm, N, metric, flags, sim, like, (cudaStream_t)stream);
    }
    RowSet* rs = &c->base;
    int boundary_fix = 0;
    if (metric == FWI_METRIC_CC_SHIFT) {
        if (simul && !norm) rs = &c->hrflat; else rs = &c->hr;
        if (!rs->built) { rc = build_rowset(c, *rs, rs == &c->hr ? 1 : 2); if (rc) return rc; }
        if (simul && norm) {
            // data constants of the normalised flattened interpolated array come from variant 2
            if (!c->hrflat.built) { rc = build_rowset(c, c->hrflat, 2); if (rc) return rc; }
            boundary_fix = 1;
        }
    }
    int mode;
    if (metric == FWI_METRIC_VR || metric == FWI_METRIC_GAU) mode = norm ? MODE_MOM_MAX : MODE_SSE;
    else mode = (simul && norm) ? MODE_MOM_MAX : MODE_MOM;

    EvalParams p{};
    p.rows = rs->rows; p.gbar = rs->gbar; p.tc = rs->tc; p.fc = rs->fc;
    if (boundary_fix) { p.fc.D1[1] = c->hrflat.fc.D1[1]; p.fc.D2[1] = c->hrflat.fc.D2[1]; }
    p.phase = c->phase_dev; p.M = M; p.ldm = ldm; p.frac = frac; p.nfrac = nfrac; p.N = N; p.K = c->K; p.Tv = rs->Tv;
    p.metric = metric; p.flags = flags; p.boundary_fix = boundary_fix; p.sim = sim; p.like = like;

    if (flags & FWI_FLAG_GRAM) {
        FWI_REQUIRE(!norm, "fwi_mc_eval: the Gram mode cannot normalise traces (it never forms them); drop FWI_FLAG_GRAM or FWI_FLAG_NORMALISED");
        FWI_REQUIRE(c->NM == 1 && rs->gram, "fwi_mc_eval: the Gram mode supports single-medium Green's functions only");
        const int NS = c->C * (c->C + 1) / 2, PT = 2 * NS + 3 * c->C;
        const size_t smem = (size_t)c->K * PT * sizeof(double);
        FWI_REQUIRE(smem <= 200 * 1024, "fwi_mc_eval: K=%d traces exceed the shared-memory Gram buffer", c->K);
        cudaStream_t gst = (cudaStream_t)stream;
        const unsigned blocks = (unsigned)ceil_div(N, 128);
#define GRAM(CV) do { if (smem > 48 * 1024) FWI_CUDA(cudaFuncSetAttribute(mc_gram_kernel<CV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
                      mc_gram_kernel<CV><<<blocks, 128, smem, gst>>>(rs->gram, p); } while (0)
        if (c->C == 3) GRAM(3); else if (c->C == 6) GRAM(6); else GRAM(9);
#undef GRAM
        FWI_CUDA(cudaGetLastError());
        return FWI_OK;
    }
    // samples per lane: 4 when there is enough work to fill the machine twice over, else fewer; the wide kernels (8 per
    // lane, 4 for two media) for big batches (see launch_eval_s)
    int S = 4;
    const int64_t full = (int64_t)c->sm_count * 2 * 128;
    if (N < full) S = 2;
    if (N < full / 4) S = 1;
    const bool big = N >= 4 * full;
    if (big) S = 8;                          // the wide kernels
    { const char* e = getenv("FWI_MC_S"); if (e && S > atoi(e) && atoi(e) >= 1) S = atoi(e); }     // tuning aid
    // big batches: one sample group per warp, every warp walks all K traces (no block-level synchronisation);
    // small batches are latency-bound: the warps of a CTA share one sample group and split the traces.  The
    // cross-boundary patch of flattened CC-shift carries state from trace to trace, so it never splits.
    int nw = (S == 8) ? 4 : 8, ks = 1;
    if (!big && !boundary_fix) { nw = pick_warps(c->K); ks = nw; }
    else if (!boundary_fix && S == 8) ks = 2;     // measured at N = 2e6 / 4e6: ks 1: 175, 2: 215, 4: 189 M samples/s (finer CTA tail)
    p.ks = ks;
    cudaStream_t st = (cudaStream_t)stream;
    if (c->NM == 1) {
        if (c->C == 3) return launch_eval_m<3, 1>(p, mode, S, nw, st);
        if (c->C == 6) return launch_eval_m<6, 1>(p, mode, S, nw, st);
        return launch_eval_m<9, 1>(p, mode, S, nw, st);
    }
    if (c->C == 3) return launch_eval_m<3, 2>(p, mode, S, nw, st);
    if (c->C == 6) return launch_eval_m<6, 2>(p, mode, S, nw, st);
    return launch_eval_m<9, 2>(p, mode, S, nw, st);
}

int fwi_mc_transform_draws(int type, const float* draws, int64_t ldn, int64_t N, float amp, float* out, int64_t ldo,
                           void* stream) {
    FWI_REQUIRE(type >= 0 && type <= 6, "fwi_mc_transform_draws: unknown inversion type %d", type);
    FWI_REQUIRE(draws && out && N >= 0 && ldn >= N && ldo >= N, "fwi_mc_transform_draws: bad pointers / sizes");
    if (N == 0) return FWI_OK;
    mc_transform_kernel<<<(unsigned)ceil_div(N, 128), 128, 0, (cudaStream_t)stream>>>(type, draws, ldn, N, amp, out, ldo);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

// Persistent per-device partials buffer for fwi_mc_reduce (a stream-ordered allocation around a synchronising call is
// handed back to the driver every time, which costs milliseconds once tens of GB are allocated).  One caller per device
// at a time: the call synchronises before it returns.
static void* reduce_scratch(size_t bytes) {
    static void* buf[64] = {};
    static size_t cap[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (cap[dev] < bytes) {
        if (buf[dev]) cudaFree(buf[dev]);
        buf[dev] = nullptr; cap[dev] = 0;
        if (cudaMalloc(&buf[dev], bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        cap[dev] = bytes;
    }
    return buf[dev];
}

int fwi_mc_reduce(const float* L, int64_t N, double* sum_host, int64_t* argmax_host, float* max_host, void* stream) {
    FWI_REQUIRE(L && N >= 1, "fwi_mc_reduce: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (int)std::min<int64_t>(1024, ceil_div(N, 1024));
    char* scratch = (char*)reduce_scratch(1024 * (sizeof(double) + sizeof(long long) + sizeof(float)));
    FWI_REQUIRE(scratch, "fwi_mc_reduce: no device scratch");
    double* psum = (double*)scratch;
    long long* parg = (long long*)(scratch + 1024 * sizeof(double));
    float* pmax = (float*)(scratch + 1024 * (sizeof(double) + sizeof(long long)));
    mc_reduce_kernel<<<blocks, 256, 0, st>>>(L, N, psum, pmax, parg);
    FWI_CUDA(cudaGetLastError());
    std::vector<double> hs(blocks); std::vector<float> hm(blocks); std::vector<long long> ha(blocks);
    FWI_CUDA(cudaMemcpyAsync(hs.data(), psum, blocks * sizeof(double), cudaMemcpyDeviceToHost, st));
    FWI_CUDA(cudaMemcpyAsync(hm.data(), pmax, blocks * sizeof(float), cudaMemcpyDeviceToHost, st));
    FWI_CUDA(cudaMemcpyAsync(ha.data(), parg, blocks * sizeof(long long), cudaMemcpyDeviceToHost, st));
    FWI_CUDA(cudaStreamSynchronize(st));
    double s = 0.0; float mx = -INFINITY; long long am = -1;
    for (int b = 0; b < blocks; ++b) {
        s += hs[b];
        if (hm[b] > mx || (hm[b] == mx && ha[b] >= 0 && (am < 0 || ha[b] < am))) { mx = hm[b]; am = ha[b]; }
    }
    if (sum_host) *sum_host = s;
    if (argmax_host) *argmax_host = am;
    if (max_host) *max_host = mx;
    return FWI_OK;
}

int fwi_mc_sample_eval(fwi_mc_ctx* c, int type, uint64_t seed, int64_t first, int64_t N, float amp, int metric, int flags,
                       int nfrac, float* MTs, int64_t ldn, float* sim, float* L, double* sumL, int64_t* argmax,
                       float* maxL, void* stream) {
    FWI_REQUIRE(c && c->uploaded, "fwi_mc_sample_eval: context has no data (call fwi_mc_upload)");
    FWI_REQUIRE(type >= 0 && type <= 6, "fwi_mc_sample_eval: unknown inversion type %d", type);
    FWI_REQUIRE(type_components(type) == c->C, "fwi_mc_sample_eval: inversion type %d produces %d components but the Green's functions have %d", type, type_components(type), c->C);
    FWI_REQUIRE(MTs && sim && L && N >= 0 && ldn >= N && first >= 0, "fwi_mc_sample_eval: bad pointers / sizes");
    FWI_REQUIRE((c->NM == 1 && nfrac == 0) || (c->NM == 2 && (nfrac == 1 || nfrac == 3)), "fwi_mc_sample_eval: nfrac=%d inconsistent with n_media=%d", nfrac, c->NM);
    if (N == 0) { if (sumL) *sumL = 0.0; if (argmax) *argmax = -1; if (maxL) *maxL = 0.f; return FWI_OK; }
    DeviceGuard g(c->device);
    cudaStream_t st = (cudaStream_t)stream;
    mc_sample_kernel<<<(unsigned)ceil_div(N, 128), 128, 0, st>>>(type, seed, first, N, amp, nfrac, MTs, ldn);
    FWI_CUDA(cudaGetLastError());
    const int rows = type_components(type) + (type_combined(type) ? 1 : 0);
    const float* frac = nfrac ? MTs + (int64_t)rows * ldn : nullptr;
    int rc = fwi_mc_eval(c, MTs, ldn, frac, nfrac, N, metric, flags, sim, L, stream);
    if (rc) return rc;
    if (sumL || argmax || maxL) return fwi_mc_reduce(L, N, sumL, argmax, maxL, stream);
    return FWI_OK;
}

int fwi_mc_normalise(const float* L, int64_t N, double sumL, float* MTp, void* stream) {
    FWI_REQUIRE(L && MTp && N >= 0, "fwi_mc_normalise: bad arguments");
    if (!(sumL > 0.0)) { set_error("fwi_mc_normalise: sum of likelihoods is %g - no adequate solution (FWI:1206-1208)", sumL); return FWI_EZEROPROB; }
    if (N == 0) return FWI_OK;
    // MTp = L * p_model / p_data with p_model = 1/N and p_data = sum(p_model * L)  ==  L / sum(L)
    mc_normalise_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, (cudaStream_t)stream>>>(L, N, 1.0 / sumL, MTp);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

__global__ void mc_stage_kernel(const double* __restrict__ Mh, int64_t N, int C, int n_comp, float* __restrict__ M) {
    // (N, n_comp) float64 sample-major -> (C, N) fp32, missing trailing components zero (FWI:262)
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * C) return;
    const int c = (int)(i / N);
    const int64_t n = i % N;
    M[i] = (c < n_comp) ? (float)Mh[n * n_comp + c] : 0.f;
}
__global__ void mc_unstage_kernel(const float* __restrict__ s, int64_t N, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) out[i] = (double)s[i];
}

int fwi_mc_eval_host(fwi_mc_ctx* c, const double* M_host, int64_t N, int n_comp, const double* frac_host, int nfrac,
                     int metric, int flags, double* sim_host) {
    FWI_REQUIRE(c && c->uploaded, "fwi_mc_eval_host: context has no data (call fwi_mc_upload)");
    FWI_REQUIRE(M_host && sim_host && N >= 1, "fwi_mc_eval_host: bad arguments");
    FWI_REQUIRE(n_comp >= 1 && n_comp <= c->C, "fwi_mc_eval_host: n_comp=%d exceeds C=%d", n_comp, c->C);
    DeviceGuard g(c->device);
    if (c->stage_cap < N) {
        if (c->stage_M) cudaFree(c->stage_M);
        if (c->stage_sim) cudaFree(c->stage_sim);
        if (c->stage_frac) cudaFree(c->stage_frac);
        c->stage_M = c->stage_sim = c->stage_frac = nullptr;
        FWI_CUDA(cudaMalloc(&c->stage_M, (size_t)N * c->C * sizeof(float)));
        FWI_CUDA(cudaMalloc(&c->stage_sim, (size_t)N * sizeof(float)));
        FWI_CUDA(cudaMalloc(&c->stage_frac, (size_t)N * 3 * sizeof(float)));
        c->stage_cap = N;
    }
    const int64_t need = (int64_t)N * (n_comp + 3) * sizeof(double);
    if (c->dstage_bytes < need) {
        if (c->dstage) cudaFree(c->dstage);
        c->dstage = nullptr; c->dstage_bytes = 0;
        FWI_CUDA(cudaMalloc(&c->dstage, (size_t)need));
        c->dstage_bytes = need;
    }
    double* dbuf = c->dstage;
    int rc = FWI_OK;
    do {
        if (cudaMemcpy(dbuf, M_host, (size_t)N * n_comp * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) { rc = FWI_ECUDA; break; }
        mc_stage_kernel<<<(unsigned)ceil_div(N * c->C, 256), 256>>>(dbuf, N, c->C, n_comp, c->stage_M);
        const float* frac = nullptr;
        if (frac_host && nfrac > 0) {
            double* fb = dbuf + (size_t)N * n_comp;
            if (cudaMemcpy(fb, frac_host, (size_t)N * nfrac * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) { rc = FWI_ECUDA; break; }
            mc_stage_kernel<<<(unsigned)ceil_div(N * nfrac, 256), 256>>>(fb, N, nfrac, nfrac, c->stage_frac);
            frac = c->stage_frac;
        }
        rc = fwi_mc_eval(c, c->stage_M, N, frac, frac ? nfrac : 0, N, metric, flags, c->stage_sim, nullptr, nullptr);
        if (rc) break;
        mc_unstage_kernel<<<(unsigned)ceil_div(N, 256), 256>>>(c->stage_sim, N, dbuf);
        if (cudaMemcpy(sim_host, dbuf, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess) { rc = FWI_ECUDA; break; }
    } while (0);
    if (rc == FWI_ECUDA) set_error("fwi_mc_eval_host: CUDA copy failed: %s", cudaGetErrorString(cudaGetLastError()));
    return rc;
}


int fwi_mc_prepare(const double* raw_dev, int K, int C, int T, int n_media, const int* shift_dev, int zero_head,
                   const int* cut_start_dev, int cut_len, double scale1, double scale2, double* out_dev, void* stream) {
    FWI_REQUIRE(raw_dev && out_dev && K >= 1 && C >= 1 && T >= 1 && (n_media == 1 || n_media == 2), "fwi_mc_prepare: bad arguments");
    FWI_REQUIRE(cut_start_dev == nullptr || cut_len >= 1, "fwi_mc_prepare: cut_len must be >= 1 when cut_start is given");
    const int Tout = cut_start_dev ? cut_len : T;
    const int64_t total = (int64_t)K * C * Tout * n_media;
    mc_prepare_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, (cudaStream_t)stream>>>(raw_dev, K, C, T, n_media, shift_dev, zero_head,
                                                                                      cut_start_dev, Tout, scale1, scale2, out_dev);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}


int fwi_mc_posterior_hist(int mode, const float* MTs_dev, int64_t ldn, const float* MTp_dev, const int64_t* idx_dev, int64_t n,
                          int row0, double* hist_dev, void* stream) {
    FWI_REQUIRE(mode >= 0 && mode <= 2 && MTs_dev && hist_dev && n >= 0 && ldn >= 1 && row0 >= 0, "fwi_mc_posterior_hist: bad arguments");
    FWI_REQUIRE(mode == 2 || MTp_dev, "fwi_mc_posterior_hist: MTp_dev is required for modes 0 and 1");
    const int nbins = (mode == 0) ? 36 * 72 : (mode == 1 ? 202 : 122 * 41);   // np.arange(-pi/2, pi/2 + bs, bs) has 122 labels
    cudaStream_t st = (cudaStream_t)stream;
    FWI_CUDA(cudaMemsetAsync(hist_dev, 0, nbins * sizeof(double), st));
    if (n == 0) return FWI_OK;
    const int blocks = (int)std::min<int64_t>(296, ceil_div(n, 256));
    mc_hist_kernel<<<blocks, 256, nbins * sizeof(double), st>>>(mode, MTs_dev, ldn, MTp_dev, (const long long*)idx_dev, n, row0, hist_dev, nbins);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}


int fwi_mc_lstsq(int device, const double* G_host, const double* d_host, int K, int C, int T, double* M_host) {
    FWI_REQUIRE(G_host && d_host && M_host && K >= 1 && T >= 1, "fwi_mc_lstsq: bad arguments");
    FWI_REQUIRE(C == 3 || C == 6 || C == 9, "fwi_mc_lstsq: C must be 3, 6 or 9 (got %d)", C);
    int ndev = 0;
    FWI_CUDA(cudaGetDeviceCount(&ndev));
    FWI_REQUIRE(device >= 0 && device < ndev, "fwi_mc_lstsq: device %d out of range (%d visible)", device, ndev);
    DeviceGuard g(device);
    const size_t nG = (size_t)K * C * T, nd = (size_t)K * T;
    const int NS = C * (C + 1) / 2;
    double* buf = nullptr;
    FWI_CUDA(cudaMalloc(&buf, (nG + nd + NS + C + C + 1) * sizeof(double)));
    double *dG = buf, *dd = buf + nG, *acc = dd + nd, *dm = acc + NS + C;
    int* st = (int*)(dm + C);
    int rc = FWI_OK;
    do {
        if (cudaMemcpy(dG, G_host, nG * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(dd, d_host, nd * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemset(acc, 0, (NS + C) * sizeof(double)) != cudaSuccess) { rc = FWI_ECUDA; break; }
        const unsigned blocks = (unsigned)std::min<int64_t>(296, ceil_div((int64_t)nd, 128));
        if (C == 3) { mc_normal_eq_kernel<3><<<blocks, 128>>>(dG, dd, K, T, acc); mc_cholesky_kernel<3><<<1, 32>>>(acc, dm, st); }
        else if (C == 6) { mc_normal_eq_kernel<6><<<blocks, 128>>>(dG, dd, K, T, acc); mc_cholesky_kernel<6><<<1, 32>>>(acc, dm, st); }
        else { mc_normal_eq_kernel<9><<<blocks, 128>>>(dG, dd, K, T, acc); mc_cholesky_kernel<9><<<1, 32>>>(acc, dm, st); }
        int hst = 0;
        if (cudaMemcpy(M_host, dm, C * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess ||
            cudaMemcpy(&hst, st, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) { rc = FWI_ECUDA; break; }
        if (hst) { set_error("fwi_mc_lstsq: the Green's functions are rank deficient (non-positive Cholesky pivot)"); rc = FWI_EINVAL; }
    } while (0);
    if (rc == FWI_ECUDA) set_error("fwi_mc_lstsq: CUDA failure: %s", cudaGetErrorString(cudaGetLastError()));
    cudaFree(buf);
    return rc;
}

int fwi_diag_fp32_peak(int device, double* tflops_out) {
    FWI_REQUIRE(tflops_out, "fwi_diag_fp32_peak: NULL output");
    int ndev = 0;
    FWI_CUDA(cudaGetDeviceCount(&ndev));
    FWI_REQUIRE(device >= 0 && device < ndev, "fwi_diag_fp32_peak: device %d out of range (%d visible)", device, ndev);
    DeviceGuard g(device);
    cudaDeviceProp prop;
    FWI_CUDA(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    float* out = nullptr;
    FWI_CUDA(cudaMalloc(&out, (size_t)blocks * threads * sizeof(float)));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {           // first repetition warms the clocks up
        cudaEventRecord(e0);
        fp32_fma_probe_kernel<<<blocks, threads>>>(out, iters, 1.0f + rep);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    const cudaError_t err = cudaGetLastError();
    cudaFree(out);
    if (err != cudaSuccess) { set_error("fwi_diag_fp32_peak: %s", cudaGetErrorString(err)); return FWI_ECUDA; }
    *tflops_out = 2.0 * 64.0 * iters * (double)blocks * threads / (best * 1e-3) / 1e12;
    return FWI_OK;
}

}  // extern "C"
