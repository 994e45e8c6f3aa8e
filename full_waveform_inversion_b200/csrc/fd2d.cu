// Track B, 2-D: leapfrog acoustic step with fused source injection / receiver sampling, forward-field
// snapshotting and adjoint imaging, for sm_100a.
//
//   w_n     = lap(u_n) + f_n
//   u_{n+1} = g * (2 u_n - g * u_{n-1} + m * w_n)           (oracle/fd_oracle.py, spec B1-B3)
//
// Data layout: every field is [nz][px] fp32, x contiguous, px = nx rounded up to 32 floats so each row
// starts on a 128-byte line; no ghost cells in memory.  The (BX+8) x (BZ+8) input tile of u_n is staged
// into shared memory by ONE TMA tiled load per CTA (cp.async.bulk.tensor.2d); the hardware zero-fills
// the part of the box that falls outside the grid, which is the Dirichlet halo.  Each lane owns four
// consecutive x points (one float4), reads its x-neighbours as two more float4 from the tile, and keeps
// the nine z-neighbours in a register window that rotates down the column, so shared memory is read
// ~4 x 16 B per float4 of output.  u_{n-1} and m are touched once per point straight from global
// (coalesced float4) and u_{n+1} overwrites u_{n-1} in place: 16 B of algorithmic traffic per update.
// The forward pass can stream w_n to an HBM snapshot (evict-first stores); the adjoint pass reads it
// back and accumulates the zero-lag cross-correlation in the same kernel.  The Born (linearised) step reads it back as the
// source term of the scattered field: du_{n+1} = g (2 du_n - g du_{n-1} + m lap(du_n) + dm w_n)  (spec B5).
// A plan may make row z = 0 a free surface (spec B6, fwi_fd2d_set_free_surface): every step kernel has an FS instance in which
// the CTAs at z = 0 replace the zero halo above the grid by the odd mirror u[-k] = -u[k]; all other CTAs run unchanged code.
#include "fd_common.cuh"
#include <vector>
#include <algorithm>
#include <cmath>
#include <cstring>

namespace fwi {

// ADJ2: image this step AND the previous one (deferred).  BORN: a scattered (linearised) step whose source term is
// dm * w_n, w_n read from the background sweep's snapshot (spec B5, tests/born_reference.py)
enum { STEP_FWD = 0, STEP_FWD_SAVE = 1, STEP_ADJ = 2, STEP_ADJ2 = 3, STEP_BORN = 4 };
}  // namespace fwi
#include "fd3d.cuh"
#include "fd2d_tb2.cuh"
namespace fwi {

struct Step2DArgs {
    float* oldnew;        // u_{n-1} in, u_{n+1} out (in place)
    const float* m;
    const float* gx;
    const float* gz;
    float* snap;          // w_n: written (FWD_SAVE) or read (ADJ)
    const float* snap_prev; // ADJ2: snapshot paired with the field of the previous adjoint step (= u_n of this launch)
    float* acc;           // imaging accumulator (ADJ)
    int nx, nz, px;
    PointListDev inj;     // sources (forward) / receivers (adjoint)
    const float* inj_vals;
    PointListDev rec;     // receivers to sample (forward only; tile_ptr == nullptr otherwise)
    float* rec_out;
    const float* dm;      // BORN: model perturbation dm = (2 m / v) dv, pitched like m
};

// rows of u_{n-1} / m requested before the dependency wait.  ms per 1000-step gradient at 1000x3000: 0 rows 17.0, 1 row
// 16.2, 2 rows 16.0 (80 registers, still 6 CTAs per SM); prefetching the adjoint's snapshot row as well: 16.5 - 19.0
constexpr int kPrefetchRows = 2;
// The PDL trigger is left implicit (when this grid's CTAs exit): an explicit early griddepcontrol.launch_dependents parks the
// whole next grid at its dependency wait and releases all CTAs in the same instant, which lines up their load / compute /
// store phases and costs L2 bandwidth (ms per 5000-step gradient: no PDL 85.5, implicit 84.5, after the dense part 88.6,
// at the top 101).
// No minimum-blocks bound: ptxas settles at 80 registers (3 CTAs of 256 threads per SM); with an explicit minimum of 1 it takes 110.
// FS: free surface at z = 0 (spec B6, tests/free_surface_reference.py): the top row of CTAs replaces the zero-filled rows
// above the grid by the odd mirror u[-k] = -u[k] before computing; every other CTA runs the FS = false code.
template <int BZ, int NW, int MODE, bool FS>
__global__ void __launch_bounds__(NW * 32) fd2d_step_kernel(const __grid_constant__ CUtensorMap tm_cur, Step2DArgs a) {
    constexpr int BX = 128, SX = BX + 2 * kHalo, SZ = BZ + 2 * kHalo, RPW = BZ / NW;
    static_assert(BZ % NW == 0, "rows must split evenly over warps");
    extern __shared__ __align__(128) float tile[];          // [SZ][SX]
    __shared__ __align__(8) uint64_t bar;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tx0 = blockIdx.x * BX, tz0 = blockIdx.y * BZ;
    const int x = tx0 + 4 * lane;
    const int zw = tz0 + warp * RPW;
    const bool col_ok = x < a.px;
    // ---- prologue that does not depend on the previous time step: with programmatic dependent launch this part of
    //      step n+1 runs while step n is still draining (the launch latency and the tail of a 6 us kernel overlap)
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
        fence_proxy_async();
    }
    float4 gx4 = make_float4(1.f, 1.f, 1.f, 1.f);
    if (col_ok) gx4 = ld4(a.gx + x);
    // (prefetching the adjoint's snapshot rows into L2 from here was measured: 17.3 vs 17.0 ms per 1000-step gradient, not kept;
    //  so was a bulk L2 prefetch, cp.async.bulk.prefetch.L2, of the two snapshot tiles of the NEXT deferred-imaging launch
    //  issued by the propagate-only step before it: 16.5 vs 15.6 us per forward+adjoint step pair at 1000 x 3000)
    // u_{n-1} and m of this warp's first rows: neither is written by the step this launch is chained to (u_{n-1} is the
    // output of step n-2, which completed before step n-1 passed its own wait), and requesting them here takes one L2
    // round trip off the serial chain  TMA wait -> row loads -> compute
    float4 o4p[kPrefetchRows], m4p[kPrefetchRows];
#pragma unroll
    for (int r = 0; r < kPrefetchRows; ++r) {
        o4p[r] = make_float4(0.f, 0.f, 0.f, 0.f); m4p[r] = o4p[r];
        if (col_ok && zw + r < a.nz) {
            o4p[r] = ld4(a.oldnew + (size_t)(zw + r) * a.px + x);
            m4p[r] = ld4(a.m + (size_t)(zw + r) * a.px + x);
        }
    }
    griddep_wait();                 // step n complete and visible (no-op for a plain launch)
    if (threadIdx.x == 0) {
        mbar_expect_tx(&bar, SX * SZ * (uint32_t)sizeof(float));
        tma_load_2d(tile, &tm_cur, tx0 - kHalo, tz0 - kHalo, &bar);
    }
    __syncthreads();        // barrier init visible to every waiter

    mbar_wait(&bar, 0);
    if (FS && tz0 == 0) {           // uniform per CTA
        mirror_rows(tile, SX, kHalo, SX);       // tile row kHalo is z = 0; the x halo columns are mirrored too
        __syncthreads();
    }

    if (col_ok && zw < a.nz) {
        // register window over z: win[k] holds row (z - 4 + k) of this lane's float4 column
        float4 win[9];
        const float* tcol = tile + (warp * RPW) * SX + kHalo + 4 * lane;     // row z-4 of the first output row
#pragma unroll
        for (int k = 0; k < 8; ++k) win[k + 1] = ld4(tcol + k * SX);
#pragma unroll
        for (int r = 0; r < RPW; ++r) {
            const int z = zw + r;
#pragma unroll
            for (int k = 0; k < 8; ++k) win[k] = win[k + 1];
            win[8] = ld4(tcol + (r + 8) * SX);
            if (z < a.nz) {
                const float* trow = tile + (warp * RPW + r + kHalo) * SX + 4 * lane;
                const float4 L = ld4(trow), R = ld4(trow + 8);
                const float4 C = win[4];
                const float ax[12] = {L.x, L.y, L.z, L.w, C.x, C.y, C.z, C.w, R.x, R.y, R.z, R.w};
                float zc[9][4];
#pragma unroll
                for (int k = 0; k < 9; ++k) { zc[k][0] = win[k].x; zc[k][1] = win[k].y; zc[k][2] = win[k].z; zc[k][3] = win[k].w; }
                const size_t off = (size_t)z * a.px + x;
                const float4 o4 = (r < kPrefetchRows) ? o4p[r < kPrefetchRows ? r : 0] : ld4(a.oldnew + off);
                const float4 m4 = (r < kPrefetchRows) ? m4p[r < kPrefetchRows ? r : 0] : ld4(a.m + off);
                float4 w4 = make_float4(0.f, 0.f, 0.f, 0.f), d4 = w4;
                if (MODE == STEP_BORN) { w4 = ld4_stream(a.snap + off); d4 = ld4(a.dm + off); }
                const float bw[4] = {w4.x, w4.y, w4.z, w4.w}, bd[4] = {d4.x, d4.y, d4.z, d4.w};
                const float gzv = __ldg(a.gz + z);
                const float ov[4] = {o4.x, o4.y, o4.z, o4.w}, mv[4] = {m4.x, m4.y, m4.z, m4.w};
                const float gv[4] = {gx4.x * gzv, gx4.y * gzv, gx4.z * gzv, gx4.w * gzv};
                float wv[4], nv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float c = ax[4 + j];
                    float lap = (2.0f * kC0) * c;
                    lap = fmaf(kC1, (ax[3 + j] + ax[5 + j]) + (zc[3][j] + zc[5][j]), lap);
                    lap = fmaf(kC2, (ax[2 + j] + ax[6 + j]) + (zc[2][j] + zc[6][j]), lap);
                    lap = fmaf(kC3, (ax[1 + j] + ax[7 + j]) + (zc[1][j] + zc[7][j]), lap);
                    lap = fmaf(kC4, (ax[0 + j] + ax[8 + j]) + (zc[0][j] + zc[8][j]), lap);
                    wv[j] = lap;
                    // BORN: nv = g * fma(m, lap, fma(dm, w, fma(-g, o, 2 c))) - the forward update with dm * w_n added last
                    float rest = fmaf(-gv[j], ov[j], 2.0f * c);
                    if (MODE == STEP_BORN) rest = fmaf(bd[j], bw[j], rest);
                    nv[j] = gv[j] * fmaf(mv[j], lap, rest);
                }
                st4(a.oldnew + off, make_float4(nv[0], nv[1], nv[2], nv[3]));
                if (MODE == STEP_FWD_SAVE) st4_stream(a.snap + off, make_float4(wv[0], wv[1], wv[2], wv[3]));
                if (MODE == STEP_ADJ || MODE == STEP_ADJ2) {
                    const float4 s4 = ld4_stream(a.snap + off);
                    float4 c4 = ld4(a.acc + off);
                    if (MODE == STEP_ADJ2) {
                        // deferred imaging of the previous adjoint step: its field is this launch's u_n (centre value C);
                        // same fma order as two consecutive ADJ launches, so the accumulator is bit-identical
                        const float4 sp = ld4_stream(a.snap_prev + off);
                        c4.x = fmaf(C.x, sp.x, c4.x); c4.y = fmaf(C.y, sp.y, c4.y);
                        c4.z = fmaf(C.z, sp.z, c4.z); c4.w = fmaf(C.w, sp.w, c4.w);
                    }
                    c4.x = fmaf(nv[0], s4.x, c4.x); c4.y = fmaf(nv[1], s4.y, c4.y);
                    c4.z = fmaf(nv[2], s4.z, c4.z); c4.w = fmaf(nv[3], s4.w, c4.w);
                    st4(a.acc + off, c4);
                }
            }
        }
    }

    // ---- sparse fix-ups for the points this tile owns: injection, then receiver sampling ----------
    const int tid = blockIdx.y * gridDim.x + blockIdx.x;
    const int i0 = a.inj.tile_ptr ? a.inj.tile_ptr[tid] : 0, i1 = a.inj.tile_ptr ? a.inj.tile_ptr[tid + 1] : 0;
    const int r0 = a.rec.tile_ptr ? a.rec.tile_ptr[tid] : 0, r1 = a.rec.tile_ptr ? a.rec.tile_ptr[tid + 1] : 0;
    if (i1 > i0 || r1 > r0) {             // uniform per CTA
        __syncthreads();
        for (int e = i0 + threadIdx.x; e < i1; e += blockDim.x) {
            const int off = a.inj.off[e];
            const int z = off / a.px, xx = off - z * a.px;
            const float val = a.inj_vals[a.inj.id[e]];
            const float gm = a.gx[xx] * a.gz[z] * a.m[off];
            atomicAdd(a.oldnew + off, gm * val);                       // u_{n+1} += g m f
            if (MODE == STEP_FWD_SAVE) atomicAdd(a.snap + off, val);   // w_n includes f_n
            if (MODE == STEP_ADJ || MODE == STEP_ADJ2) atomicAdd(a.acc + off, gm * val * a.snap[off]);
        }
        if (r1 > r0) {
            __syncthreads();
            for (int e = r0 + threadIdx.x; e < r1; e += blockDim.x)
                a.rec_out[a.rec.id[e]] = __ldcg(a.oldnew + a.rec.off[e]);
        }
    }
}

// ------------------------------------------------------------------------------------------ small kernels
__global__ void fd_model_kernel(const float* __restrict__ v, int nz, int nx, int px, float dt_over_h,
                                float* __restrict__ m, float* __restrict__ vp) {
    const int x = blockIdx.y * blockDim.x + threadIdx.x, z = blockIdx.x;   // rows on grid.x (no 65535 limit)
    if (x >= px || z >= nz) return;
    float val = 0.f, vv = 0.f;
    if (x < nx) { vv = v[(size_t)z * nx + x]; const float c = vv * dt_over_h; val = c * c; }
    m[(size_t)z * px + x] = val;
    vp[(size_t)z * px + x] = vv;
}

// Born: dm = (2 m / v) dv in the owned columns (dm/dv of m = (v dt / h)^2, spec B5), 0 in the pad columns
__global__ void fd_dm_kernel(const float* __restrict__ dv, const float* __restrict__ m, const float* __restrict__ vp, int nz,
                             int nx, int px, float* __restrict__ dm) {
    const int x = blockIdx.y * blockDim.x + threadIdx.x, z = blockIdx.x;   // rows on grid.x (no 65535 limit)
    if (x >= px || z >= nz) return;
    const size_t o = (size_t)z * px + x;
    dm[o] = (x < nx) ? 2.0f * m[o] * dv[(size_t)z * nx + x] / vp[o] : 0.f;
}

__global__ void fd_grad_finalize_kernel(const float* __restrict__ acc, const float* __restrict__ vp, int nz, int nx,
                                        int px, float* __restrict__ grad) {
    const int x = blockIdx.y * blockDim.x + threadIdx.x, z = blockIdx.x;   // rows on grid.x (no 65535 limit)
    if (x >= nx || z >= nz) return;
    const size_t o = (size_t)z * px + x;
    grad[(size_t)z * nx + x] += 2.0f * acc[o] / vp[o];                 // dJ/dv = (2/v) I
}

__global__ void fd_unpitch_kernel(const float* __restrict__ src, int nz, int nx, int px, float* __restrict__ dst) {
    const int x = blockIdx.y * blockDim.x + threadIdx.x, z = blockIdx.x;   // rows on grid.x (no 65535 limit)
    if (x < nx && z < nz) dst[(size_t)z * nx + x] = src[(size_t)z * px + x];
}

__global__ void fd_residual_kernel(const float* __restrict__ syn, const float* __restrict__ obs, int64_t n,
                                   float* __restrict__ res, double* __restrict__ J) {
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float r = syn[i] - obs[i];
        res[i] = r;
        s += (double)r * (double)r;
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ double ws[32];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += ws[w];
        atomicAdd(J, 0.5 * t);
    }
}

// Off-grid points (spec B7, tests/offgrid_reference.py): an operator in CSR form maps time-major rows of one side to the
// other, out[n][j] = sum_{e in [ptr[j], ptr[j+1])} w[e] * in[n][col[e]], summed in CSR order so that every run gives the
// same bits.  Gather: point-major CSR, cell rows in, point rows out (traces); spread: cell-major CSR, point rows in, cell
// rows out (wavelets, residuals).  One kernel serves both; the two names keep them apart in profiles.
// A thread owns one output column and kInterpRows time rows: the lanes of a warp read their CSR entries 64 taps apart (one
// L1 wavefront per lane), so each (col, w) is loaded once for kInterpRows rows (measured at 3000 receivers x 64 taps,
// nt = 5000: 6.8 ms per gather with one row per thread).
constexpr int kInterpRows = 8;
__device__ __forceinline__ void interp_rows(const int* __restrict__ ptr, const int* __restrict__ col, const float* __restrict__ w,
                                            const float* __restrict__ in, int nin, float* __restrict__ out, int nout, int nt) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nout) return;
    const int e0 = ptr[j], e1 = ptr[j + 1];
    for (int n0 = blockIdx.y * kInterpRows; n0 < nt; n0 += gridDim.y * kInterpRows) {
        const int nn = min(kInterpRows, nt - n0);
        const float* rows = in + (size_t)n0 * nin;
        float acc[kInterpRows];
#pragma unroll
        for (int k = 0; k < kInterpRows; ++k) acc[k] = 0.f;
        for (int e = e0; e < e1; ++e) {
            const float we = w[e];
            const float* p = rows + col[e];
#pragma unroll
            for (int k = 0; k < kInterpRows; ++k)
                if (k < nn) acc[k] = fmaf(we, p[(size_t)k * nin], acc[k]);
        }
#pragma unroll
        for (int k = 0; k < kInterpRows; ++k)
            if (k < nn) out[(size_t)(n0 + k) * nout + j] = acc[k];
    }
}
__global__ void fd_interp_gather_kernel(const int* __restrict__ ptr, const int* __restrict__ col, const float* __restrict__ w,
                                        const float* __restrict__ in, int nin, float* __restrict__ out, int nout, int nt) {
    interp_rows(ptr, col, w, in, nin, out, nout, nt);
}
__global__ void fd_interp_spread_kernel(const int* __restrict__ ptr, const int* __restrict__ col, const float* __restrict__ w,
                                        const float* __restrict__ in, int nin, float* __restrict__ out, int nout, int nt) {
    interp_rows(ptr, col, w, in, nin, out, nout, nt);
}

__global__ void fd_update_kernel(float* __restrict__ v, const float* __restrict__ g, float step, float vmin, float vmax,
                                 int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = fminf(vmax, fmaxf(vmin, v[i] - step * g[i]));
}

__global__ void fd_absmax_kernel(const float* __restrict__ x, int64_t n, unsigned int* __restrict__ out) {
    float mx = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        mx = fmaxf(mx, fabsf(x[i]));
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(mx));     // non-negative floats order like uints
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int encode_tiled_f32(CUtensorMap* out, void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                     const uint32_t* box) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        FWI_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        if (!p || q != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled not available from the driver"); return FWI_ECUDA; }
        fn = (EncodeTiledFn)p;
    }
    cuuint64_t d[5]; cuuint64_t s[5]; cuuint32_t b[5]; cuuint32_t es[5];
    for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; es[i] = 1; }
    for (int i = 0; i < rank - 1; ++i) s[i] = strides_bytes[i];
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, base, d, s, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return FWI_ECUDA; }
    return FWI_OK;
}

}  // namespace fwi

using namespace fwi;

// =============================================================================================== host plan
//
// Time loops are replayed as CUDA graphs: a 1000 x 3000 step kernel runs for ~6 us, about what one
// cudaLaunchKernel costs the host, so a stream of individual launches is launch-bound.  The whole forward
// pass (nt step nodes) and the whole gradient (forward with snapshots, residual, adjoint with imaging, and the
// checkpoint copies when they are needed) are each captured ONCE per (nt, geometry size) on the plan's private
// stream and re-launched for every shot.  That requires every pointer inside the graph to be stable, so the
// graph only touches plan-owned buffers: wavelet / observed data are copied into staging buffers before the
// launch, synthetics are copied out after it, and the sparse source / receiver lists keep their allocations
// (set_geometry rewrites their contents in place).
namespace {

// A device array the plan owns, `cap` elements.  ensure() is the one place that reallocates plan memory: captured graphs
// hold the old address, so every reallocation drops them.  `slack`: allocate n + n/2 + 16 elements, so that a later
// geometry of similar size reuses the array; otherwise exactly max(n, 1).
template <typename T> struct DevArray {
    T* d = nullptr;
    size_t cap = 0;
    int ensure(fwi_fd2d* p, size_t n, bool slack = false);
    void release() { if (d) cudaFree(d); d = nullptr; cap = 0; }
};

struct PointList {
    int n = 0;
    DevArray<int> tile_ptr, off, id;
    void release() { tile_ptr.release(); off.release(); id.release(); n = 0; }
    // what a kernel reads; an absent or empty list is all null, which the kernels skip
    static PointListDev dev(const PointList* pl) {
        return (pl && pl->n) ? PointListDev{pl->tile_ptr.d, pl->off.d, pl->id.d} : PointListDev{nullptr, nullptr, nullptr};
    }
};

// A sparse operator in CSR form (fd_interp_*_kernel): rows[j] sums w[e] * in[col[e]] over e in [ptr[j], ptr[j+1]).
struct Csr {
    int rows = 0;
    DevArray<int> ptr, col;
    DevArray<float> w;
    void release() { ptr.release(); col.release(); w.release(); rows = 0; }
};

// Off-grid points of one side (spec B7, fwi_fd*_set_positions): `npts` points whose taps land on the side's unique cells,
// which are what the step kernels' point lists hold.  by_point (point -> cells) gathers traces, by_cell (cell -> points)
// spreads wavelets and residuals.  npts = -1: the integer geometry is set, and a point is its cell.
struct Interp {
    int npts = -1;
    Csr by_point, by_cell;
    void release() { by_point.release(); by_cell.release(); npts = -1; }
};

// The step-kernel families: the one-step tile kernel, the two-steps-per-pass kernel (temporal blocking, "tb2") and the
// 3-D kernel.  A tb2 plan also runs the tile kernel, for the odd step of a sweep and for fwi_fd_step.
enum Family { kTile, kTb2, k3D };

// One built shape of a family: tile rows (bz / cz / by), warps per CTA, dynamic shared memory per CTA, and its kernel for
// each free-surface setting (0 off, 1 on: spec B6) and mode, indexed by STEP_FWD .. STEP_BORN (null where the family has no
// such mode).  The tables below are the only list of the shapes the library builds.
template <typename Kernel> struct StepShape {
    int rows, warps;
    size_t smem;
    Kernel fn[2][5];
};
using TileShape = StepShape<void (*)(CUtensorMap, Step2DArgs)>;
using Tb2Shape = StepShape<void (*)(CUtensorMap, CUtensorMap, CUtensorMap, Tb2Args)>;
using Fd3Shape = StepShape<void (*)(CUtensorMap, CUtensorMap, CUtensorMap, Step3DArgs)>;

constexpr int kBX = 128;
template <int BZ, int NW> TileShape tile_shape() {
    return {BZ, NW, (size_t)(kBX + 2 * kHalo) * (BZ + 2 * kHalo) * sizeof(float),
            {{fd2d_step_kernel<BZ, NW, STEP_FWD, false>, fd2d_step_kernel<BZ, NW, STEP_FWD_SAVE, false>,
              fd2d_step_kernel<BZ, NW, STEP_ADJ, false>, fd2d_step_kernel<BZ, NW, STEP_ADJ2, false>,
              fd2d_step_kernel<BZ, NW, STEP_BORN, false>},
             {fd2d_step_kernel<BZ, NW, STEP_FWD, true>, fd2d_step_kernel<BZ, NW, STEP_FWD_SAVE, true>,
              fd2d_step_kernel<BZ, NW, STEP_ADJ, true>, fd2d_step_kernel<BZ, NW, STEP_ADJ2, true>,
              fd2d_step_kernel<BZ, NW, STEP_BORN, true>}}};
}
constexpr int kTb2Warps = 8;          // (4 warps at 24 rows measured 8 % slower)
template <int CZ> Tb2Shape tb2_shape() {
    return {CZ, kTb2Warps, ((size_t)(CZ + 16) * kT2W0 + 2 * (size_t)(CZ + 8) * kT2W1) * sizeof(float),
            {{fd2d_tb2_kernel<CZ, kTb2Warps, STEP_FWD, false>, fd2d_tb2_kernel<CZ, kTb2Warps, STEP_FWD_SAVE, false>,
              fd2d_tb2_kernel<CZ, kTb2Warps, STEP_ADJ, false>, nullptr, nullptr},
             {fd2d_tb2_kernel<CZ, kTb2Warps, STEP_FWD, true>, fd2d_tb2_kernel<CZ, kTb2Warps, STEP_FWD_SAVE, true>,
              fd2d_tb2_kernel<CZ, kTb2Warps, STEP_ADJ, true>, nullptr, nullptr}}};
}
template <int BY> Fd3Shape fd3_shape() {
    return {BY, T3<BY>::Threads / 32, T3<BY>::Smem,
            {{fd3d_step_kernel<STEP_FWD, BY, false>, fd3d_step_kernel<STEP_FWD_SAVE, BY, false>,
              fd3d_step_kernel<STEP_ADJ, BY, false>, fd3d_step_kernel<STEP_ADJ2, BY, false>,
              fd3d_step_kernel<STEP_BORN, BY, false>},
             {fd3d_step_kernel<STEP_FWD, BY, true>, fd3d_step_kernel<STEP_FWD_SAVE, BY, true>,
              fd3d_step_kernel<STEP_ADJ, BY, true>, fd3d_step_kernel<STEP_ADJ2, BY, true>,
              fd3d_step_kernel<STEP_BORN, BY, true>}}};
}
// The one-step kernel is built for exactly these (rows, warps per CTA): the round-1 sweep's winner and three heights of 7 rows
// per warp among which one has tiles that fill whole waves.  pick_tile() breaks ties by this order.
// (5 and 7 warps per CTA measured 1.5x slower at 1000 x 3000)
static const TileShape kTileShapes[] = {tile_shape<32, 4>(), tile_shape<28, 4>(), tile_shape<42, 6>(), tile_shape<56, 8>()};
static const Tb2Shape kTb2Shapes[] = {tb2_shape<32>(), tb2_shape<24>()};
static const Fd3Shape kFd3Shapes[] = {fd3_shape<16>(), fd3_shape<14>()};     // the first row is the single-GPU tile height

template <typename Shape, size_t N> const Shape* find_shape(const Shape (&table)[N], int rows, int warps) {
    for (const auto& k : table)
        if (k.rows == rows && k.warps == warps) return &k;
    return nullptr;
}

// The plan's shot-level operations (fwi_fd2d_forward, _gradient, _born, _gauss_newton).
enum Op { kForward, kGradient, kBorn, kGaussNewton };

// How an operation divides its nt steps: nseg segments of seg steps, the last one possibly shorter.  Gradient and
// Gauss-Newton: checkpoint segments (nseg = 1: every snapshot is stored); Born: segments of S steps; forward: one segment.
struct Split { int seg, nseg; };

struct State { int c, o; };      // fld[] indices of u_n and u_{n-1}

struct GraphEntry {
    Op op;
    int nt, nsrc, nrec;          // cells that sources / receivers inject into / sample
    int psrc, prec;              // off-grid points (Interp::npts; -1 with the integer geometry)
    Split split;
    cudaGraphExec_t exec;
    int64_t kernels;
    State end;                   // the forward state the graph's last forward sweep leaves behind
};

}  // namespace

struct fwi_fd2d {
    int device = 0, nz = 0, ny = 1, nx = 0, px = 0, nabs = 0;   // ny == 1: 2-D plan; rows() = nz * ny
    float h = 0, dt = 0, alpha = 0;
    int tiles_y = 1, zchunk = 0, nzch = 1;                      // 3-D tiling: 128 x fd3->rows columns, z chunks
    const Fd3Shape* fd3 = kFd3Shapes;
    float* gy = nullptr;
    CUtensorMap tm3[8], tm3_old[8], tm3_m;
    // slab decomposition over peer memory (3-D only)
    int z_own0 = 0, z_own1 = 0;                 // owned planes of the local grid; 0,0 = whole grid
    void* peer_arena[2] = {nullptr, nullptr};   // IPC-opened arenas of the upper / lower neighbour
    size_t peer_fld_off[2][8] = {};             // byte offsets of the neighbours' wavefield buffers in their arenas
    size_t peer_flags_off[2] = {0, 0};
    int peer_up_z = 0;
    bool peer_ipc[2] = {false, false};          // opened with cudaIpcOpenMemHandle (else: another plan of this process)
    int* sync_area = nullptr;                   // SlabSync words (fd3d.cuh) inside the arena; the step id lives there
    int last_desc = 0;                          // the last z chunk marches downwards (slab with a lower neighbour)
    long long slab_timeout_cycles = 4000000000LL;   // bounded spin on a neighbour's flag (~2 s; FWI_SLAB_TIMEOUT_MS)
    bool peers() const { return peer_arena[0] || peer_arena[1]; }
    Family family = kTile;
    const TileShape* tile = kTileShapes;        // the one-step tile kernel's shape (2-D plans)
    int tiles_x = 0, tiles_z = 0;
    int sm_count = 148;
    CUtensorMap tb_cur[8], tb_old[8], tb_m;     // two-steps-per-pass kernel
    const Tb2Shape* tb2 = kTb2Shapes;
    int tiles_x2 = 0, tiles_z2 = 0;
    float *m = nullptr, *vp = nullptr, *gx = nullptr, *gz = nullptr;
    void* arena = nullptr;
    float* fld[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // forward 0..3, adjoint 4..7 (one-step kernels use 0/1 and 4/5)
    CUtensorMap tmap[8];
    float* acc = nullptr;
    DevArray<float> snap, ckpt, resid, syn, obs, wav;
    DevArray<float> dm;               // Born: pitched dm = (2 m / v) dv
    double* d_J = nullptr;
    PointList src, rec;
    PointList src_ext2, src_own2, rec_ext2, rec_own2;   // tb2: binned by the 120 x cz core tiles (+-4 for *_ext2)
    int nsrc = 0, nrec = 0;           // source / receiver cells: the columns of p->wav, p->syn, p->resid
    Interp isrc, irec;                // off-grid points (spec B7) over those cells
    DevArray<float> pts;              // off grid: gradient synthetics / Gauss-Newton J dv at the receivers
    DevArray<float> pres;             // off grid: the residual at the receivers
    size_t mem_limit = 0;             // 0 = automatic (fraction of free memory)
    bool pdl = true;                  // chain 2-D steps with programmatic dependent launch (FWI_PDL=0 turns it off)
    bool pdl_chain = false;           // false right after a kernel that rewrites what a step reads BEFORE its dependency wait (m)
    int split_nt = -1; Split split{0, 0}; size_t split_limit = 0;   // cached storage decision of the last gradient
    int fwd_c = 0, fwd_o = 1;         // fld[] indices of u_n and u_{n-1} after the last forward
    bool model_set = false;
    bool free_surface = false;        // spec B6: odd mirror above z = 0, no sponge on the top face (fwi_fd2d_set_free_surface)
    bool use_graphs = true;
    bool defer_imaging = true;        // tile and 3-D kernels: image two adjoint steps per accumulator update
    int64_t launches = 0;
    cudaStream_t work = nullptr;
    cudaEvent_t ev_in = nullptr, ev_out = nullptr, ev_geom = nullptr;
    bool geom_pending = false;        // set_geometry queued uploads on `work` that a caller-driven step has not yet waited for
    // pinned host staging for the point lists: three slots used in turn, so set_geometry never waits for the shot that
    // is still running (its uploads are queued behind that shot's graph) and never reads freed pageable memory
    struct Stage { int* host = nullptr; size_t cap = 0, used = 0; cudaEvent_t done = nullptr; bool busy = false; } stage[3];
    int stage_cur = 0;
    std::vector<GraphEntry> graphs;
    int rows() const { return nz * ny; }
    size_t plane() const { return (size_t)nz * ny * px; }
};

// Sponge profile (oracle/fd_oracle.py sponge_profile), float64 on the host then rounded once, padded with 1.  `free_top`
// drops the strip at index 0: a free surface is not damped (spec B6).
static std::vector<float> sponge_profile(int n, int padded, int nabs, float alpha, bool free_top) {
    std::vector<float> prof(padded, 1.0f);
    for (int i = 0; i < std::min(nabs, n); ++i) {
        const double t = (double)alpha * (nabs - i) / nabs;
        const float val = (float)std::exp(-t * t);
        if (!free_top) prof[i] = std::min(prof[i], val);
        prof[n - 1 - i] = std::min(prof[n - 1 - i], val);
    }
    return prof;
}

static void drop_graphs(fwi_fd2d* p) {
    for (auto& g : p->graphs) cudaGraphExecDestroy(g.exec);
    p->graphs.clear();
}

template <typename T> int DevArray<T>::ensure(fwi_fd2d* p, size_t n, bool slack) {
    if (d && n <= cap) return FWI_OK;
    release();
    drop_graphs(p);
    const size_t want = slack ? n + n / 2 + 16 : std::max<size_t>(n, 1);
    FWI_CUDA(cudaMalloc(&d, want * sizeof(T)));
    cap = want;
    return FWI_OK;
}

static void clear_geometry(fwi_fd2d* p) {
    drop_graphs(p);                   // they hold the addresses of the lists released here
    p->src.release(); p->rec.release();
    p->src_ext2.release(); p->src_own2.release(); p->rec_ext2.release(); p->rec_own2.release();
    p->isrc.release(); p->irec.release();
    p->nsrc = p->nrec = 0;
}

// Receivers as the caller sees them: traces, observed data and residuals have this many columns.
static int rec_points(const fwi_fd2d* p) { return p->irec.npts >= 0 ? p->irec.npts : p->nrec; }

static int make_tmaps3(fwi_fd2d* p) {
    p->tiles_x = (p->nx + k3BX - 1) / k3BX;
    // Tile height and z chunks.  One CTA per SM is resident (170 KB of plane rings) and every chunk re-reads 8 halo planes;
    // for a tile height BY and a chunk count the model cost is  waves x (planes per chunk + 8) x BY.  Single-GPU plans keep
    // BY = 16 (0.96 of the HBM roofline at 512^3); peer-memory slabs, whose few chunks make the last wave's tail expensive,
    // take the cheaper of 16 and 14 (512-wide planes: 4 x 37 = 148 tiles of 14 rows, one per SM).  FWI_FD3D_BY overrides.
    {
        const int nzo = (p->z_own1 > 0 ? p->z_own1 : p->nz) - p->z_own0;
        // peer-memory slabs: with a lower neighbour and two or more chunks the last chunk marches downwards, so that both
        // boundaries are pushed early; a 4-plane boundary must not straddle two chunks
        // (measured on 8 GPUs, 64 planes per rank, us per launch: one chunk 93.0 / 95.7 with 14- / 16-row tiles, two chunks
        // 97.9 / 100.1 - a single chunk re-reads 8 instead of 16 halo planes, which outweighs pushing the lower boundary
        // at the end of the launch; the model charges that late push 3 %; 4 GPUs, 128 planes per rank: 152.4 vs 157.2 us)
        int force_by = 0;
        if (const char* e = getenv("FWI_FD3D_BY")) force_by = atoi(e);
        const Fd3Shape* best_k = kFd3Shapes;
        int best = 1;
        double best_cost = 1e300;
        for (const auto& k : kFd3Shapes) {
            if (force_by ? k.rows != force_by : (&k != kFd3Shapes && !p->peers())) continue;
            const int txy = p->tiles_x * ((p->ny + k.rows - 1) / k.rows);
            for (int nzch = 1; nzch <= std::max(1, nzo / 8); ++nzch) {
                const int zc = (nzo + nzch - 1) / nzch;
                const int real = (nzo + zc - 1) / zc;
                if (p->peers() && nzo - (real - 1) * zc < kHalo) continue;
                const double waves = std::ceil((double)txy * real / p->sm_count);
                const double late_push = (p->peer_arena[1] && real == 1) ? 1.03 : 1.0;
                const double cost = waves * (zc + 2 * kHalo) * k.rows * late_push;
                if (cost < best_cost - 1e-9) { best_cost = cost; best = nzch; best_k = &k; }
            }
        }
        p->fd3 = best_k;
        p->tiles_y = (p->ny + p->fd3->rows - 1) / p->fd3->rows;
        p->zchunk = (nzo + best - 1) / best;
        p->nzch = (nzo + p->zchunk - 1) / p->zchunk;
        p->last_desc = (p->peer_arena[1] && p->nzch >= 2) ? 1 : 0;   // (never the chunk at z = 0, see fd3d_step_kernel FS)
    }
    for (int i = 0; i < 8; ++i) {
        const uint64_t dims[3] = {(uint64_t)p->nx, (uint64_t)p->ny, (uint64_t)p->nz};
        const uint64_t strides[2] = {(uint64_t)p->px * sizeof(float), (uint64_t)p->px * p->ny * sizeof(float)};
        const uint32_t box[3] = {(uint32_t)k3SX, (uint32_t)(p->fd3->rows + 2 * kHalo), 1u};
        int rc = encode_tiled_f32(&p->tm3[i], p->fld[i], 3, dims, strides, box);
        if (rc) return rc;
        const uint64_t dims_p[3] = {(uint64_t)p->px, (uint64_t)p->ny, (uint64_t)p->nz};
        const uint32_t box_o[3] = {(uint32_t)k3BX, (uint32_t)p->fd3->rows, 1u};
        rc = encode_tiled_f32(&p->tm3_old[i], p->fld[i], 3, dims_p, strides, box_o);
        if (rc) return rc;
        if (i == 0 && (rc = encode_tiled_f32(&p->tm3_m, p->m, 3, dims_p, strides, box_o))) return rc;
    }
    return FWI_OK;
}

static int make_tmaps(fwi_fd2d* p) {
    if (p->family == k3D) return make_tmaps3(p);
    const int cz = p->tb2->rows;
    p->tiles_x2 = (p->nx + kT2CX - 1) / kT2CX;
    p->tiles_z2 = (p->nz + cz - 1) / cz;
    {
        const uint64_t dims[2] = {(uint64_t)p->nx, (uint64_t)p->nz};
        const uint64_t dims_p[2] = {(uint64_t)p->px, (uint64_t)p->nz};
        const uint64_t strides[1] = {(uint64_t)p->px * sizeof(float)};
        const uint32_t box_c[2] = {(uint32_t)kT2W0, (uint32_t)(cz + 16)}, box_o[2] = {(uint32_t)kT2W1, (uint32_t)(cz + 8)};
        for (int i = 0; i < 8; ++i) {
            int rc = encode_tiled_f32(&p->tb_cur[i], p->fld[i], 2, dims, strides, box_c);
            if (rc) return rc;
            rc = encode_tiled_f32(&p->tb_old[i], p->fld[i], 2, dims_p, strides, box_o);
            if (rc) return rc;
        }
        int rc = encode_tiled_f32(&p->tb_m, p->m, 2, dims_p, strides, box_o);
        if (rc) return rc;
    }
    for (int i = 0; i < 8; ++i) {
        const uint64_t dims[2] = {(uint64_t)p->nx, (uint64_t)p->nz};
        const uint64_t strides[1] = {(uint64_t)p->px * sizeof(float)};
        const uint32_t box[2] = {(uint32_t)(kBX + 2 * kHalo), (uint32_t)(p->tile->rows + 2 * kHalo)};
        int rc = encode_tiled_f32(&p->tmap[i], p->fld[i], 2, dims, strides, box);
        if (rc) return rc;
    }
    return FWI_OK;
}

// ---- pinned staging of the point lists ---------------------------------------------------------------------------
static int stage_begin(fwi_fd2d* p, size_t need_ints) {
    p->stage_cur = (p->stage_cur + 1) % 3;
    auto& sl = p->stage[p->stage_cur];
    if (!sl.done) FWI_CUDA(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    if (sl.busy) { FWI_CUDA(cudaEventSynchronize(sl.done)); sl.busy = false; }      // uploads of three set_geometry calls ago
    if (sl.cap < need_ints) {
        if (sl.host) cudaFreeHost(sl.host);
        sl.host = nullptr; sl.cap = 0;
        const size_t cap = need_ints + need_ints / 2 + 1024;
        FWI_CUDA(cudaMallocHost(&sl.host, cap * sizeof(int)));
        sl.cap = cap;
    }
    sl.used = 0;
    return FWI_OK;
}
// Ensures `a` holds v.size() elements and queues their upload through the slot stage_begin sized (floats travel through
// the int slot bit for bit).  Contents are rewritten in place on the work stream, ordered after the previous shot's graph.
template <typename T> static int stage_upload(fwi_fd2d* p, DevArray<T>& a, const std::vector<T>& v, bool slack) {
    static_assert(sizeof(T) == sizeof(int), "the staging slots hold 4-byte words");
    int rc = a.ensure(p, v.size(), slack);
    if (rc || v.empty()) return rc;
    auto& sl = p->stage[p->stage_cur];
    int* h = sl.host + sl.used;
    memcpy(h, v.data(), v.size() * sizeof(T));
    sl.used += v.size();
    FWI_CUDA(cudaMemcpyAsync(a.d, h, v.size() * sizeof(T), cudaMemcpyHostToDevice, p->work));
    return FWI_OK;
}
static int stage_end(fwi_fd2d* p) {
    auto& sl = p->stage[p->stage_cur];
    FWI_CUDA(cudaEventRecord(sl.done, p->work));
    sl.busy = true;
    FWI_CUDA(cudaEventRecord(p->ev_geom, p->work));
    p->geom_pending = true;
    return FWI_OK;
}

// Bins points by the CTA tiles of a kernel family: (z, y, x) tile size and count, and the first plane of the z tiles (the
// 3-D kernel's z chunks start at the slab's first owned plane).  Bin (tz, ty, tx) is the CTA (tx, ty, tz) of the launch.
struct TileGrid { int size[3], count[3], z0; };

static TileGrid tile_grid(const fwi_fd2d* p, Family f) {
    if (f == k3D) return {{p->zchunk, p->fd3->rows, k3BX}, {p->nzch, p->tiles_y, p->tiles_x}, p->z_own0};
    if (f == kTb2) return {{p->tb2->rows, 1, kT2CX}, {p->tiles_z2, 1, p->tiles_x2}, 0};
    return {{p->tile->rows, 1, kBX}, {p->tiles_z, 1, p->tiles_x}, 0};
}

static int check_points(const fwi_fd2d* p, int n, const int* iz, const int* iy, const int* ix, const char* what) {
    const int z_own1 = p->z_own1 > 0 ? p->z_own1 : p->nz;
    for (int i = 0; i < n; ++i) {
        const int yy = iy ? iy[i] : 0;
        FWI_REQUIRE(iz[i] >= 0 && iz[i] < p->nz && ix[i] >= 0 && ix[i] < p->nx && yy >= 0 && yy < p->ny, "%s %d at (z=%d, y=%d, x=%d) is outside the %d x %d x %d grid", what, i, iz[i], yy, ix[i], p->nz, p->ny, p->nx);
        // a slab computes only its owned planes; the neighbours overwrite the ghost planes
        FWI_REQUIRE(iz[i] >= p->z_own0 && iz[i] < z_own1, "%s %d at z=%d is outside the planes [%d, %d) this slab owns", what, i, iz[i], p->z_own0, z_own1);
        // the free surface holds p = 0: a point on it would inject into, or record, a row that stays 0
        FWI_REQUIRE(!p->free_surface || iz[i] >= 1, "%s %d at (z=%d, y=%d, x=%d) lies on the free surface; sources and receivers need z >= 1", what, i, iz[i], yy, ix[i]);
    }
    return FWI_OK;
}

struct HostList { std::vector<int> tile_ptr, off, id; };

// Lists each (checked) point in every tile whose core widened by `reach` on each side holds it: reach 0 gives the single
// owning tile, kHalo the tb2 kernel's extended list.  A counting sort keeps the points of a bin in input order.
static void bin_points(const fwi_fd2d* p, const TileGrid& g, int reach, int n, const int* iz, const int* iy, const int* ix,
                       HostList& out) {
    const int nbins = g.count[0] * g.count[1] * g.count[2];
    std::vector<int>& tile_ptr = out.tile_ptr;
    tile_ptr.assign(nbins + 1, 0);
    std::vector<std::pair<int, int>> hits;      // (bin, point) in input order
    hits.reserve(n);
    for (int i = 0; i < n; ++i) {
        const int c[3] = {iz[i] - g.z0, iy ? iy[i] : 0, ix[i]};
        int lo[3], hi[3];
        for (int d = 0; d < 3; ++d) {
            lo[d] = std::max(0, (c[d] - reach) / g.size[d]);
            hi[d] = std::min(g.count[d] - 1, (c[d] + reach) / g.size[d]);
        }
        for (int tz = lo[0]; tz <= hi[0]; ++tz)
            for (int ty = lo[1]; ty <= hi[1]; ++ty)
                for (int tx = lo[2]; tx <= hi[2]; ++tx) {
                    const int b = (tz * g.count[1] + ty) * g.count[2] + tx;
                    hits.push_back({b, i});
                    tile_ptr[b + 1]++;
                }
    }
    for (int t = 0; t < nbins; ++t) tile_ptr[t + 1] += tile_ptr[t];
    std::vector<int> fill(tile_ptr.begin(), tile_ptr.end() - 1);
    out.off.resize(tile_ptr[nbins]);
    out.id.resize(tile_ptr[nbins]);
    for (const auto& h : hits) {
        const int i = h.second, e = fill[h.first]++;
        out.off[e] = (iz[i] * p->ny + (iy ? iy[i] : 0)) * p->px + ix[i];
        out.id[e] = i;
    }
}

// Launches the kernel of `mode` of a step-kernel shape, its free-surface instance when `fs`.  With `pdl` it is chained to
// the previous kernel on the stream by a programmatic edge (also inside captured graphs) and orders itself behind its
// predecessor with griddepcontrol.wait.
template <typename Kernel, typename... Args>
static int launch_shape(const StepShape<Kernel>& k, int mode, bool fs, dim3 grid, bool pdl, cudaStream_t st, const Args&... args) {
    FWI_REQUIRE(k.fn[fs][mode], "fd2d: the %d-row kernel has no step mode %d", k.rows, mode);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = dim3(k.warps * 32); cfg.dynamicSmemBytes = k.smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    FWI_CUDA(cudaLaunchKernelEx(&cfg, k.fn[fs][mode], args...));
    return FWI_OK;
}

static int launch_step(fwi_fd2d* p, int mode, int cur, float* oldnew, const PointList* inj, const float* inj_vals,
                       const PointList* rec, float* rec_out, float* snap, cudaStream_t st, const float* snap_prev = nullptr) {
    p->launches++;
    if (p->family != k3D) {
        Step2DArgs a{};
        a.oldnew = oldnew; a.m = p->m; a.gx = p->gx; a.gz = p->gz; a.snap = snap; a.acc = p->acc; a.snap_prev = snap_prev;
        a.nx = p->nx; a.nz = p->nz; a.px = p->px;
        a.inj = PointList::dev(inj);
        a.inj_vals = inj_vals;
        a.rec = PointList::dev(rec);
        a.rec_out = rec_out;
        a.dm = p->dm.d;
        const bool pdl = p->pdl && p->pdl_chain;
        p->pdl_chain = true;
        return launch_shape(*p->tile, mode, p->free_surface, dim3(p->tiles_x, p->tiles_z), pdl, st, p->tmap[cur], a);
    }
    Step3DArgs a{};
    a.oldnew = oldnew; a.m = p->m; a.gx = p->gx; a.gy = p->gy; a.gz = p->gz; a.snap = snap; a.acc = p->acc; a.snap_prev = snap_prev;
    a.nx = p->nx; a.ny = p->ny; a.nz = p->nz; a.px = p->px; a.zchunk = p->zchunk;
    a.inj = PointList::dev(inj);
    a.inj_vals = inj_vals;
    a.rec = PointList::dev(rec);
    a.rec_out = rec_out;
    a.z_own0 = p->z_own0; a.z_own1 = p->z_own1 > 0 ? p->z_own1 : p->nz;
    int oi = -1;
    for (int i = 0; i < 8; ++i) if (p->fld[i] == oldnew) oi = i;
    FWI_REQUIRE(oi >= 0, "fd3d: output buffer is not one of the plan's wavefields");
    a.last_desc = p->last_desc;
    a.peer_up = p->peer_arena[0] ? (float*)((char*)p->peer_arena[0] + p->peer_fld_off[0][oi]) : nullptr;
    a.peer_dn = p->peer_arena[1] ? (float*)((char*)p->peer_arena[1] + p->peer_fld_off[1][oi]) : nullptr;
    a.peer_up_z = p->peer_up_z;
    a.sync = p->sync_area;
    a.flag_peer_up = p->peer_arena[0] ? (int*)((char*)p->peer_arena[0] + p->peer_flags_off[0]) + kSyncFlagDn : nullptr;   // I am its lower neighbour
    a.flag_peer_dn = p->peer_arena[1] ? (int*)((char*)p->peer_arena[1] + p->peer_flags_off[1]) + kSyncFlagUp : nullptr;   // I am its upper neighbour
    a.timeout_cycles = p->slab_timeout_cycles;
    a.dm = p->dm.d;
    // (programmatic dependent launch was measured on this kernel too: 2 % at 128^3, nothing from 256^3 up - not used)
    return launch_shape(*p->fd3, mode, p->free_surface, dim3(p->tiles_x, p->tiles_y, p->nzch), false, st, p->tm3[cur], p->tm3_old[oi], p->tm3_m, a);
}

static void other_two(const State& s, int base, int& a, int& b) {
    int f[2], k = 0;
    for (int i = base; i < base + 4 && k < 2; ++i) if (i != s.c && i != s.o) f[k++] = i;
    a = f[0]; b = f[1];
}

static int launch_tb2(fwi_fd2d* p, int mode, const State& s, int jc, int jd, const PointList* inj_ext, const PointList* inj_own,
                      const float* inj1, const float* inj2, const PointList* rec, float* rec1, float* rec2, float* snap1, float* snap2,
                      cudaStream_t st) {
    p->launches++;
    Tb2Args a{};
    a.out_new = p->fld[jc]; a.out_mid = p->fld[jd]; a.gx = p->gx; a.gz = p->gz; a.m = p->m; a.snap1 = snap1; a.snap2 = snap2; a.acc = p->acc;
    a.nx = p->nx; a.nz = p->nz; a.px = p->px;
    a.inj_ext = PointList::dev(inj_ext);
    a.inj_own = PointList::dev(inj_own);
    a.inj1 = inj1; a.inj2 = inj2;
    a.rec = PointList::dev(rec);
    a.rec1 = rec1; a.rec2 = rec2;
    const bool pdl = p->pdl && p->pdl_chain;      // the pass loads m before its dependency wait
    p->pdl_chain = true;
    return launch_shape(*p->tb2, mode, p->free_surface, dim3(p->tiles_x2, p->tiles_z2), pdl, st, p->tb_cur[s.c], p->tb_old[s.o], p->tb_m, a);
}

// forward time loop over steps [n0, n1); `s` holds the fld[] indices of (u_n, u_{n-1}) on entry and on return
static int run_forward(fwi_fd2d* p, const float* wavelet, int n0, int n1, float* traces, bool save, size_t snap_base,
                       State& s, cudaStream_t st) {
    const size_t pl = p->plane();
    p->pdl_chain = false;             // (segment of) a sweep starts behind memsets / checkpoint copies: full dependency
    int n = n0;
    if (p->family == kTb2) {
        for (; n + 1 < n1; n += 2) {
            int jc, jd;
            other_two(s, 0, jc, jd);
            float* s1 = save ? p->snap.d + (size_t)(n - snap_base) * pl : nullptr;
            int rc = launch_tb2(p, save ? STEP_FWD_SAVE : STEP_FWD, s, jc, jd, &p->src_ext2, &p->src_own2, wavelet + (size_t)n * p->nsrc,
                                wavelet + (size_t)(n + 1) * p->nsrc, traces ? &p->rec_own2 : nullptr,
                                traces ? traces + (size_t)n * p->nrec : nullptr, traces ? traces + (size_t)(n + 1) * p->nrec : nullptr,
                                s1, save ? s1 + pl : nullptr, st);
            if (rc) return rc;
            s = State{jc, jd};
        }
    }
    // a leftover single step behind a two-steps-per-pass launch reads u_{n-1} written by that very pass: no chaining
    if (p->family == kTb2) p->pdl_chain = false;
    for (; n < n1; ++n) {
        float* snap = save ? p->snap.d + (size_t)(n - snap_base) * pl : nullptr;
        int rc = launch_step(p, save ? STEP_FWD_SAVE : STEP_FWD, s.c, p->fld[s.o], &p->src, wavelet + (size_t)n * p->nsrc,
                             traces ? &p->rec : nullptr, traces ? traces + (size_t)n * p->nrec : nullptr, snap, st);
        if (rc) return rc;
        s = State{s.o, s.c};
    }
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

// adjoint steps for trace rows n1-1 down to n0 (fields fld[4..7])
static int run_adjoint(fwi_fd2d* p, const float* resid, int n0, int n1, size_t snap_base, State& s, cudaStream_t st) {
    const size_t pl = p->plane();
    p->pdl_chain = false;             // first adjoint step follows the residual kernel and the field memsets
    int n = n1 - 1;
    if (p->family == kTb2) {
        for (; n - 1 >= n0; n -= 2) {
            int jc, jd;
            other_two(s, 4, jc, jd);
            int rc = launch_tb2(p, STEP_ADJ, s, jc, jd, &p->rec_ext2, &p->rec_own2, resid + (size_t)n * p->nrec, resid + (size_t)(n - 1) * p->nrec,
                                nullptr, nullptr, nullptr, p->snap.d + (size_t)(n - snap_base) * pl, p->snap.d + (size_t)(n - 1 - snap_base) * pl, st);
            if (rc) return rc;
            s = State{jc, jd};
        }
    }
    if (p->family != kTb2 && p->defer_imaging) {
        // deferred imaging: the first step of a pair only propagates (17 B/pt of traffic instead of 29), the second one
        // images both fields, touching the accumulator once per two steps
        for (; n - 1 >= n0; n -= 2) {
            int rc = launch_step(p, STEP_FWD, s.c, p->fld[s.o], &p->rec, resid + (size_t)n * p->nrec, nullptr, nullptr, nullptr, st);
            if (rc) return rc;
            s = State{s.o, s.c};
            rc = launch_step(p, STEP_ADJ2, s.c, p->fld[s.o], &p->rec, resid + (size_t)(n - 1) * p->nrec, nullptr, nullptr,
                             p->snap.d + (size_t)(n - 1 - snap_base) * pl, st, p->snap.d + (size_t)(n - snap_base) * pl);
            if (rc) return rc;
            s = State{s.o, s.c};
        }
    }
    if (p->family == kTb2) p->pdl_chain = false;          // see run_forward: leftover step behind a two-step pass
    for (; n >= n0; --n) {
        int rc = launch_step(p, STEP_ADJ, s.c, p->fld[s.o], &p->rec, resid + (size_t)n * p->nrec, nullptr, nullptr,
                             p->snap.d + (size_t)(n - snap_base) * pl, st);
        if (rc) return rc;
        s = State{s.o, s.c};
    }
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

// scattered (Born) steps [n0, n1) on fld[4..5], one-step kernel in every 2-D family: dm * w_n is the source term, w_n the
// snapshot the background sweep of the same steps saved at n - snap_base; no injection, receivers sample du_{n+1}.
// The first launch may be chained to the background sweep: before its dependency wait a Born step reads only du_{n-1} and
// m, which that sweep does not write.
static int run_born(fwi_fd2d* p, int n0, int n1, size_t snap_base, State& s, float* traces, cudaStream_t st) {
    const size_t pl = p->plane();
    for (int n = n0; n < n1; ++n) {
        int rc = launch_step(p, STEP_BORN, s.c, p->fld[s.o], nullptr, nullptr, &p->rec, traces + (size_t)n * p->nrec,
                             p->snap.d + (size_t)(n - snap_base) * pl, st);
        if (rc) return rc;
        s = State{s.o, s.c};
    }
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

// Off-grid points (spec B7): out (nt, op.rows) = in (nt, nin) through the CSR operator `op`, gathering (cells -> points)
// or spreading (points -> cells).
static int launch_interp(fwi_fd2d* p, bool gather, const Csr& op, const float* in, int nin, float* out, int nt, cudaStream_t st) {
    if (!op.rows || nt < 1) return FWI_OK;
    const dim3 grid((op.rows + 127) / 128, std::min((nt + kInterpRows - 1) / kInterpRows, 65535));
    if (gather) fd_interp_gather_kernel<<<grid, 128, 0, st>>>(op.ptr.d, op.col.d, op.w.d, in, nin, out, op.rows, nt);
    else fd_interp_spread_kernel<<<grid, 128, 0, st>>>(op.ptr.d, op.col.d, op.w.d, in, nin, out, op.rows, nt);
    FWI_CUDA(cudaGetLastError());
    p->launches += 1;
    return FWI_OK;
}

// ---- peer-memory slabs: what may be overwritten when ---------------------------------------------------------------
// A neighbour stores its boundary planes of launch k into THIS GPU's ghost planes of the buffer launch k writes.  Before a
// run (or a checkpointed segment) rewrites wavefields, a one-thread kernel waits until the neighbours have pushed
// everything up to the current step id, so no late push of the previous sweep lands on freshly written planes; and the
// ghost planes of the buffer that holds u_{n-1} are never written locally, because the neighbours' FIRST launch of the
// new sweep pushes into exactly those planes and may run ahead of this GPU's memset / restore.
static int slab_fence(fwi_fd2d* p, cudaStream_t st) {
    if (!p->peers()) return FWI_OK;
    fd3d_slab_sync_kernel<<<1, 32, 0, st>>>(p->sync_area, p->peer_arena[0] != nullptr, p->peer_arena[1] != nullptr, p->slab_timeout_cycles);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}
static void own_range(const fwi_fd2d* p, size_t& off, size_t& n) {      // floats of the planes a rank may write itself
    if (p->peers()) { off = (size_t)p->z_own0 * p->ny * p->px; n = (size_t)(p->z_own1 - p->z_own0) * p->ny * p->px; }
    else { off = 0; n = p->plane(); }
}
static int zero_state(fwi_fd2d* p, int cur, int old, cudaStream_t st) {
    int rc = slab_fence(p, st);
    if (rc) return rc;
    size_t off, n;
    own_range(p, off, n);
    FWI_CUDA(cudaMemsetAsync(p->fld[cur], 0, p->plane() * sizeof(float), st));
    FWI_CUDA(cudaMemsetAsync(p->fld[old] + off, 0, n * sizeof(float), st));
    return FWI_OK;
}
static int restore_state(fwi_fd2d* p, const State& c, const float* ck_cur, const float* ck_old, cudaStream_t st) {
    int rc = slab_fence(p, st);
    if (rc) return rc;
    size_t off, n;
    own_range(p, off, n);
    FWI_CUDA(cudaMemcpyAsync(p->fld[c.c], ck_cur, p->plane() * sizeof(float), cudaMemcpyDeviceToDevice, st));
    FWI_CUDA(cudaMemcpyAsync(p->fld[c.o] + off, ck_old + off, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return FWI_OK;
}

// The forward pass as a sequence of stream operations on `st` (captured into a graph or run directly).  Each record_*
// leaves in `fs` the forward state after the last forward sweep it records.
static int record_forward(fwi_fd2d* p, int nt, cudaStream_t st, State& fs) {
    int rc = zero_state(p, 0, 1, st);
    if (rc) return rc;
    fs = State{0, 1};
    return run_forward(p, p->wav.d, 0, nt, p->nrec ? p->syn.d : nullptr, false, 0, fs, st);
}

// Born modelling of one shot: per segment of S steps the background forward saves its S snapshots (traces -> p->syn)
// and the scattered sweep over the same steps consumes them (traces -> p->resid).  Both states carry over from one
// segment to the next, so no checkpoints are needed and S changes no result.
static int record_born(fwi_fd2d* p, int nt, int S, cudaStream_t st, State& fs) {
    int rc = zero_state(p, 0, 1, st);
    if (rc || (rc = zero_state(p, 4, 5, st))) return rc;
    fs = State{0, 1};
    State bs{4, 5};
    for (int n0 = 0; n0 < nt; n0 += S) {
        const int n1 = std::min(nt, n0 + S);
        if ((rc = run_forward(p, p->wav.d, n0, n1, p->syn.d, true, n0, fs, st))) return rc;
        if ((rc = run_born(p, n0, n1, n0, bs, p->resid.d, st))) return rc;
    }
    return FWI_OK;
}

// The gradient of one shot as a sequence of stream operations on `st`: forward (+ snapshots or checkpoints),
// residual, adjoint with imaging.  Reads p->wav / p->obs, leaves synthetics in p->syn, I in p->acc, J in p->d_J.
// gauss_newton: every forward segment (or the single full forward) saves its snapshots and is followed by the Born
// sweep over it, which writes J dv into p->resid in place of the residual; the adjoint then images J^T J dv.
// With checkpoints, the last forward sweep is the recompute of the first segment.
static int record_gradient(fwi_fd2d* p, int nt, int seg, int nseg, cudaStream_t st, State& fs, bool gauss_newton) {
    const size_t pl = p->plane();
    const size_t ntr = (size_t)nt * p->nrec;
    int rc = zero_state(p, 0, 1, st);
    if (rc) return rc;
    fs = State{0, 1};
    State bs{4, 5};
    std::vector<State> seg_state(nseg, fs);
    if (gauss_newton && (rc = zero_state(p, 4, 5, st))) return rc;
    if (nseg == 1) {
        rc = run_forward(p, p->wav.d, 0, nt, p->nrec ? p->syn.d : nullptr, true, 0, fs, st);
        if (rc) return rc;
        if (gauss_newton && (rc = run_born(p, 0, nt, 0, bs, p->resid.d, st))) return rc;
    } else {
        for (int s = 0; s < nseg; ++s) {
            if ((rc = slab_fence(p, st))) return rc;       // the ghost planes of u_n must have arrived before they are saved
            FWI_CUDA(cudaMemcpyAsync(p->ckpt.d + (size_t)(2 * s) * pl, p->fld[fs.c], pl * sizeof(float), cudaMemcpyDeviceToDevice, st));
            FWI_CUDA(cudaMemcpyAsync(p->ckpt.d + (size_t)(2 * s + 1) * pl, p->fld[fs.o], pl * sizeof(float), cudaMemcpyDeviceToDevice, st));
            seg_state[s] = fs;
            const int n0 = s * seg, n1 = std::min(nt, (s + 1) * seg);
            rc = run_forward(p, p->wav.d, n0, n1, p->nrec ? p->syn.d : nullptr, gauss_newton, n0, fs, st);
            if (rc) return rc;
            if (gauss_newton && (rc = run_born(p, n0, n1, n0, bs, p->resid.d, st))) return rc;
        }
    }
    FWI_CUDA(cudaMemsetAsync(p->d_J, 0, sizeof(double), st));
    if (p->irec.npts >= 0) {
        // off grid (spec B7): the misfit lives at the receivers and the adjoint sources are W^T r at the cells.  Gather the
        // synthetics (Gauss-Newton: J dv), take the residual there, spread it (J dv) back into p->resid.
        const int np = p->irec.npts;
        const size_t ntp = (size_t)nt * np;
        if ((rc = launch_interp(p, true, p->irec.by_point, gauss_newton ? p->resid.d : p->syn.d, p->nrec, p->pts.d, nt, st))) return rc;
        if (ntp && !gauss_newton) {
            fd_residual_kernel<<<(unsigned)std::min<size_t>(1024, (ntp + 255) / 256), 256, 0, st>>>(p->pts.d, p->obs.d, (int64_t)ntp, p->pres.d, p->d_J);
            FWI_CUDA(cudaGetLastError());
            p->launches += 1;
        }
        if ((rc = launch_interp(p, false, p->irec.by_cell, gauss_newton ? p->pts.d : p->pres.d, np, p->resid.d, nt, st))) return rc;
    } else if (ntr && !gauss_newton) {
        fd_residual_kernel<<<(unsigned)std::min<size_t>(1024, (ntr + 255) / 256), 256, 0, st>>>(p->syn.d, p->obs.d, (int64_t)ntr, p->resid.d, p->d_J);
        FWI_CUDA(cudaGetLastError());
        p->launches += 1;
    }
    if ((rc = zero_state(p, 4, 5, st))) return rc;
    FWI_CUDA(cudaMemsetAsync(p->acc, 0, pl * sizeof(float), st));
    State as{4, 5};
    if (nseg == 1) {
        rc = run_adjoint(p, p->resid.d, 0, nt, 0, as, st);
        if (rc) return rc;
    } else {
        for (int s = nseg - 1; s >= 0; --s) {
            const int n0 = s * seg, n1 = std::min(nt, (s + 1) * seg);
            fs = seg_state[s];
            if ((rc = restore_state(p, fs, p->ckpt.d + (size_t)(2 * s) * pl, p->ckpt.d + (size_t)(2 * s + 1) * pl, st))) return rc;
            rc = run_forward(p, p->wav.d, n0, n1, nullptr, true, n0, fs, st);     // recompute w_n for this segment
            if (rc) return rc;
            rc = run_adjoint(p, p->resid.d, n0, n1, n0, as, st);
            if (rc) return rc;
        }
    }
    return FWI_OK;
}

static int record(fwi_fd2d* p, Op op, int nt, const Split& split, cudaStream_t st, State& fs) {
    if (op == kForward) return record_forward(p, nt, st, fs);
    if (op == kBorn) return record_born(p, nt, split.seg, st, fs);
    return record_gradient(p, nt, split.seg, split.nseg, st, fs, op == kGaussNewton);
}

// Cached graph of a time loop, keyed by (op, nt, cells and off-grid points of both sides, split); captured and instantiated on first use.
static int get_graph(fwi_fd2d* p, Op op, int nt, const Split& split, GraphEntry** out) {
    for (auto& g : p->graphs)
        if (g.op == op && g.nt == nt && g.nsrc == p->nsrc && g.nrec == p->nrec && g.psrc == p->isrc.npts && g.prec == p->irec.npts && g.split.seg == split.seg && g.split.nseg == split.nseg) { *out = &g; return FWI_OK; }
    cudaGraph_t graph = nullptr;
    FWI_CUDA(cudaStreamBeginCapture(p->work, cudaStreamCaptureModeThreadLocal));
    const int64_t l0 = p->launches;
    State end{0, 1};
    int rc = record(p, op, nt, split, p->work, end);
    cudaError_t e = cudaStreamEndCapture(p->work, &graph);
    const int64_t kernels = p->launches - l0;
    p->launches = l0;
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess) { set_error("stream capture failed: %s", cudaGetErrorString(e)); return FWI_ECUDA; }
    cudaGraphExec_t exec = nullptr;
    e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) { set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(e)); return FWI_ECUDA; }
    if (p->graphs.size() >= 6) { cudaGraphExecDestroy(p->graphs.front().exec); p->graphs.erase(p->graphs.begin()); }
    p->graphs.push_back(GraphEntry{op, nt, p->nsrc, p->nrec, p->isrc.npts, p->irec.npts, split, exec, kernels, end});
    *out = &p->graphs.back();
    return FWI_OK;
}

// Run an operation's time loop either directly on the work stream or as a cached graph, and note which buffers then
// hold u_n and u_{n-1} of its last forward sweep.
static int run_cached(fwi_fd2d* p, Op op, int nt, const Split& split) {
    p->pdl_chain = false;             // the first step of a sweep follows memsets / copies / foreign kernels: full dependency
    State end{0, 1};
    int rc;
    if (!p->use_graphs) {
        if ((rc = record(p, op, nt, split, p->work, end))) return rc;
    } else {
        GraphEntry* g = nullptr;
        if ((rc = get_graph(p, op, nt, split, &g))) return rc;
        FWI_CUDA(cudaGraphLaunch(g->exec, p->work));
        p->launches += g->kernels;
        end = g->end;
    }
    p->fwd_c = end.c; p->fwd_o = end.o;
    return FWI_OK;
}

static int enter(fwi_fd2d* p, cudaStream_t user) {       // work stream waits for everything queued on the caller's
    FWI_CUDA(cudaEventRecord(p->ev_in, user));
    FWI_CUDA(cudaStreamWaitEvent(p->work, p->ev_in, 0));
    return FWI_OK;
}
static int leave(fwi_fd2d* p, cudaStream_t user) {       // ... and the caller's stream waits for the work stream
    FWI_CUDA(cudaEventRecord(p->ev_out, p->work));
    FWI_CUDA(cudaStreamWaitEvent(user, p->ev_out, 0));
    return FWI_OK;
}

template <typename Shape, size_t N> static int allow_smem(const Shape (&table)[N]) {
    for (const auto& k : table)
        for (const auto& row : k.fn)
            for (auto fn : row)
                if (fn) FWI_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem));
    return FWI_OK;
}

extern "C" {

static int init_plan(fwi_fd2d* p, int device, int nz, int ny, int nx, float h, float dt, int nabs, float alpha);
extern "C" int fwi_fd2d_destroy(fwi_fd2d* p);

static int create_plan(int device, int nz, int ny, int nx, float h, float dt, int nabs, float alpha, fwi_fd2d** out) {
    FWI_REQUIRE(out != nullptr, "fwi_fd_create: out is NULL");
    FWI_REQUIRE(nz >= 1 && nx >= 1 && ny >= 1, "fwi_fd_create: grid must be at least 1 x 1 (got %d x %d x %d)", nz, ny, nx);
    FWI_REQUIRE((int64_t)nz * ny * ((nx + 31) & ~31) < (int64_t)2147483647, "fwi_fd_create: grid too large for 32-bit point offsets");
    FWI_REQUIRE(h > 0.f && dt > 0.f, "fwi_fd2d_create: h and dt must be positive");
    FWI_REQUIRE(nabs >= 0 && alpha >= 0.f, "fwi_fd2d_create: nabs and alpha must be non-negative");
    int ndev = 0;
    FWI_CUDA(cudaGetDeviceCount(&ndev));
    FWI_REQUIRE(device >= 0 && device < ndev, "fwi_fd2d_create: device %d out of range (%d visible)", device, ndev);
    DeviceGuard g(device);
    auto* p = new fwi_fd2d();
    p->family = ny > 1 ? k3D : kTile;
    const int rc = init_plan(p, device, nz, ny, nx, h, dt, nabs, alpha);
    if (rc) { fwi_fd2d_destroy(p); return rc; }          // nothing half-built leaks
    *out = p;
    return FWI_OK;
}

static int init_plan(fwi_fd2d* p, int device, int nz, int ny, int nx, float h, float dt, int nabs, float alpha) {
    p->device = device; p->nz = nz; p->ny = ny; p->nx = nx; p->h = h; p->dt = dt; p->nabs = nabs; p->alpha = alpha;
    p->px = (nx + 31) & ~31;
    p->tiles_x = (nx + kBX - 1) / kBX;
    p->tiles_z = (nz + p->tile->rows - 1) / p->tile->rows;
    const size_t pl = p->plane();
    FWI_CUDA(cudaStreamCreateWithFlags(&p->work, cudaStreamNonBlocking));
    FWI_CUDA(cudaEventCreateWithFlags(&p->ev_in, cudaEventDisableTiming));
    FWI_CUDA(cudaEventCreateWithFlags(&p->ev_out, cudaEventDisableTiming));
    FWI_CUDA(cudaEventCreateWithFlags(&p->ev_geom, cudaEventDisableTiming));
    // one arena for everything the step kernels re-read every step, hottest first; its layout decides where the
    // fields land in the L2, and the step timings were measured with exactly this order:
    //   [m, acc, fld0, fld1, fld4, fld5 | fld2, fld3, fld6, fld7, vp]
    const size_t plb = (pl * sizeof(float) + 255) & ~(size_t)255;
    FWI_CUDA(cudaMalloc(&p->arena, 11 * plb + 256));
    FWI_CUDA(cudaMemset(p->arena, 0, 11 * plb + 256));
    p->sync_area = (int*)((char*)p->arena + 11 * plb);
    {
        char* a = (char*)p->arena;
        const int order[8] = {0, 1, 4, 5, 2, 3, 6, 7};
        p->m = (float*)a; p->acc = (float*)(a + plb);
        for (int k = 0; k < 8; ++k) p->fld[order[k]] = (float*)(a + (2 + k) * plb);
        p->vp = (float*)(a + 10 * plb);
    }
    { const char* e = getenv("FWI_PDL"); if (e && e[0] == '0') p->pdl = false; }
    FWI_CUDA(cudaMalloc(&p->gx, p->px * sizeof(float)));
    FWI_CUDA(cudaMalloc(&p->gz, nz * sizeof(float)));
    FWI_CUDA(cudaMalloc(&p->gy, ny * sizeof(float)));
    FWI_CUDA(cudaMalloc(&p->d_J, sizeof(double)));
    std::vector<float> gxh = sponge_profile(nx, p->px, nabs, alpha, false), gzh = sponge_profile(nz, nz, nabs, alpha, false),
                       gyh = (ny > 1) ? sponge_profile(ny, ny, nabs, alpha, false) : std::vector<float>(1, 1.0f);
    FWI_CUDA(cudaMemcpy(p->gy, gyh.data(), ny * sizeof(float), cudaMemcpyHostToDevice));
    FWI_CUDA(cudaMemcpy(p->gx, gxh.data(), p->px * sizeof(float), cudaMemcpyHostToDevice));
    FWI_CUDA(cudaMemcpy(p->gz, gzh.data(), nz * sizeof(float), cudaMemcpyHostToDevice));
    cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, device);
    int rc = make_tmaps(p);
    if (rc) return rc;
    // the tb2 and 3-D kernels take more than the default 48 KB of dynamic shared memory (the tile kernel stays below it)
    if ((rc = allow_smem(kTb2Shapes)) || (rc = allow_smem(kFd3Shapes))) return rc;
    return FWI_OK;
}

// Tile height of the one-step kernel.  All tiles of a step are resident at once (3-6 CTAs per SM), so a step lasts as long as
// the SM with the most tiles: 1000 x 3000 in 128 x 32 tiles is 768 tiles = 5.2 per SM, i.e. 28 SMs carry 6 and set the pace
// (0.865 balance), while 42-row tiles are 576 = 3.9 per SM (0.97) with less halo (50 rows read for 42 instead of 40 for 32).
// Model cost: ceil(tiles / SMs) x (rows + 4) - the 8 halo rows are loaded but not computed.  Measured at 1000 x 3000, us per
// forward+adjoint step pair: 32 rows 16.67, 28: 15.34, 42: 15.50, 56: 15.56 (forward step 6.77 / 5.83 / 5.94 / 5.85); at
// 1500 x 3000: 27.9 / 25.9 / 26.1 / 26.8.  The kernels are bit-identical, only the decomposition differs.
static const TileShape* pick_tile(int nz, int nx, int sms) {
    const long tx = (nx + kBX - 1) / kBX;
    const TileShape* pick = kTileShapes;
    double best = 1e300;
    for (const auto& k : kTileShapes) {
        const long tiles = tx * ((nz + k.rows - 1) / k.rows);
        const double cost = (double)((tiles + sms - 1) / sms) * (k.rows + 4);
        if (cost < best - 1e-9) { best = cost; pick = &k; }
    }
    return pick;
}

int fwi_fd2d_create(int device, int nz, int nx, float h, float dt, int nabs, float alpha, fwi_fd2d** out) {
    int rc = create_plan(device, nz, 1, nx, h, dt, nabs, alpha, out);
    if (rc) return rc;
    // Default step kernel by grid size (tools/variant_bench.py, us per forward+adjoint step pair, tile vs two-steps-per-pass):
    //   250x3000 12.8 vs 7.8 | 500x3000 14.6 vs 11.5 | 1000x3000 18.0 vs 19.6 | 2000x3000 41.9 vs 42.7 | 3000x3000 79.7 vs 60.4
    // Small grids are launch-bound (half the launches wins), grids whose fields leave the L2 are HBM-bound (12.7 instead
    // of 17 B per step wins); in between the one-step tile kernel streams from L2 faster than tb2 can compute.
    // fwi_fd2d_set_tile / set_tb2 override this.
    const char* e = getenv("FWI_FD2D_VARIANT");
    const bool force_tile = e && !strcmp(e, "tile");
    const double pts = (double)nz * nx;
    if (!force_tile && nz >= 32 && nx >= 128) {
        if (pts <= 2.0e6) rc = fwi_fd2d_set_tb2(*out, 24);
        else if (pts > 7.5e6) rc = fwi_fd2d_set_tb2(*out, 32);
        if (rc) { fwi_fd2d_destroy(*out); *out = nullptr; return rc; }
    }
    if ((*out)->family == kTile && nz >= 32) {
        const TileShape* t = pick_tile(nz, nx, (*out)->sm_count);
        rc = fwi_fd2d_set_tile(*out, t->rows, t->warps);
        if (rc) { fwi_fd2d_destroy(*out); *out = nullptr; }
    }
    return rc;
}

int fwi_fd3d_create(int device, int nz, int ny, int nx, float h, float dt, int nabs, float alpha, fwi_fd2d** out) {
    FWI_REQUIRE(ny >= 2, "fwi_fd3d_create: ny must be >= 2 (use fwi_fd2d_create for 2-D grids)");
    return create_plan(device, nz, ny, nx, h, dt, nabs, alpha, out);
}

int fwi_fd2d_destroy(fwi_fd2d* p) {
    if (!p) return FWI_OK;
    DeviceGuard g(p->device);
    if (p->work) cudaStreamSynchronize(p->work);
    drop_graphs(p);
    cudaFree(p->arena); cudaFree(p->gx); cudaFree(p->gz); cudaFree(p->gy); cudaFree(p->d_J);
    for (DevArray<float>* a : {&p->snap, &p->ckpt, &p->resid, &p->syn, &p->obs, &p->wav, &p->dm, &p->pts, &p->pres}) a->release();
    clear_geometry(p);
    for (int s = 0; s < 2; ++s) if (p->peer_arena[s] && p->peer_ipc[s]) cudaIpcCloseMemHandle(p->peer_arena[s]);
    if (p->ev_in) cudaEventDestroy(p->ev_in);
    if (p->ev_out) cudaEventDestroy(p->ev_out);
    if (p->ev_geom) cudaEventDestroy(p->ev_geom);
    for (auto& sl : p->stage) { if (sl.host) cudaFreeHost(sl.host); if (sl.done) cudaEventDestroy(sl.done); }
    if (p->work) cudaStreamDestroy(p->work);
    delete p;
    return FWI_OK;
}

int fwi_fd2d_set_tile(fwi_fd2d* p, int bz, int nw) {
    FWI_REQUIRE(p, "fwi_fd2d_set_tile: NULL plan");
    const TileShape* t = find_shape(kTileShapes, bz, nw);
    FWI_REQUIRE(t, "fwi_fd2d_set_tile: unsupported (bz=%d, nw=%d)", bz, nw);
    FWI_REQUIRE(p->family != k3D, "fwi_fd2d_set_tile: 2-D plans only");
    DeviceGuard g(p->device);
    FWI_CUDA(cudaStreamSynchronize(p->work));
    drop_graphs(p);
    p->family = kTile; p->tile = t;
    p->tiles_z = (p->nz + bz - 1) / bz;
    clear_geometry(p);                // tile binning changed
    return make_tmaps(p);
}

int fwi_fd2d_set_tb2(fwi_fd2d* p, int cz) {
    FWI_REQUIRE(p, "fwi_fd2d_set_tb2: NULL plan");
    const Tb2Shape* t = find_shape(kTb2Shapes, cz, kTb2Warps);
    FWI_REQUIRE(t, "fwi_fd2d_set_tb2: unsupported core rows %d", cz);
    FWI_REQUIRE(p->family != k3D, "fwi_fd2d_set_tb2: 2-D plans only");
    DeviceGuard g(p->device);
    FWI_CUDA(cudaStreamSynchronize(p->work));
    drop_graphs(p);
    p->family = kTb2; p->tb2 = t;
    clear_geometry(p);
    return make_tmaps(p);
}

int fwi_fd2d_set_free_surface(fwi_fd2d* p, int enable) {
    FWI_REQUIRE(p, "fwi_fd2d_set_free_surface: NULL plan");
    FWI_REQUIRE(!enable || !p->peer_arena[0], "fwi_fd2d_set_free_surface: this slab has an upper neighbour; only the slab that owns z = 0 has the surface");
    DeviceGuard g(p->device);
    FWI_CUDA(cudaStreamSynchronize(p->work));
    drop_graphs(p);
    p->free_surface = enable != 0;
    const std::vector<float> gzh = sponge_profile(p->nz, p->nz, p->nabs, p->alpha, p->free_surface);
    FWI_CUDA(cudaMemcpy(p->gz, gzh.data(), p->nz * sizeof(float), cudaMemcpyHostToDevice));
    clear_geometry(p);                // the geometry is checked against the surface when it is set
    return FWI_OK;
}

int fwi_fd2d_set_graphs(fwi_fd2d* p, int enable) {
    FWI_REQUIRE(p, "fwi_fd2d_set_graphs: NULL plan");
    p->use_graphs = enable != 0;
    return FWI_OK;
}

int fwi_fd2d_set_memory_limit(fwi_fd2d* p, uint64_t bytes) {
    FWI_REQUIRE(p, "fwi_fd2d_set_memory_limit: NULL plan");
    p->mem_limit = (size_t)bytes;
    return FWI_OK;
}

int fwi_fd2d_set_model(fwi_fd2d* p, const float* v_dev, void* stream) {
    FWI_REQUIRE(p && v_dev, "fwi_fd2d_set_model: NULL argument");
    DeviceGuard g(p->device);
    cudaStream_t user = (cudaStream_t)stream;
    int rc = enter(p, user);
    if (rc) return rc;
    dim3 grid(p->rows(), (p->px + 127) / 128);
    fd_model_kernel<<<grid, 128, 0, p->work>>>(v_dev, p->rows(), p->nx, p->px, p->dt / p->h, p->m, p->vp);
    FWI_CUDA(cudaGetLastError());
    p->model_set = true;
    p->pdl_chain = false;             // the next step must not start reading m while this kernel is still writing it
    return leave(p, user);
}

// ---- off-grid points (spec B7, tests/offgrid_reference.py) ---------------------------------------------------------
// Kaiser window parameter of the windowed-sinc taps: the b on a 0.01 grid that minimises
// E(b) = max |sum_k w_k(f) exp(i kappa d_k) - 1| over kappa in [0, 2 pi / 3], f in [0, 1)  (E(4.06) = 8.79e-3).
constexpr double kKaiserB = 4.06;

// One axis's taps of a coordinate x in cell units on n cells: (index, weight) in ascending index, float64.  An integral x is
// one tap of weight 1; otherwise 8 taps at floor(x) - 3 .. floor(x) + 4 of Hicks' Kaiser-windowed sinc with half-width 4.
// `fold` (the free-surface z axis): a tap at -k lands on +k with its weight negated, a tap on row 0 is dropped.  Taps
// outside [0, n) are dropped (the zero halo of B1); taps on one index are summed.
static std::vector<std::pair<int, double>> axis_taps(double x, int n, bool fold) {
    std::vector<std::pair<int, double>> t;
    const double fl = std::floor(x), f = x - fl;
    const int i = (int)fl;
    if (f == 0.0) { t.push_back({i, 1.0}); return t; }
    const double i0b = std::cyl_bessel_i(0.0, kKaiserB);
    for (int k = -3; k <= 4; ++k) {
        const double d = k - f, pd = M_PI * d;
        double w = std::sin(pd) / pd * std::cyl_bessel_i(0.0, kKaiserB * std::sqrt(1.0 - (d / 4) * (d / 4))) / i0b;
        int j = i + k;
        if (fold && j < 0) { j = -j; w = -w; }
        if ((fold && j == 0) || j < 0 || j >= n) continue;
        auto it = std::find_if(t.begin(), t.end(), [j](const std::pair<int, double>& e) { return e.first == j; });
        if (it != t.end()) it->second += w;
        else t.push_back({j, w});
    }
    std::sort(t.begin(), t.end());
    return t;
}

struct HostCsr { std::vector<int> ptr, col; std::vector<float> w; };

// One side's off-grid points as cells and the two CSR forms of the operator W (points x cells).
struct SideTaps {
    std::vector<int> cz, cy, cx;                          // the unique cells, in ascending linear offset
    HostCsr by_point, by_cell;
};

static int build_side(const fwi_fd2d* p, int n, const double* z, const double* y, const double* x, const char* what, SideTaps& s) {
    const double dims[3] = {(double)p->nz, (double)p->ny, (double)p->nx};
    std::vector<std::pair<int64_t, std::pair<int, double>>> taps;        // (cell offset, (point, weight)), point-major
    s.by_point.ptr.assign(1, 0);
    for (int i = 0; i < n; ++i) {
        const double c[3] = {z[i], y ? y[i] : 0.0, x[i]};
        FWI_REQUIRE(std::isfinite(c[0]) && std::isfinite(c[1]) && std::isfinite(c[2]), "%s %d at (z=%g, y=%g, x=%g) is not finite", what, i, c[0], c[1], c[2]);
        for (int d = 0; d < 3; ++d)
            FWI_REQUIRE(c[d] >= 0.0 && c[d] <= dims[d] - 1, "%s %d at (z=%g, y=%g, x=%g) is outside the %d x %d x %d grid (each coordinate must lie in [0, n - 1])", what, i, c[0], c[1], c[2], p->nz, p->ny, p->nx);
        FWI_REQUIRE(!p->free_surface || c[0] > 0.0, "%s %d at (z=%g, y=%g, x=%g) lies on the free surface; off-grid points need z > 0", what, i, c[0], c[1], c[2]);
        const auto tz = axis_taps(c[0], p->nz, p->free_surface), ty = axis_taps(c[1], p->ny, false), tx = axis_taps(c[2], p->nx, false);
        for (const auto& a : tz)
            for (const auto& b : ty)
                for (const auto& e : tx)
                    taps.push_back({((int64_t)a.first * p->ny + b.first) * p->nx + e.first, {i, a.second * b.second * e.second}});
        s.by_point.ptr.push_back((int)taps.size());
    }
    std::vector<int64_t> cells(taps.size());
    for (size_t e = 0; e < taps.size(); ++e) cells[e] = taps[e].first;
    std::sort(cells.begin(), cells.end());
    cells.erase(std::unique(cells.begin(), cells.end()), cells.end());
    const int nc = (int)cells.size();
    s.cz.resize(nc); s.cy.resize(nc); s.cx.resize(nc);
    for (int c = 0; c < nc; ++c) {
        s.cx[c] = (int)(cells[c] % p->nx);
        s.cy[c] = (int)(cells[c] / p->nx % p->ny);
        s.cz[c] = (int)(cells[c] / p->nx / p->ny);
    }
    // a point's taps come in ascending cell order and never repeat a cell (axis_taps merged them per axis)
    s.by_point.col.resize(taps.size()); s.by_point.w.resize(taps.size());
    s.by_cell.ptr.assign(nc + 1, 0);
    for (size_t e = 0; e < taps.size(); ++e) {
        s.by_point.col[e] = (int)(std::lower_bound(cells.begin(), cells.end(), taps[e].first) - cells.begin());
        s.by_point.w[e] = (float)taps[e].second.second;
        s.by_cell.ptr[s.by_point.col[e] + 1]++;
    }
    for (int c = 0; c < nc; ++c) s.by_cell.ptr[c + 1] += s.by_cell.ptr[c];
    std::vector<int> fill(s.by_cell.ptr.begin(), s.by_cell.ptr.end() - 1);
    s.by_cell.col.resize(taps.size()); s.by_cell.w.resize(taps.size());
    for (size_t e = 0; e < taps.size(); ++e) {                           // points of a cell in ascending order
        const int k = fill[s.by_point.col[e]]++;
        s.by_cell.col[k] = taps[e].second.first;
        s.by_cell.w[k] = s.by_point.w[e];
    }
    return FWI_OK;
}

// ---- installing a geometry: build it on the host, then commit it, so that a rejected one leaves the plan as it was ----
// The cells of both sides binned into every point list the plan's family runs and, off grid, both sides' operators.
struct HostGeometry {
    int nsrc = 0, nrec = 0;                   // cells
    int psrc = -1, prec = -1;                 // off-grid points (Interp::npts)
    HostList src, rec, src_ext2, src_own2, rec_ext2, rec_own2;
    SideTaps s, r;
};

// Checks the cells, all sources and then all receivers, and bins them for every kernel family the plan runs.
static int bin_geometry(const fwi_fd2d* p, int nsrc, const int* src_z, const int* src_y, const int* src_x, int nrec,
                        const int* rec_z, const int* rec_y, const int* rec_x, HostGeometry& g) {
    int rc = check_points(p, nsrc, src_z, src_y, src_x, "source");
    if (rc || (rc = check_points(p, nrec, rec_z, rec_y, rec_x, "receiver"))) return rc;
    g.nsrc = nsrc; g.nrec = nrec;
    const TileGrid step = tile_grid(p, p->family == k3D ? k3D : kTile);     // tb2 plans run the tile kernel for single steps
    bin_points(p, step, 0, nsrc, src_z, src_y, src_x, g.src);
    bin_points(p, step, 0, nrec, rec_z, rec_y, rec_x, g.rec);
    if (p->family == kTb2) {
        const TileGrid pass = tile_grid(p, kTb2);
        bin_points(p, pass, kHalo, nsrc, src_z, src_y, src_x, g.src_ext2);
        bin_points(p, pass, 0, nsrc, src_z, src_y, src_x, g.src_own2);
        bin_points(p, pass, kHalo, nrec, rec_z, rec_y, rec_x, g.rec_ext2);
        bin_points(p, pass, 0, nrec, rec_z, rec_y, rec_x, g.rec_own2);
    }
    return FWI_OK;
}

// (slack: the tb2 extended lists vary a little from shot to shot)
static int upload_list(fwi_fd2d* p, PointList& pl, const HostList& h) {
    int rc = stage_upload(p, pl.tile_ptr, h.tile_ptr, false);
    if (!rc) rc = stage_upload(p, pl.off, h.off, true);
    if (!rc) rc = stage_upload(p, pl.id, h.id, true);
    return rc;
}
static int upload_csr(fwi_fd2d* p, Csr& c, const HostCsr& h) {
    int rc = stage_upload(p, c.ptr, h.ptr, true);
    if (!rc) rc = stage_upload(p, c.col, h.col, true);
    if (!rc) rc = stage_upload(p, c.w, h.w, true);
    return rc;
}

// Uploads every array of a built geometry through one staging slot, then switches the plan to it.  A failed CUDA call
// leaves the plan without a geometry rather than with parts of two.
static int commit_geometry(fwi_fd2d* p, const HostGeometry& g) {
    DeviceGuard dg(p->device);
    const std::pair<PointList*, const HostList*> lists[] = {{&p->src, &g.src}, {&p->rec, &g.rec}, {&p->src_ext2, &g.src_ext2},
                                                            {&p->src_own2, &g.src_own2}, {&p->rec_ext2, &g.rec_ext2}, {&p->rec_own2, &g.rec_own2}};
    const std::pair<Csr*, const HostCsr*> ops[] = {{&p->isrc.by_point, &g.s.by_point}, {&p->isrc.by_cell, &g.s.by_cell},
                                                   {&p->irec.by_point, &g.r.by_point}, {&p->irec.by_cell, &g.r.by_cell}};
    const int nlists = p->family == kTb2 ? 6 : 2, nops = g.psrc >= 0 ? 4 : 0;
    size_t ints = 0;
    for (int k = 0; k < nlists; ++k) ints += lists[k].second->tile_ptr.size() + lists[k].second->off.size() + lists[k].second->id.size();
    for (int k = 0; k < nops; ++k) ints += ops[k].second->ptr.size() + ops[k].second->col.size() + ops[k].second->w.size();
    if (g.nsrc != p->nsrc || g.nrec != p->nrec) drop_graphs(p);
    int rc = stage_begin(p, ints);
    for (int k = 0; k < nlists && !rc; ++k) rc = upload_list(p, *lists[k].first, *lists[k].second);
    for (int k = 0; k < nops && !rc; ++k) rc = upload_csr(p, *ops[k].first, *ops[k].second);
    if (!rc) {
        for (int k = 0; k < nlists; ++k) lists[k].first->n = lists[k].second->tile_ptr.back();
        for (int k = 0; k < nops; ++k) ops[k].first->rows = (int)ops[k].second->ptr.size() - 1;
        p->nsrc = g.nsrc; p->nrec = g.nrec;
        p->isrc.npts = g.psrc; p->irec.npts = g.prec;
        rc = stage_end(p);
    }
    if (rc) clear_geometry(p);
    return rc;
}

static int set_geometry(fwi_fd2d* p, int nsrc, const int* src_z, const int* src_y, const int* src_x, int nrec,
                        const int* rec_z, const int* rec_y, const int* rec_x) {
    FWI_REQUIRE(p, "fwi_fd_set_geometry: NULL plan");
    FWI_REQUIRE(nsrc >= 0 && nrec >= 0 && (nsrc == 0 || (src_z && src_x)) && (nrec == 0 || (rec_z && rec_x)), "fwi_fd_set_geometry: bad arguments");
    HostGeometry g;                           // (psrc = prec = -1: points are cells again)
    const int rc = bin_geometry(p, nsrc, src_z, src_y, src_x, nrec, rec_z, rec_y, rec_x, g);
    return rc ? rc : commit_geometry(p, g);
}

static int set_positions(fwi_fd2d* p, int nsrc, const double* src_z, const double* src_y, const double* src_x, int nrec,
                         const double* rec_z, const double* rec_y, const double* rec_x) {
    FWI_REQUIRE(p, "fwi_fd_set_positions: NULL plan");
    FWI_REQUIRE(nsrc >= 0 && nrec >= 0 && (nsrc == 0 || (src_z && src_x)) && (nrec == 0 || (rec_z && rec_x)), "fwi_fd_set_positions: bad arguments");
    // a point's taps may straddle two slabs, and a slab's residual would miss the part of a trace another rank samples
    FWI_REQUIRE(!p->peers(), "fwi_fd_set_positions: not available on a plan connected as a peer-memory slab");
    HostGeometry g;
    int rc = build_side(p, nsrc, src_z, src_y, src_x, "source", g.s);
    if (rc || (rc = build_side(p, nrec, rec_z, rec_y, rec_x, "receiver", g.r)) ||
        (rc = bin_geometry(p, (int)g.s.cz.size(), g.s.cz.data(), g.s.cy.data(), g.s.cx.data(), (int)g.r.cz.size(), g.r.cz.data(),
                           g.r.cy.data(), g.r.cx.data(), g)))
        return rc;
    g.psrc = nsrc; g.prec = nrec;
    return commit_geometry(p, g);
}

int fwi_fd2d_set_positions(fwi_fd2d* p, int nsrc, const double* src_z, const double* src_x, int nrec, const double* rec_z,
                           const double* rec_x) {
    FWI_REQUIRE(p && p->ny == 1, "fwi_fd2d_set_positions: needs a 2-D plan");
    return set_positions(p, nsrc, src_z, nullptr, src_x, nrec, rec_z, nullptr, rec_x);
}

int fwi_fd3d_set_positions(fwi_fd2d* p, int nsrc, const double* src_z, const double* src_y, const double* src_x, int nrec,
                           const double* rec_z, const double* rec_y, const double* rec_x) {
    FWI_REQUIRE(p && p->ny > 1, "fwi_fd3d_set_positions: needs a 3-D plan");
    FWI_REQUIRE((nsrc == 0 || src_y) && (nrec == 0 || rec_y), "fwi_fd3d_set_positions: y coordinates missing");
    return set_positions(p, nsrc, src_z, src_y, src_x, nrec, rec_z, rec_y, rec_x);
}

int fwi_fd2d_set_geometry(fwi_fd2d* p, int nsrc, const int* src_z, const int* src_x, int nrec, const int* rec_z,
                          const int* rec_x) {
    FWI_REQUIRE(p && p->ny == 1, "fwi_fd2d_set_geometry: needs a 2-D plan");
    return set_geometry(p, nsrc, src_z, nullptr, src_x, nrec, rec_z, nullptr, rec_x);
}

int fwi_fd3d_set_geometry(fwi_fd2d* p, int nsrc, const int* src_z, const int* src_y, const int* src_x, int nrec,
                          const int* rec_z, const int* rec_y, const int* rec_x) {
    FWI_REQUIRE(p && p->ny > 1, "fwi_fd3d_set_geometry: needs a 3-D plan");
    FWI_REQUIRE((nsrc == 0 || src_y) && (nrec == 0 || rec_y), "fwi_fd3d_set_geometry: y indices missing");
    return set_geometry(p, nsrc, src_z, src_y, src_x, nrec, rec_z, rec_y, rec_x);
}

// ---- the shot-level operations -------------------------------------------------------------------------------------
// Steps per Born segment: the background sweep saves this many snapshots, then the scattered sweep reads them back.
// (profiles/r3_born_bench.txt, ms per Born shot at 1000 x 3000, nt = 5000: see DESIGN.md)
constexpr int kBornSeg = 128;

// Forward-field storage in planes: the memory limit, or 85 % of the free memory plus the floats the plan holds in
// buffers it may reallocate (`reclaim`).
static int storage_budget(fwi_fd2d* p, size_t reclaim, size_t& budget, size_t& planes) {
    budget = p->mem_limit;
    if (!budget) {
        size_t fr = 0, tot = 0;
        FWI_CUDA(cudaMemGetInfo(&fr, &tot));
        budget = (size_t)((fr + reclaim * sizeof(float)) * 0.85);
    }
    planes = budget / (p->plane() * sizeof(float));
    return FWI_OK;
}

// Storage decision and buffers of an operation over nt steps (no launches).
// Gradient and Gauss-Newton hold every w_n in HBM if it fits, else checkpoint.  The decision is cached per (nt, limit):
// cudaMemGetInfo takes a driver-wide lock and was measured stalling the host for 5 - 90 ms every few calls, which showed
// up as sporadic slow shots.  Born runs in segments of S = min(nt, kBornSeg, planes the budget allows) steps; it only
// queries free memory when the snapshot buffer cannot already hold min(nt, kBornSeg) planes.
static int prepare(fwi_fd2d* p, Op op, int nt, Split& split) {
    const size_t pl = p->plane(), ntr = (size_t)nt * p->nrec, ntp = (size_t)nt * rec_points(p);
    const bool adjoint = op == kGradient || op == kGaussNewton;
    split = Split{nt, 1};
    int rc;
    if (adjoint && p->split_nt == nt && p->split_limit == p->mem_limit) {
        split = p->split;
    } else if (adjoint) {
        size_t budget = 0, planes = 0;
        if ((rc = storage_budget(p, p->snap.cap + p->ckpt.cap, budget, planes))) return rc;
        if ((size_t)nt > planes) {
            // segment length S with S + 2*ceil(nt/S) planes minimal-ish: start from sqrt(2 nt)
            split.seg = std::max(1, (int)std::ceil(std::sqrt(2.0 * nt)));
            split.nseg = (nt + split.seg - 1) / split.seg;
            FWI_REQUIRE((size_t)split.seg + 2 * (size_t)split.nseg <= planes, "fwi_fd2d_gradient: %zu bytes are not enough even with checkpointing (need %zu planes of %zu bytes)", budget, (size_t)split.seg + 2 * (size_t)split.nseg, pl * sizeof(float));
        }
    } else if (op == kBorn) {
        const int S = std::min(nt, kBornSeg);
        size_t budget = 0, planes = (size_t)S;
        if ((p->mem_limit || p->snap.cap < (size_t)S * pl) && (rc = storage_budget(p, p->snap.cap, budget, planes))) return rc;
        FWI_REQUIRE(planes >= 1, "fwi_fd2d_born: the memory limit holds no snapshot plane of %zu bytes", pl * sizeof(float));
        split.seg = (int)std::min<size_t>((size_t)S, planes);
        split.nseg = (nt + split.seg - 1) / split.seg;
    }
    if (op != kForward && (rc = p->snap.ensure(p, (size_t)split.seg * pl))) return rc;
    if (adjoint && split.nseg > 1 && (rc = p->ckpt.ensure(p, (size_t)split.nseg * 2 * pl))) return rc;
    if (op != kForward && (rc = p->resid.ensure(p, ntr))) return rc;
    if ((rc = p->syn.ensure(p, ntr))) return rc;
    if (adjoint && (rc = p->obs.ensure(p, ntp))) return rc;
    if (adjoint && p->irec.npts >= 0 &&
        ((rc = p->pts.ensure(p, ntp)) || (rc = p->pres.ensure(p, ntp)))) return rc;
    if ((rc = p->wav.ensure(p, (size_t)nt * p->nsrc))) return rc;
    if (adjoint) { p->split_nt = nt; p->split_limit = p->mem_limit; p->split = split; }      // buffers exist now
    if ((op == kBorn || op == kGaussNewton) && (rc = p->dm.ensure(p, pl))) return rc;
    return FWI_OK;
}

// grad (dense grid) += (2 / v) * imaging accumulator
static int launch_finalize(fwi_fd2d* p, float* grad, cudaStream_t st) {
    dim3 grid(p->rows(), (p->nx + 127) / 128);
    fd_grad_finalize_kernel<<<grid, 128, 0, st>>>(p->acc, p->vp, p->rows(), p->nx, p->px, grad);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

// dm = (2 m / v) dv into the plan-owned pitched buffer, on the work stream ahead of the time loop (captured graphs keep
// the buffer's address)
static int stage_dm(fwi_fd2d* p, const float* dv_dev) {
    dim3 grid(p->rows(), (p->px + 127) / 128);
    fd_dm_kernel<<<grid, 128, 0, p->work>>>(dv_dev, p->m, p->vp, p->rows(), p->nx, p->px, p->dm.d);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

// One shot's device arrays (misfit: host).  A null pointer is an input the operation does not read or an output the
// caller does not want.
struct ShotIO {
    const float* wavelet = nullptr;
    const float* obs = nullptr;
    const float* dv = nullptr;
    float* image = nullptr;           // dense grid += (2 / v) I: the gradient, or J^T J dv
    float* traces = nullptr;          // synthetics
    float* dtraces = nullptr;         // Born traces J dv
    double* misfit = nullptr;         // J = 1/2 sum r^2; waits for the shot
};

// Trace rows (nt, receivers) of a shot into the caller's `dst` from the cell rows `cells`: a copy on the grid; off grid
// (spec B7) gathered to the receivers, or, with `gathered`, copied from p->pts, where the graph already gathered them.
static int copy_traces(fwi_fd2d* p, float* dst, const float* cells, bool gathered, int nt) {
    const size_t n = (size_t)nt * rec_points(p);
    if (!n) return FWI_OK;
    if (p->irec.npts >= 0 && !gathered) return launch_interp(p, true, p->irec.by_point, cells, p->nrec, dst, nt, p->work);
    FWI_CUDA(cudaMemcpyAsync(dst, p->irec.npts >= 0 ? p->pts.d : cells, n * sizeof(float), cudaMemcpyDeviceToDevice, p->work));
    return FWI_OK;
}

// One shot of `op` on the plan's work stream, ordered after everything queued on `stream` and before what follows on it.
static int run_shot(fwi_fd2d* p, Op op, int nt, void* stream, const ShotIO& io) {
    DeviceGuard g(p->device);
    cudaStream_t user = (cudaStream_t)stream;
    Split split;
    int rc;
    if ((rc = prepare(p, op, nt, split)) || (rc = enter(p, user))) return rc;
    const size_t nw = (size_t)nt * p->nsrc, ntp = (size_t)nt * rec_points(p);
    if (p->isrc.npts >= 0) {          // off grid (spec B7): the cells' wavelets are W_s^T times the points'
        if ((rc = launch_interp(p, false, p->isrc.by_cell, io.wavelet, p->isrc.npts, p->wav.d, nt, p->work))) return rc;
    } else if (nw) {
        FWI_CUDA(cudaMemcpyAsync(p->wav.d, io.wavelet, nw * sizeof(float), cudaMemcpyDeviceToDevice, p->work));
    }
    if (io.obs && ntp) FWI_CUDA(cudaMemcpyAsync(p->obs.d, io.obs, ntp * sizeof(float), cudaMemcpyDeviceToDevice, p->work));
    if (io.dv && (rc = stage_dm(p, io.dv))) return rc;
    if ((rc = run_cached(p, op, nt, split))) return rc;
    if (io.image) {
        if ((rc = launch_finalize(p, io.image, p->work))) return rc;
        p->launches += 1;
    }
    if (io.dtraces && (rc = copy_traces(p, io.dtraces, p->resid.d, op == kGaussNewton, nt))) return rc;
    if (io.traces && (rc = copy_traces(p, io.traces, p->syn.d, op == kGradient, nt))) return rc;
    if (io.misfit) FWI_CUDA(cudaMemcpyAsync(io.misfit, p->d_J, sizeof(double), cudaMemcpyDeviceToHost, p->work));
    if ((rc = leave(p, user))) return rc;
    if (io.misfit) FWI_CUDA(cudaStreamSynchronize(p->work));
    return FWI_OK;
}

int fwi_fd2d_forward(fwi_fd2d* p, const float* wavelet_dev, int nt, float* traces_dev, void* stream) {
    FWI_REQUIRE(p && p->model_set, "fwi_fd2d_forward: set the model first");
    FWI_REQUIRE(nt >= 0 && (p->nsrc == 0 || wavelet_dev), "fwi_fd2d_forward: bad wavelet / nt");
    FWI_REQUIRE(p->nrec == 0 || traces_dev, "fwi_fd2d_forward: traces_dev is NULL but receivers are set");
    ShotIO io;
    io.wavelet = wavelet_dev; io.traces = traces_dev;
    return run_shot(p, kForward, nt, stream, io);
}

int fwi_fd2d_wavefield(fwi_fd2d* p, int which, float* out_dev, void* stream) {
    FWI_REQUIRE(p && out_dev && which >= 0 && which <= 2, "fwi_fd2d_wavefield: bad arguments");
    DeviceGuard g(p->device);
    cudaStream_t user = (cudaStream_t)stream;
    int rc = enter(p, user);
    if (rc) return rc;
    const float* src = (which == 0) ? p->fld[p->fwd_c] : (which == 1 ? p->fld[p->fwd_o] : p->acc);
    dim3 grid(p->rows(), (p->nx + 127) / 128);
    fd_unpitch_kernel<<<grid, 128, 0, p->work>>>(src, p->rows(), p->nx, p->px, out_dev);
    FWI_CUDA(cudaGetLastError());
    return leave(p, user);
}

// Allocate everything fwi_fd2d_forward (gradient = 0) or fwi_fd2d_gradient (1) over nt steps with the current geometry
// will need, without launching anything: keeps allocations (which synchronise the device) out of timed regions and out
// of the way of kernels that wait for another plan.
int fwi_fd_reserve(fwi_fd2d* p, int nt, int gradient) {
    FWI_REQUIRE(p && nt >= 1, "fwi_fd_reserve: bad arguments");
    DeviceGuard g(p->device);
    const Op op = gradient ? kGradient : kForward;
    Split split;
    int rc = prepare(p, op, nt, split);
    if (rc) return rc;
    if (p->use_graphs && p->model_set) {          // capture, instantiate and upload the time loop now as well
        GraphEntry* e = nullptr;
        p->pdl_chain = false;
        if ((rc = get_graph(p, op, nt, split, &e))) return rc;
        FWI_CUDA(cudaGraphUpload(e->exec, p->work));
        FWI_CUDA(cudaStreamSynchronize(p->work));
    }
    return FWI_OK;
}

int fwi_fd2d_gradient(fwi_fd2d* p, const float* wavelet_dev, const float* obs_dev, int nt, float* grad_dev,
                      float* traces_dev, double* misfit_host, void* stream) {
    FWI_REQUIRE(p && p->model_set, "fwi_fd2d_gradient: set the model first");
    FWI_REQUIRE((wavelet_dev || p->nsrc == 0) && (obs_dev || p->nrec == 0) && grad_dev && nt >= 1, "fwi_fd2d_gradient: NULL argument or nt < 1");
    FWI_REQUIRE((p->nsrc >= 1 && p->nrec >= 1) || p->z_own1 > 0, "fwi_fd2d_gradient: geometry needs at least one source and one receiver");
    ShotIO io;
    io.wavelet = wavelet_dev; io.obs = obs_dev; io.image = grad_dev; io.traces = traces_dev; io.misfit = misfit_host;
    return run_shot(p, kGradient, nt, stream, io);
}

// ---- Born modelling and Gauss-Newton Hessian-vector products (spec B5) ------------------------------------------
static int check_linearised(fwi_fd2d* p, const char* fn, const float* wavelet_dev, const float* dv_dev, const float* out_dev, int nt) {
    FWI_REQUIRE(p && p->model_set, "%s: set the model first", fn);
    FWI_REQUIRE(wavelet_dev && dv_dev && out_dev && nt >= 1, "%s: NULL argument or nt < 1", fn);
    FWI_REQUIRE(p->nsrc >= 1 && p->nrec >= 1, "%s: geometry needs at least one source and one receiver", fn);
    // the slab step-id protocol assumes the same launch sequence on every rank
    FWI_REQUIRE(!p->peers(), "%s: not available on a plan connected as a peer-memory slab", fn);
    return FWI_OK;
}

int fwi_fd2d_born(fwi_fd2d* p, const float* wavelet_dev, const float* dv_dev, int nt, float* dtraces_dev, float* traces_dev,
                  void* stream) {
    int rc = check_linearised(p, "fwi_fd2d_born", wavelet_dev, dv_dev, dtraces_dev, nt);
    if (rc) return rc;
    ShotIO io;
    io.wavelet = wavelet_dev; io.dv = dv_dev; io.dtraces = dtraces_dev; io.traces = traces_dev;
    return run_shot(p, kBorn, nt, stream, io);
}

int fwi_fd2d_gauss_newton(fwi_fd2d* p, const float* wavelet_dev, const float* dv_dev, int nt, float* hv_dev, float* dtraces_dev,
                          void* stream) {
    int rc = check_linearised(p, "fwi_fd2d_gauss_newton", wavelet_dev, dv_dev, hv_dev, nt);
    if (rc) return rc;
    ShotIO io;
    io.wavelet = wavelet_dev; io.dv = dv_dev; io.image = hv_dev; io.dtraces = dtraces_dev;     // H dv = (2 / v) I
    return run_shot(p, kGaussNewton, nt, stream, io);
}

int64_t fwi_fd2d_launch_count(fwi_fd2d* p) { return p ? p->launches : 0; }

// ---- low-level stepping API: the caller drives the time loop (used by the slab-decomposed multi-GPU path, which
// interleaves halo exchanges with single steps on the caller's stream) -----------------------------------------
int fwi_fd_set_profiles(fwi_fd2d* p, const float* gz_host, const float* gy_host, const float* gx_host) {
    FWI_REQUIRE(p, "fwi_fd_set_profiles: NULL plan");
    DeviceGuard g(p->device);
    FWI_CUDA(cudaStreamSynchronize(p->work));
    if (gz_host) FWI_CUDA(cudaMemcpy(p->gz, gz_host, p->nz * sizeof(float), cudaMemcpyHostToDevice));
    if (gy_host) FWI_CUDA(cudaMemcpy(p->gy, gy_host, p->ny * sizeof(float), cudaMemcpyHostToDevice));
    if (gx_host) FWI_CUDA(cudaMemcpy(p->gx, gx_host, p->nx * sizeof(float), cudaMemcpyHostToDevice));
    return FWI_OK;
}

void* fwi_fd_field_ptr(fwi_fd2d* p, int idx) { return (p && idx >= 0 && idx < 8) ? (void*)p->fld[idx] : nullptr; }
int fwi_fd_pitch(fwi_fd2d* p) { return p ? p->px : 0; }

int fwi_fd_reserve_snapshots(fwi_fd2d* p, int nsteps) {
    FWI_REQUIRE(p && nsteps >= 0, "fwi_fd_reserve_snapshots: bad arguments");
    DeviceGuard g(p->device);
    FWI_CUDA(cudaStreamSynchronize(p->work));
    return p->snap.ensure(p, (size_t)nsteps * p->plane());
}

// Zero the wavefield pair (0 = forward, 1 = adjoint; the adjoint pair also clears the imaging accumulator).
int fwi_fd_reset(fwi_fd2d* p, int pair, void* stream) {
    FWI_REQUIRE(p && (pair == 0 || pair == 1), "fwi_fd_reset: bad arguments");
    DeviceGuard g(p->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t pl = p->plane();
    FWI_CUDA(cudaMemsetAsync(p->fld[4 * pair], 0, pl * sizeof(float), st));
    FWI_CUDA(cudaMemsetAsync(p->fld[4 * pair + 1], 0, pl * sizeof(float), st));
    if (pair == 1) FWI_CUDA(cudaMemsetAsync(p->acc, 0, pl * sizeof(float), st));
    return FWI_OK;
}

// One leapfrog step on `stream`.  mode: 0 forward, 1 forward + snapshot[snap_index], 2 adjoint + imaging with
// snapshot[snap_index].  `cur` (0/1) says which buffer of the pair holds u_n; u_{n+1} lands in the other one.
// inj_vals_dev: this step's injected values (sources for modes 0/1, receiver residuals for mode 2);
// rec_out_dev: this step's trace row (modes 0/1, nullable).
int fwi_fd_step(fwi_fd2d* p, int mode, int cur, const float* inj_vals_dev, float* rec_out_dev, int64_t snap_index, void* stream) {
    FWI_REQUIRE(p && p->model_set, "fwi_fd_step: set the model first");
    FWI_REQUIRE(mode >= 0 && mode <= 2 && (cur == 0 || cur == 1), "fwi_fd_step: bad mode / cur");
    FWI_REQUIRE(p->irec.npts < 0, "fwi_fd_step: the plan holds off-grid positions (fwi_fd*_set_positions); single steps take the integer geometry");
    p->pdl_chain = false;             // caller-driven loop: other kernels (halo exchange, resets) sit between the steps
    FWI_REQUIRE(mode == 0 || (snap_index >= 0 && (size_t)(snap_index + 1) * p->plane() <= p->snap.cap), "fwi_fd_step: snapshot %lld not reserved", (long long)snap_index);
    DeviceGuard g(p->device);
    if (p->geom_pending) {
        // (not while the caller captures a graph: it synchronised before starting the capture, and an event recorded
        // outside a capture must not be waited for inside it)
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        FWI_CUDA(cudaStreamIsCapturing((cudaStream_t)stream, &cs));
        if (cs == cudaStreamCaptureStatusNone) { FWI_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, p->ev_geom, 0)); p->geom_pending = false; }
    }
    const int base = (mode == STEP_ADJ) ? 4 : 0;
    float* snap = (mode == 0) ? nullptr : p->snap.d + (size_t)snap_index * p->plane();
    int rc = launch_step(p, mode, base + cur, p->fld[base + (cur ^ 1)], mode == STEP_ADJ ? &p->rec : &p->src, inj_vals_dev,
                         (mode != STEP_ADJ && rec_out_dev) ? &p->rec : nullptr, rec_out_dev, snap, (cudaStream_t)stream);
    if (rc) return rc;
    FWI_CUDA(cudaGetLastError());
    if (mode != STEP_ADJ) { p->fwd_c = cur ^ 1; p->fwd_o = cur; }
    return FWI_OK;
}

// ---- slab decomposition over NVLink peer memory (3-D): the step kernel itself stores its boundary planes into the
// neighbours' ghost planes and publishes a step id; the next launch of the neighbour waits for it. -------------------
int fwi_fd_slab_info(fwi_fd2d* p, void* ipc_handle_out /*64 bytes*/, uint64_t* offsets_out /*9: 8 wavefield buffers + sync area*/) {
    FWI_REQUIRE(p && ipc_handle_out && offsets_out, "fwi_fd_slab_info: bad arguments");
    DeviceGuard g(p->device);
    cudaIpcMemHandle_t h;
    FWI_CUDA(cudaIpcGetMemHandle(&h, p->arena));
    memcpy(ipc_handle_out, &h, sizeof(h));
    for (int i = 0; i < 8; ++i) offsets_out[i] = (uint64_t)((char*)p->fld[i] - (char*)p->arena);
    offsets_out[8] = (uint64_t)((char*)p->sync_area - (char*)p->arena);
    return FWI_OK;
}

static int slab_finish_connect(fwi_fd2d* p, int z_own0, int z_own1, int up_ghost_z) {
    p->z_own0 = z_own0; p->z_own1 = z_own1; p->peer_up_z = up_ghost_z;
    if (const char* e = getenv("FWI_SLAB_TIMEOUT_MS")) { const double ms = atof(e); if (ms > 0) p->slab_timeout_cycles = (long long)(ms * 1.9e6); }
    clear_geometry(p);                // z chunking (and so the point binning) changes
    return make_tmaps(p);
}

// own planes [z_own0, z_own1) of the local grid; neighbour handles (null = no neighbour on that side); up_ghost_z = first
// ghost plane index, in the upper neighbour's local grid, that receives this rank's first four owned planes.
int fwi_fd_slab_connect(fwi_fd2d* p, int z_own0, int z_own1, const void* up_handle, const uint64_t* up_offsets, int up_ghost_z,
                        const void* dn_handle, const uint64_t* dn_offsets) {
    FWI_REQUIRE(p && p->ny > 1, "fwi_fd_slab_connect: needs a 3-D plan");
    FWI_REQUIRE(z_own0 >= 0 && z_own1 <= p->nz && z_own1 - z_own0 >= 2 * kHalo, "fwi_fd_slab_connect: owned range [%d, %d) invalid for nz=%d", z_own0, z_own1, p->nz);
    FWI_REQUIRE(!p->free_surface || !up_handle, "fwi_fd_slab_connect: a free-surface plan cannot have an upper neighbour; only the slab that owns z = 0 has the surface");
    DeviceGuard g(p->device);
    FWI_CUDA(cudaStreamSynchronize(p->work));
    drop_graphs(p);
    const void* hs[2] = {up_handle, dn_handle};
    const uint64_t* offs[2] = {up_offsets, dn_offsets};
    for (int s = 0; s < 2; ++s) {
        if (!hs[s]) continue;
        FWI_REQUIRE(offs[s], "fwi_fd_slab_connect: offsets missing");
        cudaIpcMemHandle_t h;
        memcpy(&h, hs[s], sizeof(h));
        FWI_CUDA(cudaIpcOpenMemHandle(&p->peer_arena[s], h, cudaIpcMemLazyEnablePeerAccess));
        p->peer_ipc[s] = true;
        for (int i = 0; i < 8; ++i) p->peer_fld_off[s][i] = (size_t)offs[s][i];
        p->peer_flags_off[s] = (size_t)offs[s][8];
    }
    return slab_finish_connect(p, z_own0, z_own1, up_ghost_z);
}

// Same protocol between plans of ONE process (peers are other plans on this or a peer-accessible device): used by the
// single-GPU protocol test, where two small plans run on two streams of the same GPU.
int fwi_fd_slab_connect_local(fwi_fd2d* p, int z_own0, int z_own1, fwi_fd2d* up, int up_ghost_z, fwi_fd2d* dn) {
    FWI_REQUIRE(p && p->ny > 1, "fwi_fd_slab_connect_local: needs a 3-D plan");
    FWI_REQUIRE(z_own0 >= 0 && z_own1 <= p->nz && z_own1 - z_own0 >= 2 * kHalo, "fwi_fd_slab_connect_local: owned range [%d, %d) invalid for nz=%d", z_own0, z_own1, p->nz);
    FWI_REQUIRE(!p->free_surface || !up, "fwi_fd_slab_connect_local: a free-surface plan cannot have an upper neighbour; only the slab that owns z = 0 has the surface");
    DeviceGuard g(p->device);
    FWI_CUDA(cudaStreamSynchronize(p->work));
    drop_graphs(p);
    fwi_fd2d* nb[2] = {up, dn};
    for (int s = 0; s < 2; ++s) {
        if (!nb[s]) continue;
        FWI_REQUIRE(nb[s]->ny == p->ny && nb[s]->px == p->px, "fwi_fd_slab_connect_local: neighbour has a different plane shape");
        p->peer_arena[s] = nb[s]->arena;
        p->peer_ipc[s] = false;
        for (int i = 0; i < 8; ++i) p->peer_fld_off[s][i] = (size_t)((char*)nb[s]->fld[i] - (char*)nb[s]->arena);
        p->peer_flags_off[s] = (size_t)((char*)nb[s]->sync_area - (char*)nb[s]->arena);
    }
    return slab_finish_connect(p, z_own0, z_own1, up_ghost_z);
}

int fwi_fd_slab_set_timeout(fwi_fd2d* p, double milliseconds) {
    FWI_REQUIRE(p && milliseconds > 0, "fwi_fd_slab_set_timeout: bad arguments");
    p->slab_timeout_cycles = (long long)(milliseconds * 1.9e6);      // clock64 ticks at ~1.9 GHz
    drop_graphs(p);                                                   // the timeout is a kernel argument
    return FWI_OK;
}

// Clears the error flag after the caller has dealt with a timeout (all ranks together, with the device idle).
int fwi_fd_slab_clear_error(fwi_fd2d* p) {
    FWI_REQUIRE(p, "fwi_fd_slab_clear_error: NULL plan");
    DeviceGuard g(p->device);
    FWI_CUDA(cudaDeviceSynchronize());
    FWI_CUDA(cudaMemset(p->sync_area + kSyncError, 0, sizeof(int)));
    return FWI_OK;
}

int fwi_fd_slab_error(fwi_fd2d* p, int* error_out) {
    FWI_REQUIRE(p && error_out, "fwi_fd_slab_error: bad arguments");
    DeviceGuard g(p->device);
    FWI_CUDA(cudaMemcpy(error_out, p->sync_area + kSyncError, sizeof(int), cudaMemcpyDeviceToHost));
    return FWI_OK;
}

// grad_dev (dense grid) += (2 / v) * imaging accumulator
int fwi_fd_finalize_gradient(fwi_fd2d* p, float* grad_dev, void* stream) {
    FWI_REQUIRE(p && grad_dev, "fwi_fd_finalize_gradient: bad arguments");
    DeviceGuard g(p->device);
    return launch_finalize(p, grad_dev, (cudaStream_t)stream);
}


// Small persistent device scratch per GPU for the plan-less reductions below.  (cudaMallocAsync / cudaFreeAsync around a
// synchronising call hands the block back to the driver every time: measured 8 ms per call with 25 GB allocated, which
// was 40 % of a config-3 line search.)  One caller per device at a time: both users synchronise before returning.
static void* device_scratch() {
    static void* scratch[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (!scratch[dev] && cudaMalloc(&scratch[dev], 256) != cudaSuccess) { cudaGetLastError(); scratch[dev] = nullptr; }
    return scratch[dev];
}

int fwi_fd_misfit(const float* syn_dev, const float* obs_dev, int64_t n, float* resid_dev, double* misfit_host, void* stream) {
    FWI_REQUIRE(syn_dev && obs_dev && resid_dev && misfit_host && n >= 0, "fwi_fd_misfit: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    double* dJ = (double*)device_scratch();
    FWI_REQUIRE(dJ, "fwi_fd_misfit: no device scratch");
    FWI_CUDA(cudaMemsetAsync(dJ, 0, sizeof(double), st));
    if (n > 0) fd_residual_kernel<<<(unsigned)std::min<int64_t>(1024, (n + 255) / 256), 256, 0, st>>>(syn_dev, obs_dev, n, resid_dev, dJ);
    FWI_CUDA(cudaGetLastError());
    FWI_CUDA(cudaMemcpyAsync(misfit_host, dJ, sizeof(double), cudaMemcpyDeviceToHost, st));
    FWI_CUDA(cudaStreamSynchronize(st));
    return FWI_OK;
}

int fwi_fd_model_update(float* v_dev, const float* grad_dev, int64_t n, float step, float vmin, float vmax, void* stream) {
    FWI_REQUIRE(v_dev && grad_dev && n >= 0 && vmin <= vmax, "fwi_fd_model_update: bad arguments");
    if (n > 0) fd_update_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(v_dev, grad_dev, step, vmin, vmax, n);
    FWI_CUDA(cudaGetLastError());
    return FWI_OK;
}

int fwi_fd_absmax(const float* x_dev, int64_t n, float* out_host, void* stream) {
    FWI_REQUIRE(x_dev && out_host && n >= 1, "fwi_fd_absmax: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned int* d = (unsigned int*)device_scratch();
    FWI_REQUIRE(d, "fwi_fd_absmax: no device scratch");
    d += 16;                                             // its own slot (the misfit uses the first 8 bytes)
    FWI_CUDA(cudaMemsetAsync(d, 0, sizeof(unsigned int), st));
    fd_absmax_kernel<<<(unsigned)std::min<int64_t>(1024, (n + 255) / 256), 256, 0, st>>>(x_dev, n, d);
    FWI_CUDA(cudaGetLastError());
    unsigned int h = 0;
    FWI_CUDA(cudaMemcpyAsync(&h, d, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    FWI_CUDA(cudaStreamSynchronize(st));
    memcpy(out_host, &h, sizeof(float));
    return FWI_OK;
}

}  // extern "C"
