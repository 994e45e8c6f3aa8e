// Track B, 2-D: temporally blocked step kernel - TWO leapfrog steps per pass.
//
// A CTA owns a 120 (x) x CZ (z) core tile.  One TMA transaction group stages, on one mbarrier,
//     u_n      on the core +- 8  (136 x (CZ+16) box, out-of-grid zero-filled = Dirichlet),
//     u_{n-1}  on the core +- 4  (128 x (CZ+8) box)   and   m on the core +- 4,
// then
//   step 1: u_{n+1} = g (2 u_n - g u_{n-1} + m (lap u_n + f_n)) on the core +- 4 (128 columns = 32 lanes x float4),
//           written over u_{n-1} IN SHARED MEMORY (the update is pointwise in u_{n-1});
//           sources falling in the core +- 4 are injected into the shared copy;
//   step 2: u_{n+2} = g (2 u_{n+1} - g u_n + m (lap u_{n+1} + f_{n+1})) on the core, straight from shared memory.
// Both new time levels of the core go to a second pair of global buffers (neighbouring CTAs still read the halo
// of the input pair), so the host ping-pongs between two buffer pairs.  Per two steps a point costs one read of
// u_n (x1.7 halo), u_{n-1} (x1.33), m (x1.33) and two writes: ~12.7 B per step instead of ~17, half the launches,
// and the adjoint touches its imaging accumulator once per two steps.  Redundant arithmetic: 1.17x.
// z-neighbours rotate through a register window, x-neighbours are two extra LDS.128, as in the one-step kernel.
#pragma once
#include "fd_common.cuh"

namespace fwi {

constexpr int kT2CX = 120;                 // core columns (30 lanes x float4)
constexpr int kT2W1 = 128;                 // step-1 columns
constexpr int kT2W0 = 136;                 // u_n box columns

struct Tb2Args {
    float* out_new;        // u_{n+2}
    float* out_mid;        // u_{n+1}
    const float* gx;
    const float* gz;
    const float* m;        // global m (fix-ups only)
    float* snap1;          // w of sub-step 1 (forward: written; adjoint: read)
    float* snap2;          // w of sub-step 2
    float* acc;
    int nx, nz, px;
    PointListDev inj_ext;  // injection points binned by the tiles whose core +- 4 contains them (duplicates across tiles)
    PointListDev inj_own;  // injection points binned by owning core tile
    const float* inj1;     // value row of sub-step 1 / 2
    const float* inj2;
    PointListDev rec;      // receivers binned by owning core tile (forward only)
    float* rec1;
    float* rec2;
};

// FS: free surface at z = 0 (spec B6).  The top row of CTAs mirrors the u_n rows above the surface after the TMA arrives,
// and the u_{n+1} rows above it again after step 1 and its injection; step 1's own values above the surface are discarded.
template <int CZ, int NW, int MODE, bool FS>
__global__ void __launch_bounds__(NW * 32) fd2d_tb2_kernel(const __grid_constant__ CUtensorMap tm_cur,
                                                            const __grid_constant__ CUtensorMap tm_old,
                                                            const __grid_constant__ CUtensorMap tm_m, Tb2Args a) {
    constexpr int Z0 = CZ + 16, Z1 = CZ + 8;
    constexpr int RP1 = Z1 / NW, RP2 = CZ / NW;
    static_assert(Z1 % NW == 0 && CZ % NW == 0, "rows must split evenly over the warps");
    extern __shared__ __align__(128) float smem[];
    float* sCur = smem;                         // [Z0][136]
    float* sOld = smem + Z0 * kT2W0;            // [Z1][128]  u_{n-1}, then u_{n+1}
    float* sM = sOld + Z1 * kT2W1;              // [Z1][128]
    __shared__ __align__(8) uint64_t bar;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * kT2CX, z0 = blockIdx.y * CZ;
    // Prologue that does not depend on the previous pass (programmatic dependent launch, see fd2d_step_kernel): the
    // barrier, the sponge profile and the TMA load of m, which never changes inside a sweep.
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
        fence_proxy_async();
        mbar_expect_tx(&bar, (Z0 * kT2W0 + 2 * Z1 * kT2W1) * (uint32_t)sizeof(float));
        tma_load_2d(sM, &tm_m, x0 - 4, z0 - 4, &bar);
    }
    const int x = x0 - 4 + 4 * lane;                         // first column of this lane's float4 (step-1 frame)
    float gxs[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) gxs[q] = __ldg(a.gx + min(max(x + q, 0), a.px - 1));
    const int tid = blockIdx.y * gridDim.x + blockIdx.x;
    griddep_wait();                                          // the previous pass is complete and visible
    if (threadIdx.x == 0) {
        tma_load_2d(sCur, &tm_cur, x0 - 8, z0 - 8, &bar);
        tma_load_2d(sOld, &tm_old, x0 - 4, z0 - 4, &bar);
    }
    __syncthreads();

    mbar_wait(&bar, 0);
    if (FS && z0 == 0) {                                     // uniform per CTA; sCur row 8 is z = 0
        mirror_rows(sCur, kT2W0, 8, kT2W0);
        __syncthreads();
    }

    // ------------------------------------------------------------------ step 1 on the core +- 4
    {
        const int r0 = warp * RP1;                           // first R1 row of this warp; R1 row r <-> z = z0 - 4 + r
        float4 win[9];
        const float* tcol = sCur + r0 * kT2W0 + 4 + 4 * lane;   // sCur row (r0 + k) <-> z - 4 + k of the first output
#pragma unroll
        for (int k = 0; k < 8; ++k) win[k + 1] = ld4(tcol + k * kT2W0);
#pragma unroll
        for (int r = 0; r < RP1; ++r) {
            const int row = r0 + r, z = z0 - 4 + row;
#pragma unroll
            for (int k = 0; k < 8; ++k) win[k] = win[k + 1];
            win[8] = ld4(tcol + (r + 8) * kT2W0);
            const float* trow = sCur + (row + 4) * kT2W0 + 4 * lane;
            const float4 L = ld4(trow), R = ld4(trow + 8), C = win[4];
            const float ax[12] = {L.x, L.y, L.z, L.w, C.x, C.y, C.z, C.w, R.x, R.y, R.z, R.w};
            float zc[9][4];
#pragma unroll
            for (int k = 0; k < 9; ++k) { zc[k][0] = win[k].x; zc[k][1] = win[k].y; zc[k][2] = win[k].z; zc[k][3] = win[k].w; }
            const float4 o4 = ld4(sOld + row * kT2W1 + 4 * lane), m4 = ld4(sM + row * kT2W1 + 4 * lane);
            const float ov[4] = {o4.x, o4.y, o4.z, o4.w}, mv[4] = {m4.x, m4.y, m4.z, m4.w};
            const float gzv = __ldg(a.gz + min(max(z, 0), a.nz - 1));
            float wv[4], nv[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float c = ax[4 + q], g = gxs[q] * gzv;
                float lap = (2.0f * kC0) * c;
                lap = fmaf(kC1, (ax[3 + q] + ax[5 + q]) + (zc[3][q] + zc[5][q]), lap);
                lap = fmaf(kC2, (ax[2 + q] + ax[6 + q]) + (zc[2][q] + zc[6][q]), lap);
                lap = fmaf(kC3, (ax[1 + q] + ax[7 + q]) + (zc[1][q] + zc[7][q]), lap);
                lap = fmaf(kC4, (ax[0 + q] + ax[8 + q]) + (zc[0][q] + zc[8][q]), lap);
                wv[q] = lap;
                nv[q] = g * fmaf(mv[q], lap, fmaf(-g, ov[q], 2.0f * c));
            }
            st4(sOld + row * kT2W1 + 4 * lane, make_float4(nv[0], nv[1], nv[2], nv[3]));
            if (MODE == STEP_FWD_SAVE) {
                // w_n of the core points goes to the snapshot (lanes 1..30, rows 4 .. CZ+3 of R1)
                if (lane >= 1 && lane <= 30 && row >= 4 && row < CZ + 4 && z < a.nz && x < a.px)
                    st4_stream(a.snap1 + (size_t)z * a.px + x, make_float4(wv[0], wv[1], wv[2], wv[3]));
            }
        }
    }
    __syncthreads();
    // sources / residuals of sub-step 1 that fall into the core +- 4 are injected into the shared copy of u_{n+1}
    {
        const int i0 = a.inj_ext.tile_ptr ? a.inj_ext.tile_ptr[tid] : 0, i1 = a.inj_ext.tile_ptr ? a.inj_ext.tile_ptr[tid + 1] : 0;
        if (i1 > i0) {
            for (int e = i0 + threadIdx.x; e < i1; e += blockDim.x) {
                const int off = a.inj_ext.off[e];
                const int z = off / a.px, xx = off - z * a.px;
                const float val = a.inj1[a.inj_ext.id[e]];
                const float gm = a.gx[xx] * a.gz[z] * a.m[off];
                atomicAdd(sOld + (z - (z0 - 4)) * kT2W1 + (xx - (x0 - 4)), gm * val);
                const bool own = (z >= z0 && z < z0 + CZ && xx >= x0 && xx < x0 + kT2CX);
                if (MODE == STEP_FWD_SAVE && own) atomicAdd(a.snap1 + off, val);      // w_n includes f_n
            }
            __syncthreads();
        }
    }
    if (FS && z0 == 0) {                                     // sOld row 4 is z = 0; the injected u_{n+1} is mirrored
        mirror_rows(sOld, kT2W1, 4, kT2W1);
        __syncthreads();
    }

    // ------------------------------------------------------------------ step 2 on the core
    {
        const int r0 = warp * RP2;                           // core row; sOld row (r0 + r + 4) is the centre
        const bool lane_ok = (lane >= 1 && lane <= 30) && x < a.px;
        float4 win[9];
        const float* tcol = sOld + r0 * kT2W1 + 4 * lane;    // sOld row (r0 + k) <-> core row r0 - 4 + k
#pragma unroll
        for (int k = 0; k < 8; ++k) win[k + 1] = ld4(tcol + k * kT2W1);
#pragma unroll
        for (int r = 0; r < RP2; ++r) {
            const int crow = r0 + r, z = z0 + crow;
#pragma unroll
            for (int k = 0; k < 8; ++k) win[k] = win[k + 1];
            win[8] = ld4(tcol + (r + 8) * kT2W1);
            if (lane_ok && z < a.nz) {
                // x neighbours of u_{n+1}: columns x-4 .. x+7 of sOld row crow+4 (lanes 1..30 stay inside the 128 columns)
                const float* trow = sOld + (crow + 4) * kT2W1 + 4 * lane;
                const float4 L = ld4(trow - 4), R = ld4(trow + 4), C = win[4];
                const float ax[12] = {L.x, L.y, L.z, L.w, C.x, C.y, C.z, C.w, R.x, R.y, R.z, R.w};
                float zc[9][4];
#pragma unroll
                for (int k = 0; k < 9; ++k) { zc[k][0] = win[k].x; zc[k][1] = win[k].y; zc[k][2] = win[k].z; zc[k][3] = win[k].w; }
                const float4 o4 = ld4(sCur + (crow + 8) * kT2W0 + 4 + 4 * lane);       // u_n at the same point
                const float4 m4 = ld4(sM + (crow + 4) * kT2W1 + 4 * lane);
                const float ov[4] = {o4.x, o4.y, o4.z, o4.w}, mv[4] = {m4.x, m4.y, m4.z, m4.w};
                const float gzv = __ldg(a.gz + z);
                float wv[4], nv[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float c = ax[4 + q], g = gxs[q] * gzv;
                    float lap = (2.0f * kC0) * c;
                    lap = fmaf(kC1, (ax[3 + q] + ax[5 + q]) + (zc[3][q] + zc[5][q]), lap);
                    lap = fmaf(kC2, (ax[2 + q] + ax[6 + q]) + (zc[2][q] + zc[6][q]), lap);
                    lap = fmaf(kC3, (ax[1 + q] + ax[7 + q]) + (zc[1][q] + zc[7][q]), lap);
                    lap = fmaf(kC4, (ax[0 + q] + ax[8 + q]) + (zc[0][q] + zc[8][q]), lap);
                    wv[q] = lap;
                    nv[q] = g * fmaf(mv[q], lap, fmaf(-g, ov[q], 2.0f * c));
                }
                const size_t off = (size_t)z * a.px + x;
                st4(a.out_new + off, make_float4(nv[0], nv[1], nv[2], nv[3]));
                st4(a.out_mid + off, C);                                               // u_{n+1}, injection included
                if (MODE == STEP_FWD_SAVE) st4_stream(a.snap2 + off, make_float4(wv[0], wv[1], wv[2], wv[3]));
                if (MODE == STEP_ADJ) {
                    const float4 s1 = ld4_stream(a.snap1 + off), s2 = ld4_stream(a.snap2 + off);
                    float4 c4 = ld4(a.acc + off);
                    c4.x = fmaf(nv[0], s2.x, fmaf(C.x, s1.x, c4.x)); c4.y = fmaf(nv[1], s2.y, fmaf(C.y, s1.y, c4.y));
                    c4.z = fmaf(nv[2], s2.z, fmaf(C.z, s1.z, c4.z)); c4.w = fmaf(nv[3], s2.w, fmaf(C.w, s1.w, c4.w));
                    st4(a.acc + off, c4);
                }
            }
        }
    }

    // ------------------------------------------------------------------ owner fix-ups: sub-step-1 receivers, sub-step-2 injection + receivers
    const int j0 = a.inj_own.tile_ptr ? a.inj_own.tile_ptr[tid] : 0, j1 = a.inj_own.tile_ptr ? a.inj_own.tile_ptr[tid + 1] : 0;
    const int r0 = a.rec.tile_ptr ? a.rec.tile_ptr[tid] : 0, r1 = a.rec.tile_ptr ? a.rec.tile_ptr[tid + 1] : 0;
    if (j1 > j0 || r1 > r0) {
        for (int e = r0 + threadIdx.x; e < r1; e += blockDim.x) {        // trace row of sub-step 1 from the shared u_{n+1}
            const int off = a.rec.off[e];
            const int z = off / a.px, xx = off - z * a.px;
            a.rec1[a.rec.id[e]] = sOld[(z - (z0 - 4)) * kT2W1 + (xx - (x0 - 4))];
        }
        __syncthreads();
        for (int e = j0 + threadIdx.x; e < j1; e += blockDim.x) {
            const int off = a.inj_own.off[e];
            const int z = off / a.px, xx = off - z * a.px;
            const float val = a.inj2[a.inj_own.id[e]];
            const float gm = a.gx[xx] * a.gz[z] * a.m[off];
            atomicAdd(a.out_new + off, gm * val);
            if (MODE == STEP_FWD_SAVE) atomicAdd(a.snap2 + off, val);
            if (MODE == STEP_ADJ) atomicAdd(a.acc + off, gm * val * a.snap2[off]);
        }
        if (r1 > r0) {
            __syncthreads();
            for (int e = r0 + threadIdx.x; e < r1; e += blockDim.x) a.rec2[a.rec.id[e]] = __ldcg(a.out_new + a.rec.off[e]);
        }
    }
}

}  // namespace fwi
