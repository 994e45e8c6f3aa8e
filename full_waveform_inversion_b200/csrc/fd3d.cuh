// Track B, 3-D: 25-point (8th-order) leapfrog step, marching along z with a TMA plane pipeline.
//
// Layout [nz][ny][px] fp32, x contiguous.  A CTA owns a 128 (x) x 16 (y) column of the grid over a chunk of z and
// marches through it plane by plane:
//   * two dedicated producer warps (one elected lane each) feed shared memory by TMA with full/empty mbarrier pairs:
//     the first keeps a ring of NP = 8 u_n planes filled (one 136 x 24 x 1 box per z plane, halo included,
//     out-of-grid zero-filled = Dirichlet), the second a 4-deep ring of u_{n-1} / m planes (128 x 16 x 1 boxes).
//     They are separate warps on purpose: a single producer that blocks on one ring's empty barrier also holds back
//     the other ring's loads, which cost 25 % of the step (290 -> 390 Gpt/s at 512^3);
//   * 8 consumer warps own two y rows each, a lane owns a float4 of x.  The nine z-neighbours of every output live
//     in a register window that rotates as the march advances (one LDS.128 per new plane); the x and y neighbours
//     come from the centre plane, which is still in the ring four planes behind the newest one;
//   * u_{n+1} overwrites u_{n-1} in place (plain per-warp global loads of u_{n-1} / m instead of the second ring cost
//     40 % of the step); snapshot write / snapshot read + imaging are fused exactly as in 2-D; the CTA applies its own
//     source / receiver points at the end; the Born step reads w_n and dm from global memory beside the adjoint's
//     operands (not through the u_{n-1} / m ring) and adds dm * w_n inside the update.
// Algorithmic traffic: 16 B per point update (+ halo re-reads that hit L2).
#pragma once
#include "fd_common.cuh"

namespace fwi {

constexpr int k3BX = 128, k3NP = 8;                                // tile width, u_n ring depth
constexpr int k3RPW = 2;                                            // y rows per consumer warp
constexpr int k3SX = k3BX + 2 * kHalo;                              // 136
constexpr int k3NO = 4, k3OmLead = 5, k3Prod = 2;                   // u_{n-1}/m plane ring depth; issued 3 planes before use; producer warps
// The tile height BY is a template parameter: 16 rows (8 consumer warps) or 14 rows (7 consumer warps).  512-wide planes
// give 4 x 32 = 128 tiles of 16 rows but 4 x 37 = 148 tiles of 14 rows - exactly one per SM, which removes the 25 % tail of
// a second wave that only 108 CTAs fill (measured on 4-GPU slabs: 0.78 -> see DESIGN.md); fwi_fd2d picks per plan.
template <int BY> struct T3 {
    static constexpr int CW = BY / k3RPW;                           // consumer warps
    static constexpr int SY = BY + 2 * kHalo;
    static constexpr int PlaneFloats = k3SX * SY;                   // BY = 16: 3264 floats = 13056 B; BY = 14: 2992 floats = 11968 B
    static constexpr int PlaneStride = (PlaneFloats + 31) / 32 * 32; // ring slots start on 128-byte lines (TMA destination alignment)
    static constexpr int OmFloats = k3BX * BY;
    static constexpr int Threads = (CW + k3Prod) * 32;
    static constexpr size_t Smem = ((size_t)k3NP * PlaneStride + (size_t)k3NO * 2 * OmFloats) * sizeof(float);
    static_assert(BY % k3RPW == 0 && (OmFloats * 4) % 128 == 0, "u_{n-1} / m planes must stay 128-byte multiples");
};

struct Step3DArgs {
    float* oldnew;
    const float* m;
    const float* gx;
    const float* gy;
    const float* gz;
    float* snap;
    const float* snap_prev;   // ADJ2: snapshot paired with the previous adjoint step's field (= u_n of this launch)
    float* acc;
    int nx, ny, nz, px, zchunk;
    PointListDev inj;
    const float* inj_vals;
    PointListDev rec;
    float* rec_out;
    // ---- slab decomposition over NVLink peer memory (all null / zero for a single-GPU plan) -----------------------
    int z_own0, z_own1;        // owned plane range of the local grid (ghost planes lie outside and are never computed)
    int last_desc;             // 1: the last z chunk marches downwards, so that the lower boundary planes come first
    float* peer_up;            // the upper / lower neighbour's copy of `oldnew` (peer-mapped), or null
    float* peer_dn;
    int peer_up_z;             // first ghost plane (in the upper neighbour's local grid) that receives my first 4 owned planes
    int* sync;                 // this GPU's sync words (SlabSync below)
    int* flag_peer_up;         // where I announce "boundary planes of launch k pushed" to the upper / lower neighbour
    int* flag_peer_dn;
    long long timeout_cycles;  // bounded spin on a neighbour's flag
    const float* dm;           // BORN: model perturbation dm = (2 m / v) dv, pitched like m
};

// sync words of one plan (ints inside its arena; the neighbours write [0] / [1] through their peer mapping)
enum SlabSync { kSyncFlagUp = 0,   // written by the upper neighbour: its launch k has pushed my upper ghost planes
                kSyncFlagDn = 1,   // same from the lower neighbour
                kSyncDoneAll = 2,  // CTAs of the running launch that have finished
                kSyncError = 3,    // a wait timed out: every later launch returns at once, the host raises
                kSyncStep = 4,     // launches completed so far - the step id lives on the device, so the time loop
                                   // can be replayed from a CUDA graph
                kSyncDoneUp = 5,   // CTAs that have pushed their share of the upper / lower boundary planes
                kSyncDoneDn = 6 };

__device__ __forceinline__ int ld_acquire_sys(const int* p) {
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(int* p, int v) {
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ---- slab protocol helpers -----------------------------------------------------------------------------------------
// One consumer warp / the whole CTA reports that its share of a boundary side is in the neighbour's memory; the last
// reporter of the side publishes the step id there (system-scope release).  Callers have fenced their peer stores.
__device__ __forceinline__ void slab_side_done(const Step3DArgs& a, int side, unsigned ctas_on_side, int signal_id) {
    unsigned int* cnt = (unsigned int*)(a.sync + (side == 0 ? kSyncDoneUp : kSyncDoneDn));
    __threadfence();
    if (atomicAdd(cnt, 1u) == ctas_on_side - 1) {
        *cnt = 0;
        __threadfence_system();
        st_release_sys(side == 0 ? a.flag_peer_up : a.flag_peer_dn, signal_id);
    }
}

// Waits (one thread) until the neighbours have pushed everything up to launch `need`; used before a run's memsets /
// checkpoint restores so that no late push of the previous run lands on freshly written ghost planes.
__global__ void fd3d_slab_sync_kernel(int* sync, int has_up, int has_dn, long long timeout_cycles) {
    if (threadIdx.x != 0 || sync[kSyncError]) return;
    const int need = sync[kSyncStep];
    for (int side = 0; side < 2; ++side) {
        if ((side == 0 && !has_up) || (side == 1 && !has_dn)) continue;
        const long long t0 = clock64();
        while (ld_acquire_sys(sync + side) < need) {
            if (clock64() - t0 > timeout_cycles) { atomicExch(sync + kSyncError, 1); return; }
            __nanosleep(200);
        }
    }
}

// FS: free surface at z = 0 (spec B6).  For a plane z < 0 the producer loads plane -z and the consumers negate it as it enters
// their register windows (u[-k] = -u[k]); centre planes never lie above the surface, so the x / y neighbours are unchanged.
// The planes above the surface are the first four of the chunk that starts at z = 0, which marches upwards: a chunk marches
// downwards only when it is the last of two or more, and chunks hold at least 8 planes (make_tmaps3), so a downward march
// ends at z >= 4.  The producer handles both directions; the consumers test only while priming (testing every plane of the
// march as well raised the ADJ2 instance's spills from 24 to 92 bytes at BY = 16).
template <int MODE, int BY, bool FS>
__global__ void __launch_bounds__(T3<BY>::Threads, 1) fd3d_step_kernel(const __grid_constant__ CUtensorMap tm_cur,
                                                                       const __grid_constant__ CUtensorMap tm_old,
                                                                       const __grid_constant__ CUtensorMap tm_m, Step3DArgs a) {
    constexpr int k3BY = BY, k3CW = T3<BY>::CW, k3PlaneFloats = T3<BY>::PlaneFloats, k3PlaneStride = T3<BY>::PlaneStride, k3OmFloats = T3<BY>::OmFloats;
    extern __shared__ __align__(128) float ring[];                   // [NP][SY][SX] u_n planes, then [NO][2][BY][BX] u_{n-1} / m planes
    float* om_ring = ring + (size_t)k3NP * k3PlaneStride;
    __shared__ __align__(8) uint64_t full_bar[k3NP], empty_bar[k3NP], om_full[k3NO], om_empty[k3NO];
    __shared__ int slab_state[4];                  // [0] step id of this launch, [1] abort, [2]/[3] consumer warps done with the upper / lower boundary

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * k3BX, y0 = blockIdx.y * k3BY;
    const int zc0 = a.z_own0 + blockIdx.z * a.zchunk, zc1 = min(a.z_own1, zc0 + a.zchunk);
    const int nout = zc1 - zc0;                   // output planes of this CTA
    const int nplanes = nout + 2 * kHalo;         // planes zc0-4 .. zc1+3
    // march direction: upwards in z, except the last chunk of a slab with a lower neighbour, which marches downwards so
    // that BOTH boundaries of the slab are computed (and pushed to the neighbours) in the first four iterations of
    // their CTAs and the NVLink transfer + the neighbours' wait hide behind the interior planes.  The stencil is
    // symmetric in z, so the register window works unchanged in either direction.
    const bool desc = a.last_desc && blockIdx.z == gridDim.z - 1;
    const int zbeg = desc ? zc1 - 1 : zc0, zstep = desc ? -1 : 1;       // output plane j is z = zbeg + zstep * j
    const bool slab = a.peer_up != nullptr || a.peer_dn != nullptr;
    const int cta = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    const int i0 = a.inj.tile_ptr ? a.inj.tile_ptr[cta] : 0, i1 = a.inj.tile_ptr ? a.inj.tile_ptr[cta + 1] : 0;
    const int r0 = a.rec.tile_ptr ? a.rec.tile_ptr[cta] : 0, r1 = a.rec.tile_ptr ? a.rec.tile_ptr[cta + 1] : 0;
    // which boundary sides this CTA owns (zchunk >= 8 in slab mode, so a 4-plane boundary never straddles two chunks)
    const bool own_up = a.peer_up && blockIdx.z == 0, own_dn = a.peer_dn && blockIdx.z == gridDim.z - 1;
    // CTAs with injection points report their sides only after the sparse fix-ups (a source may sit in a boundary plane)
    const bool early = i1 == i0;

    if (threadIdx.x == 0) {
        slab_state[0] = 0; slab_state[1] = 0; slab_state[2] = 0; slab_state[3] = 0;
        if (slab) {
            // The step id lives on the device (launches completed so far): this launch needs the neighbours' pushes of
            // launch `id` and publishes `id + 1`.  Ghost planes of u_n are written by the neighbours straight into this
            // GPU's memory; only the CTAs that read them wait (bounded spin: a dead neighbour raises the error flag).
            const int id = a.sync[kSyncStep];
            slab_state[0] = id;
            if (a.sync[kSyncError]) slab_state[1] = 1;
            else {
                for (int side = 0; side < 2; ++side) {
                    if (!(side == 0 ? own_up : own_dn)) continue;
                    const long long t0 = clock64();
                    while (ld_acquire_sys(a.sync + side) < id) {
                        if (clock64() - t0 > a.timeout_cycles) { atomicExch(a.sync + kSyncError, 1); slab_state[1] = 1; break; }
                        __nanosleep(100);
                    }
                }
                // peer GPUs wrote the ghost planes with generic-proxy stores; TMA reads them through the async proxy
                asm volatile("fence.proxy.async;" ::: "memory");
            }
        }
#pragma unroll
        for (int i = 0; i < k3NP; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], k3CW); }
#pragma unroll
        for (int i = 0; i < k3NO; ++i) { mbar_init(&om_full[i], 1); mbar_init(&om_empty[i], k3CW); }
        fence_mbar_init();
        fence_proxy_async();
    }
    __syncthreads();
    if (slab_state[1]) return;                     // a neighbour is gone: do not compute on stale ghosts, do not spin again
    const int signal_id = slab_state[0] + 1;
    const unsigned ctas_per_side = gridDim.x * gridDim.y;

    if (warp >= k3CW) {
        // ---------------- producer warp(s): one lane feeds the u_n plane ring, one the u_{n-1} / m ring
        const bool do_u = warp == k3CW, do_om = warp == k3CW + k3Prod - 1;
        if (lane == 0) {
            // tick t: u_n plane t, then the u_{n-1} / m planes of output row t - k3OmLead (3 planes before they are used)
            for (int t = 0; t < nplanes + k3OmLead; ++t) {
                if (do_u && t < nplanes) {
                    const int slot = t % k3NP;
                    if (t >= k3NP) mbar_wait(&empty_bar[slot], ((t / k3NP) - 1) & 1);
                    mbar_expect_tx(&full_bar[slot], k3PlaneFloats * (uint32_t)sizeof(float));
                    const int zp = zbeg + zstep * (t - kHalo);
                    tma_load_3d(ring + (size_t)slot * k3PlaneStride, &tm_cur, x0 - kHalo, y0 - kHalo, (FS && zp < 0) ? -zp : zp, &full_bar[slot]);
                }
                const int j = t - k3OmLead;
                if (do_om && j >= 0 && j < nout) {
                    const int slot = j % k3NO;
                    if (j >= k3NO) mbar_wait(&om_empty[slot], ((j / k3NO) - 1) & 1);
                    float* dst = om_ring + (size_t)slot * 2 * k3OmFloats;
                    mbar_expect_tx(&om_full[slot], 2 * k3OmFloats * (uint32_t)sizeof(float));
                    tma_load_3d(dst, &tm_old, x0, y0, zbeg + zstep * j, &om_full[slot]);
                    tma_load_3d(dst + k3OmFloats, &tm_m, x0, y0, zbeg + zstep * j, &om_full[slot]);
                }
            }
        }
    } else {
        // ---------------- consumer warps
        const int x = x0 + 4 * lane;
        const int yl = k3RPW * warp;                   // first of this warp's rows inside the tile
        const bool col_ok = x < a.px;
        float4 gx4 = make_float4(1.f, 1.f, 1.f, 1.f);
        if (col_ok) gx4 = ld4(a.gx + x);
        float gyv[k3RPW];
#pragma unroll
        for (int r = 0; r < k3RPW; ++r) gyv[r] = (y0 + yl + r < a.ny) ? __ldg(a.gy + y0 + yl + r) : 1.f;

        float4 win[k3RPW][9];
        auto own = [&](int p, int r) {                 // this lane's element of row r in ring plane p
            return ld4(ring + (size_t)(p % k3NP) * k3PlaneStride + (yl + r + kHalo) * k3SX + kHalo + 4 * lane);
        };
        auto neg = [](float4 v) { return make_float4(-v.x, -v.y, -v.z, -v.w); };
        // prime with planes 0..7 (the four behind the first output plane and the first four); planes 0..3 are never
        // centre planes -> release them
        for (int p = 0; p < 2 * kHalo; ++p) {
            mbar_wait(&full_bar[p % k3NP], (p / k3NP) & 1);
#pragma unroll
            for (int r = 0; r < k3RPW; ++r) {
                win[r][p + 1] = own(p, r);
                if (FS && zbeg + zstep * (p - kHalo) < 0) win[r][p + 1] = neg(win[r][p + 1]);     // mirrored plane -z
            }
            if (p < kHalo) {
                __syncwarp();
                if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&empty_bar[p % k3NP])) : "memory");
            }
        }
        // byte distance from a point of `oldnew` to its copy in the neighbour's ghost planes
        const long long dup = a.peer_up ? (long long)((char*)(a.peer_up + (size_t)(a.peer_up_z - a.z_own0) * a.ny * a.px) - (char*)a.oldnew) : 0;
        const long long ddn = a.peer_dn ? (long long)((char*)a.peer_dn - (char*)(a.oldnew + (size_t)(a.z_own1 - kHalo) * a.ny * a.px)) : 0;
        for (int iz = 0; iz < nout; ++iz) {
            const int z = zbeg + zstep * iz;
            const int ptop = iz + 2 * kHalo, pmid = iz + kHalo;
            // global operands first: their latency overlaps the barrier wait and the shared-memory reads
            float4 o4[k3RPW], m4[k3RPW], s4[k3RPW], c4[k3RPW], sp4[k3RPW], d4[k3RPW];
            size_t off[k3RPW];
            bool ok[k3RPW];
#pragma unroll
            for (int r = 0; r < k3RPW; ++r) {
                const int y = y0 + yl + r;
                ok[r] = col_ok && y < a.ny;
                off[r] = ((size_t)z * a.ny + y) * a.px + x;
                if (ok[r]) {
                    if (MODE == STEP_ADJ || MODE == STEP_ADJ2) { s4[r] = ld4_stream(a.snap + off[r]); c4[r] = ld4(a.acc + off[r]); }
                    if (MODE == STEP_ADJ2) sp4[r] = ld4_stream(a.snap_prev + off[r]);
                    if (MODE == STEP_BORN) { s4[r] = ld4_stream(a.snap + off[r]); d4[r] = ld4(a.dm + off[r]); }
                }
            }
            const float gzv = __ldg(a.gz + z);
            mbar_wait(&full_bar[ptop % k3NP], (ptop / k3NP) & 1);
            mbar_wait(&om_full[iz % k3NO], (iz / k3NO) & 1);
            {
                const float* om = om_ring + (size_t)(iz % k3NO) * 2 * k3OmFloats + (yl * k3BX) + 4 * lane;
#pragma unroll
                for (int r = 0; r < k3RPW; ++r) { o4[r] = ld4(om + r * k3BX); m4[r] = ld4(om + k3OmFloats + r * k3BX); }
            }
#pragma unroll
            for (int r = 0; r < k3RPW; ++r) {
#pragma unroll
                for (int k = 0; k < 8; ++k) win[r][k] = win[r][k + 1];
                win[r][8] = own(ptop, r);
            }
            // slab mode: the 4 owned planes next to a neighbour are also stored straight into its ghost planes (NVLink)
            const bool bu = a.peer_up && z < a.z_own0 + kHalo, bd = a.peer_dn && z >= a.z_own1 - kHalo;
            const float* mid = ring + (size_t)(pmid % k3NP) * k3PlaneStride;
            float4 yc[8 + k3RPW];                        // rows yl-4 .. yl+3+RPW of the centre plane, this lane's float4
#pragma unroll
            for (int k = 0; k < 8 + k3RPW; ++k) yc[k] = ld4(mid + (yl + k) * k3SX + kHalo + 4 * lane);
#pragma unroll
            for (int r = 0; r < k3RPW; ++r) {
                const float* row = mid + (yl + r + kHalo) * k3SX + 4 * lane;
                const float4 L = ld4(row), R = ld4(row + 8);
                const float4 C = yc[r + 4];
                const float ax[12] = {L.x, L.y, L.z, L.w, C.x, C.y, C.z, C.w, R.x, R.y, R.z, R.w};
                const float gg = gyv[r] * gzv;
                const float gv[4] = {gx4.x * gg, gx4.y * gg, gx4.z * gg, gx4.w * gg};
                const float ov[4] = {o4[r].x, o4[r].y, o4[r].z, o4[r].w}, mv[4] = {m4[r].x, m4[r].y, m4[r].z, m4[r].w};
                float wv[4], nv[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float c = ax[4 + q];
                    auto comp = [&](const float4& v) { return q == 0 ? v.x : (q == 1 ? v.y : (q == 2 ? v.z : v.w)); };
                    float lap = (3.0f * kC0) * c;
                    lap = fmaf(kC1, ((ax[3 + q] + ax[5 + q]) + (comp(yc[r + 3]) + comp(yc[r + 5]))) + (comp(win[r][3]) + comp(win[r][5])), lap);
                    lap = fmaf(kC2, ((ax[2 + q] + ax[6 + q]) + (comp(yc[r + 2]) + comp(yc[r + 6]))) + (comp(win[r][2]) + comp(win[r][6])), lap);
                    lap = fmaf(kC3, ((ax[1 + q] + ax[7 + q]) + (comp(yc[r + 1]) + comp(yc[r + 7]))) + (comp(win[r][1]) + comp(win[r][7])), lap);
                    lap = fmaf(kC4, ((ax[0 + q] + ax[8 + q]) + (comp(yc[r + 0]) + comp(yc[r + 8]))) + (comp(win[r][0]) + comp(win[r][8])), lap);
                    wv[q] = lap;
                    // BORN: nv = g * fma(m, lap, fma(dm, w, fma(-g, o, 2 c))), the same order as the 2-D kernel
                    float rest = fmaf(-gv[q], ov[q], 2.0f * c);
                    if (MODE == STEP_BORN) rest = fmaf(comp(d4[r]), comp(s4[r]), rest);
                    nv[q] = gv[q] * fmaf(mv[q], lap, rest);
                }
                if (ok[r]) {
                    const float4 n4 = make_float4(nv[0], nv[1], nv[2], nv[3]);
                    st4(a.oldnew + off[r], n4);
                    if (bu) st4((float*)((char*)(a.oldnew + off[r]) + dup), n4);
                    if (bd) st4((float*)((char*)(a.oldnew + off[r]) + ddn), n4);
                    if (MODE == STEP_FWD_SAVE) st4_stream(a.snap + off[r], make_float4(wv[0], wv[1], wv[2], wv[3]));
                    if (MODE == STEP_ADJ || MODE == STEP_ADJ2) {
                        float4 c = c4[r];
                        if (MODE == STEP_ADJ2) {      // deferred imaging of the previous adjoint step (its field is this launch's u_n)
                            c.x = fmaf(C.x, sp4[r].x, c.x); c.y = fmaf(C.y, sp4[r].y, c.y);
                            c.z = fmaf(C.z, sp4[r].z, c.z); c.w = fmaf(C.w, sp4[r].w, c.w);
                        }
                        c.x = fmaf(nv[0], s4[r].x, c.x); c.y = fmaf(nv[1], s4[r].y, c.y);
                        c.z = fmaf(nv[2], s4[r].z, c.z); c.w = fmaf(nv[3], s4[r].w, c.w);
                        st4(a.acc + off[r], c);
                    }
                }
            }
            // the centre plane is dead now (later outputs see it only through the register windows)
            __syncwarp();
            if (lane == 0) {
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&empty_bar[pmid % k3NP])) : "memory");
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&om_empty[iz % k3NO])) : "memory");
            }
            // a boundary side is complete for this warp after its 4th plane: the last consumer warp of the CTA reports the
            // CTA, the last CTA of the side publishes the step id to the neighbour - long before the march ends
            if (bu || bd) {
                // (the chunk that owns the upper boundary always marches upwards)
                const bool fin_up = bu && z == a.z_own0 + kHalo - 1, fin_dn = bd && z == (desc ? a.z_own1 - kHalo : a.z_own1 - 1);
                if (early && (fin_up || fin_dn)) {
                    __threadfence_system();            // every lane: its peer stores are visible system-wide
                    __syncwarp();
                    if (lane == 0) {
                        if (fin_up && atomicAdd(&slab_state[2], 1) == k3CW - 1) slab_side_done(a, 0, ctas_per_side, signal_id);
                        if (fin_dn && atomicAdd(&slab_state[3], 1) == k3CW - 1) slab_side_done(a, 1, ctas_per_side, signal_id);
                    }
                }
            }
        }
    }

    // ---- sparse fix-ups for the points this CTA owns: injection, then receiver sampling -------------------
    if (i1 > i0 || r1 > r0) {
        __syncthreads();
        for (int e = i0 + threadIdx.x; e < i1; e += blockDim.x) {
            const int off = a.inj.off[e];
            const int zy = off / a.px, xx = off - zy * a.px;
            const int z = zy / a.ny, y = zy - z * a.ny;
            const float val = a.inj_vals[a.inj.id[e]];
            const float gm = a.gx[xx] * a.gy[y] * a.gz[z] * a.m[off];
            atomicAdd(a.oldnew + off, gm * val);
            if (MODE == STEP_FWD_SAVE) atomicAdd(a.snap + off, val);
            if (MODE == STEP_ADJ || MODE == STEP_ADJ2) atomicAdd(a.acc + off, gm * val * a.snap[off]);
        }
        if (r1 > r0 || (slab && i1 > i0)) __syncthreads();
        for (int e = r0 + threadIdx.x; e < r1; e += blockDim.x) a.rec_out[a.rec.id[e]] = __ldcg(a.oldnew + a.rec.off[e]);
        if (slab && i1 > i0) {
            // injected cells inside a boundary plane: refresh the neighbour's ghost copy with the final value, then report
            // the sides this CTA owns (it did not report them during the march)
            for (int e = i0 + threadIdx.x; e < i1; e += blockDim.x) {
                const int off = a.inj.off[e];
                const int zy = off / a.px, xx = off - zy * a.px;
                const int z = zy / a.ny, y = zy - z * a.ny;
                const float v = __ldcg(a.oldnew + off);
                if (a.peer_up && z < a.z_own0 + kHalo) a.peer_up[((size_t)(a.peer_up_z + z - a.z_own0) * a.ny + y) * a.px + xx] = v;
                if (a.peer_dn && z >= a.z_own1 - kHalo) a.peer_dn[((size_t)(z - (a.z_own1 - kHalo)) * a.ny + y) * a.px + xx] = v;
            }
            __threadfence_system();
            __syncthreads();
            if (threadIdx.x == 0) {
                if (own_up) slab_side_done(a, 0, ctas_per_side, signal_id);
                if (own_dn) slab_side_done(a, 1, ctas_per_side, signal_id);
            }
        }
    }

    // ---- slab mode: the last CTA of the launch advances the device-resident step id --------------------------------
    if (slab) {
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned int* done = (unsigned int*)(a.sync + kSyncDoneAll);
            const unsigned total = gridDim.x * gridDim.y * gridDim.z;
            __threadfence();
            if (atomicAdd(done, 1u) == total - 1) {
                *done = 0;
                a.sync[kSyncStep] = signal_id;
                __threadfence();
            }
        }
    }
}

}  // namespace fwi
