/*
 * fwi_b200.h - C ABI of libfwi_b200.so (sm_100a).
 *
 * Plain pointers and sizes only; no torch / C++ types cross this boundary.  The Python
 * host layer (full_waveform_inversion_b200/) binds these with ctypes; INTEGRATION.md shows
 * the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative FWI_E* code; the message of the
 *     last failure (per thread) is available from fwi_last_error().  Nothing calls exit()
 *     (the reference's convention is print + sys.exit(), e.g. full_waveform_inversion.py:124-125,
 *     :1206-1208; SURVEY 8b / q9).
 *   - "dev" pointers are device memory on the handle's GPU, "host" pointers are host memory.
 *     The caller owns every buffer it passes; handles own their internal device copies.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Calls are
 *     asynchronous on that stream unless the parameter list contains a host output.
 *   - a handle is not thread-safe; use one handle per GPU / per thread.
 *
 * Track A  = the Monte-Carlo source-inversion path that exists in the reference
 *            (full_waveform_inversion.py, cited FWI:<line>).
 * Track B  = the acoustic finite-difference / adjoint path BASELINE.json names; the reference
 *            has no counterpart (SURVEY 0), so those entry points cite the self-oracle
 *            oracle/fd_oracle.py instead.
 */
#ifndef FWI_B200_H
#define FWI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FWI_OK            0
#define FWI_EINVAL       -1   /* bad argument / unsupported combination          */
#define FWI_ECUDA        -2   /* a CUDA runtime / driver call failed              */
#define FWI_ENOMEM       -3   /* device allocation failed                         */
#define FWI_EZEROPROB    -4   /* sum of likelihoods is 0 (reference: NaN probe, FWI:1206) */
#define FWI_ESTATE       -5   /* call order violated (e.g. adjoint before forward) */

const char* fwi_last_error(void);
int fwi_version(void);                      /* 100*major + minor                        */
int fwi_device_count(void);                 /* number of visible CUDA devices (0 = none) */

/* ===================================================================== Track A */

/* comparison_metric (FWI:56) */
enum { FWI_METRIC_VR = 0, FWI_METRIC_CC = 1, FWI_METRIC_PCC = 2, FWI_METRIC_CC_SHIFT = 3, FWI_METRIC_GAU = 4 };
/* flags */
enum {
    FWI_FLAG_NORMALISED   = 1,  /* perform_normallised_waveform_inversion (FWI:53)      */
    FWI_FLAG_SIMULTANEOUS = 2,  /* compare_all_waveforms_simultaneously  (FWI:54)       */
    FWI_FLAG_STRICT_REF   = 4,  /* reproduce quirk q1: per-trace 'gau' returns 0 (FWI:659-661, 678-682) */
    FWI_FLAG_TENSOR       = 16, /* require the tensor-core path (tcgen05 3 x TF32, TMEM epilogue): error if the case is not covered */
    FWI_FLAG_NO_TENSOR    = 32, /* keep the CUDA-core fp32 kernels (the tensor-core path is the default for N >= 256) */
    FWI_FLAG_GRAM         = 8   /* Gram-matrix mode (a different algorithm, SURVEY 7): un-normalised metrics only,
                                   O(K C^2) per sample in float64, no synthetic traces formed; one medium only */
};
/* inversion_type (FWI:52), in the order of the reference's dispatch FWI:734-751 */
enum {
    FWI_TYPE_FULL_MT = 0, FWI_TYPE_DC = 1, FWI_TYPE_SINGLE_FORCE = 2, FWI_TYPE_DC_SF_COUPLE = 3,
    FWI_TYPE_DC_SF_NO_COUPLING = 4, FWI_TYPE_DC_CRACK_COUPLE = 5, FWI_TYPE_SF_CRACK_NO_COUPLING = 6
};

typedef struct fwi_mc_ctx fwi_mc_ctx;

/* Create a context for K traces x C source components x T samples; n_media = 1 or 2
 * (two-media Green's functions, FWI:133).  Replaces the implicit "arrays in scope" state of
 * PARALLEL_worker_mc_inv (FWI:686-711). */
int fwi_mc_create(int device, int K, int C, int T, int n_media, fwi_mc_ctx** out);
int fwi_mc_destroy(fwi_mc_ctx* ctx);

/* Upload the problem.  G_host: float64 C-order (K,C,T) or (K,C,T,2) exactly as the reference
 * holds it (FWI:85, FWI:133); d_host: float64 (K,T) (FWI:84).  phase_index_host: NULL, or K ints
 * in {0:P,1:S,2:surface} enabling per-phase media fractions (FWI:717-727).  Converts once to the
 * fp32 device layout (rows [k][t][c..] with t-major rows so one 16-byte load feeds 4 FMAs) and
 * precomputes the per-trace data constants. Synchronous. */
int fwi_mc_upload(fwi_mc_ctx* ctx, const double* G_host, const double* d_host, const int* phase_index_host);

/* forward_model (FWI:253-264), batched: traces_dev[n][k][t] = sum_c G[k,c,t] * M[c][n].
 * M_dev is (rows >= n_comp, ldm) fp32 with the sample index contiguous - the reference's own
 * MTs layout (FWI:794).  n_comp <= C reproduces the len(M) truncation of FWI:262.
 * media_frac_dev: NULL or (nfrac, ldm) with nfrac = 1 (FWI:730) or 3 (FWI:719-721). */
int fwi_mc_forward(fwi_mc_ctx* ctx, const float* M_dev, int64_t ldm, int n_comp,
                   const float* media_frac_dev, int nfrac, int64_t N, float* traces_dev, void* stream);

/* forward_model + compare_synth_to_real_waveforms (FWI:752-755, UNP:222-232) for N samples.
 * similarity_dev[n] receives the raw similarity; likelihood_dev (nullable) receives
 * exp(-(1-s)/2) (FWI:774). */
int fwi_mc_eval(fwi_mc_ctx* ctx, const float* M_dev, int64_t ldm, const float* media_frac_dev, int nfrac,
                int64_t N, int metric, int flags, float* similarity_dev, float* likelihood_dev, void* stream);

/* Raw-draw -> source-tensor transform of the seven generators (FWI:282-510), exposed so the
 * deterministic arithmetic can be tested on replayed draws.  draws_dev is (n_draws, ldn) fp32 in
 * the reference's consumption order; out rows: C tensor rows (x amplitude, FWI:735-751) then,
 * for combined types, the amp-frac row (FWI:851-852). */
int fwi_mc_transform_draws(int inversion_type, const float* draws_dev, int64_t ldn, int64_t N,
                           float amplitude, float* out_dev, int64_t ldo, void* stream);
int fwi_mc_type_components(int inversion_type);   /* 3, 6 or 9                      */
int fwi_mc_type_draws(int inversion_type);        /* raw draws consumed per sample  */
int fwi_mc_type_rows(int inversion_type);         /* components (+1 for combined types) */

/* The whole worker loop (FWI:713-774) for global sample indices [first, first+N): Philox-4x32-10
 * keyed by (seed, global sample index) so results do not depend on how samples are sharded over
 * GPUs (fixes q4, FWI:824-827).  MTs_dev: (fwi_mc_type_rows + nfrac, ldn) fp32, row order of
 * FWI:851-862.  L_dev[n] = likelihood.  Host outputs (nullable): sum of L in float64 (FWI:847),
 * the index (relative to `first`) and value of the largest L (FWI:1217).  Synchronises `stream`
 * if any host output is requested. */
int fwi_mc_sample_eval(fwi_mc_ctx* ctx, int inversion_type, uint64_t seed, int64_t first, int64_t N,
                       float amplitude, int metric, int flags, int nfrac, float* MTs_dev, int64_t ldn,
                       float* similarity_dev, float* L_dev, double* sumL_host, int64_t* argmax_host,
                       float* maxL_host, void* stream);

/* MTp = L * p_model / p_data with p_model = 1/N_total (FWI:811, 847-848).  sumL is the global
 * sum (after the cross-GPU reduction).  Returns FWI_EZEROPROB when sumL == 0 (q9). */
int fwi_mc_normalise(const float* L_dev, int64_t N, double sumL, float* MTp_dev, void* stream);

/* Reduce L over a device array: sum (float64), argmax and max. Synchronises `stream`. */
int fwi_mc_reduce(const float* L_dev, int64_t N, double* sum_host, int64_t* argmax_host, float* max_host,
                  void* stream);

/* Host-buffer convenience used by the drop-in shim and by bench.py's e2e leg: copies M (N x C,
 * float64, sample-major like a stack of reference M vectors) host->device, evaluates, copies the
 * similarities back.  Everything, copies included, happens inside the call. */
int fwi_mc_eval_host(fwi_mc_ctx* ctx, const double* M_host, int64_t N, int n_comp, const double* media_frac_host,
                     int nfrac, int metric, int flags, double* similarity_host);

/* perform_inversion (FWI:242-250): least-squares source vector of the stacked (K*T) x C system, float64 normal
 * equations + Cholesky on the device.  G_host (K,C,T), d_host (K,T), M_host (C).  Synchronous. */
int fwi_mc_lstsq(int device, const double* G_host, const double* d_host, int K, int C, int T, double* M_host);

/* Measurement aid (SURVEY 8d, Track A roofline): achieved FP32 FMA throughput of `device` in TFLOP/s from a register-only
 * FMA kernel (8 independent chains per thread).  Synchronous, ~10 ms. */
int fwi_diag_fp32_peak(int device, double* tflops_out);

/* Input preparation (SURVEY 8f row f2): the Green's-function conditioning of load_input_data /
 * get_overall_real_and_green_func_data (FWI:92-111, FWI:178-196) as one device op.  raw_dev: float64 (K,C,T) or
 * (K,C,T,2); shift_dev: K integer sample shifts (np.roll, FWI:97) or NULL; zero_head: zero the wrapped head
 * (FWI:98-99); cut_start_dev: K window starts or NULL, cut_len the common window length (FWI:104-111);
 * scale1, scale2: unit factors applied in this order (FWI:178/192 then FWI:196).  out_dev: float64
 * (K,C,Tout[,2]), Tout = cut_len or T.  Bit-identical to the NumPy operations it replaces. */
int fwi_mc_prepare(const double* raw_dev, int K, int C, int T, int n_media, const int* shift_dev, int zero_head,
                   const int* cut_start_dev, int cut_len, double scale1, double scale2, double* out_dev, void* stream);

/* Posterior reductions (SURVEY 8f row f4): the per-sample Python loops of plot_full_waveform_inversion.py (PLOT)
 * as float64 histogram kernels over the device-resident MTs (rows, ldn) / MTp.  idx_dev: NULL (all n samples) or
 * n int64 sample indices (e.g. the top fraction by MTp, PLOT:517-520, PLOT:1003-1007).
 *   mode 0: theta-phi 5-degree bins of the force vector in rows row0..row0+2, weighted by MTp -> hist[36*72] (PLOT:522-555)
 *   mode 1: 1 % bins of the amp-frac row (row0) f and 1-f weighted by MTp, zero-probability samples skipped
 *           -> hist[2*101] (PLOT:943-961; the reference then doubles the edge bins, PLOT:963-966 - left to the caller)
 *   mode 2: lune delta-gamma bins (pi/120) of the 6-vector in rows row0..row0+5, counts -> hist[122*41] (PLOT:1011-1059) */
int fwi_mc_posterior_hist(int mode, const float* MTs_dev, int64_t ldn, const float* MTp_dev, const int64_t* idx_dev, int64_t n,
                          int row0, double* hist_dev, void* stream);

/* ===================================================================== Track B (2-D acoustic)
 * No reference counterpart exists (SURVEY 0): the specification these entry points implement is
 * frozen in oracle/fd_oracle.py (sections B1-B4 of its header), which is what each comment cites. */

typedef struct fwi_fd2d fwi_fd2d;

/* Plan for an nz x nx grid (x contiguous), cell size h, time step dt, Cerjan sponge of `nabs` cells with
 * strength `alpha` on all four sides (fd_oracle.sponge).  Allocates the wavefield pairs, the imaging
 * accumulator and the TMA descriptors. */
int fwi_fd2d_create(int device, int nz, int nx, float h, float dt, int nabs, float alpha, fwi_fd2d** out);
int fwi_fd2d_destroy(fwi_fd2d* plan);
/* Select the one-tile-per-CTA step kernel with bz tile rows and nw warps per CTA: (32, 4), or 7 rows per warp:
 * (28, 4), (42, 6), (56, 8); any other pair is FWI_EINVAL.  fwi_fd2d_create picks, for L2-resident grids, the height
 * whose tiles fill whole waves of the GPU's SMs (all shapes give bit-identical fields).  Clears the geometry. */
int fwi_fd2d_set_tile(fwi_fd2d* plan, int bz, int nw);
/* Select the temporally blocked kernel: two leapfrog steps per pass on 120 x cz core tiles (cz 24 or 32, else FWI_EINVAL);
 * an odd leftover step runs the one-step tile kernel.  Clears the geometry. */
int fwi_fd2d_set_tb2(fwi_fd2d* plan, int cz);
/* Free surface at z = 0 (spec B6, off by default; 2-D and 3-D plans): the values above the grid's first row (plane) are
 * the odd mirror u[-k] = -u[k] instead of 0, and the sponge does not damp that face.  Rebuilds the z sponge profile (a
 * later fwi_fd_set_profiles still overrides it), clears the geometry and drops the cached graphs.  While it is on,
 * fwi_fd*_set_geometry rejects sources and receivers at z = 0 (FWI_EINVAL), and the plan cannot be connected as a slab
 * with an upper neighbour, nor enabled on one: only the slab that owns global z = 0 has the surface. */
int fwi_fd2d_set_free_surface(fwi_fd2d* plan, int enable);
/* Replay the time loops as cached CUDA graphs (default on) or as individual launches (0). */
int fwi_fd2d_set_graphs(fwi_fd2d* plan, int enable);
/* Cap (bytes) on the forward-field storage used by fwi_fd2d_gradient; 0 = 85 % of free HBM.  When all nt
 * snapshots do not fit, the gradient switches to two-level checkpointing (recompute per segment).
 * fwi_fd2d_gauss_newton follows the same rule; fwi_fd2d_born keeps at most min(nt, 128) snapshots and takes fewer
 * when the cap holds fewer planes (same results); a cap below one plane is FWI_EINVAL. */
int fwi_fd2d_set_memory_limit(fwi_fd2d* plan, uint64_t bytes);
/* v_dev: (nz, nx) fp32 velocities, dense.  Builds m = (v dt / h)^2 in the pitched layout (fd_oracle B1). */
int fwi_fd2d_set_model(fwi_fd2d* plan, const float* v_dev, void* stream);
/* One shot's acquisition: integer grid indices of sources and receivers (host arrays; fd_oracle B2).
 * On FWI_EINVAL the plan keeps the geometry it had. */
int fwi_fd2d_set_geometry(fwi_fd2d* plan, int nsrc, const int* src_z_host, const int* src_x_host,
                          int nrec, const int* rec_z_host, const int* rec_x_host);
/* Forward model: nt leapfrog steps from rest; wavelet_dev (nt, nsrc); traces_dev (nt, nrec) receives
 * u_{n+1} at the receivers (fd_oracle.Problem.forward).  Source injection and receiver sampling are fused
 * into the step kernel. */
int fwi_fd2d_forward(fwi_fd2d* plan, const float* wavelet_dev, int nt, float* traces_dev, void* stream);
/* Copy a field out as dense (nz, nx): which = 0 u_n, 1 u_{n-1} (after the last forward sweep), 2 imaging sum I.
 * After a forward, a Born call or a gradient / Gauss-Newton product that stored every snapshot, that is u_nt, u_{nt-1};
 * after a checkpointed gradient / Gauss-Newton product it is u_S, u_{S-1}, where the recompute of the first segment of
 * S steps ended. */
int fwi_fd2d_wavefield(fwi_fd2d* plan, int which, float* out_dev, void* stream);
/* One shot's misfit and gradient (fd_oracle.Problem.misfit_and_gradient): forward with w_n kept in HBM
 * (or checkpointed), residual = synthetic - observed, adjoint back-propagation with the zero-lag
 * cross-correlation accumulated in the step kernel, then grad_dev (nz, nx) += (2 / v) * I.
 * traces_dev (nullable) receives the synthetics; misfit_host (nullable) receives J = 1/2 sum r^2
 * (requesting it synchronises the stream). */
int fwi_fd2d_gradient(fwi_fd2d* plan, const float* wavelet_dev, const float* obs_dev, int nt, float* grad_dev,
                      float* traces_dev, double* misfit_host, void* stream);
/* Born (linearised) modelling: dtraces_dev (nt, nrec) = J dv for the velocity perturbation dv_dev (dense, grid-shaped);
 * traces_dev (nullable) receives the background synthetics, bit-identical to fwi_fd2d_forward.  (spec B5, tests/born_reference.py) */
int fwi_fd2d_born(fwi_fd2d* plan, const float* wavelet_dev, const float* dv_dev, int nt, float* dtraces_dev,
                  float* traces_dev, void* stream);
/* Gauss-Newton Hessian-vector product: hv_dev (grid-shaped) += J^T J dv; dtraces_dev (nullable) receives J dv.
 * Same snapshot storage / checkpointing rule as fwi_fd2d_gradient.  (spec B5, tests/born_reference.py)
 * Both return FWI_EINVAL on a plan connected as a peer-memory slab. */
int fwi_fd2d_gauss_newton(fwi_fd2d* plan, const float* wavelet_dev, const float* dv_dev, int nt, float* hv_dev,
                          float* dtraces_dev, void* stream);
int64_t fwi_fd2d_launch_count(fwi_fd2d* plan);
/* Allocate what fwi_fd2d_forward (gradient = 0) or fwi_fd2d_gradient (1) over nt steps will need with the current
 * geometry, without launching anything (allocations synchronise the device: keep them out of timed regions). */
int fwi_fd_reserve(fwi_fd2d* plan, int nt, int gradient);

/* 3-D plans (nz x ny x nx, x contiguous; fd_oracle works in any dimension).  A 3-D plan is used with the same
 * fwi_fd2d_set_model / _forward / _gradient / _wavefield / _set_memory_limit / _set_graphs / _destroy entry points
 * (dense arrays are then (nz, ny, nx)); only creation and geometry differ. */
int fwi_fd3d_create(int device, int nz, int ny, int nx, float h, float dt, int nabs, float alpha, fwi_fd2d** out);
int fwi_fd3d_set_geometry(fwi_fd2d* plan, int nsrc, const int* src_z_host, const int* src_y_host, const int* src_x_host,
                          int nrec, const int* rec_z_host, const int* rec_y_host, const int* rec_x_host);     /* step-kernel launches so far (bench bookkeeping) */
/* Off-grid geometry (spec B7, tests/offgrid_reference.py): sources and receivers at float coordinates in cell units (host
 * arrays; 10.5 lies half-way between rows 10 and 11), each coordinate in [0, n - 1] of its axis, z > 0 with a free surface.
 * A point with a fractional coordinate is a tensor product of 8 Kaiser-windowed sinc taps per fractional axis (b = 4.06);
 * an integral coordinate is one tap.  Taps outside the grid are dropped; with a free surface a tap at row -k folds onto
 * row k with its weight negated and a tap on row 0 is dropped.  Sources inject wavelet x weight at every tap cell,
 * receivers record sum weight x u_{n+1} over their taps, and the misfit, gradient, Born and Gauss-Newton products are
 * taken at the points.  Replaces any geometry; fwi_fd*_set_geometry replaces it in turn.  Wavelets, observed data and
 * traces keep their (nt, points) layout.  Each shot operation then adds, on top of its step kernels: one spread of the
 * wavelet; a gradient or Gauss-Newton product one gather and one spread of the residual (J dv) inside its graph; a
 * forward or Born call one gather per trace array it returns.  FWI_EINVAL, naming the point, for a coordinate that is
 * not finite, outside the grid or at z <= 0 under a free surface; FWI_EINVAL on a plan connected as a peer-memory slab;
 * fwi_fd_step is FWI_EINVAL while the plan holds positions.  On FWI_EINVAL the plan keeps the geometry it had. */
int fwi_fd2d_set_positions(fwi_fd2d* plan, int nsrc, const double* src_z_host, const double* src_x_host,
                           int nrec, const double* rec_z_host, const double* rec_x_host);
int fwi_fd3d_set_positions(fwi_fd2d* plan, int nsrc, const double* src_z_host, const double* src_y_host,
                           const double* src_x_host, int nrec, const double* rec_z_host, const double* rec_y_host,
                           const double* rec_x_host);

/* Low-level stepping API: the caller drives the time loop, one leapfrog step per call on the caller's stream.
 * Used by the slab-decomposed multi-GPU path (acoustic.SlabPropagator), which exchanges the 4-plane halos of the
 * slab with its neighbours over NCCL/NVLink between steps. */
int fwi_fd_set_profiles(fwi_fd2d* plan, const float* gz_host, const float* gy_host, const float* gx_host); /* override sponge profiles (nullable each) */
void* fwi_fd_field_ptr(fwi_fd2d* plan, int idx);   /* wavefield buffer idx: 0/1 forward pair, 4/5 adjoint pair; layout [rows][pitch] */
int fwi_fd_pitch(fwi_fd2d* plan);                  /* floats per row (nx rounded up to 32) */
int fwi_fd_reserve_snapshots(fwi_fd2d* plan, int nsteps);
int fwi_fd_reset(fwi_fd2d* plan, int pair, void* stream);   /* zero pair 0 (forward) or 1 (adjoint + imaging sum) */
/* mode 0 forward, 1 forward + store w_n in snapshot[snap_index], 2 adjoint + imaging against snapshot[snap_index];
 * cur (0/1) = buffer of the pair holding u_n; inj_vals_dev = this step's source values (or receiver residuals);
 * rec_out_dev = this step's trace row (nullable). */
int fwi_fd_step(fwi_fd2d* plan, int mode, int cur, const float* inj_vals_dev, float* rec_out_dev, int64_t snap_index,
                void* stream);
int fwi_fd_finalize_gradient(fwi_fd2d* plan, float* grad_dev, void* stream);   /* grad += (2/v) I */
/* Slab decomposition over NVLink peer memory (3-D plans, one process per GPU): every rank exports its arena
 * (fwi_fd_slab_info: a cudaIpcMemHandle_t plus the byte offsets of the 8 wavefield buffers and of the sync area),
 * the host layer swaps them between neighbours (torch.distributed), and fwi_fd_slab_connect maps the neighbours'
 * memory.  From then on a step computes only the owned planes [z_own0, z_own1), stores its 4 boundary planes
 * straight into the neighbours' ghost planes from inside the step kernel and publishes a step id that the
 * neighbours' next launch waits for - compute and halo exchange are one kernel, no collective call per step. */
int fwi_fd_slab_info(fwi_fd2d* plan, void* ipc_handle_out, uint64_t* offsets_out);
int fwi_fd_slab_connect(fwi_fd2d* plan, int z_own0, int z_own1, const void* up_handle, const uint64_t* up_offsets, int up_ghost_z,
                        const void* dn_handle, const uint64_t* dn_offsets);
int fwi_fd_slab_error(fwi_fd2d* plan, int* error_out);       /* 1 if a launch timed out waiting for a neighbour */
/* Once connected, the ordinary fwi_fd2d_forward / fwi_fd2d_gradient entry points run the slab: step ids live in device
 * memory (so the time loops replay from CUDA graphs), both boundaries are computed and pushed in the first four
 * iterations of their CTAs (the last z chunk marches downwards), the gradient checkpoints per rank when the
 * snapshots do not fit, and a rank without sources or receivers is allowed.  After a timeout every later launch
 * returns at once until fwi_fd_slab_clear_error (all ranks, device idle). */
int fwi_fd_slab_set_timeout(fwi_fd2d* plan, double milliseconds);      /* bounded spin on a neighbour's flag (default 2 s) */
int fwi_fd_slab_clear_error(fwi_fd2d* plan);
/* The same protocol between plans of one process (peers = other plans; null = no neighbour on that side). */
int fwi_fd_slab_connect_local(fwi_fd2d* plan, int z_own0, int z_own1, fwi_fd2d* up, int up_ghost_z, fwi_fd2d* dn);

/* residual = syn - obs, J = 1/2 sum residual^2 (fd_oracle.misfit). Synchronises. */
int fwi_fd_misfit(const float* syn_dev, const float* obs_dev, int64_t n, float* resid_dev, double* misfit_host,
                  void* stream);
/* v <- clip(v - step * grad, vmin, vmax)   (fd_oracle.model_update, B4) */
int fwi_fd_model_update(float* v_dev, const float* grad_dev, int64_t n, float step, float vmin, float vmax,
                        void* stream);
/* max |x| (used for the step-length rule of B4). Synchronises. */
int fwi_fd_absmax(const float* x_dev, int64_t n, float* out_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FWI_B200_H */
