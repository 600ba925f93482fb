/*
 * smoke_b200.h -- C ABI of libsmoke_sm100.so: the B200 (sm_100a) implementation of SmokePhysAI's
 * grid smoke step (reference: src/physics/navier_stokes.py, smoke_simulator.py, fractal_generator.py).
 *
 * The reference has no FFI / plugin interface: its boundary is the Python class surface
 * (SURVEY.md s8b).  This header is the boundary one level below it -- what the Python classes in
 * smokephysai_b200/ bind with ctypes, and what any other host language would bind instead.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless the name ends in _host
 *   - the caller owns all memory; the library never allocates, frees or keeps a pointer after a call
 *   - every entry point returns 0 on success, else a negative SMK_E* code or a positive cudaError_t;
 *     smk_last_error_string() (thread-local) describes the last failure; nothing throws or exits
 *   - all work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*); no hidden syncs
 *   - fields are fp32, row-major [row=y][col=x] with an element pitch that is a multiple of 4 and a
 *     16-byte aligned base (float4 access); `batch` independent simulations are `stride_*` elements apart.
 *     The frames of smk_step_ex / smk_run_steps_ex may be f16 or bf16 instead (SMK_FRAME_*): same layout,
 *     pitch and strides counted in elements of the frame type, base aligned to 4 such elements
 *   - arithmetic follows the reference's fp32 association with no FMA contraction (built -fmad=false),
 *     true division for /dt, so results are bit-identical to the reference's CPU path
 */
#ifndef SMOKE_B200_H
#define SMOKE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMK_ABI_VERSION 7

#if defined(__GNUC__)
#define SMK_API __attribute__((visibility("default")))
#else
#define SMK_API
#endif

enum {
    SMK_OK = 0,
    SMK_EINVAL = -1,      /* null pointer, bad dimension, bad pitch/alignment */
    SMK_EUNSUPPORTED = -2 /* configuration outside what the kernels handle */
};

/* Geometry of one (batched) simulation state.  navier_stokes.py:21-35:
 *   u[h+1][w]  v[h][w+1]  p[h][w]  density[h][w]   (+ div[h][w], frames[h][w] share the p layout) */
typedef struct smk_grid {
    int32_t h, w;        /* cells: grid_size = (h, w)                           navier_stokes.py:21 */
    int32_t batch;       /* independent simulations (1 for the reference's scalar API)            */
    int32_t pitch_u;     /* elements between rows of u                                            */
    int32_t pitch_v;     /* elements between rows of v                                            */
    int32_t pitch_c;     /* elements between rows of p / density / div / frame                    */
    int64_t stride_u;    /* elements between consecutive simulations' u                           */
    int64_t stride_v;
    int64_t stride_c;
    /* Row-slab decomposition (large single grids split over GPUs).  The arrays hold h local cell rows
     * (ghost rows included) that start at global cell row row0 of a gh-row grid.  gh == 0 means "not a
     * slab" (row0 = 0, gh = h).  Only the advection (absolute fp32 coordinates, global edge tests) and the
     * emitter splat look at these; every other phase is a purely local stencil. */
    int32_t row0, gh;
} smk_grid_t;

/* Slab advection guard: cells in local rows [need_lo, need_hi) must gather only from local rows
 * [valid_lo, valid_hi) of the advected field; otherwise *overflow_flag (device int32) is set to 1. */
typedef struct smk_slab_check {
    int32_t need_lo, need_hi, valid_lo, valid_hi;
    int32_t* overflow_flag;
} smk_slab_check_t;

/* One Gaussian emitter, add_smoke_source(x, y, radius, intensity): navier_stokes.py:37 */
typedef struct smk_source {
    int32_t x, y, radius;
    float intensity;
} smk_source_t;

/* Whole-step state: ping-pong copies of every field; cur_* say which copy is live and are updated
 * (on the host, in this struct) by smk_step / smk_run_steps. */
typedef struct smk_state {
    float* u[2];
    float* v[2];
    float* d[2];
    float* p[2];
    float* div;
    int32_t cur_u, cur_v, cur_d, cur_p;
} smk_state_t;

/* Scalar coefficients, pre-rounded on the host exactly as the reference's Python does:
 *   dt    = float32(self.dt)
 *   c_uv  = float32(self.dt * self.viscosity)            navier_stokes.py:72 via :158-159
 *   c_d   = float32(self.dt * (self.viscosity * 0.1))    navier_stokes.py:72 via :160
 *   decay = 0.995f                                       navier_stokes.py:171                   */
typedef struct smk_params {
    float dt, c_uv, c_d, decay;
    int32_t jacobi_iters;       /* 20 in the reference (navier_stokes.py:139)                      */
    int32_t sweeps_per_launch;  /* temporal-blocking depth T; 0 = library default                  */
    int32_t step_kernel;        /* smk_step / smk_run_steps: SMK_STEP_AUTO, _PHASES or _FUSED      */
} smk_params_t;

/* How smk_step / smk_run_steps execute a step.  Results are bit-identical either way.
 *   SMK_STEP_PHASES  one kernel per phase (any grid size)
 *   SMK_STEP_FUSED   the whole simulation on one SM -- u, v, density in shared memory, pressure in registers --
 *                    for all the steps of the call in a single launch; grids of at most 128 x 128 cells only
 *                    (SMK_EUNSUPPORTED otherwise)
 *   SMK_STEP_AUTO    fused when the grid qualifies and the call carries enough simulations for one-simulation-per-SM
 *                    execution to win: 128 x 128 cells and at least 12 simulations (48 for a single-step call), or
 *                    at least 96 x 96 cells and 96 simulations; the phase kernels otherwise                  */
enum { SMK_STEP_AUTO = 0, SMK_STEP_PHASES = 1, SMK_STEP_FUSED = 2 };

SMK_API int smk_version(void);
SMK_API const char* smk_last_error_string(void);
/* sm_count, compute capability major*10+minor and max opt-in shared memory of the current device */
SMK_API int smk_device_info(int32_t* sm_count, int32_t* cc, int32_t* smem_optin);
/* number of kernels this library has launched in this process so far (monotonic, all threads) */
SMK_API int smk_launch_count(int64_t* count);
/* make `device` current for this thread inside the library's (statically linked) CUDA runtime */
SMK_API int smk_set_device(int32_t device);

/* The library reads its tuning / test switches (SMK_PDL, SMK_FUSED_SLICE, SMK_FUSED_CLUSTER, SMK_JACOBI_PACKED,
 * SMK_JACOBI_STREAM, SMK_JACOBI_TILE, SMK_FDD_BULK, SMK_ADVECT_TILED, SMK_PROJECT_FUSED) from the environment once, at
 * the first launch that needs one; smk_reload_env reads them again (tests change them between cases). */
SMK_API int smk_reload_env(void);

/* Per-kernel device timing, for bench.py's roofline line: while a profile is open every kernel the library
 * launches is bracketed by a pair of CUDA events recorded on the launching stream.  smk_profile_end
 * synchronises those events, adds the elapsed milliseconds and launch counts up per phase, and closes the
 * profile.  Process-wide, not re-entrant; off by default (no events, no overhead). */
enum {
    SMK_PH_SPLAT = 0, SMK_PH_FORCES_DIFFUSE_DIV, SMK_PH_JACOBI, SMK_PH_PROJECT,
    SMK_PH_ADVECT_U, SMK_PH_ADVECT_V, SMK_PH_ADVECT_D, SMK_PH_OTHER, SMK_PH_STEP_FUSED, SMK_PH_HALO, SMK_PH_PROJECT_ADVECT_U,
    SMK_PH_HALO_UNPACK, SMK_PH_COUNT
};
SMK_API int smk_profile_begin(int32_t max_records);
SMK_API int smk_profile_end(double* ms_per_phase_host, int64_t* launches_per_phase_host, int32_t nphases);

/* a2  add_smoke_source (navier_stokes.py:37-48), batched: simulation b applies sources
 *     [offsets[b], offsets[b+1]) in list order (order matters where emitters overlap). */
SMK_API int smk_splat_sources(const smk_grid_t* g, float* density, const smk_source_t* sources,
                      const int32_t* offsets, void* stream);

/* a4  diffusion_step (navier_stokes.py:50-72) on one field [batch][rows][cols]; c = float32(dt*viscosity) */
SMK_API int smk_diffuse(const float* in, float* out, int32_t rows, int32_t cols, int32_t pitch,
                int32_t batch, int64_t stride, float c, void* stream);

/* a3+a4+a5 fused: buoyancy (:154-155), the three diffusions (:158-160) and the divergence (:136)
 *     in one pass; div may be NULL. */
SMK_API int smk_forces_diffuse_div(const smk_grid_t* g, const float* u, const float* v, const float* d,
                           float* u_out, float* v_out, float* d_out, float* div,
                           float dt, float c_uv, float c_d, void* stream);

/* a5  divergence alone (navier_stokes.py:136) */
SMK_API int smk_divergence(const smk_grid_t* g, const float* u, const float* v, float* div, float dt, void* stream);

/* a6  K Jacobi sweeps (navier_stokes.py:139-145), T sweeps fused per launch (temporal blocking, pressure
 *     tile held in registers).  Ping-pongs between p and p_scratch; *result_in_scratch tells where the
 *     final field is.  T = 0 picks the default. */
SMK_API int smk_jacobi(const smk_grid_t* g, const float* div, float* p, float* p_scratch,
               int32_t K, int32_t T, int32_t* result_in_scratch_host, void* stream);

/* a7  gradient subtract in place (navier_stokes.py:148-149) */
SMK_API int smk_project(const smk_grid_t* g, const float* p, float* u, float* v, float dt, void* stream);

/* a8  bilinear_interpolate (navier_stokes.py:111-131) at n arbitrary (y, x); mode 0 plain,
 *     1 = interpolate_velocity_u (x+0.5 clamped, :97-102), 2 = interpolate_velocity_v (y+0.5 clamped, :104-109) */
SMK_API int smk_bilerp(const float* field, int32_t rows, int32_t cols, int32_t pitch,
               const float* y, const float* x, float* out, int64_t n, int32_t mode, void* stream);

/* a10 advection_step (navier_stokes.py:74-95) of one field [batch][rows][cols] by (u, v) of grid g.
 *     scale != 1 multiplies the result (the 0.995 decay of :171); frame (may be NULL) receives
 *     out + fmul*out when fmul != NULL (fractal_generator.py:62) else a copy of out (:173). */
SMK_API int smk_advect(const smk_grid_t* g, const float* field, float* out, int32_t rows, int32_t cols,
               int32_t pitch, int64_t stride, const float* u, const float* v, float dt,
               float scale, float* frame, int64_t frame_stride, const float* fmul, void* stream);
/*     the same on a row slab (g->gh != 0): coordinates and edge tests are global, memory is local;
 *     chk (may be NULL) guards the gather reach. */
SMK_API int smk_advect_slab(const smk_grid_t* g, const float* field, float* out, int32_t rows, int32_t cols,
                    int32_t pitch, const float* u, const float* v, float dt, float scale,
                    const smk_slab_check_t* chk, void* stream);

/* a3-a11 one full step() / n steps (navier_stokes.py:151-173) over the state.  frames (may be NULL):
 *     [batch][nsteps][h][pitch_c] returned copies, multiplied by (1+fmul) when fmul != NULL.
 *     Not available on a slab grid (the host interleaves halo exchanges between the phases).
 *     Every step entry point (smk_step, smk_step_ex, smk_run_steps, smk_run_steps_ex, smk_run_steps_reset_ex,
 *     smk_run_steps_src_ex, smk_run_steps_sched_ex) checks a call the same way -- frames, grid, all nine state pointers (div included), cur_*,
 *     jacobi_iters, dt, step_kernel -- and refuses a malformed one before anything is enqueued. */
SMK_API int smk_step(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm,
             float* frame, int64_t frame_stride, const float* fmul, void* stream);
SMK_API int smk_run_steps(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps,
                  float* frames, int64_t frame_step_stride, int64_t frame_batch_stride,
                  const float* fmul, void* stream);
/*     the same with the frames in another element type: frame_format SMK_FRAME_F32 (what smk_step / smk_run_steps write),
 *     SMK_FRAME_F16 or SMK_FRAME_BF16.  A half-precision frame element is the fp32 one rounded once to nearest-even
 *     (overflow gives +-inf, subnormals are kept), converted in the kernel that writes the frame: no extra launch, and
 *     the state is bit-identical whatever the format.  frame / frames: base aligned to 4 elements of the frame type;
 *     strides in elements of that type, multiples of 4.  A format outside the enum or a misaligned frame is SMK_EINVAL,
 *     before anything is enqueued. */
enum { SMK_FRAME_F32 = 0, SMK_FRAME_F16 = 1, SMK_FRAME_BF16 = 2 };
SMK_API int smk_step_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm,
                        void* frame, int64_t frame_stride, const float* fmul, int32_t frame_format, void* stream);
SMK_API int smk_run_steps_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps,
                             void* frames, int64_t frame_step_stride, int64_t frame_batch_stride,
                             const float* fmul, int32_t frame_format, void* stream);
/*     the same on a freshly reset state: u, v, p all zeros and the density zeros plus the emitters of smk_splat_sources(g,
 *     density, sources, offsets) (sources and offsets may both be NULL: no emitters), whatever the live copies hold now.
 *     When the call runs on k_step_fused (one SM per simulation), that kernel builds the reset state on chip instead of
 *     reading it -- no memset, no splat launch -- and *consumed_host is 1; the live copies then hold the state after the
 *     steps, and the other copies and div are left as they were.  Otherwise nothing is enqueued and *consumed_host is 0:
 *     the caller resets, splats and runs smk_run_steps_ex itself.  nsteps = 1 with frame_step_stride 0 is smk_step_ex. */
SMK_API int smk_run_steps_reset_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps,
                                   void* frames, int64_t frame_step_stride, int64_t frame_batch_stride,
                                   const float* fmul, int32_t frame_format, const smk_source_t* sources,
                                   const int32_t* offsets, int32_t* consumed_host, void* stream);
/*     smk_run_steps_ex with continuous sources: the emitters of (sources, offsets) -- smk_splat_sources' format, both NULL for
 *     none -- are added to the density at the head of EVERY step, before the buoyancy, exactly as smk_splat_sources followed by
 *     smk_step_ex would add them (bit-identical frames and state).  Frame t is the density after step t, written before the splat
 *     of step t + 1; the state left after the call carries no trailing splat.  On k_step_fused and k_step_cluster the emitters
 *     are splatted on chip (no extra launch); on the phase kernels one k_splat launch precedes each step.  The records are read
 *     during the launch and must stay valid until it completes.
 *     reset = 1: the call starts from a freshly reset state splatted with (reset_sources, reset_offsets) (both may be NULL), under
 *     smk_run_steps_reset_ex's contract: consumed on chip by k_step_fused (*consumed_host = 1, one launch for the reset, the
 *     one-shot splat and the continuous sources) or nothing is enqueued (*consumed_host = 0) and the caller resets, splats and
 *     calls again with reset = 0.  Returns SMK_EINVAL before enqueuing anything for nsteps < 1, unpaired sources / offsets,
 *     reset_sources without reset, or a NULL consumed_host. */
SMK_API int smk_run_steps_src_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps,
                                 void* frames, int64_t frame_step_stride, int64_t frame_batch_stride,
                                 const float* fmul, int32_t frame_format, const smk_source_t* sources, const int32_t* offsets,
                                 int32_t reset, const smk_source_t* reset_sources, const int32_t* reset_offsets,
                                 int32_t* consumed_host, void* stream);
/*     smk_run_steps_src_ex with a source schedule: emitters that move or change intensity from step to step.  With
 *     offsets_step_stride = g->batch, offsets holds nsteps * batch + 1 entries, step-major, and step t (0 .. nsteps - 1 of this
 *     call) of simulation b adds records [offsets[t * batch + b], offsets[t * batch + b + 1]) at its head, exactly as
 *     smk_splat_sources with that row followed by smk_step_ex would (bit-identical frames and state, same frame and reset
 *     contract as smk_run_steps_src_ex).  An emitter with radius < 0 adds
 *     nothing, which pads rows of different lengths to one width.  Any other stride, or a non-zero stride without sources,
 *     is SMK_EINVAL before anything is enqueued.  smk_run_steps_src_ex is this entry with offsets_step_stride = 0. */
SMK_API int smk_run_steps_sched_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps,
                                   void* frames, int64_t frame_step_stride, int64_t frame_batch_stride,
                                   const float* fmul, int32_t frame_format, const smk_source_t* sources, const int32_t* offsets,
                                   int32_t offsets_step_stride, int32_t reset, const smk_source_t* reset_sources,
                                   const int32_t* reset_offsets, int32_t* consumed_host, void* stream);
/*     1 when a call of nsteps steps (smk_step: 1) would take the fused single-launch path for this grid and params */
SMK_API int smk_step_is_fused(const smk_grid_t* g, const smk_params_t* prm, int32_t nsteps, int32_t* fused_host);
/* Host-only (no GPU needed): the time-sliced schedule smk_run_steps gives the fused kernel when `nsims` simulations of
 *     `nsteps` steps do not fill whole waves of SMs.  The nsims x nsteps simulation-steps, simulation-major, are cut into
 *     pieces of piece_len steps; every item {simulation, first step, end step, 0} is one CTA, listed in launch order.  An
 *     item with first step > 0 waits for the item of lower index that ends at that step.  items_host holds 4 int32 per
 *     item, `capacity` items; *count_host receives the number of items (SMK_EINVAL if capacity is too small). */
SMK_API int smk_fused_plan(int32_t nsims, int32_t nsteps, int32_t piece_len, int32_t* items_host, int32_t capacity, int32_t* count_host);

/* diagnostics: per simulation {max|div|, sum div^2} of the un-normalised divergence of (u, v);
 *     out[2*batch] must be zeroed by the caller; warp-shuffle + atomic reduction. */
SMK_API int smk_div_norms(const smk_grid_t* g, const float* u, const float* v, float* out, void* stream);

/*     per simulation {max|p' - p|, sum (p' - p)^2} where p' is one more Jacobi sweep (navier_stokes.py:139-145) over
 *     (p, div): the residual of the pressure iteration after the K sweeps of a step.  out[2*batch] zeroed by the caller. */
SMK_API int smk_jacobi_residual(const smk_grid_t* g, const float* div, const float* p, float* out, void* stream);

/* a13 FractalGenerator fields (fractal_generator.py:12-62).  Output index [a][b], a < na (= w), b < nb (= h),
 *     as torch.meshgrid(x_w, y_h, indexing='ij') lays them out.  Any of the three outputs may be NULL:
 *       perlin = (sum_o 0.5^o sin(2^o px[a]) cos(2^o py[b]) + 1) / 2                      (:12-31)
 *       mandel = escape_count(z <- z^2 + mx[a] + i my[b], |z| <= 2) / iterations          (:33-51)
 *       mul    = intensity * (0.7*perlin + 0.3*mandel)                                    (:59,:62)
 *     px/py/mx/my are the torch.linspace grids, made on the host exactly as the reference makes them
 *     (ATen's CPU linspace is ISA-dependent in the last ulp, and the escape count is sensitive to it). */
SMK_API int smk_fractal_fields(float* perlin, float* mandel, float* mul, int32_t na, int32_t nb, int32_t pitch,
                       float intensity, int32_t iterations,
                       const float* px, const float* py, const float* mx, const float* my, void* stream);
/* out = field + mul*field (fractal_generator.py:62) */
SMK_API int smk_apply_mul(const float* field, const float* mul, float* out, int32_t rows, int32_t cols,
                  int32_t pitch, int32_t batch, int64_t stride, void* stream);

/* SmokeSimulator.get_chaos_features ingredients (smoke_simulator.py:47-140) for nframes frames that are
 * frame_stride elements apart, each [h][pitch]:
 *   box_counts[nframes][5]  boxes of side 2,4,8,16,32 holding a pixel above the frame mean       (:89-124)
 *   hist[nframes][nbins]    torch.histogram(frame, bins=nbins, range=(lo, hi)) counts; edges[nbins+1] is the
 *                           torch.linspace(lo, hi, nbins+1) the reference's bin search uses       (:126-140)
 *   mean_out[nframes]       frame mean (may be NULL)
 * box_counts and hist are overwritten. */
SMK_API int smk_frame_features(const float* frames, int64_t frame_stride, int32_t nframes, int32_t h, int32_t w,
                       int32_t pitch, const float* edges, int32_t nbins, float lo, float hi,
                       int32_t* box_counts, int32_t* hist, float* mean_out, void* stream);
/*   sumsq[n] = ||frame[n+1] - frame[n]||^2 (double), n < nframes-1: the distances of compute_lyapunov_exponent (:67-87) */
SMK_API int smk_frame_distances(const float* frames, int64_t frame_stride, int32_t nframes, int32_t h, int32_t w,
                        int32_t pitch, double* sumsq, void* stream);

/* ---- slab halo exchange over NCCL, driven from C (SURVEY.md s8e: rows are contiguous, one send and one receive
 *      of rows x pitch floats per neighbour and field) -----------------------------------------------------
 * The library does not link NCCL: smk_nccl_load finds the libnccl.so.2 already in the process (PyTorch's) or at
 * libpath_host; without it these entry points return SMK_EUNSUPPORTED.  Typical use: every rank calls
 * smk_nccl_load; rank 0 calls smk_nccl_unique_id and broadcasts the 128 bytes over the host's own channel
 * (torch.distributed); every rank calls smk_nccl_comm_init (collective, blocks until all ranks arrive); then one
 * smk_nccl_exchange per exchange phase of the step: all blocks of the call form one ncclGroup on `stream`.
 * NCCL errors are returned as 1000 + ncclResult_t. */
typedef struct smk_halo_block {
    void* ptr;          /* device pointer of the first element of the block                          */
    int64_t count;      /* fp32 elements (rows x pitch)                                              */
    int32_t peer;       /* rank of the neighbour                                                     */
    int32_t is_send;    /* 1: ncclSend, 0: ncclRecv                                                  */
} smk_halo_block_t;
SMK_API int smk_nccl_load(const char* libpath_host, int32_t* version_host);
SMK_API int smk_nccl_unique_id(void* id128_host);
SMK_API int smk_nccl_comm_init(const void* id128_host, int32_t rank, int32_t world, void** comm_out_host);
SMK_API int smk_nccl_comm_destroy(void* comm);
SMK_API int smk_nccl_exchange(void* comm, const smk_halo_block_t* blocks_host, int32_t nblocks, void* stream);

/* ---- slab halo exchange by direct peer stores over NVLink, and the slab step issued from C (csrc/peer_halo.cu) -----------
 * Every rank owns a mailbox in device memory: for each of its two neighbours two slots (exchange number & 1) of four field
 * regions (u, v, density, p; field_stride elements apart), and one arrival counter per neighbour.  The mailbox is exported
 * with smk_ipc_export, the 64-byte handle travels over the host's own channel (torch.distributed), the neighbours map it with
 * smk_ipc_open.  smk_peer_push copies this rank's boundary rows into the neighbours' mailboxes (16-byte peer stores) and bumps
 * their counters (st.release.sys); smk_peer_unpack waits for this rank's counters (ld.acquire.sys) and copies its mailbox
 * slots into the ghost rows.  link[0] is the upper neighbour (rank - 1), link[1] the lower one (rank + 1); a side without a
 * neighbour has remote_mailbox == NULL.  Offsets and counts are in fp32 elements relative to the base of the field, multiples
 * of 4 (whole rows of a pitch that is a multiple of 4); field order u, v, density, p.  seq points at two zero-initialised
 * uint32 in this rank's memory (exchanges completed; scratch).  All ranks must issue the same sequence of exchanges. */
typedef struct smk_peer_link {
    float* remote_mailbox;      /* the neighbour's region that receives FROM this rank, slot 0 (peer-mapped)         */
    uint32_t* remote_flag;      /* the neighbour's counter this rank bumps after a push (peer-mapped)                */
    float* local_mailbox;       /* this rank's region that receives from that neighbour, slot 0                      */
    uint32_t* local_flag;       /* this rank's counter that neighbour bumps                                          */
    int64_t send_off[4], send_count[4];   /* rows this rank owns that the neighbour stores as ghost rows             */
    int64_t recv_off[4], recv_count[4];   /* this rank's ghost rows on that side                                     */
} smk_peer_link_t;
typedef struct smk_peer_comm {
    smk_peer_link_t link[2];
    int64_t field_stride;       /* elements between the field regions of a slot (>= the largest count)               */
    int64_t parity_stride;      /* elements between the two slots of a region (>= 4 * field_stride)                  */
    uint32_t* seq;
} smk_peer_comm_t;
/*     handle + byte offset of `ptr` inside its device allocation (cudaIpcGetMemHandle works on allocation bases) */
SMK_API int smk_ipc_export(const void* ptr, void* handle64_host, int64_t* offset_host);
SMK_API int smk_ipc_open(const void* handle64_host, int64_t offset, void** ptr_out_host);
SMK_API int smk_ipc_close(void* ptr, int64_t offset);
/*     field_base_host[4]: device pointers of the live u, v, density, p of this rank; NULL entries are not exchanged */
SMK_API int smk_peer_push(const smk_peer_comm_t* c, float* const* field_base_host, void* stream);
SMK_API int smk_peer_unpack(const smk_peer_comm_t* c, float* const* field_base_host, void* stream);
/* One step() (navier_stokes.py:151-173) of a row slab in a single call: [peer exchange of u, v, density, p when comm != NULL],
 *     forces + diffusion + divergence, the Jacobi launches, gradient subtract, the three advections with their reach guards
 *     (chk_* may be NULL).  With comm the caller's halo must be at least jacobi_iters + 4 rows (one exchange per step).  comm == NULL
 *     steps a slab whose ghost rows the caller refreshed itself, or an undecomposed grid (gh == 0).
 *     flags (comm != NULL): SMK_SLAB_PUSH_HEAD -- push this rank's boundary rows at the head of the step (the plain exchange);
 *     SMK_SLAB_PUSH_TAIL -- push the boundary rows the NEXT step needs from the middle of this step's density advection (the rows
 *     to send are advected first), so that the transfer overlaps compute; the next call then omits SMK_SLAB_PUSH_HEAD.  All ranks
 *     pass the same flags, and nothing may change the fields between a PUSH_TAIL step and the step that consumes it. */
#define SMK_SLAB_PUSH_HEAD 1
#define SMK_SLAB_PUSH_TAIL 2
SMK_API int smk_slab_step(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, const smk_peer_comm_t* comm, int32_t flags,
                          const smk_slab_check_t* chk_u, const smk_slab_check_t* chk_v, const smk_slab_check_t* chk_d, void* stream);

/*     the tail of that step alone: gradient subtract (:148-149) + advection of u, v, density (:166-168) + decay (:171) on the live
 *     copies, which flip.  On big fields the gradient subtract is fused into the u and v advections (SMK_PROJECT_FUSED=0 disables). */
SMK_API int smk_project_advect(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm,
                               const smk_slab_check_t* chk_u, const smk_slab_check_t* chk_v, const smk_slab_check_t* chk_d, void* stream);

/* ---- reverse mode: adjoints of the step's phases (csrc/adjoint.cu), composed by smokephysai_b200/autodiff.py -------------------
 * Each entry is the transpose of one forward phase, linearised at the forward values it is given; gradients follow torch autograd
 * through the reference's ops (floor: no gradient; torch.clamp passes it where lo <= x <= hi; bilinear weights from the clamped
 * integer corners).  Gradient buffers have the layout of the field they belong to (pads zero).  No float atomics: two calls on the
 * same inputs give bitwise-equal results.  SMK_EUNSUPPORTED on a slab grid (gh != 0). */

/*     adjoint of smk_advect (field [batch][rows][cols] advected by (u, v)).  The effective output gradient is
 *       e = (g_out + (g_frame + fmul*g_frame)) * scale      (g_out, g_frame and fmul may each be NULL: zero / no fractal)
 *     with g_frame [batch][h][pitch_c] frame_stride apart and fmul [h][pitch_c] (cell-centred fields only).  g_field receives the
 *     field gradient (written, or added when accumulate != 0); the gradients through the back-trace are added into g_u and g_v.
 *     g_field may alias g_u or g_v and g_out may alias any output.  workspace: 16 + 32*batch*rows*cols bytes, 16-byte aligned. */
SMK_API int smk_advect_adjoint(const smk_grid_t* g, const float* field, int32_t rows, int32_t cols, int32_t pitch, int64_t stride,
                               const float* u, const float* v, float dt, float scale,
                               const float* g_out, const float* g_frame, int64_t frame_stride, const float* fmul,
                               float* g_field, int32_t accumulate, float* g_u, float* g_v, void* workspace, void* stream);
/*     adjoint of smk_project: g_p = g_p_in + the transpose of the gradient subtract applied to (g_u, g_v); g_p_in may be NULL (zero).
 *     The gradients of u and v pass through unchanged. */
SMK_API int smk_project_adjoint(const smk_grid_t* g, const float* g_u, const float* g_v, const float* g_p_in, float* g_p, float dt,
                                void* stream);
/*     adjoint of K Jacobi sweeps (smk_jacobi): from the gradient g_p_in of the swept pressure, g_p (of the pressure before the sweeps,
 *     ring cells included) and g_div (of the divergence).  T as smk_jacobi.  workspace: 5 fields of batch * F floats, F = stride_c
 *     (h * pitch_c when batch == 1), 16-byte aligned; NULL allowed when K == 0. */
SMK_API int smk_jacobi_adjoint(const smk_grid_t* g, const float* g_p_in, float* g_p, float* g_div, int32_t K, int32_t T,
                               float* workspace, void* stream);
/*     adjoint of smk_forces_diffuse_div: from the gradients of (u_out, v_out, d_out, div), those of (u, v, d) before the buoyancy and
 *     the diffusions.  Outputs must not alias inputs. */
SMK_API int smk_forces_diffuse_div_adjoint(const smk_grid_t* g, const float* g_u_diff, const float* g_v_diff, const float* g_d_diff,
                                           const float* g_div, float* g_u, float* g_v, float* g_d, float dt, float c_uv, float c_d,
                                           void* stream);
/*     intensity gradient of smk_splat_sources: g_intensity[k] = sum over emitter k's footprint of g_density * its splat weight,
 *     for the nsources = offsets[batch] emitters of (sources, offsets); a fixed-order tree per emitter. */
SMK_API int smk_splat_sources_adjoint(const smk_grid_t* g, const float* g_density, const smk_source_t* sources,
                                      const int32_t* offsets, int32_t nsources, float* g_intensity, void* stream);
/*     the same with accumulate = 1: g_intensity[k] += that sum (one rounded add per call, so successive calls sum in call order);
 *     accumulate = 0 is smk_splat_sources_adjoint. */
SMK_API int smk_splat_sources_adjoint_ex(const smk_grid_t* g, const float* g_density, const smk_source_t* sources,
                                         const int32_t* offsets, int32_t nsources, int32_t accumulate, float* g_intensity,
                                         void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SMOKE_B200_H */
