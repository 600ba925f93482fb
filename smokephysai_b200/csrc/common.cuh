// common.cuh -- shared device helpers and the internal launcher prototypes of libsmoke_sm100.so.
//
// Arithmetic contract (SURVEY.md s8a "parity traps"): every fp32 operation is rounded once, in the
// association the reference's torch expressions imply.  The library is compiled with -fmad=false, so
// nvcc never contracts a*b+c; division is IEEE (-prec-div=true default).  Do not add fast-math flags.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "../../include/smoke_b200.h"

namespace smk {

// ---- frame output in SMK_FRAME_F32 / _F16 / _BF16 ----------------------------------------------------------------
// A frame element is the fp32 value the step computes (fractal factor applied), rounded once to the frame type,
// round-to-nearest-even, just before the store (cvt.rn: overflow -> inf, subnormals kept, nothing saturates).  `frame`
// points at the frame base, `k` counts elements of the frame type; `fmt` is uniform over the launch, so the branch
// never diverges.  frame_st4 needs k to be a multiple of 4 (16-byte fp32 / 8-byte half stores).
__device__ __forceinline__ unsigned pack_h2(const __half2 h) { return *reinterpret_cast<const unsigned*>(&h); }
__device__ __forceinline__ unsigned pack_b2(const __nv_bfloat162 h) { return *reinterpret_cast<const unsigned*>(&h); }
__device__ __forceinline__ void frame_st4(void* frame, const size_t k, const float4 v, const int fmt)
{
    if (fmt == SMK_FRAME_F16)
        *reinterpret_cast<uint2*>(static_cast<__half*>(frame) + k) =
            make_uint2(pack_h2(__floats2half2_rn(v.x, v.y)), pack_h2(__floats2half2_rn(v.z, v.w)));
    else if (fmt == SMK_FRAME_BF16)
        *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(frame) + k) =
            make_uint2(pack_b2(__floats2bfloat162_rn(v.x, v.y)), pack_b2(__floats2bfloat162_rn(v.z, v.w)));
    else
        *reinterpret_cast<float4*>(static_cast<float*>(frame) + k) = v;
}
__device__ __forceinline__ void* frame_offset(void* frame, const size_t k, const int fmt)
{
    return static_cast<char*>(frame) + k * (fmt == SMK_FRAME_F32 ? 4 : 2);
}
__device__ __forceinline__ void frame_st1(void* frame, const size_t k, const float v, const int fmt)
{
    if (fmt == SMK_FRAME_F16)       static_cast<__half*>(frame)[k] = __float2half_rn(v);
    else if (fmt == SMK_FRAME_BF16) static_cast<__nv_bfloat16*>(frame)[k] = __float2bfloat16_rn(v);
    else                            static_cast<float*>(frame)[k] = v;
}

__device__ __forceinline__ int clampi(int a, int lo, int hi) { return min(max(a, lo), hi); }
// torch.clamp(x, lo, hi) == min(max(x, lo), hi)
__device__ __forceinline__ float clampf(float a, float lo, float hi) { return fminf(fmaxf(a, lo), hi); }

// a8: bilinear_interpolate (navier_stokes.py:111-131) with a sampler f(row, col) over a Hg x Wg field.
// Corner indices are clamped AFTER the +1 (:116-123), weights come from the clamped corners (:125-128),
// the sum is ((wa*f00 + wb*f01) + wc*f10) + wd*f11 (:130-131).
template <class Sampler>
__device__ __forceinline__ float bilerp(const Sampler& f, int Hg, int Wg, float y, float x)
{
    int x0 = (int)floorf(x), y0 = (int)floorf(y);
    int x1 = x0 + 1, y1 = y0 + 1;
    x0 = clampi(x0, 0, Wg - 1); x1 = clampi(x1, 0, Wg - 1);
    y0 = clampi(y0, 0, Hg - 1); y1 = clampi(y1, 0, Hg - 1);
    const float ax = (float)x1 - x, bx = x - (float)x0;
    const float ay = (float)y1 - y, by = y - (float)y0;
    const float wa = ax * ay, wb = bx * ay, wc = ax * by, wd = bx * by;
    float s = wa * f(y0, x0) + wb * f(y0, x1);
    s = s + wc * f(y1, x0);
    s = s + wd * f(y1, x1);
    return s;
}

// a9: interpolate_velocity_u at integer (i, j) (navier_stokes.py:97-102), closed form.
// x = min(j+0.5, w-1): for j <= w-2 the weights are 0.5/0.5 along x; along y the weight pair is (1, 0)
// unless i is U's last row, where the clamped y1 == y0 makes both 0.  The zero-weight terms only add +-0.
template <class Sampler>
__device__ __forceinline__ float interp_u_at(const Sampler& U, int h, int w, int i, int j)
{
    if (j > w - 2 || i > h - 1) return 0.0f;       // U has h+1 rows: last row index is h
    return 0.5f * U(i, j) + 0.5f * U(i, j + 1);
}
// interpolate_velocity_v at integer (i, j) (navier_stokes.py:104-109): 0.5*(V[i][j] + V[i+1][j]) for
// i <= h-2 and j <= w-1 (V has w+1 columns), else 0.
template <class Sampler>
__device__ __forceinline__ float interp_v_at(const Sampler& V, int h, int w, int i, int j)
{
    if (i > h - 2 || j > w - 1) return 0.0f;
    return 0.5f * V(i, j) + 0.5f * V(i + 1, j);
}

struct GlobalField {
    const float* __restrict__ p; int pitch;
    __device__ __forceinline__ float operator()(int i, int j) const { return __ldg(p + (size_t)i * pitch + j); }
};

// ---- programmatic dependent launch -------------------------------------------------------------------------
// The phase-per-kernel path is a chain of dependent kernels on one stream (10 per step at 1024^2, K = 100), each a few
// microseconds long: the gap between "last CTA of kernel n exits" and "first CTA of kernel n + 1 runs" is paid ten
// times per step.  Kernels of the chain are launched with cudaLaunchAttributeProgrammaticStreamSerialization and start with
// pdl_prologue(): griddepcontrol.wait blocks until the previous kernel has completed and its writes are visible (so every
// global access of the kernel stays ordered after it), griddepcontrol.launch_dependents lets the NEXT kernel's CTAs
// be scheduled as soon as this kernel's CTAs have all started, so its launch latency and prologue overlap this kernel.
// SMK_PDL=0 launches the chain the classic way.  A kernel launched without the attribute runs pdl_prologue() as no-ops.
__device__ __forceinline__ void pdl_prologue()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
bool pdl_enabled(cudaStream_t s);
template <class... P, class... A>
inline void launch_chain(void (*kernel)(P...), const dim3 grid, const dim3 block, const size_t smem, cudaStream_t s, A&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr = {};
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr; cfg.numAttrs = pdl_enabled(s) ? 1 : 0;
    (void)cudaLaunchKernelEx(&cfg, kernel, P(args)...);          // errors are picked up by check_launch()
}

// add_smoke_source at one cell (navier_stokes.py:45-48): acc plus emitter e's Gaussian when cell (i, j) lies within its radius.
// k_splat, the reset start of k_step_fused and the continuous emitters of k_step_fused / k_step_cluster add a cell's emitters
// through this, in list order: bit-identical densities.
__device__ __forceinline__ float splat_add(float acc, const int i, const int j, const smk_source_t& e)
{
    const long long dx = (long long)j - e.x, dy = (long long)i - e.y;
    const float dist = sqrtf((float)(dx * dx + dy * dy));            // navier_stokes.py:45
    if (dist <= (float)e.radius) {                                   // :46
        const double r3 = (double)e.radius / 3.0;
        const float denom = (float)(2.0 * (r3 * r3));
        const float d2 = dist * dist;
        acc = acc + e.intensity * expf((-d2) / denom);               // :48
    }
    return acc;
}

// Tuning / test switches from the environment, read ONCE per process (getenv is not free and not thread-safe against
// setenv; a launch must not pay for it) and again only on smk_reload_env(), which the tests call after changing a variable.
// SMK_ENV_UNSET marks a variable that is not set: the launcher then picks by its own rule.
constexpr int SMK_ENV_UNSET = -2147483647 - 1;
struct EnvCfg {
    int pdl;             // SMK_PDL            0: no programmatic dependent launch
    int fused_slice;     // SMK_FUSED_SLICE    0: one CTA per simulation, n > 0: time-sliced schedule with pieces of n steps
    int fused_cluster;   // SMK_FUSED_CLUSTER  0: never split a simulation over a CTA cluster, 2: always (when supported)
    int jacobi_packed;   // SMK_JACOBI_PACKED  0: scalar in-place kernel, else mask of packed row pairs
    int jacobi_stream;   // SMK_JACOBI_STREAM  0 off / 1 LDGSTS / 2 TMA staging of the streaming kernel
    int jacobi_tile;     // SMK_JACOBI_TILE    1: 64 x 128 (8 warps), 2: 128 x 128, 3: 64 x 128 (16 warps)
    int fdd_bulk;        // SMK_FDD_BULK       0 / 1: staging path of k_forces_diffuse_div
    int advect_tiled;    // SMK_ADVECT_TILED   0 / 1: direct / shared-memory tiled advection
    int project_fused;   // SMK_PROJECT_FUSED  0: k_project + k_advect(u) as two kernels even where the fused one applies
    int push_stream;     // SMK_PUSH_STREAM    0: the push a slab step issues for the next step stays on the caller's stream
    int advect_tma;      // SMK_ADVECT_TMA     0: interior tiles of k_advect_tiled stage with cp.async like the others (default: TMA)
    int splat_big;       // SMK_SPLAT_BIG      0 / 1: k_splat / k_splat_big (128 x 64 cells per CTA) whatever the grid size
};
const EnvCfg& env();

// thread-local error string + checks (abi.cu)
int fail(int code, const char* fmt, ...);
int check_launch(const char* what);
// optional per-kernel event timing (smk_profile_begin/end): one scope object around each launch
void prof_mark(int phase, cudaStream_t s, bool stop);
struct ProfScope {
    int phase; cudaStream_t s;
    ProfScope(int phase_, cudaStream_t s_) : phase(phase_), s(s_) { prof_mark(phase, s, false); }
    ~ProfScope() { prof_mark(phase, s, true); }
};
bool aligned16(const void* p);
int check_grid(const smk_grid_t* g, const char* who);

// launchers (one per kernel family); all asynchronous on `s`
int launch_splat(const smk_grid_t* g, float* density, const smk_source_t* src, const int32_t* off, cudaStream_t s);
int launch_diffuse(const float* in, float* out, int rows, int cols, int pitch, int batch, int64_t stride, float c, cudaStream_t s);
int launch_forces_diffuse_div(const smk_grid_t* g, const float* u, const float* v, const float* d,
                              float* uo, float* vo, float* dout, float* div, float dt, float c_uv, float c_d, cudaStream_t s);
int launch_divergence(const smk_grid_t* g, const float* u, const float* v, float* div, float dt, cudaStream_t s);
int launch_jacobi(const smk_grid_t* g, const float* div, float* p, float* scratch, int K, int T, int* in_scratch, cudaStream_t s);
int launch_project(const smk_grid_t* g, const float* p, float* u, float* v, float dt, cudaStream_t s);
int launch_bilerp(const float* f, int rows, int cols, int pitch, const float* y, const float* x, float* out, int64_t n, int mode, cudaStream_t s);
// part (tiled kernel only, see advect_is_tiled): band_n > 0 -> only the tile rows [band_lo, band_lo + band_n); else every tile row
// except those of the (up to two, ascending, disjoint) bands [skip_lo[k], skip_lo[k] + skip_n[k])
struct AdvectPart { int band_lo, band_n, skip_lo[2], skip_n[2]; };
// frame / frame_stride / frame_format: the (fractal-scaled) copy of the result, SMK_FRAME_*, stride in elements of that type
int launch_advect(const smk_grid_t* g, const float* field, float* out, int rows, int cols, int pitch, int64_t stride,
                  const float* u, const float* v, float dt, float scale, void* frame, int64_t frame_stride,
                  const float* fmul, const smk_slab_check_t* chk, cudaStream_t s, int proj = 0, const float* p = nullptr, float* vout = nullptr,
                  const AdvectPart* part = nullptr, int frame_format = SMK_FRAME_F32);
bool advect_can_fuse_project(const smk_grid_t* g);
// 128-byte CUtensorMap of a (pitch, rows, batch) fp32 tensor read / written in box_cols x box_rows x 1 boxes (jacobi.cu); false when
// the driver entry point is missing or the shape cannot be encoded
struct alignas(64) TmaMap { unsigned long long opaque[16]; };
bool tma_map_3d(void* map128, const float* base, int pitch, int rows, int batch, int64_t batch_stride, int box_rows, int box_cols);
bool advect_is_tiled(const smk_grid_t* g, int rows, int cols);
int advect_tile_rows();
int launch_div_norms(const smk_grid_t* g, const float* u, const float* v, float* out, cudaStream_t s);
int launch_jacobi_residual(const smk_grid_t* g, const float* div, const float* p, float* out, cudaStream_t s);
int launch_fractal_fields(float* perlin, float* mandel, float* mul, int na, int nb, int pitch, float intensity, int iterations,
                          const float* px, const float* py, const float* mx, const float* my, cudaStream_t s);
int launch_frame_features(const float* frames, int64_t frame_stride, int nframes, int h, int w, int pitch,
                          const float* edges, int nbins, float lo, float hi, int* box_counts, int* hist, float* mean_out, cudaStream_t s);
int launch_frame_distances(const float* frames, int64_t frame_stride, int nframes, int h, int w, int pitch, double* sumsq, cudaStream_t s);
bool fused_supported(const smk_grid_t* g);
bool fused_full_size(const smk_grid_t* g);   // 128 x 128 cells at the natural pitches: the k_step_fused<true, ..> / k_step_cluster grid
int pick_cluster(int batch);          // CTAs per simulation k_step_cluster would use for `batch` 128 x 128 simulations (0: one CTA each)

// One call of the step entry points (smk_step*, smk_run_steps*), everything but the grid, state and params: abi.cu's
// run_steps validates it and runs it on the phase kernels or on launch_steps_fused.
struct StepCall {
    int nsteps = 1;
    void* frames = nullptr;                   // may be NULL; strides in elements of frame_format (SMK_FRAME_*)
    int64_t frame_step_stride = 0, frame_batch_stride = 0;
    const float* fmul = nullptr;
    int frame_format = SMK_FRAME_F32;
    const smk_source_t* csrc = nullptr;       // emitters splatted at the head of every step (NULL: none); step t of simulation b
    const int32_t* coff = nullptr;            //   adds records [coff[t * cstride + b], coff[t * cstride + b + 1])
    int cstride = 0;                          // 0: one list for every step (continuous sources); batch: a schedule, a row per step
    bool reset = false;                       // start from a reset state splatted once with (rsrc, roff): k_step_fused only
    const smk_source_t* rsrc = nullptr;
    const int32_t* roff = nullptr;
};
int launch_steps_fused(const smk_grid_t* g, const smk_state_t* st, const smk_params_t* prm, const StepCall& c, cudaStream_t s);
// One step on the phase kernels (peer_halo.cu), for a whole grid or a row slab whose ghost rows are current: the continuous
// emitters (csrc / coff), buoyancy + diffusion + divergence, the Jacobi sweeps, the gradient subtract and the three advections.
// All per-call inputs may be NULL: the frame (whole grids), the reach guards chk_* and the comm of the tail push (slabs).
int phase_step(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, const smk_source_t* csrc, const int32_t* coff,
               void* frame, int64_t frame_stride, const float* fmul, int frame_format,
               const smk_slab_check_t* chk_u, const smk_slab_check_t* chk_v, const smk_slab_check_t* chk_d,
               const smk_peer_comm_t* push_comm, cudaStream_t s);
int fused_plan(int nsims, int nsteps, int piece_len, int32_t* items, int capacity, int* count);
int launch_apply_mul(const float* f, const float* mul, float* out, int rows, int cols, int pitch, int batch, int64_t stride, cudaStream_t s);

}  // namespace smk
