// abi.cu -- the extern "C" surface of libsmoke_sm100.so (include/smoke_b200.h): argument validation,
// thread-local error string, and the one runner behind the step entry points (navier_stokes.py:151-173).
#include <atomic>
#include <mutex>
#include <cstdarg>
#include <cstdio>
#include <vector>
#include <cstdlib>
#include "common.cuh"

namespace smk {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

// ---- environment switches: read once, re-read on smk_reload_env() ------------------------------------------
static EnvCfg g_env;
static std::atomic<int> g_env_ready{0};
static std::mutex g_env_mutex;
static int env_int(const char* name)
{
    const char* e = getenv(name);
    return (e && e[0]) ? atoi(e) : SMK_ENV_UNSET;
}
static void env_read_locked()
{
    EnvCfg c;
    c.pdl = env_int("SMK_PDL");
    c.fused_slice = env_int("SMK_FUSED_SLICE");
    c.fused_cluster = env_int("SMK_FUSED_CLUSTER");
    c.jacobi_packed = env_int("SMK_JACOBI_PACKED");
    c.jacobi_stream = env_int("SMK_JACOBI_STREAM");
    c.jacobi_tile = env_int("SMK_JACOBI_TILE");
    c.fdd_bulk = env_int("SMK_FDD_BULK");
    c.advect_tiled = env_int("SMK_ADVECT_TILED");
    c.project_fused = env_int("SMK_PROJECT_FUSED");
    c.push_stream = env_int("SMK_PUSH_STREAM");
    c.splat_big = env_int("SMK_SPLAT_BIG");
    c.advect_tma = env_int("SMK_ADVECT_TMA");
    g_env = c;
    g_env_ready.store(1, std::memory_order_release);
}
const EnvCfg& env()
{
    if (!g_env_ready.load(std::memory_order_acquire)) {
        std::lock_guard<std::mutex> lock(g_env_mutex);
        if (!g_env_ready.load(std::memory_order_relaxed)) env_read_locked();
    }
    return g_env;
}

// SMK_PDL=0 switches programmatic dependent launch off; never inside a stream capture (plain kernel nodes there)
bool pdl_enabled(cudaStream_t s)
{
    if (env().pdl == 0) return false;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone;
}

int check_launch(const char* what)
{
    g_launches.fetch_add(1, std::memory_order_relaxed);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail((int)e, "%s: %s", what, cudaGetErrorString(e));
    return SMK_OK;
}

// ---- per-kernel event timing ---------------------------------------------------------------------------
struct ProfRec { int phase; cudaEvent_t a, b; };
static std::atomic<bool> g_prof_on{false};
static std::vector<ProfRec> g_prof;          // records in use
static std::vector<cudaEvent_t> g_prof_pool; // pre-created events (2 per record)
static size_t g_prof_used = 0;

void prof_mark(int phase, cudaStream_t s, bool stop)
{
    if (!g_prof_on.load(std::memory_order_relaxed)) return;
    if (!stop) {
        if (g_prof_used + 2 > g_prof_pool.size()) return;      // pool exhausted: later launches go untimed
        ProfRec r{phase, g_prof_pool[g_prof_used], g_prof_pool[g_prof_used + 1]};
        g_prof_used += 2;
        cudaEventRecord(r.a, s);
        g_prof.push_back(r);
    } else if (!g_prof.empty() && g_prof.back().phase == phase) {
        cudaEventRecord(g_prof.back().b, s);
    }
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int check_grid(const smk_grid_t* g, const char* who)
{
    if (!g) return fail(SMK_EINVAL, "%s: grid is NULL", who);
    if (g->h < 1 || g->w < 1) return fail(SMK_EINVAL, "%s: bad grid %d x %d", who, g->h, g->w);
    if (g->batch < 1 || g->batch > 65535) return fail(SMK_EINVAL, "%s: batch %d outside [1, 65535]", who, g->batch);
    if (g->pitch_u < g->w || g->pitch_c < g->w || g->pitch_v < g->w + 1)
        return fail(SMK_EINVAL, "%s: pitch smaller than the row (u %d, v %d, c %d for w=%d)", who, g->pitch_u, g->pitch_v, g->pitch_c, g->w);
    if ((g->pitch_u | g->pitch_v | g->pitch_c) & 3)
        return fail(SMK_EINVAL, "%s: pitches must be multiples of 4 elements (u %d, v %d, c %d)", who, g->pitch_u, g->pitch_v, g->pitch_c);
    if ((g->stride_u | g->stride_v | g->stride_c) & 3)
        return fail(SMK_EINVAL, "%s: batch strides must be multiples of 4 elements", who);
    if (g->batch > 1 && (g->stride_u < (int64_t)(g->h + 1) * g->pitch_u || g->stride_v < (int64_t)g->h * g->pitch_v ||
                         g->stride_c < (int64_t)g->h * g->pitch_c))
        return fail(SMK_EINVAL, "%s: batch stride smaller than one field", who);
    if (g->gh != 0 && (g->row0 < 0 || g->row0 + g->h > g->gh))
        return fail(SMK_EINVAL, "%s: slab rows [%d, %d) outside the global grid of %d rows", who, g->row0, g->row0 + g->h, g->gh);
    if (g->gh == 0 && g->row0 != 0) return fail(SMK_EINVAL, "%s: row0 set without gh", who);
    return SMK_OK;
}

int check_solid(const smk_grid_t* g, const uint8_t* solid, int64_t solid_stride, const char* who)
{
    if (solid && reinterpret_cast<uintptr_t>(solid) % 4) return fail(SMK_EINVAL, "%s: solid is not 4-byte aligned", who);
    if (solid_stride != 0 && (!solid || solid_stride != (int64_t)g->h * g->pitch_c))
        return fail(SMK_EINVAL, "%s: solid_batch_stride must be 0 or h * pitch_c (%lld) with a mask, got %lld", who,
                    (long long)g->h * g->pitch_c, (long long)solid_stride);
    if (solid && g->gh != 0) return fail(SMK_EUNSUPPORTED, "%s: solid cells are not available on a slab grid (gh != 0)", who);
    return SMK_OK;
}

static int check_ptrs(const char* who, std::initializer_list<const void*> ps)
{
    int k = 0;
    for (const void* p : ps) {
        if (!p) return fail(SMK_EINVAL, "%s: pointer argument %d is NULL", who, k);
        if (!aligned16(p)) return fail(SMK_EINVAL, "%s: pointer argument %d is not 16-byte aligned", who, k);
        ++k;
    }
    return SMK_OK;
}

}  // namespace smk

using namespace smk;

#define SMK_TRY(x) do { const int rc_ = (x); if (rc_ != SMK_OK) return rc_; } while (0)

extern "C" {

int smk_version(void) { return SMK_ABI_VERSION; }

const char* smk_last_error_string(void) { return g_err; }

int smk_device_info(int32_t* sm_count, int32_t* cc, int32_t* smem_optin)
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    cudaDeviceProp p;
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&p, dev);
    if (e != cudaSuccess) return fail((int)e, "smk_device_info: %s", cudaGetErrorString(e));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc) *cc = p.major * 10 + p.minor;
    if (smem_optin) *smem_optin = (int32_t)p.sharedMemPerBlockOptin;
    return SMK_OK;
}

int smk_launch_count(int64_t* count)
{
    if (!count) return fail(SMK_EINVAL, "smk_launch_count: NULL");
    *count = g_launches.load(std::memory_order_relaxed);
    return SMK_OK;
}

int smk_set_device(int32_t device)
{
    const cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail((int)e, "smk_set_device(%d): %s", device, cudaGetErrorString(e));
    return SMK_OK;
}

int smk_reload_env(void)
{
    std::lock_guard<std::mutex> lock(g_env_mutex);
    env_read_locked();
    return SMK_OK;
}

int smk_profile_begin(int32_t max_records)
{
    if (max_records < 1 || max_records > (1 << 20)) return fail(SMK_EINVAL, "smk_profile_begin: max_records %d", max_records);
    if (g_prof_on.load()) return fail(SMK_EINVAL, "smk_profile_begin: a profile is already open");
    while (g_prof_pool.size() < 2 * (size_t)max_records) {
        cudaEvent_t e;
        const cudaError_t rc = cudaEventCreate(&e);
        if (rc != cudaSuccess) return fail((int)rc, "smk_profile_begin: %s", cudaGetErrorString(rc));
        g_prof_pool.push_back(e);
    }
    g_prof.clear();
    g_prof.reserve(max_records);
    g_prof_used = 0;
    g_prof_on.store(true);
    return SMK_OK;
}

int smk_profile_end(double* ms, int64_t* launches, int32_t nphases)
{
    if (!g_prof_on.load()) return fail(SMK_EINVAL, "smk_profile_end: no profile is open");
    g_prof_on.store(false);
    if (!ms || !launches || nphases < SMK_PH_COUNT) return fail(SMK_EINVAL, "smk_profile_end: need %d phase slots", SMK_PH_COUNT);
    for (int k = 0; k < nphases; ++k) { ms[k] = 0.0; launches[k] = 0; }
    for (const ProfRec& r : g_prof) {
        cudaError_t rc = cudaEventSynchronize(r.b);
        float t = 0.f;
        if (rc == cudaSuccess) rc = cudaEventElapsedTime(&t, r.a, r.b);
        if (rc != cudaSuccess) return fail((int)rc, "smk_profile_end: %s", cudaGetErrorString(rc));
        ms[r.phase] += (double)t;
        launches[r.phase] += 1;
    }
    g_prof.clear();
    return SMK_OK;
}

int smk_splat_sources(const smk_grid_t* g, float* density, const smk_source_t* sources, const int32_t* offsets, void* stream)
{
    SMK_TRY(check_grid(g, "smk_splat_sources"));
    SMK_TRY(check_ptrs("smk_splat_sources", {density}));
    if (!sources || !offsets) return fail(SMK_EINVAL, "smk_splat_sources: sources/offsets NULL");
    return launch_splat(g, density, sources, offsets, (cudaStream_t)stream);
}

int smk_diffuse(const float* in, float* out, int32_t rows, int32_t cols, int32_t pitch, int32_t batch, int64_t stride,
                float c, void* stream)
{
    if (rows < 1 || cols < 1 || pitch < cols || batch < 1 || batch > 65535)
        return fail(SMK_EINVAL, "smk_diffuse: bad shape %d x %d pitch %d batch %d", rows, cols, pitch, batch);
    if (!in || !out || in == out) return fail(SMK_EINVAL, "smk_diffuse: in/out NULL or aliased (the stencil is out of place)");
    return launch_diffuse(in, out, rows, cols, pitch, batch, stride, c, (cudaStream_t)stream);
}

int smk_forces_diffuse_div(const smk_grid_t* g, const float* u, const float* v, const float* d,
                           float* u_out, float* v_out, float* d_out, float* div, float dt, float c_uv, float c_d, void* stream)
{
    SMK_TRY(check_grid(g, "smk_forces_diffuse_div"));
    SMK_TRY(check_ptrs("smk_forces_diffuse_div", {u, v, d, u_out, v_out, d_out}));
    if (u == u_out || v == v_out || d == d_out) return fail(SMK_EINVAL, "smk_forces_diffuse_div: outputs must not alias inputs");
    if (!(dt != 0.0f)) return fail(SMK_EINVAL, "smk_forces_diffuse_div: dt must be non-zero");
    return launch_forces_diffuse_div(g, u, v, d, u_out, v_out, d_out, div, dt, c_uv, c_d, (cudaStream_t)stream);
}

int smk_divergence(const smk_grid_t* g, const float* u, const float* v, float* div, float dt, void* stream)
{
    SMK_TRY(check_grid(g, "smk_divergence"));
    SMK_TRY(check_ptrs("smk_divergence", {u, v, div}));
    return launch_divergence(g, u, v, div, dt, (cudaStream_t)stream);
}

int smk_jacobi(const smk_grid_t* g, const float* div, float* p, float* p_scratch, int32_t K, int32_t T,
               int32_t* result_in_scratch_host, void* stream)
{
    SMK_TRY(check_grid(g, "smk_jacobi"));
    SMK_TRY(check_ptrs("smk_jacobi", {div, p, p_scratch}));
    if (p == p_scratch) return fail(SMK_EINVAL, "smk_jacobi: p and p_scratch must differ");
    if (K < 0 || T < 0) return fail(SMK_EINVAL, "smk_jacobi: negative K or T");
    if (!result_in_scratch_host) return fail(SMK_EINVAL, "smk_jacobi: result_in_scratch_host is NULL");
    int flag = 0;
    const int rc = launch_jacobi(g, div, p, p_scratch, K, T, &flag, (cudaStream_t)stream);
    *result_in_scratch_host = flag;
    return rc;
}

int smk_jacobi_obst(const smk_grid_t* g, const float* div, float* p, float* p_scratch, const uint8_t* solid, int64_t solid_batch_stride,
                    int32_t K, int32_t T, int32_t* result_in_scratch_host, void* stream)
{
    SMK_TRY(check_grid(g, "smk_jacobi_obst"));
    SMK_TRY(check_ptrs("smk_jacobi_obst", {div, p, p_scratch}));
    if (p == p_scratch) return fail(SMK_EINVAL, "smk_jacobi_obst: p and p_scratch must differ");
    if (K < 0 || T < 0) return fail(SMK_EINVAL, "smk_jacobi_obst: negative K or T");
    if (!result_in_scratch_host) return fail(SMK_EINVAL, "smk_jacobi_obst: result_in_scratch_host is NULL");
    if (!solid || reinterpret_cast<uintptr_t>(solid) % 4) return fail(SMK_EINVAL, "smk_jacobi_obst: solid is NULL or not 4-byte aligned");
    if (solid_batch_stride != 0 && solid_batch_stride != (int64_t)g->h * g->pitch_c)
        return fail(SMK_EINVAL, "smk_jacobi_obst: solid_batch_stride must be 0 or h * pitch_c, got %lld", (long long)solid_batch_stride);
    int flag = 0;
    const int rc = launch_jacobi(g, div, p, p_scratch, K, T, &flag, (cudaStream_t)stream, solid, solid_batch_stride);
    *result_in_scratch_host = flag;
    return rc;
}

int smk_project(const smk_grid_t* g, const float* p, float* u, float* v, float dt, void* stream)
{
    SMK_TRY(check_grid(g, "smk_project"));
    SMK_TRY(check_ptrs("smk_project", {p, u, v}));
    return launch_project(g, p, u, v, dt, (cudaStream_t)stream);
}

int smk_project_ex(const smk_grid_t* g, const float* p, float* u, float* v, float dt, const uint8_t* solid, int64_t solid_batch_stride,
                   void* stream)
{
    SMK_TRY(check_grid(g, "smk_project_ex"));
    SMK_TRY(check_ptrs("smk_project_ex", {p, u, v}));
    SMK_TRY(check_solid(g, solid, solid_batch_stride, "smk_project_ex"));
    if (!solid) return launch_project(g, p, u, v, dt, (cudaStream_t)stream);
    return launch_project_obst(g, p, u, v, solid, solid_batch_stride, dt, (cudaStream_t)stream);
}

int smk_obstacle_faces(const smk_grid_t* g, float* u, float* v, float* div, const uint8_t* solid, int64_t solid_batch_stride, float dt,
                       void* stream)
{
    SMK_TRY(check_grid(g, "smk_obstacle_faces"));
    SMK_TRY(check_ptrs("smk_obstacle_faces", {u, v}));
    if (!solid) return fail(SMK_EINVAL, "smk_obstacle_faces: solid is NULL");
    SMK_TRY(check_solid(g, solid, solid_batch_stride, "smk_obstacle_faces"));
    if (div && !aligned16(div)) return fail(SMK_EINVAL, "smk_obstacle_faces: div is not 16-byte aligned");
    if (div && !(dt != 0.0f)) return fail(SMK_EINVAL, "smk_obstacle_faces: dt must be non-zero");
    return launch_obstacle_faces(g, u, v, div, solid, solid_batch_stride, dt, (cudaStream_t)stream);
}

int smk_obstacle_cells(const smk_grid_t* g, float* d, void* frame, int64_t frame_stride, int32_t frame_format, const uint8_t* solid,
                       int64_t solid_batch_stride, void* stream)
{
    SMK_TRY(check_grid(g, "smk_obstacle_cells"));
    SMK_TRY(check_ptrs("smk_obstacle_cells", {d}));
    if (!solid) return fail(SMK_EINVAL, "smk_obstacle_cells: solid is NULL");
    SMK_TRY(check_solid(g, solid, solid_batch_stride, "smk_obstacle_cells"));
    if (frame_format != SMK_FRAME_F32 && frame_format != SMK_FRAME_F16 && frame_format != SMK_FRAME_BF16)
        return fail(SMK_EINVAL, "smk_obstacle_cells: bad frame_format %d", frame_format);
    if (frame && g->batch > 1 && frame_stride < (int64_t)g->h * g->pitch_c)
        return fail(SMK_EINVAL, "smk_obstacle_cells: frame_stride smaller than one frame");
    return launch_obstacle_cells(g, d, frame, frame_stride, frame_format, solid, solid_batch_stride, (cudaStream_t)stream);
}

int smk_bilerp(const float* field, int32_t rows, int32_t cols, int32_t pitch, const float* y, const float* x,
               float* out, int64_t n, int32_t mode, void* stream)
{
    if (!field || !y || !x || !out) return fail(SMK_EINVAL, "smk_bilerp: NULL pointer");
    if (rows < 1 || cols < 1 || pitch < cols || n < 0 || mode < 0 || mode > 2)
        return fail(SMK_EINVAL, "smk_bilerp: bad arguments (%d x %d pitch %d n %lld mode %d)", rows, cols, pitch, (long long)n, mode);
    return launch_bilerp(field, rows, cols, pitch, y, x, out, n, mode, (cudaStream_t)stream);
}

int smk_advect(const smk_grid_t* g, const float* field, float* out, int32_t rows, int32_t cols, int32_t pitch, int64_t stride,
               const float* u, const float* v, float dt, float scale, float* frame, int64_t frame_stride,
               const float* fmul, void* stream)
{
    SMK_TRY(check_grid(g, "smk_advect"));
    if (!field || !out || !u || !v) return fail(SMK_EINVAL, "smk_advect: NULL pointer");
    if (field == out) return fail(SMK_EINVAL, "smk_advect: the gather is out of place, field == out");
    if (out == u || out == v) return fail(SMK_EINVAL, "smk_advect: out aliases a velocity input");
    if (rows < 1 || cols < 1 || pitch < cols) return fail(SMK_EINVAL, "smk_advect: bad field shape %d x %d pitch %d", rows, cols, pitch);
    // the velocities are u[h+1][w], v[h][w+1] by the grid's own definition; a field larger than either would index past them
    if (rows > g->h + 1 || cols > g->w + 1)
        return fail(SMK_EINVAL, "smk_advect: a %d x %d field does not fit the %d x %d cell grid (at most %d x %d)", rows, cols, g->h, g->w, g->h + 1, g->w + 1);
    if (frame && (rows != g->h || cols != g->w)) return fail(SMK_EINVAL, "smk_advect: frame output needs a cell-centred field");
    return launch_advect(g, field, out, rows, cols, pitch, stride, u, v, dt, scale, frame, frame_stride, fmul, nullptr, (cudaStream_t)stream);
}

int smk_advect_slab(const smk_grid_t* g, const float* field, float* out, int32_t rows, int32_t cols, int32_t pitch,
                    const float* u, const float* v, float dt, float scale, const smk_slab_check_t* chk, void* stream)
{
    SMK_TRY(check_grid(g, "smk_advect_slab"));
    if (g->gh == 0) return fail(SMK_EINVAL, "smk_advect_slab: the grid is not a slab (gh == 0)");
    if (g->batch != 1) return fail(SMK_EUNSUPPORTED, "smk_advect_slab: batch must be 1");
    if (!field || !out || !u || !v) return fail(SMK_EINVAL, "smk_advect_slab: NULL pointer");
    if (field == out || out == u || out == v) return fail(SMK_EINVAL, "smk_advect_slab: out aliases an input");
    if (rows < 1 || cols < 1 || pitch < cols) return fail(SMK_EINVAL, "smk_advect_slab: bad field shape %d x %d pitch %d", rows, cols, pitch);
    if (rows > g->h + 1 || cols > g->w + 1)
        return fail(SMK_EINVAL, "smk_advect_slab: a %d x %d field does not fit the %d x %d cell slab", rows, cols, g->h, g->w);
    if (chk && (!chk->overflow_flag || chk->need_lo > chk->need_hi || chk->valid_lo > chk->valid_hi))
        return fail(SMK_EINVAL, "smk_advect_slab: bad check ranges");
    return launch_advect(g, field, out, rows, cols, pitch, 0, u, v, dt, scale, nullptr, 0, nullptr, chk, (cudaStream_t)stream);
}

// The kernels a step call runs on: one launch per phase per step, or all the steps in one launch of k_step_fused (one CTA per
// simulation, or the time-sliced schedule) or of k_step_cluster (a cluster of CTAs per simulation).
enum StepPlan { PLAN_PHASES, PLAN_FUSED, PLAN_CLUSTER };

// SMK_STEP_AUTO: the fused kernel runs one simulation per SM, so it pays off when a call carries enough work per
// launch -- several steps (the state stays on chip between them), or a single step of at least 32 simulations.
// One step of a few simulations is faster spread over all SMs by the phase kernels (tools/step_latency.py: 37 us
// against 45 us per step() at batch 1; the fused launch also reads and writes the state, ~10 us).
// Solid cells (obstacles) are applied by the phase kernels only: with them the plan is always PLAN_PHASES.
static int pick_step_kernel(const smk_grid_t* g, const smk_params_t* prm, int nsteps, StepPlan* plan, bool solid = false)
{
    *plan = PLAN_PHASES;
    if (prm->step_kernel == SMK_STEP_PHASES) return SMK_OK;
    if (prm->step_kernel != SMK_STEP_AUTO && prm->step_kernel != SMK_STEP_FUSED)
        return fail(SMK_EINVAL, "smk_step: step_kernel %d is not SMK_STEP_AUTO/_PHASES/_FUSED", prm->step_kernel);
    if (solid) {
        if (prm->step_kernel == SMK_STEP_FUSED)
            return fail(SMK_EUNSUPPORTED, "smk_step: SMK_STEP_FUSED does not apply solid obstacles (the phase kernels do)");
        return SMK_OK;
    }
    if (fused_supported(g)) {
        // One simulation per SM pays when there are enough simulations to fill the SMs; a few simulations are faster on the
        // phase kernels spread over all SMs, whose launch gaps programmatic dependent launch has removed.  Measured per step
        // (tools/step_latency_sizes.py, K = 20): 128 x 128: 1 simulation 27.6 us on the phase path against 30.0 fused (20-step
        // calls), 8 simulations equal, 32 simulations 38.7 against 30.0; single-step calls 39.8 against 45.3 at 32 simulations.
        // 96 x 96 (generic fused kernel): 32 simulations 36.8 against 47.8, 148 simulations 77 against 63.  Below 96 x 96
        // the phase path always wins (64 x 64: 52 against 65 us per step of 148 simulations).
        // Round 2: a few full-size simulations (up to 33) run on clusters of four CTAs (k_step_cluster): 27.3 us per step at K = 40 for
        // 1 .. 32 simulations against 36.6 .. 48.4 on the phase path (tools/cluster_latency.py), so those take the fused path too.
        const bool full = fused_full_size(g);
        const bool big_enough = (long)g->h * g->w >= 96L * 96L;
        const int need = full ? (nsteps >= 2 ? 12 : 48) : 96;
        const bool clustered = full && pick_cluster(g->batch) != 0;
        if (prm->step_kernel == SMK_STEP_FUSED || clustered || (big_enough && g->batch >= need))
            *plan = clustered ? PLAN_CLUSTER : PLAN_FUSED;
        return SMK_OK;
    }
    if (prm->step_kernel == SMK_STEP_FUSED)
        return fail(SMK_EUNSUPPORTED, "smk_step: SMK_STEP_FUSED needs a non-slab grid of at most 128 x 128 cells, got %d x %d", g->h, g->w);
    return SMK_OK;
}

int smk_step_is_fused(const smk_grid_t* g, const smk_params_t* prm, int32_t nsteps, int32_t* fused_host)
{
    SMK_TRY(check_grid(g, "smk_step_is_fused"));
    if (!prm || !fused_host) return fail(SMK_EINVAL, "smk_step_is_fused: NULL");
    StepPlan plan = PLAN_PHASES;
    SMK_TRY(pick_step_kernel(g, prm, nsteps, &plan));
    *fused_host = plan != PLAN_PHASES;
    return SMK_OK;
}

int smk_fused_plan(int32_t nsims, int32_t nsteps, int32_t piece_len, int32_t* items_host, int32_t capacity, int32_t* count_host)
{
    if (!count_host || (capacity > 0 && !items_host)) return fail(SMK_EINVAL, "smk_fused_plan: NULL");
    if (nsims <= 0 || nsteps <= 0 || piece_len <= 0 || capacity < 0 || (int64_t)nsims * nsteps > 0x3fffffff)
        return fail(SMK_EINVAL, "smk_fused_plan: nsims %d, nsteps %d, piece_len %d", nsims, nsteps, piece_len);
    int n = 0;
    const int rc = fused_plan(nsims, nsteps, piece_len, items_host, capacity, &n);
    *count_host = n;
    return rc;
}

// frames of SMK_FRAME_F32 / _F16 / _BF16: bytes per element; the kernels store 4 elements at a time (16 or 8 bytes)
static int frame_elem_size(int32_t fmt) { return fmt == SMK_FRAME_F32 ? 4 : 2; }
static int check_frames(const char* who, const void* frames, int64_t stride0, int64_t stride1, int32_t fmt)
{
    if (fmt != SMK_FRAME_F32 && fmt != SMK_FRAME_F16 && fmt != SMK_FRAME_BF16)
        return fail(SMK_EINVAL, "%s: frame_format %d is not SMK_FRAME_F32/_F16/_BF16", who, fmt);
    if (!frames) return SMK_OK;
    if (reinterpret_cast<uintptr_t>(frames) % (4u * frame_elem_size(fmt)))
        return fail(SMK_EINVAL, "%s: frame base is not aligned to 4 elements of the frame type (%d B)", who, 4 * frame_elem_size(fmt));
    if ((stride0 | stride1) & 3) return fail(SMK_EINVAL, "%s: frame strides must be multiples of 4 elements", who);
    return SMK_OK;
}

}  // extern "C"

// The one body behind every step entry point: checks the whole call before anything is enqueued, then runs it on the kernels
// pick_step_kernel chose.  A reset is consumed (*consumed = 1) only on k_step_fused; elsewhere nothing is enqueued and the
// caller resets and calls again without one.
static int run_steps(const char* who, const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, const StepCall& c,
                     int32_t* consumed, cudaStream_t s)
{
    SMK_TRY(check_frames(who, c.frames, c.frame_step_stride, c.frame_batch_stride, c.frame_format));
    if (c.nsteps < 0) return fail(SMK_EINVAL, "%s: negative nsteps", who);
    if (!g || !st || !prm) return fail(SMK_EINVAL, "%s: grid/state/params NULL", who);
    if ((c.csrc == nullptr) != (c.coff == nullptr)) return fail(SMK_EINVAL, "%s: sources and offsets go together", who);
    if (c.cstride != 0 && (!c.csrc || c.cstride != g->batch))
        return fail(SMK_EINVAL, "%s: offsets_step_stride must be 0 or the batch (%d) with sources, got %d", who, g->batch, c.cstride);
    if ((c.rsrc == nullptr) != (c.roff == nullptr)) return fail(SMK_EINVAL, "%s: reset_sources and reset_offsets go together", who);
    if (!c.reset && c.rsrc) return fail(SMK_EINVAL, "%s: reset_sources without a reset", who);
    if ((c.fu == nullptr) != (c.fv == nullptr)) return fail(SMK_EINVAL, "%s: force_u and force_v go together", who);
    if ((c.fu && !aligned16(c.fu)) || (c.fv && !aligned16(c.fv))) return fail(SMK_EINVAL, "%s: force_u / force_v not 16-byte aligned", who);
    if (c.fstep != 0 && c.fstep != 1) return fail(SMK_EINVAL, "%s: force_per_step must be 0 or 1, got %d", who, c.fstep);
    if (c.fstep && !c.fu) return fail(SMK_EINVAL, "%s: force_per_step = 1 without forcing", who);
    SMK_TRY(check_grid(g, who));
    if (c.solid && reinterpret_cast<uintptr_t>(c.solid) % 4) return fail(SMK_EINVAL, "%s: solid is not 4-byte aligned", who);
    if (c.sstride != 0 && (!c.solid || c.sstride != (int64_t)g->h * g->pitch_c))
        return fail(SMK_EINVAL, "%s: solid_batch_stride must be 0 or h * pitch_c (%lld) with a mask, got %lld", who,
                    (long long)g->h * g->pitch_c, (long long)c.sstride);
    if (g->gh != 0 && (g->gh != g->h || g->row0 != 0))
        return fail(SMK_EUNSUPPORTED, "%s: slab grids are stepped phase by phase with halo exchanges in between", who);
    SMK_TRY(check_ptrs(who, {st->u[0], st->u[1], st->v[0], st->v[1], st->d[0], st->d[1], st->p[0], st->p[1], st->div}));
    if ((st->cur_u | st->cur_v | st->cur_d | st->cur_p) & ~1) return fail(SMK_EINVAL, "%s: cur_* must be 0 or 1", who);
    if (prm->jacobi_iters < 0) return fail(SMK_EINVAL, "%s: negative jacobi_iters", who);
    if (!(prm->dt != 0.0f)) return fail(SMK_EINVAL, "%s: dt must be non-zero", who);
    StepPlan plan = PLAN_PHASES;
    SMK_TRY(pick_step_kernel(g, prm, c.nsteps, &plan, c.solid != nullptr));
    if (c.nsteps == 0 || (c.reset && plan != PLAN_FUSED)) return SMK_OK;
    if (plan != PLAN_PHASES) {
        SMK_TRY(launch_steps_fused(g, st, prm, c, s));
        if (c.reset) *consumed = 1;
        return SMK_OK;
    }
    const int64_t step_bytes = c.frame_step_stride * frame_elem_size(c.frame_format);
    const int64_t fu_step = c.fstep ? (int64_t)g->batch * g->stride_u : 0, fv_step = c.fstep ? (int64_t)g->batch * g->stride_v : 0;
    for (int t = 0; t < c.nsteps; ++t)
        SMK_TRY(phase_step(g, st, prm, c.csrc, c.coff ? c.coff + (int64_t)t * c.cstride : nullptr,
                           c.fu ? c.fu + t * fu_step : nullptr, c.fv ? c.fv + t * fv_step : nullptr, c.solid, c.sstride,
                           c.frames ? static_cast<char*>(c.frames) + (int64_t)t * step_bytes : nullptr,
                           c.frame_batch_stride, c.fmul, c.frame_format, nullptr, nullptr, nullptr, nullptr, s));
    return SMK_OK;
}

extern "C" {

int smk_step(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, float* frame, int64_t frame_stride,
             const float* fmul, void* stream)
{
    return smk_step_ex(g, st, prm, frame, frame_stride, fmul, SMK_FRAME_F32, stream);
}

int smk_step_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, void* frame, int64_t frame_stride,
                const float* fmul, int32_t frame_format, void* stream)
{
    StepCall c;
    c.frames = frame; c.frame_batch_stride = frame_stride; c.fmul = fmul; c.frame_format = frame_format;
    return run_steps("smk_step", g, st, prm, c, nullptr, (cudaStream_t)stream);
}

int smk_run_steps(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps,
                  float* frames, int64_t frame_step_stride, int64_t frame_batch_stride, const float* fmul, void* stream)
{
    return smk_run_steps_ex(g, st, prm, nsteps, frames, frame_step_stride, frame_batch_stride, fmul, SMK_FRAME_F32, stream);
}

int smk_run_steps_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps, void* frames,
                     int64_t frame_step_stride, int64_t frame_batch_stride, const float* fmul, int32_t frame_format, void* stream)
{
    StepCall c;
    c.nsteps = nsteps; c.frames = frames; c.frame_step_stride = frame_step_stride; c.frame_batch_stride = frame_batch_stride;
    c.fmul = fmul; c.frame_format = frame_format;
    return run_steps("smk_run_steps", g, st, prm, c, nullptr, (cudaStream_t)stream);
}

int smk_run_steps_reset_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps, void* frames,
                           int64_t frame_step_stride, int64_t frame_batch_stride, const float* fmul, int32_t frame_format,
                           const smk_source_t* sources, const int32_t* offsets, int32_t* consumed_host, void* stream)
{
    if (!consumed_host) return fail(SMK_EINVAL, "smk_run_steps_reset_ex: consumed_host is NULL");
    *consumed_host = 0;
    StepCall c;
    c.nsteps = nsteps; c.frames = frames; c.frame_step_stride = frame_step_stride; c.frame_batch_stride = frame_batch_stride;
    c.fmul = fmul; c.frame_format = frame_format; c.reset = true; c.rsrc = sources; c.roff = offsets;
    return run_steps("smk_run_steps_reset_ex", g, st, prm, c, consumed_host, (cudaStream_t)stream);
}

int smk_run_steps_src_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps, void* frames,
                         int64_t frame_step_stride, int64_t frame_batch_stride, const float* fmul, int32_t frame_format,
                         const smk_source_t* sources, const int32_t* offsets, int32_t reset, const smk_source_t* reset_sources,
                         const int32_t* reset_offsets, int32_t* consumed_host, void* stream)
{
    return smk_run_steps_sched_ex(g, st, prm, nsteps, frames, frame_step_stride, frame_batch_stride, fmul, frame_format, sources,
                                  offsets, 0, reset, reset_sources, reset_offsets, consumed_host, stream);
}

int smk_run_steps_sched_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps, void* frames,
                           int64_t frame_step_stride, int64_t frame_batch_stride, const float* fmul, int32_t frame_format,
                           const smk_source_t* sources, const int32_t* offsets, int32_t offsets_step_stride, int32_t reset,
                           const smk_source_t* reset_sources, const int32_t* reset_offsets, int32_t* consumed_host, void* stream)
{
    return smk_run_steps_force_ex(g, st, prm, nsteps, frames, frame_step_stride, frame_batch_stride, fmul, frame_format, sources,
                                  offsets, offsets_step_stride, nullptr, nullptr, 0, reset, reset_sources, reset_offsets,
                                  consumed_host, stream);
}

int smk_run_steps_force_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps, void* frames,
                           int64_t frame_step_stride, int64_t frame_batch_stride, const float* fmul, int32_t frame_format,
                           const smk_source_t* sources, const int32_t* offsets, int32_t offsets_step_stride,
                           const float* force_u, const float* force_v, int32_t force_per_step, int32_t reset,
                           const smk_source_t* reset_sources, const int32_t* reset_offsets, int32_t* consumed_host, void* stream)
{
    return smk_run_steps_obst_ex(g, st, prm, nsteps, frames, frame_step_stride, frame_batch_stride, fmul, frame_format, sources,
                                 offsets, offsets_step_stride, force_u, force_v, force_per_step, nullptr, 0, reset, reset_sources,
                                 reset_offsets, consumed_host, stream);
}

int smk_run_steps_obst_ex(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, int32_t nsteps, void* frames,
                          int64_t frame_step_stride, int64_t frame_batch_stride, const float* fmul, int32_t frame_format,
                          const smk_source_t* sources, const int32_t* offsets, int32_t offsets_step_stride,
                          const float* force_u, const float* force_v, int32_t force_per_step, const uint8_t* solid,
                          int64_t solid_batch_stride, int32_t reset, const smk_source_t* reset_sources, const int32_t* reset_offsets,
                          int32_t* consumed_host, void* stream)
{
    const char* who = solid ? "smk_run_steps_obst_ex" : "smk_run_steps_force_ex";
    if (!consumed_host) return fail(SMK_EINVAL, "%s: consumed_host is NULL", who);
    *consumed_host = 0;
    if (reset != 0 && reset != 1) return fail(SMK_EINVAL, "%s: reset must be 0 or 1, got %d", who, reset);
    if (nsteps < 1) return fail(SMK_EINVAL, "%s: nsteps must be >= 1, got %d", who, nsteps);
    StepCall c;
    c.nsteps = nsteps; c.frames = frames; c.frame_step_stride = frame_step_stride; c.frame_batch_stride = frame_batch_stride;
    c.fmul = fmul; c.frame_format = frame_format; c.csrc = sources; c.coff = offsets; c.cstride = offsets_step_stride;
    c.fu = force_u; c.fv = force_v; c.fstep = force_per_step;
    c.solid = solid; c.sstride = solid_batch_stride;
    c.reset = reset == 1; c.rsrc = reset_sources; c.roff = reset_offsets;
    return run_steps(who, g, st, prm, c, consumed_host, (cudaStream_t)stream);
}

int smk_add_forcing(const smk_grid_t* g, float* u, float* v, const float* du, const float* dv, void* stream)
{
    SMK_TRY(check_grid(g, "smk_add_forcing"));
    SMK_TRY(check_ptrs("smk_add_forcing", {u, v, du, dv}));
    return launch_add_forcing(g, u, v, du, dv, (cudaStream_t)stream);
}

int smk_div_norms(const smk_grid_t* g, const float* u, const float* v, float* out, void* stream)
{
    SMK_TRY(check_grid(g, "smk_div_norms"));
    SMK_TRY(check_ptrs("smk_div_norms", {u, v}));
    if (!out) return fail(SMK_EINVAL, "smk_div_norms: out NULL");
    return launch_div_norms(g, u, v, out, (cudaStream_t)stream);
}

int smk_jacobi_residual(const smk_grid_t* g, const float* div, const float* p, float* out, void* stream)
{
    SMK_TRY(check_grid(g, "smk_jacobi_residual"));
    SMK_TRY(check_ptrs("smk_jacobi_residual", {div, p}));
    if (!out) return fail(SMK_EINVAL, "smk_jacobi_residual: out NULL");
    return launch_jacobi_residual(g, div, p, out, (cudaStream_t)stream);
}

int smk_jacobi_residual_ex(const smk_grid_t* g, const float* div, const float* p, const uint8_t* solid, int64_t solid_batch_stride,
                           float* out, void* stream)
{
    SMK_TRY(check_grid(g, "smk_jacobi_residual_ex"));
    SMK_TRY(check_ptrs("smk_jacobi_residual_ex", {div, p}));
    if (!out) return fail(SMK_EINVAL, "smk_jacobi_residual_ex: out NULL");
    if (solid_batch_stride != 0 && (!solid || solid_batch_stride != (int64_t)g->h * g->pitch_c))
        return fail(SMK_EINVAL, "smk_jacobi_residual_ex: solid_batch_stride must be 0 or h * pitch_c with a mask, got %lld",
                    (long long)solid_batch_stride);
    if (!solid) return launch_jacobi_residual(g, div, p, out, (cudaStream_t)stream);
    return launch_jacobi_residual_obst(g, div, p, solid, solid_batch_stride, out, (cudaStream_t)stream);
}

int smk_fractal_fields(float* perlin, float* mandel, float* mul, int32_t na, int32_t nb, int32_t pitch, float intensity,
                       int32_t iterations, const float* px, const float* py, const float* mx, const float* my, void* stream)
{
    if (!perlin && !mandel && !mul) return fail(SMK_EINVAL, "smk_fractal_fields: no output requested");
    if (((perlin || mul) && (!px || !py)) || ((mandel || mul) && (!mx || !my))) return fail(SMK_EINVAL, "smk_fractal_fields: NULL grid");
    if (na < 1 || nb < 1 || pitch < nb || iterations < 1) return fail(SMK_EINVAL, "smk_fractal_fields: bad shape %d x %d pitch %d", na, nb, pitch);
    return launch_fractal_fields(perlin, mandel, mul, na, nb, pitch, intensity, iterations, px, py, mx, my, (cudaStream_t)stream);
}

int smk_apply_mul(const float* field, const float* mul, float* out, int32_t rows, int32_t cols, int32_t pitch,
                  int32_t batch, int64_t stride, void* stream)
{
    if (!field || !mul || !out) return fail(SMK_EINVAL, "smk_apply_mul: NULL pointer");
    if (rows < 1 || cols < 1 || pitch < cols || batch < 1 || batch > 65535) return fail(SMK_EINVAL, "smk_apply_mul: bad shape");
    return launch_apply_mul(field, mul, out, rows, cols, pitch, batch, stride, (cudaStream_t)stream);
}

int smk_frame_features(const float* frames, int64_t frame_stride, int32_t nframes, int32_t h, int32_t w, int32_t pitch,
                       const float* edges, int32_t nbins, float lo, float hi, int32_t* box_counts, int32_t* hist,
                       float* mean_out, void* stream)
{
    if (!frames || !edges || !box_counts || !hist) return fail(SMK_EINVAL, "smk_frame_features: NULL pointer");
    if (nframes < 0 || h < 1 || w < 1 || pitch < w || nbins < 1 || nbins > 8192 || !(hi > lo))
        return fail(SMK_EINVAL, "smk_frame_features: bad arguments (%d frames of %d x %d pitch %d, %d bins)", nframes, h, w, pitch, nbins);
    if (nframes > 1 && frame_stride < (int64_t)h * pitch) return fail(SMK_EINVAL, "smk_frame_features: frame_stride smaller than a frame");
    return launch_frame_features(frames, frame_stride, nframes, h, w, pitch, edges, nbins, lo, hi, box_counts, hist, mean_out,
                                 (cudaStream_t)stream);
}

int smk_frame_distances(const float* frames, int64_t frame_stride, int32_t nframes, int32_t h, int32_t w, int32_t pitch,
                        double* sumsq, void* stream)
{
    if (!frames || !sumsq) return fail(SMK_EINVAL, "smk_frame_distances: NULL pointer");
    if (nframes < 0 || h < 1 || w < 1 || pitch < w) return fail(SMK_EINVAL, "smk_frame_distances: bad arguments");
    if (nframes > 1 && frame_stride < (int64_t)h * pitch) return fail(SMK_EINVAL, "smk_frame_distances: frame_stride smaller than a frame");
    return launch_frame_distances(frames, frame_stride, nframes, h, w, pitch, sumsq, (cudaStream_t)stream);
}

}  // extern "C"
