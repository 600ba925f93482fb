// stencil.cu -- every phase of step() except the Jacobi sweeps (navier_stokes.py:151-173), plus the
// emitter splat, the divergence norms and the fractal multiplier field.  All kernels are HBM/L2-bound
// stencils or gathers: coalesced row-major access, shared-memory staging with halos where a phase reuses
// neighbours, no tensor cores (nothing here is a contraction).
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include "common.cuh"

namespace smk {

// =====================================================================================================
// a3 + a4 + a5 fused: buoyancy, three diffusions, divergence -- one read of (u, v, d), one write of
// (u', v', d', div).  A CTA owns FTH x 128 cells.  The tile (+1 halo, replicate-clamped at the domain
// edge, buoyancy already added to v) is staged in shared memory with one LDG.128 + STS.128 per four cells;
// every thread then produces four consecutive cells from LDS.128 rows and stores them with STG.128.  The
// diffused u / v go to a second pair of tiles from which the divergence is formed.
// Shared column c of a staged row holds global column j0 - 4 + c (the body starts 16-byte aligned at c = 4,
// the halo columns j0-1, j0+128, j0+129 sit at c = 3, 132, 133).
// =====================================================================================================
constexpr int FTH = 16, FTW = 128, FSP = 136, FTHREADS = 256;

__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, const float4 v) { *reinterpret_cast<float4*>(p) = v; }

// diffusion_step: f + c*((((up+down)+left)+right) - 4f)                             navier_stokes.py:69-72
__device__ __forceinline__ float diff1(float f, float up, float dn, float l, float r, float c)
{
    float s = up + dn;
    s = s + l;
    s = s + r;
    return f + c * (s - 4.0f * f);
}
// The strip's left / right neighbours come from the adjacent lanes (a scalar LDS at a 4-word lane stride is a 4-way
// bank conflict); lanes 0 and 31 read the staged halo columns.  Must be called by all 32 lanes of the warp.
__device__ __forceinline__ float4 diff4(const float* up_row, const float* cur_row, const float* dn_row, int c4, float c)
{
    const float4 up = lds4(up_row + c4), cur = lds4(cur_row + c4), dn = lds4(dn_row + c4);
    float l = __shfl_up_sync(0xffffffffu, cur.w, 1), r = __shfl_down_sync(0xffffffffu, cur.x, 1);
    if (c4 == 4) l = cur_row[3];
    if (c4 == 4 + 4 * 31) r = cur_row[132];
    float4 o;
    o.x = diff1(cur.x, up.x, dn.x, l, cur.y, c);
    o.y = diff1(cur.y, up.y, dn.y, cur.x, cur.z, c);
    o.z = diff1(cur.z, up.z, dn.z, cur.y, cur.w, c);
    o.w = diff1(cur.w, up.w, dn.w, cur.z, r, c);
    return o;
}
// store the first `n` (1..4) lanes of v at p (p is 16-byte aligned)
__device__ __forceinline__ void st4_partial(float* p, const float4 v, int n)
{
    if (n >= 4) { st4(p, v); return; }
    if (n > 0) p[0] = v.x;
    if (n > 1) p[1] = v.y;
    if (n > 2) p[2] = v.z;
}

// Interior tiles (the staged window lies strictly inside the fields, every cell gets buoyancy, nothing is clamped or
// partially stored) take a different staging path: all 1870 16-byte chunks of the three windows are put in flight at
// once with cp.async and awaited once -- the generic path's LDG -> STS loop serialises six DRAM round trips per warp,
// which is what bound the kernel (long-scoreboard stalls, 44 % of DRAM peak) -- and the buoyancy is then added in
// shared memory by the thread that copied the chunk.
// one box of a (pitch, rows, batch) tensor map -> shared memory, completion counted in bytes on an mbarrier
__device__ __forceinline__ void at_tma_box(void* smem_dst, const TmaMap* map, const int x, const int y, const int z, unsigned long long* bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 :: "r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(map), "r"(x), "r"(y), "r"(z),
                    "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
// thread 0 of a CTA: initialise the mbarrier and arm it for `bytes` of TMA traffic
__device__ __forceinline__ void tma_bar_arm(unsigned long long* bar, const unsigned bytes)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bar_wait(unsigned long long* bar, const unsigned parity)
{
    unsigned done = 0;
    while (!done)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}

__device__ __forceinline__ void fdd_cp_async16(float* smem_dst, const float* gmem_src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}

struct FddTile {                // su, sv, sd start on 128-byte boundaries (TMA destinations of the interior tiles)
    float su[FTH + 3][FSP];     // u rows i0-1 .. i0+FTH+1
    float pad0[(128 - sizeof(float) * (FTH + 3) * FSP % 128) % 128 / sizeof(float)];
    float sv[FTH + 2][FSP];     // v + buoyancy, rows i0-1 .. i0+FTH
    float pad1[(128 - sizeof(float) * (FTH + 2) * FSP % 128) % 128 / sizeof(float)];
    float sd[FTH + 2][FSP];     // density, same rows
    float pad2[(128 - sizeof(float) * (FTH + 2) * FSP % 128) % 128 / sizeof(float)];
    float su1[FTH + 1][FTW];    // diffused u, rows i0 .. i0+FTH
    float sv1[FTH][FTW + 4];    // diffused v, cols j0 .. j0+128
};

template <bool INTERIOR>
__device__ __forceinline__ void fdd_tile(FddTile& T, const float* __restrict__ U, const float* __restrict__ V, const float* __restrict__ D,
                                         float* __restrict__ Uo, float* __restrict__ Vo, float* __restrict__ Do, float* __restrict__ DIV,
                                         const int h, const int w, const int pu, const int pv, const int pc,
                                         const float dt, const float c_uv, const float c_d, const int i0, const int j0,
                                         const int b, const TmaMap* mU, const TmaMap* mV, const TmaMap* mD, unsigned long long* bar)
{
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const int c0 = j0 + 4 * lane;                  // first global column of this lane's float4
    const int c4 = 4 + 4 * lane;                   // its shared-memory column

    if (INTERIOR) {
        // shared column c holds global column j0 - 4 + c: whole 16-byte chunks [j0-4, j0+132) of every staged row
        constexpr int NCH = FSP / 4;               // 34 chunks per row
        if (bar) {
            // TMA: the three windows as three box loads issued by one thread (round 2; the 1870 LDGSTS of the path below and their
            // address arithmetic were ~13 % of the kernel's instructions)
            if (threadIdx.x == 0) {
                tma_bar_arm(bar, sizeof(float) * ((FTH + 3) + 2 * (FTH + 2)) * FSP);
                at_tma_box(&T.su[0][0], mU, j0 - 4, i0 - 1, b, bar);
                at_tma_box(&T.sv[0][0], mV, j0 - 4, i0 - 1, b, bar);
                at_tma_box(&T.sd[0][0], mD, j0 - 4, i0 - 1, b, bar);
            }
            __syncthreads();
            tma_bar_wait(bar, 0u);
        } else {
        for (int k = threadIdx.x; k < (FTH + 3) * NCH; k += FTHREADS) {
            const int r = k / NCH, c = (k - r * NCH) * 4;
            fdd_cp_async16(&T.su[r][c], U + ((size_t)(i0 - 1 + r) * pu + (j0 - 4 + c)));
        }
        for (int k = threadIdx.x; k < (FTH + 2) * NCH; k += FTHREADS) {
            const int r = k / NCH, c = (k - r * NCH) * 4;
            fdd_cp_async16(&T.sv[r][c], V + ((size_t)(i0 - 1 + r) * pv + (j0 - 4 + c)));
            fdd_cp_async16(&T.sd[r][c], D + ((size_t)(i0 - 1 + r) * pc + (j0 - 4 + c)));
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        // buoyancy: v[:, :-1] += dt * (density * 0.1) (navier_stokes.py:154-155) on the chunks this thread copied (cp.async: a thread
        // sees its own copies after wait_group; TMA: every thread sees everything after the mbarrier)
        for (int k = threadIdx.x; k < (FTH + 2) * NCH; k += FTHREADS) {
            const int r = k / NCH, c = (k - r * NCH) * 4;
            float4 x = lds4(&T.sv[r][c]);
            const float4 y = lds4(&T.sd[r][c]);
            x.x = x.x + dt * (y.x * 0.1f); x.y = x.y + dt * (y.y * 0.1f);
            x.z = x.z + dt * (y.z * 0.1f); x.w = x.w + dt * (y.w * 0.1f);
            st4(&T.sv[r][c], x);
        }
    } else {
        // ---- stage u ------------------------------------------------------------------------------------
        for (int r = wp; r < FTH + 3; r += FTHREADS / 32) {
            const float* row = U + (size_t)clampi(i0 - 1 + r, 0, h) * pu;
            float4 x;
            if (c0 + 3 < w) x = ld4(row + c0);
            else {
                x.x = __ldg(row + min(c0, w - 1)); x.y = __ldg(row + min(c0 + 1, w - 1));
                x.z = __ldg(row + min(c0 + 2, w - 1)); x.w = __ldg(row + min(c0 + 3, w - 1));
            }
            st4(&T.su[r][c4], x);
            if (lane < 2) T.su[r][lane == 0 ? 3 : 132] = __ldg(row + clampi(lane == 0 ? j0 - 1 : j0 + 128, 0, w - 1));
        }
        // ---- stage v (+ buoyancy: v[:, :-1] += dt * (density * 0.1), navier_stokes.py:154-155) and density ----
        for (int r = wp; r < FTH + 2; r += FTHREADS / 32) {
            const int gi = clampi(i0 - 1 + r, 0, h - 1);
            const float* vrow = V + (size_t)gi * pv;
            const float* drow = D + (size_t)gi * pc;
            float4 x, y;
            if (c0 + 3 < w) {
                x = ld4(vrow + c0); y = ld4(drow + c0);
                x.x = x.x + dt * (y.x * 0.1f); x.y = x.y + dt * (y.y * 0.1f);
                x.z = x.z + dt * (y.z * 0.1f); x.w = x.w + dt * (y.w * 0.1f);
            } else {
                float vv[4], dd[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int cjv = min(c0 + k, w), cjd = min(cjv, w - 1);
                    dd[k] = __ldg(drow + cjd);
                    vv[k] = __ldg(vrow + cjv);
                    if (cjv < w) vv[k] = vv[k] + dt * (dd[k] * 0.1f);
                }
                x = make_float4(vv[0], vv[1], vv[2], vv[3]); y = make_float4(dd[0], dd[1], dd[2], dd[3]);
            }
            st4(&T.sv[r][c4], x); st4(&T.sd[r][c4], y);
            if (lane < 3) {
                const int sc = lane == 0 ? 3 : 131 + lane;
                const int cjv = clampi(lane == 0 ? j0 - 1 : j0 + 127 + lane, 0, w), cjd = min(cjv, w - 1);
                const float dv = __ldg(drow + cjd);
                float vv = __ldg(vrow + cjv);
                if (cjv < w) vv = vv + dt * (dv * 0.1f);
                T.sv[r][sc] = vv; T.sd[r][sc] = dv;
            }
        }
    }
    __syncthreads();

    // ---- diffusion ------------------------------------------------------------------------------------
    for (int r = wp; r <= FTH; r += FTHREADS / 32) {                    // u rows i0 .. i0+FTH
        const int i = i0 + r;
        const float4 o = diff4(T.su[r], T.su[r + 1], T.su[r + 2], c4, c_uv);
        st4(&T.su1[r][4 * lane], o);
        if (INTERIOR) { if (r < FTH) st4(Uo + (size_t)i * pu + c0, o); }
        else if (i <= h && (r < FTH || i == h)) st4_partial(Uo + (size_t)i * pu + c0, o, w - c0);
    }
    for (int r = wp; r < FTH; r += FTHREADS / 32) {                     // v and density rows i0 .. i0+FTH-1
        const int i = i0 + r;
        const float4 o = diff4(T.sv[r], T.sv[r + 1], T.sv[r + 2], c4, c_uv);
        st4(&T.sv1[r][4 * lane], o);
        const float4 q = diff4(T.sd[r], T.sd[r + 1], T.sd[r + 2], c4, c_d);
        if (INTERIOR) {
            st4(Vo + (size_t)i * pv + c0, o);
            st4(Do + (size_t)i * pc + c0, q);
        } else if (i < h) {
            st4_partial(Vo + (size_t)i * pv + c0, o, w + 1 - c0);
            st4_partial(Do + (size_t)i * pc + c0, q, w - c0);
        }
    }
    if (threadIdx.x < FTH) {                                            // v column j0+128 (the staggered extra column)
        const int r = threadIdx.x, i = i0 + r;
        const float o = diff1(T.sv[r + 1][132], T.sv[r][132], T.sv[r + 2][132], T.sv[r + 1][131], T.sv[r + 1][133], c_uv);
        T.sv1[r][128] = o;
        if (!INTERIOR && i < h && j0 + 128 == w) Vo[(size_t)i * pv + w] = o;
    }
    if (DIV == nullptr) return;
    __syncthreads();
    // ---- div = (((u[i+1][j] - u[i][j]) + v[i][j+1]) - v[i][j]) / dt                    navier_stokes.py:136
    for (int r = wp; r < FTH; r += FTHREADS / 32) {
        const int i = i0 + r;
        if (!INTERIOR && i >= h) break;
        const float4 ua = lds4(&T.su1[r][4 * lane]), ub = lds4(&T.su1[r + 1][4 * lane]);
        const float4 va = lds4(&T.sv1[r][4 * lane]);
        float vr = __shfl_down_sync(0xffffffffu, va.x, 1);                 // v[i][j+1] of the strip's last cell: next lane
        if (lane == 31) vr = T.sv1[r][128];
        float4 o;
        o.x = (((ub.x - ua.x) + va.y) - va.x) / dt;
        o.y = (((ub.y - ua.y) + va.z) - va.y) / dt;
        o.z = (((ub.z - ua.z) + va.w) - va.z) / dt;
        o.w = (((ub.w - ua.w) + vr) - va.w) / dt;
        if (INTERIOR) st4(DIV + (size_t)i * pc + c0, o);
        else st4_partial(DIV + (size_t)i * pc + c0, o, w - c0);
    }
}

__global__ void __launch_bounds__(FTHREADS)
k_forces_diffuse_div(const float* __restrict__ U, const float* __restrict__ V, const float* __restrict__ D,
                     float* __restrict__ Uo, float* __restrict__ Vo, float* __restrict__ Do, float* __restrict__ DIV,
                     const int h, const int w, const int pu, const int pv, const int pc,
                     const long long su_, const long long sv_, const long long sc_,
                     const float dt, const float c_uv, const float c_d, const int bulk,
                     const __grid_constant__ TmaMap mU, const __grid_constant__ TmaMap mV, const __grid_constant__ TmaMap mD)
{
    pdl_prologue();
    __shared__ __align__(128) FddTile T;
    __shared__ __align__(8) unsigned long long tma_bar;
    const int i0 = blockIdx.y * FTH, j0 = blockIdx.x * FTW;
    const size_t b = blockIdx.z;
    U += b * su_; Uo += b * su_; V += b * sv_; Vo += b * sv_; D += b * sc_; Do += b * sc_;
    if (DIV) DIV += b * sc_;
    // interior: rows i0-1 .. i0+FTH+1 of u and i0-1 .. i0+FTH of v, density exist; columns j0-4 .. j0+131 are cells
    // that take buoyancy (< w) and lie inside every pitch; no output row or column is the last of its field
    // (bulk: only on grids of several CTA waves -- on small ones the extra shared-memory pass of the buoyancy costs more
    // latency than the serialised loads: 16.1 against 14.2 us at 1024^2, 334 against 446 us at 8192^2)
    const bool interior = bulk && i0 >= 1 && i0 + FTH + 1 <= h - 1 && j0 >= 4 && j0 + FTW + 4 <= w && j0 + FTW + 4 <= pu && j0 + FTW + 4 <= pc;
    // bulk == 2: interior tiles stage by TMA
    if (interior) fdd_tile<true>(T, U, V, D, Uo, Vo, Do, DIV, h, w, pu, pv, pc, dt, c_uv, c_d, i0, j0, (int)b, &mU, &mV, &mD, bulk == 2 ? &tma_bar : nullptr);
    else          fdd_tile<false>(T, U, V, D, Uo, Vo, Do, DIV, h, w, pu, pv, pc, dt, c_uv, c_d, i0, j0, (int)b, &mU, &mV, &mD, nullptr);
}

int launch_forces_diffuse_div(const smk_grid_t* g, const float* u, const float* v, const float* d,
                              float* uo, float* vo, float* dout, float* div, float dt, float c_uv, float c_d, cudaStream_t s)
{
    dim3 grid((g->w + FTW - 1) / FTW, (g->h + FTH - 1) / FTH, g->batch);
    ProfScope prof_(SMK_PH_FORCES_DIFFUSE_DIV, s);
    int bulk = (int64_t)g->h * g->w * g->batch >= ((int64_t)6 << 20) ? 1 : 0;
    if (env().fdd_bulk != SMK_ENV_UNSET) bulk = env().fdd_bulk;             // tests force a staging path on small grids: 0 / 1 (cp.async) / 2 (TMA)
    else if (bulk) bulk = 2;
    TmaMap mU, mV, mD;
    memset(&mU, 0, sizeof mU); memset(&mV, 0, sizeof mV); memset(&mD, 0, sizeof mD);
    if (bulk == 2 && !(tma_map_3d(&mU, u, g->pitch_u, g->h + 1, g->batch, g->stride_u, FTH + 3, FSP) &&
                       tma_map_3d(&mV, v, g->pitch_v, g->h, g->batch, g->stride_v, FTH + 2, FSP) &&
                       tma_map_3d(&mD, d, g->pitch_c, g->h, g->batch, g->stride_c, FTH + 2, FSP)))
        bulk = 1;                                                            // no tensor map: cp.async
    launch_chain(k_forces_diffuse_div, grid, dim3(FTHREADS), 0, s, u, v, d, uo, vo, dout, div, g->h, g->w, g->pitch_u, g->pitch_v, g->pitch_c,
                                                   g->stride_u, g->stride_v, g->stride_c, dt, c_uv, c_d, bulk, mU, mV, mD);
    return check_launch("k_forces_diffuse_div");
}

// ---- a4 alone: diffusion_step on one field (unit hook for NavierStokesSimulator.diffusion_step) -------
__global__ void k_diffuse(const float* __restrict__ F, float* __restrict__ O, const int rows, const int cols,
                          const int pitch, const long long stride, const float c)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= rows || j >= cols) return;
    F += (size_t)blockIdx.z * stride; O += (size_t)blockIdx.z * stride;
    const int iu = max(i - 1, 0), id = min(i + 1, rows - 1), jl = max(j - 1, 0), jr = min(j + 1, cols - 1);
    const float f = F[(size_t)i * pitch + j];
    float s = F[(size_t)iu * pitch + j] + F[(size_t)id * pitch + j];
    s = s + F[(size_t)i * pitch + jl];
    s = s + F[(size_t)i * pitch + jr];
    O[(size_t)i * pitch + j] = f + c * (s - 4.0f * f);
}

int launch_diffuse(const float* in, float* out, int rows, int cols, int pitch, int batch, int64_t stride, float c, cudaStream_t s)
{
    dim3 grid((cols + 31) / 32, (rows + 7) / 8, batch), blk(32, 8);
    ProfScope prof_(SMK_PH_OTHER, s);
    k_diffuse<<<grid, blk, 0, s>>>(in, out, rows, cols, pitch, stride, c);
    return check_launch("k_diffuse");
}

// ---- a5 alone ----------------------------------------------------------------------------------------
__global__ void k_divergence(const float* __restrict__ U, const float* __restrict__ V, float* __restrict__ DIV,
                             const int h, const int w, const int pu, const int pv, const int pc,
                             const long long su_, const long long sv_, const long long sc_, const float dt)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= h || j >= w) return;
    const size_t b = blockIdx.z;
    U += b * su_; V += b * sv_; DIV += b * sc_;
    float s = U[(size_t)(i + 1) * pu + j] - U[(size_t)i * pu + j];
    s = s + V[(size_t)i * pv + j + 1];
    s = s - V[(size_t)i * pv + j];
    DIV[(size_t)i * pc + j] = s / dt;
}

int launch_divergence(const smk_grid_t* g, const float* u, const float* v, float* div, float dt, cudaStream_t s)
{
    dim3 grid((g->w + 31) / 32, (g->h + 7) / 8, g->batch), blk(32, 8);
    ProfScope prof_(SMK_PH_OTHER, s);
    k_divergence<<<grid, blk, 0, s>>>(u, v, div, g->h, g->w, g->pitch_u, g->pitch_v, g->pitch_c,
                                      g->stride_u, g->stride_v, g->stride_c, dt);
    return check_launch("k_divergence");
}

// ---- a7: gradient subtract, in place (navier_stokes.py:148-149) -----------------------------------------
// One thread per four consecutive cells of a row: LDG.128 of p (this row and the row above), u and v,
// the pressure to the left of the group through a warp shuffle, STG.128 of u and v.
__global__ void __launch_bounds__(256)
k_project(const float* __restrict__ P, float* __restrict__ U, float* __restrict__ V,
          const int h, const int w, const int pu, const int pv, const int pc,
          const long long su_, const long long sv_, const long long sc_, const float dt)
{
    pdl_prologue();
    const int c0 = (blockIdx.x * 32 + threadIdx.x) * 4, i = blockIdx.y * 8 + threadIdx.y;
    const size_t b = blockIdx.z;
    P += b * sc_; U += b * su_; V += b * sv_;
    const bool in = i < h && c0 < w;
    float4 p4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const bool full = in && c0 + 3 < w;
    const float* prow = P + (size_t)i * pc;
    if (full) p4 = ld4(prow + c0);
    else if (in) {
        p4.x = prow[c0];
        if (c0 + 1 < w) p4.y = prow[c0 + 1];
        if (c0 + 2 < w) p4.z = prow[c0 + 2];
    }
    float pl = __shfl_up_sync(0xffffffffu, p4.w, 1);
    if (!in) return;
    if (threadIdx.x == 0 && c0 > 0) pl = prow[c0 - 1];
    const int n = w - c0;                                    // valid columns in this group (>= 1)
    if (i >= 1) {        // u[1:-1, :] -= dt * (p[1:, :] - p[:-1, :])
        const float* qrow = prow - pc;
        float* urow = U + (size_t)i * pu + c0;
        if (full) {
            const float4 q4 = ld4(qrow + c0);
            float4 u4 = *reinterpret_cast<const float4*>(urow);
            u4.x = u4.x - dt * (p4.x - q4.x); u4.y = u4.y - dt * (p4.y - q4.y);
            u4.z = u4.z - dt * (p4.z - q4.z); u4.w = u4.w - dt * (p4.w - q4.w);
            st4(urow, u4);
        } else {
            const float pp[3] = {p4.x, p4.y, p4.z};
            for (int k = 0; k < n && k < 3; ++k) urow[k] = urow[k] - dt * (pp[k] - qrow[c0 + k]);
        }
    }
    {                    // v[:, 1:-1] -= dt * (p[:, 1:] - p[:, :-1])
        float* vrow = V + (size_t)i * pv + c0;
        if (full) {
            float4 v4 = *reinterpret_cast<const float4*>(vrow);
            if (c0 > 0) v4.x = v4.x - dt * (p4.x - pl);
            v4.y = v4.y - dt * (p4.y - p4.x); v4.z = v4.z - dt * (p4.z - p4.y); v4.w = v4.w - dt * (p4.w - p4.z);
            st4(vrow, v4);
        } else {
            const float pp[4] = {pl, p4.x, p4.y, p4.z};
            for (int k = 0; k < n && k < 3; ++k)
                if (c0 + k > 0) vrow[k] = vrow[k] - dt * (pp[k + 1] - pp[k]);
        }
    }
}

int launch_project(const smk_grid_t* g, const float* p, float* u, float* v, float dt, cudaStream_t s)
{
    dim3 grid((g->w + 127) / 128, (g->h + 7) / 8, g->batch), blk(32, 8);
    ProfScope prof_(SMK_PH_PROJECT, s);
    launch_chain(k_project, grid, blk, 0, s, p, u, v, g->h, g->w, g->pitch_u, g->pitch_v, g->pitch_c,
                                   g->stride_u, g->stride_v, g->stride_c, dt);
    return check_launch("k_project");
}

// ---- a8: bilinear_interpolate at arbitrary coordinates (unit hook) ---------------------------------------
__global__ void k_bilerp(const float* __restrict__ F, const int rows, const int cols, const int pitch,
                         const float* __restrict__ Y, const float* __restrict__ X, float* __restrict__ O,
                         const long long n, const int mode)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    float y = Y[k], x = X[k];
    if (mode == 1) x = clampf(x + 0.5f, 0.0f, (float)(cols - 1));        // navier_stokes.py:100-101
    if (mode == 2) y = clampf(y + 0.5f, 0.0f, (float)(rows - 1));        // navier_stokes.py:107-108
    const GlobalField f{F, pitch};
    O[k] = bilerp(f, rows, cols, y, x);
}

int launch_bilerp(const float* f, int rows, int cols, int pitch, const float* y, const float* x, float* out, int64_t n, int mode, cudaStream_t s)
{
    if (n <= 0) return SMK_OK;
    ProfScope prof_(SMK_PH_OTHER, s);
    k_bilerp<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(f, rows, cols, pitch, y, x, out, n, mode);
    return check_launch("k_bilerp");
}

// ---- a10 (+a9, a11 epilogue): advection_step of one field by (u, v) ---------------------------------------
// One thread per four consecutive cells of a row.  The velocity samples at the cell (a9: the closed form of
// interpolate_velocity_u/v on the integer grid) come from three LDG.128; the back-traced bilinear gather (a8)
// is four scalar loads per cell through the read-only path (for dt*|velocity| of a few cells they hit L1).
// px, py are clamped to the field before the floor, so the lower corner needs no clamp and the upper corner a
// single min; the corner coordinates stay in fp32 (exact below 2^24), which removes every int->float convert.
struct AdvectArgs {
    const float* F; float* O; int rows, cols, pitch; long long stride;
    const float* U; const float* V; int h, w, pu, pv; long long su_, sv_;
    float dt; int has_scale; float scale;
    void* frame; long long frame_stride; int frame_pitch; const float* fmul;      // frame: SMK_FRAME_* elements (frame_format)
    int frame_format;
    unsigned ngroups; unsigned long long magic;          // row = (idx * magic) >> 40 == idx / ngroups (+ fix-up)
    int row0, gh;                                        // slab: global row of local row 0, global cell rows
    int need_lo, need_hi, valid_lo, valid_hi; int* overflow;
    const float* P; int pc; long long sc_;               // k_advect_tiled<.., 1>: pressure for the fused gradient subtract,
    float* Vout;                                         // and where the projected v goes (a different array than V)
    // k_advect_tiled on a part of the tile rows (smk_slab_step computes the rows it sends to its neighbours first): the launch
    // covers tile rows ty0 + blockIdx.y, stepping over the rows [skip_lo[k], skip_lo[k] + skip_n[k]) of up to two bands
    int ty0, skip_lo[2], skip_n[2];
    int use_tma;                                         // k_advect_tiled: interior tiles stage their windows with TMA box loads
};

template <bool SLAB>
__global__ void __launch_bounds__(256)
k_advect(const AdvectArgs a)
{
    pdl_prologue();
    const unsigned idx = blockIdx.x * 256u + threadIdx.x;
    unsigned row = (unsigned)(((unsigned long long)idx * a.magic) >> 40);
    if (row * a.ngroups > idx) --row;
    const int i = (int)row, c0 = (int)(idx - row * a.ngroups) * 4;
    if (i >= a.rows) return;
    const size_t b = blockIdx.y;
    const float* __restrict__ F = a.F + b * a.stride;
    const float* __restrict__ U = a.U + b * a.su_;
    const float* __restrict__ V = a.V + b * a.sv_;
    const int w = a.w, rows = a.rows, cols = a.cols, pitch = a.pitch;
    // slab: h is the GLOBAL cell-row count and gi the global row of this thread's cells; memory stays local
    const int h = SLAB ? a.gh : a.h;
    const int gi = SLAB ? i + a.row0 : i;
    const int grows = SLAB ? rows - a.h + a.gh : rows;

    // a9: u_i = 0.5*U[i][j] + 0.5*U[i][j+1] for j <= w-2 and i <= h-1, else 0      navier_stokes.py:97-102
    float ui[4] = {0.f, 0.f, 0.f, 0.f}, vi[4] = {0.f, 0.f, 0.f, 0.f};
    if (gi <= h - 1 && c0 <= w - 2) {
        const float* urow = U + (size_t)i * a.pu + c0;
        float uu[5];
        if (c0 + 4 < w) {
            const float4 t = ld4(urow);
            uu[0] = t.x; uu[1] = t.y; uu[2] = t.z; uu[3] = t.w; uu[4] = __ldg(urow + 4);
        } else {
#pragma unroll
            for (int k = 0; k < 5; ++k) uu[k] = (c0 + k < w) ? __ldg(urow + k) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (c0 + k <= w - 2) ui[k] = 0.5f * uu[k] + 0.5f * uu[k + 1];
    }
    //     v_i = 0.5*V[i][j] + 0.5*V[i+1][j] for i <= h-2 and j <= w-1, else 0      navier_stokes.py:104-109
    if (gi <= h - 2 && c0 <= w - 1 && (!SLAB || i + 1 < a.h)) {
        const float* vrow = V + (size_t)i * a.pv + c0;               // pitch_v >= w+1 rounded up to 4: in bounds
        const float4 t0 = ld4(vrow), t1 = ld4(vrow + a.pv);
        vi[0] = 0.5f * t0.x + 0.5f * t1.x;
        if (c0 + 1 <= w - 1) vi[1] = 0.5f * t0.y + 0.5f * t1.y;
        if (c0 + 2 <= w - 1) vi[2] = 0.5f * t0.z + 0.5f * t1.z;
        if (c0 + 3 <= w - 1) vi[3] = 0.5f * t0.w + 0.5f * t1.w;
    }
    const float xmax = (float)(cols - 1), ymax = (float)(grows - 1);
    const float fi = (float)gi;
    float val[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float px = (float)(c0 + k) - a.dt * ui[k];                          // :87
        float py = fi - a.dt * vi[k];                                       // :88
        px = fminf(fmaxf(px, 0.0f), xmax);                                  // :91
        py = fminf(fmaxf(py, 0.0f), ymax);                                  // :92
        // a8 (:111-131) with x0 = floor(px) already inside [0, cols-1]
        const float fx0 = floorf(px), fy0 = floorf(py);
        const float fx1 = fminf(fx0 + 1.0f, xmax), fy1 = fminf(fy0 + 1.0f, ymax);
        const int x0 = (int)fx0;
        int y0 = (int)fy0;
        const int dx = (fx1 != fx0) ? 1 : 0;
        int dy = (fy1 != fy0) ? pitch : 0;
        if (SLAB) {                                                         // global -> local row, kept inside the slab
            y0 -= a.row0;
            const int y1 = y0 + (dy ? 1 : 0);
            if (i >= a.need_lo && i < a.need_hi && (y0 < a.valid_lo || y1 >= a.valid_hi) && a.overflow) *a.overflow = 1;
            if (y1 > rows - 1) dy = 0;
            y0 = clampi(y0, 0, rows - 1);
        }
        const float ax = fx1 - px, bx = px - fx0, ay = fy1 - py, by = py - fy0;
        const float* q = F + (y0 * pitch + x0);
        const float f00 = __ldg(q), f01 = __ldg(q + dx), f10 = __ldg(q + dy), f11 = __ldg(q + dy + dx);
        float s = (ax * ay) * f00 + (bx * ay) * f01;
        s = s + (ax * by) * f10;
        s = s + (bx * by) * f11;
        if (a.has_scale) s = s * a.scale;                                   // :171
        val[k] = (c0 + k < cols) ? s : 0.0f;
    }
    // pitch is a multiple of 4, so the whole group lies inside the (padded) row: one STG.128, zeros in the padding
    st4(a.O + b * a.stride + (size_t)i * pitch + c0, make_float4(val[0], val[1], val[2], val[3]));
    if (a.frame) {                                                          // :173 (+ fractal_generator.py:62)
        float4 fr = make_float4(val[0], val[1], val[2], val[3]);
        if (a.fmul) {
            const float4 m = ld4(a.fmul + (size_t)i * a.frame_pitch + c0);
            fr.x = fr.x + m.x * fr.x; fr.y = fr.y + m.y * fr.y; fr.z = fr.z + m.z * fr.z; fr.w = fr.w + m.w * fr.w;
        }
        frame_st4(a.frame, b * a.frame_stride + (size_t)i * a.frame_pitch + c0, fr, a.frame_format);
    }
}

// ---- the same on a shared-memory tile ---------------------------------------------------------------------------
// k_advect above is bound by instruction issue and L1 wavefronts, not by DRAM (77 % issue slots, 76 % L1 data pipe,
// 41 % DRAM at 8192^2; the same rate when the fields fit in L2): ~100 instructions per cell, a third of them 64-bit
// address arithmetic and edge predicates, and a 4-cells-per-thread layout that spreads each scalar gather of a warp
// over 512 B.  Here a CTA stages, with 16-byte cp.async copies, the 16 x 128 cell tile it produces -- the velocity
// rows it samples and the advected field with a 4-cell halo -- and then works like the fused kernel's advection:
// cyclic cell mapping (lane l owns cells l, l+32, l+64, l+96 of a row: every shared-memory gather of a warp hits 32
// consecutive banks for sub-cell displacements), 32-bit shared-memory offsets, two cells at a time as f32x2 pairs
// (every add that consumes a product stays scalar: ptxas contracts packed mul + add even under --fmad=false).
// The code is instantiated twice: INTERIOR tiles (every cell, its velocity samples and the whole staged window lie
// strictly inside the field: no edge predicate anywhere) and the general case.  A back-trace that leaves the staged
// window (more than about three cells) falls back to global loads for that cell pair; results are identical.
constexpr int AT_R = 16, AT_C = 128, AT_HB = 4;
constexpr int AT_FP = AT_C + 2 * AT_HB, AT_FR = AT_R + 2 * AT_HB;      // staged field window: 24 rows x 136 columns
constexpr int AT_UP = AT_C + 4, AT_VP = AT_C;                          // u tile 16 x 129 (pitch 132), v tile 17 x 128

struct AdvectTile {                                                    // every array starts on a 128-byte boundary (TMA destinations)
    float sF[AT_FR][AT_FP];
    float sU[AT_R][AT_UP];
    float sV[AT_R + 1][AT_VP];
};
static_assert(sizeof(float) * AT_FR * AT_FP % 128 == 0 && sizeof(float) * AT_R * AT_UP % 128 == 0 && sizeof(float) * (AT_R + 1) * AT_VP % 128 == 0,
              "the staged arrays of k_advect_tiled must keep 128-byte offsets");

// ... with the gradient subtract (a7, navier_stokes.py:148-149) fused in: the pressure window behind the staged field window
// (one more row above for u's p[i-1][j], one more column to the left for v's p[i][j-1]; 16-byte aligned columns)
constexpr int AT_PR = AT_FR + 1, AT_PP = AT_FP + 8;                    // 25 rows x 144 columns: rows [i0-5, i0+20), columns [j0-8, j0+136)
struct AdvectTileP {
    AdvectTile t;
    float sP[AT_PR][AT_PP];
};

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gmem_src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ float2 neg2(const float2 a) { return make_float2(-a.x, -a.y); }


// One value of the advected field straight from global memory (the rare back-trace that leaves the staged window), with the
// gradient subtract applied on the fly when the kernel fuses it (PROJ 1: the field is u).
template <int PROJ>
__device__ __forceinline__ float advect_global(const AdvectArgs& a, const float* F, const float* P, const int y, const int x)
{
    float f = __ldg(F + ((unsigned)y * a.pitch + x));
    if (PROJ == 1 && y >= 1 && y <= a.h - 1 && x < a.w) f = f - a.dt * (__ldg(P + ((unsigned)y * a.pc + x)) - __ldg(P + ((unsigned)(y - 1) * a.pc + x)));
    return f;
}

// PROJ: 0 plain advection; 1: k_project fused into the u advection -- the staged u (the field window, which is also where an
// interior tile takes its u samples from) and the v tile are the UNPROJECTED arrays and get u -= dt (p[i][j] - p[i-1][j]),
// v -= dt (p[i][j] - p[i][j-1]) in shared memory, from a pressure window staged next to them, before the advection reads them.
// Same two rounded operations per cell as k_project, so the result is bit-identical to project-then-advect.  The projected u is
// never written to memory (only this kernel reads it); the projected v tile is written to a.Vout, a DIFFERENT array than the
// one being read (other CTAs still stage unprojected rows of V), which the v and density advections then use.  A first version
// that let the v advection re-project v from p instead (no Vout) was slower: 274 against 177 us per launch at 8192^2.
template <bool SLAB, bool INTERIOR, int PROJ>
__device__ __forceinline__ void advect_tile(const AdvectArgs& a, AdvectTile& T, float (*sP)[AT_PP], const float* F, const float* U, const float* V,
                                            const float* P, float* O, const size_t b, const int i0, const int j0,
                                            const TmaMap* mF, const TmaMap* mU, const TmaMap* mV, const TmaMap* mP, unsigned long long* bar)
{
    const int tid = threadIdx.x, lane = tid & 31, wp = tid >> 5;
    const int w = a.w, rows = a.rows, cols = a.cols, pitch = a.pitch;
    const int ffmt = PROJ ? SMK_FRAME_F32 : a.frame_format;          // the fused u advection writes no frame (a.frame is NULL)

    // ---- stage: field window rows [i0-4, i0+20) x columns [j0-4, j0+132), u rows [i0, i0+16), v rows [i0, i0+17) ----
    const int wy0 = INTERIOR ? i0 - AT_HB : max(i0 - AT_HB, 0), wy1 = INTERIOR ? i0 + AT_R + AT_HB : min(i0 + AT_R + AT_HB, rows);
    const int wx0 = INTERIOR ? j0 - AT_HB : max(j0 - AT_HB, 0), wx1 = INTERIOR ? j0 + AT_C + AT_HB : min(j0 + AT_C + AT_HB, pitch);
    if (INTERIOR && a.use_tma) {
        // interior tile, TMA staging: the same windows as three box loads (four with the pressure window) issued by ONE thread --
        // no per-thread address arithmetic, no LDGSTS through the LSU pipe; every thread then waits on the mbarrier they complete on
        if (tid == 0) {
            tma_bar_arm(bar, sizeof(float) * (AT_FR * AT_FP + (AT_R + 1) * AT_VP + (PROJ ? AT_PR * AT_PP : AT_R * AT_UP)));
            at_tma_box(&T.sF[0][0], mF, j0 - AT_HB, i0 - AT_HB, (int)b, bar);
            at_tma_box(&T.sV[0][0], mV, j0, i0, (int)b, bar);
            if (PROJ) at_tma_box(&sP[0][0], mP, j0 - 8, i0 - AT_HB - 1, (int)b, bar);
            else      at_tma_box(&T.sU[0][0], mU, j0, i0, (int)b, bar);
        }
        __syncthreads();                                                   // the barrier is initialised and armed
        tma_bar_wait(bar, 0u);
    } else {
#pragma unroll
    for (int rr = 0; rr < AT_FR / 8; ++rr) {                         // warp wp copies window rows wp, wp+8, wp+16
        const int r = wp + 8 * rr, y = i0 - AT_HB + r;
        if (INTERIOR || (y >= wy0 && y < wy1)) {
            const int x = j0 - AT_HB + 4 * lane;
            const int off = y * pitch + x;                             // signed: only dereferenced where it is in range
            if (INTERIOR || (x >= wx0 && x < wx1)) cp_async16(&T.sF[r][4 * lane], F + off);
            if (lane < 2 && (INTERIOR || (x + 128 >= wx0 && x + 128 < wx1))) cp_async16(&T.sF[r][128 + 4 * lane], F + (off + 128));
        }
    }
    const int urows = a.h + 1;
    // (an interior tile of the fused u advection reads its u samples from the projected field window instead: same array)
#pragma unroll
    for (int rr = 0; rr < ((PROJ == 1 && INTERIOR) ? 0 : 2); ++rr) {
        const int r = wp + 8 * rr, y = i0 + r;
        if (INTERIOR || y < urows) {
            const float* src = U + ((unsigned)y * a.pu + j0);
            if (INTERIOR || j0 + 4 * lane < a.pu) cp_async16(&T.sU[r][4 * lane], src + 4 * lane);
            if (lane == 0 && (INTERIOR || j0 + 128 < a.pu)) cp_async16(&T.sU[r][128], src + 128);
        }
    }
#pragma unroll
    for (int rr = 0; rr < 3; ++rr) {
        const int r = wp + 8 * rr, y = i0 + r;
        if (r <= AT_R && (INTERIOR || y < a.h)) {
            if (INTERIOR || j0 + 4 * lane < a.pv) cp_async16(&T.sV[r][4 * lane], V + ((unsigned)y * a.pv + j0 + 4 * lane));
        }
    }
    if (PROJ) {
        // pressure window rows [i0-5, i0+20) x columns [j0-8, j0+136): 25 rows of 36 16-byte chunks
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
            const int r = wp + 8 * rr, y = i0 - AT_HB - 1 + r;
            if (r < AT_PR && (INTERIOR || (y >= 0 && y < a.h))) {
                const int x = j0 - 8 + 4 * lane;
                const int off = y * a.pc + x;
                if (INTERIOR || (x >= 0 && x < a.pc)) cp_async16(&sP[r][4 * lane], P + off);
                if (lane < 4 && (INTERIOR || (x + 128 >= 0 && x + 128 < a.pc))) cp_async16(&sP[r][128 + 4 * lane], P + (off + 128));
            }
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    }
    if (PROJ && INTERIOR) {
        // every staged cell is one k_project updates: four cells per LDS.128 / STS.128, no predicate
        const float dt = a.dt;
        for (int k = tid; k < AT_FR * (AT_FP / 4); k += 256) {                       // field window, 24 rows x 34 groups
            const int r = k / (AT_FP / 4), c = (k - r * (AT_FP / 4)) * 4;
            float4 f = *reinterpret_cast<const float4*>(&T.sF[r][c]);
            const float4 pc = *reinterpret_cast<const float4*>(&sP[r + 1][c + 4]);
            const float4 pa = *reinterpret_cast<const float4*>(&sP[r][c + 4]);
            f.x = f.x - dt * (pc.x - pa.x); f.y = f.y - dt * (pc.y - pa.y);
            f.z = f.z - dt * (pc.z - pa.z); f.w = f.w - dt * (pc.w - pa.w);
            *reinterpret_cast<float4*>(&T.sF[r][c]) = f;
        }
        for (int k = tid; k < (AT_R + 1) * (AT_C / 4); k += 256) {                   // v tile, 17 rows x 32 groups
            const int r = k / (AT_C / 4), c = (k - r * (AT_C / 4)) * 4;
            float4 f = *reinterpret_cast<const float4*>(&T.sV[r][c]);
            const float4 pc = *reinterpret_cast<const float4*>(&sP[r + 5][c + 8]);
            const float pl = sP[r + 5][c + 7];
            f.x = f.x - dt * (pc.x - pl); f.y = f.y - dt * (pc.y - pc.x);
            f.z = f.z - dt * (pc.z - pc.y); f.w = f.w - dt * (pc.w - pc.z);
            *reinterpret_cast<float4*>(&T.sV[r][c]) = f;
            if (r < AT_R) *reinterpret_cast<float4*>(a.Vout + b * a.sv_ + ((unsigned)(i0 + r) * a.pv + j0 + c)) = f;      // the tile's own 16 rows
        }
        __syncthreads();
    } else if (PROJ) {
        const float dt = a.dt;
        // field window: row r <-> y = i0 - 4 + r <-> sP row r + 1; column c <-> x = j0 - 4 + c <-> sP column c + 4
        for (int k = tid; k < AT_FR * AT_FP; k += 256) {
            const int r = k / AT_FP, c = k - r * AT_FP, y = i0 - AT_HB + r, x = j0 - AT_HB + c;
            if (y >= 1 && y <= a.h - 1 && x >= 0 && x < w)
                T.sF[r][c] = T.sF[r][c] - dt * (sP[r + 1][c + 4] - sP[r][c + 4]);
        }
        // u tile: row r <-> y = i0 + r <-> sP row r + 5; column c <-> x = j0 + c <-> sP column c + 8
        for (int k = tid; k < AT_R * (AT_C + 1); k += 256) {
            const int r = k / (AT_C + 1), c = k - r * (AT_C + 1), y = i0 + r, x = j0 + c;
            if (y >= 1 && y <= a.h - 1 && x < w)
                T.sU[r][c] = T.sU[r][c] - dt * (sP[r + 5][c + 8] - sP[r + 4][c + 8]);
        }
        for (int k = tid; k < (AT_R + 1) * AT_C; k += 256) {     // v tile
            const int r = k / AT_C, c = k - r * AT_C, y = i0 + r, x = j0 + c;
            if (y < a.h && x >= 1 && x <= w - 1)
                T.sV[r][c] = T.sV[r][c] - dt * (sP[r + 5][c + 8] - sP[r + 5][c + 7]);
        }
        __syncthreads();
        // the projected v of the tile's own rows (every staged 16-byte chunk: cells, column w, padding) goes to Vout ...
        float* vout = a.Vout + b * a.sv_;
        for (int k = tid; k < AT_R * (AT_C / 4); k += 256) {
            const int r = k / (AT_C / 4), c = (k - r * (AT_C / 4)) * 4, y = i0 + r, x = j0 + c;
            if (y < a.h && x < a.pv) *reinterpret_cast<float4*>(vout + ((unsigned)y * a.pv + x)) = *reinterpret_cast<const float4*>(&T.sV[r][c]);
        }
        // ... and where w is a multiple of the tile width, column w of v (which k_project leaves alone) and its padding lie
        // beyond the last tile column of u: the tiles of that column copy them
        if (j0 + AT_C == w && tid < AT_R && i0 + tid < a.h)
            *reinterpret_cast<float4*>(vout + ((unsigned)(i0 + tid) * a.pv + w)) = __ldg(reinterpret_cast<const float4*>(V + ((unsigned)(i0 + tid) * a.pv + w)));
    }

    // slab: h is the GLOBAL cell-row count and gi the global row of this thread's cells; memory stays local
    const int h = SLAB ? a.gh : a.h;
    const int grows = SLAB ? rows - a.h + a.gh : rows;
    const float2 half2 = make_float2(0.5f, 0.5f), dt2 = make_float2(a.dt, a.dt), one2 = make_float2(1.0f, 1.0f);
    const float xmax = (float)(cols - 1), ymax = (float)(grows - 1);
    const int jb = j0 + lane;
    const float* sF0 = &T.sF[0][0];
    const int wy_org = i0 - AT_HB, wx_org = j0 - AT_HB;
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
        const int ri = 2 * wp + rr, i = i0 + ri;                     // tile row, local field row (warp-uniform)
        if (!INTERIOR && i >= rows) break;
        const int gi = SLAB ? i + a.row0 : i;
        const float fi = (float)gi;
        const bool urow_ok = INTERIOR || gi <= h - 1;                              // u_i is 0 on u's last row     :97-102
        const bool vrow_ok = INTERIOR || (gi <= h - 2 && (!SLAB || i + 1 < a.h));  // v_i is 0 on the last cell row :104-109
        float val[4];
        const float* urow = (PROJ == 1 && INTERIOR) ? &T.sF[ri + AT_HB][AT_HB] : &T.sU[ri][0];
#pragma unroll
        for (int kp = 0; kp < 2; ++kp) {
            const int c = lane + 64 * kp, c1 = c + 32;                 // tile columns of the pair
            const int j = jb + 64 * kp, j1 = j + 32;
            // a9: u_i = 0.5*U[i][j] + 0.5*U[i][j+1] for j <= w-2;  v_i = 0.5*V[i][j] + 0.5*V[i+1][j] for j <= w-1; else 0
            const bool cu0 = urow_ok && (INTERIOR || j <= w - 2), cu1 = urow_ok && (INTERIOR || j1 <= w - 2);
            const bool cv0 = vrow_ok && (INTERIOR || j <= w - 1), cv1 = vrow_ok && (INTERIOR || j1 <= w - 1);
            const float2 ua = make_float2(cu0 ? urow[c] : 0.f, cu1 ? urow[c1] : 0.f);
            const float2 ub = make_float2(cu0 ? urow[c + 1] : 0.f, cu1 ? urow[c1 + 1] : 0.f);
            const float2 va = make_float2(cv0 ? T.sV[ri][c] : 0.f, cv1 ? T.sV[ri][c1] : 0.f);
            const float2 vb = make_float2(cv0 ? T.sV[ri + 1][c] : 0.f, cv1 ? T.sV[ri + 1][c1] : 0.f);
            const float2 hua = __fmul2_rn(half2, ua), hub = __fmul2_rn(half2, ub);
            const float2 hva = __fmul2_rn(half2, va), hvb = __fmul2_rn(half2, vb);
            const float2 ui = make_float2(hua.x + hub.x, hua.y + hub.y);
            const float2 vi = make_float2(hva.x + hvb.x, hva.y + hvb.y);
            const float2 du = __fmul2_rn(dt2, ui), dv = __fmul2_rn(dt2, vi);
            float2 px = make_float2((float)j - du.x, (float)j1 - du.y);                                     // :87
            float2 py = make_float2(fi - dv.x, fi - dv.y);                                                  // :88
            px.x = fminf(fmaxf(px.x, 0.0f), xmax); px.y = fminf(fmaxf(px.y, 0.0f), xmax);                   // :91
            py.x = fminf(fmaxf(py.x, 0.0f), ymax); py.y = fminf(fmaxf(py.y, 0.0f), ymax);                   // :92
            // a8 (:111-131) with x0 = floor(px) already inside [0, cols-1]
            const float2 fx0 = make_float2(floorf(px.x), floorf(px.y)), fy0 = make_float2(floorf(py.x), floorf(py.y));
            float2 fx1 = __fadd2_rn(fx0, one2), fy1 = __fadd2_rn(fy0, one2);
            const int x0a = (int)fx0.x, x0b = (int)fx0.y;
            int y0a = (int)fy0.x, y0b = (int)fy0.y;
            float2 f00, f01, f10, f11;
            bool gathered = false;
            if (INTERIOR) {
                // The window of an interior tile lies inside the field (on a slab: inside the stored rows, and -- k_advect_tiled --
                // inside the rows that are still exact, so no reach guard can fire here), so a pair whose lower corners are inside
                // the window (with room for the +1 corners) has x0 + 1 <= cols - 1 and y0 + 1 <= rows - 1: the clamps of the upper
                // corners (:121, :123) do not bind and the corner offsets are the constants 1 and AT_FP.  Only the pairs that leave
                // the window clamp, compare and gather from global memory (below).
                const int yorg = SLAB ? wy_org + a.row0 : wy_org;                    // y0 is a GLOBAL row on a slab
                const int lya = y0a - yorg, lxa = x0a - wx_org, lyb = y0b - yorg, lxb = x0b - wx_org;
                const bool inwin = ((unsigned)lya < (unsigned)(AT_FR - 1)) & ((unsigned)lxa < (unsigned)(AT_FP - 1)) &
                                   ((unsigned)lyb < (unsigned)(AT_FR - 1)) & ((unsigned)lxb < (unsigned)(AT_FP - 1));
                if (inwin) {
                    const float* qa = sF0 + (lya * AT_FP + lxa);
                    const float* qb = sF0 + (lyb * AT_FP + lxb);
                    f00 = make_float2(qa[0], qb[0]); f01 = make_float2(qa[1], qb[1]);
                    f10 = make_float2(qa[AT_FP], qb[AT_FP]); f11 = make_float2(qa[AT_FP + 1], qb[AT_FP + 1]);
                    gathered = true;
                }
            }
            if (!gathered) {
                fx1.x = fminf(fx1.x, xmax); fx1.y = fminf(fx1.y, xmax);
                fy1.x = fminf(fy1.x, ymax); fy1.y = fminf(fy1.y, ymax);
                const int dxa = (fx1.x != fx0.x) ? 1 : 0, dxb = (fx1.y != fx0.y) ? 1 : 0;
                int dya = (fy1.x != fy0.x) ? 1 : 0, dyb = (fy1.y != fy0.y) ? 1 : 0;
                if (SLAB) {                                                         // global -> local row, kept inside the slab
                    y0a -= a.row0; y0b -= a.row0;
                    const int y1a = y0a + dya, y1b = y0b + dyb;
                    if (i >= a.need_lo && i < a.need_hi && a.overflow &&
                        ((j < cols && (y0a < a.valid_lo || y1a >= a.valid_hi)) || (j1 < cols && (y0b < a.valid_lo || y1b >= a.valid_hi))))
                        *a.overflow = 1;
                    if (y1a > rows - 1) dya = 0;
                    if (y1b > rows - 1) dyb = 0;
                    y0a = clampi(y0a, 0, rows - 1); y0b = clampi(y0b, 0, rows - 1);
                }
                // both cells of the pair inside the staged window?  (an interior tile comes here with a pair that is not, unless the
                // slab clamp above just moved it back in)
                bool inwin;
                if (INTERIOR && !SLAB) inwin = false;
                else if (INTERIOR) {
                    const int lya = y0a - wy_org, lxa = x0a - wx_org, lyb = y0b - wy_org, lxb = x0b - wx_org;
                    inwin = ((unsigned)lya < (unsigned)(AT_FR - 1)) & ((unsigned)lxa < (unsigned)(AT_FP - 1)) &
                            ((unsigned)lyb < (unsigned)(AT_FR - 1)) & ((unsigned)lxb < (unsigned)(AT_FP - 1));
                } else inwin = y0a >= wy0 && y0a + dya < wy1 && x0a >= wx0 && x0a + dxa < wx1 &&
                               y0b >= wy0 && y0b + dyb < wy1 && x0b >= wx0 && x0b + dxb < wx1;
                if (inwin) {
                    const float* qa = sF0 + ((y0a - wy_org) * AT_FP + (x0a - wx_org));
                    const float* qb = sF0 + ((y0b - wy_org) * AT_FP + (x0b - wx_org));
                    const int oya = dya * AT_FP, oyb = dyb * AT_FP;
                    f00 = make_float2(qa[0], qb[0]); f01 = make_float2(qa[dxa], qb[dxb]);
                    f10 = make_float2(qa[oya], qb[oyb]); f11 = make_float2(qa[oya + dxa], qb[oyb + dxb]);
                } else {
                    if (PROJ) {
                        f00 = make_float2(advect_global<PROJ>(a, F, P, y0a, x0a), advect_global<PROJ>(a, F, P, y0b, x0b));
                        f01 = make_float2(advect_global<PROJ>(a, F, P, y0a, x0a + dxa), advect_global<PROJ>(a, F, P, y0b, x0b + dxb));
                        f10 = make_float2(advect_global<PROJ>(a, F, P, y0a + dya, x0a), advect_global<PROJ>(a, F, P, y0b + dyb, x0b));
                        f11 = make_float2(advect_global<PROJ>(a, F, P, y0a + dya, x0a + dxa), advect_global<PROJ>(a, F, P, y0b + dyb, x0b + dxb));
                    } else {
                        const float* qa = F + ((unsigned)y0a * pitch + x0a);
                        const float* qb = F + ((unsigned)y0b * pitch + x0b);
                        const int oya = dya * pitch, oyb = dyb * pitch;
                        f00 = make_float2(__ldg(qa), __ldg(qb)); f01 = make_float2(__ldg(qa + dxa), __ldg(qb + dxb));
                        f10 = make_float2(__ldg(qa + oya), __ldg(qb + oyb)); f11 = make_float2(__ldg(qa + oya + dxa), __ldg(qb + oyb + dxb));
                    }
                }
            }
            const float2 ax = __fadd2_rn(fx1, neg2(px)), bx = __fadd2_rn(px, neg2(fx0));
            const float2 ay = __fadd2_rn(fy1, neg2(py)), by = __fadd2_rn(py, neg2(fy0));
            const float2 t00 = __fmul2_rn(__fmul2_rn(ax, ay), f00), t01 = __fmul2_rn(__fmul2_rn(bx, ay), f01);
            const float2 t10 = __fmul2_rn(__fmul2_rn(ax, by), f10), t11 = __fmul2_rn(__fmul2_rn(bx, by), f11);
            float2 sum = make_float2(t00.x + t01.x, t00.y + t01.y);
            sum.x = sum.x + t10.x; sum.y = sum.y + t10.y;
            sum.x = sum.x + t11.x; sum.y = sum.y + t11.y;
            if (a.has_scale) sum = __fmul2_rn(sum, make_float2(a.scale, a.scale));                          // :171
            val[2 * kp] = sum.x; val[2 * kp + 1] = sum.y;
        }
        // coalesced scalar stores (a warp writes 128 B per instruction); the padding columns [cols, pitch) get zeros
        float* orow = O + (unsigned)i * pitch;
        if (INTERIOR) {
#pragma unroll
            for (int k = 0; k < 4; ++k) orow[jb + 32 * k] = val[k];
            if (a.frame) {                                                          // :173 (+ fractal_generator.py:62)
                const size_t frow = b * a.frame_stride + (unsigned)i * a.frame_pitch;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float fr = val[k];
                    if (a.fmul) fr = fr + __ldg(a.fmul + (unsigned)i * a.frame_pitch + jb + 32 * k) * fr;
                    frame_st1(a.frame, frow + jb + 32 * k, fr, ffmt);
                }
            }
        } else {
            const size_t frow = b * a.frame_stride + (unsigned)i * a.frame_pitch;
            const float* mrow = a.fmul ? a.fmul + (unsigned)i * a.frame_pitch : nullptr;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int j = jb + 32 * k;
                if (j < pitch) {
                    const float x = (j < cols) ? val[k] : 0.0f;
                    orow[j] = x;
                    if (a.frame && j < a.frame_pitch) {
                        float fr = x;
                        if (mrow) fr = fr + __ldg(mrow + j) * fr;
                        frame_st1(a.frame, frow + j, fr, ffmt);
                    }
                }
            }
        }
    }
}

template <bool SLAB, int PROJ>
__global__ void __launch_bounds__(256, PROJ ? 5 : 6)        // 40 registers: 6 CTAs per SM beat 4 (62 registers) by 12 % and 7 (32, spills) by 5 %; the pressure window of the fused variants leaves room for 5
k_advect_tiled(const AdvectArgs a, const __grid_constant__ TmaMap mF, const __grid_constant__ TmaMap mU, const __grid_constant__ TmaMap mV,
               const __grid_constant__ TmaMap mP)
{
    pdl_prologue();
    __shared__ __align__(128) typename std::conditional<PROJ != 0, AdvectTileP, AdvectTile>::type TT;
    __shared__ __align__(8) unsigned long long tma_bar;
    AdvectTile& T = *reinterpret_cast<AdvectTile*>(&TT);
    float (*sP)[AT_PP] = PROJ ? reinterpret_cast<float (*)[AT_PP]>(reinterpret_cast<char*>(&TT) + sizeof(AdvectTile)) : nullptr;
    int ty = (int)blockIdx.y + a.ty0;
    if (ty >= a.skip_lo[0]) ty += a.skip_n[0];
    if (ty >= a.skip_lo[1]) ty += a.skip_n[1];
    const int i0 = ty * AT_R, j0 = blockIdx.x * AT_C;
    const size_t b = blockIdx.z;
    const float* F = a.F + b * a.stride;
    const float* U = a.U + b * a.su_;
    const float* V = a.V + b * a.sv_;
    const float* P = PROJ ? a.P + b * a.sc_ : nullptr;
    float* O = a.O + b * a.stride;
    asm volatile("" : "+l"(F));
    asm volatile("" : "+l"(U));
    asm volatile("" : "+l"(V));
    asm volatile("" : "+l"(O));
    // interior tile: the staged window and the tile's u / v rows lie inside the arrays, every cell is a field cell
    // strictly before the last row / column of the (global) grid, so no sample is zeroed and nothing needs a bound
    const int gi_last = (SLAB ? a.row0 : 0) + i0 + AT_R - 1;
    const int h = SLAB ? a.gh : a.h;
    bool interior = i0 >= AT_HB && i0 + AT_R + AT_HB <= a.rows && j0 >= AT_HB && j0 + AT_C + AT_HB <= a.pitch &&
                    j0 + AT_C + 4 <= a.pu && j0 + AT_C <= a.pv && i0 + AT_R + 1 <= a.h &&
                    j0 + AT_C - 1 <= a.w - 2 && gi_last <= h - 2 && j0 + AT_C <= a.cols && j0 + AT_C <= a.frame_pitch;
    // fused gradient subtract: the pressure window lies inside p, and every staged cell is one that k_project updates
    // (u rows 1 .. h-1: the window starts at row i0 - 4 >= 1; v columns 1 .. w-1: the window starts at column j0 - 4 >= 1)
    // slab with a reach guard: the in-window gathers of an interior tile are not tested against the exact rows, so its window has to
    // lie inside them (or its rows outside the guarded ones)
    if (SLAB && a.overflow)
        interior = interior && ((i0 - AT_HB >= a.valid_lo && i0 + AT_R + AT_HB <= a.valid_hi) || i0 + AT_R <= a.need_lo || i0 >= a.need_hi);
    if (PROJ) interior = interior && i0 >= AT_HB + 1 && i0 + AT_R + AT_HB <= a.h && j0 >= 8 && j0 + AT_C + 8 <= a.pc && j0 + AT_C + AT_HB <= a.w;
    if (interior) advect_tile<SLAB, true, PROJ>(a, T, sP, F, U, V, P, O, b, i0, j0, &mF, &mU, &mV, &mP, &tma_bar);
    else          advect_tile<SLAB, false, PROJ>(a, T, sP, F, U, V, P, O, b, i0, j0, &mF, &mU, &mV, &mP, &tma_bar);
}

// proj / p / vout: 0 / NULL / NULL for the plain advection; 1 fuses the gradient subtract of the pressure p into the tiled u
// advection (field == u and v are then the UNPROJECTED arrays; the projected v is written to vout, a different array).
// advect_can_fuse_project() tells whether the launch would take the tiled kernel; callers that get `false` run k_project first.
bool advect_can_fuse_project(const smk_grid_t* g)
{
    if (env().project_fused == 0) return false;
    const int tiled = env().advect_tiled != SMK_ENV_UNSET ? env().advect_tiled : -1;
    const bool big = (int64_t)g->h * g->w * g->batch >= (int64_t)6 << 20;
    const bool forced = env().project_fused == 1 && tiled != 0;
    return (tiled == 1 || (tiled == -1 && big) || forced) && (g->h + 1 + AT_R - 1) / AT_R <= 65535;
}

// true when launch_advect (without a fused gradient subtract) would run k_advect_tiled for a field of this size
bool advect_is_tiled(const smk_grid_t* g, int rows, int cols)
{
    int tiled = -1;
    if (env().advect_tiled != SMK_ENV_UNSET) tiled = env().advect_tiled;
    const bool big = (int64_t)rows * cols * g->batch >= (int64_t)6 << 20;
    return (tiled == 1 || (tiled == -1 && big)) && (rows + AT_R - 1) / AT_R <= 65535;
}
int advect_tile_rows() { return AT_R; }

int launch_advect(const smk_grid_t* g, const float* field, float* out, int rows, int cols, int pitch, int64_t stride,
                  const float* u, const float* v, float dt, float scale, void* frame, int64_t frame_stride,
                  const float* fmul, const smk_slab_check_t* chk, cudaStream_t s, int proj, const float* p, float* vout,
                  const AdvectPart* part, int frame_format)
{
    if ((int64_t)rows * pitch >= (1ll << 31)) return fail(SMK_EUNSUPPORTED, "smk_advect: field of %d x %d exceeds 2^31 elements", rows, pitch);
    AdvectArgs a;
    a.F = field; a.O = out; a.rows = rows; a.cols = cols; a.pitch = pitch; a.stride = stride;
    a.U = u; a.V = v; a.h = g->h; a.w = g->w; a.pu = g->pitch_u; a.pv = g->pitch_v; a.su_ = g->stride_u; a.sv_ = g->stride_v;
    a.dt = dt; a.has_scale = scale != 1.0f ? 1 : 0; a.scale = scale;
    a.frame = frame; a.frame_stride = frame_stride; a.frame_pitch = g->pitch_c; a.fmul = fmul; a.frame_format = frame_format;
    a.ngroups = (unsigned)((cols + 3) / 4);
    a.magic = ((1ull << 40) + a.ngroups - 1) / a.ngroups;
    const bool slab = g->gh != 0 && (g->gh != g->h || g->row0 != 0);
    a.row0 = g->row0; a.gh = g->gh;
    a.need_lo = chk ? chk->need_lo : 0; a.need_hi = chk ? chk->need_hi : 0;
    a.valid_lo = chk ? chk->valid_lo : 0; a.valid_hi = chk ? chk->valid_hi : 0; a.overflow = chk ? chk->overflow_flag : nullptr;
    a.P = p; a.pc = g->pitch_c; a.sc_ = g->stride_c; a.Vout = vout;
    a.ty0 = 0; a.skip_lo[0] = a.skip_lo[1] = 0x7fffffff; a.skip_n[0] = a.skip_n[1] = 0;
    a.use_tma = 0;
    TmaMap mF, mU, mV, mP;
    memset(&mF, 0, sizeof mF); memset(&mU, 0, sizeof mU); memset(&mV, 0, sizeof mV); memset(&mP, 0, sizeof mP);
    // tensor maps for the tiled kernel's interior tiles (SMK_ADVECT_TMA=0: cp.async staging everywhere); any failure keeps cp.async
    auto make_maps = [&]() {
        if (env().advect_tma == 0) return;
        const int urows = g->h + 1;
        bool ok = tma_map_3d(&mF, field, pitch, rows, g->batch, stride, AT_FR, AT_FP) &&
                  tma_map_3d(&mV, v, g->pitch_v, g->h, g->batch, g->stride_v, AT_R + 1, AT_VP);
        if (ok && proj) ok = tma_map_3d(&mP, p, g->pitch_c, g->h, g->batch, g->stride_c, AT_PR, AT_PP);
        if (ok && !proj) ok = tma_map_3d(&mU, u, g->pitch_u, urows, g->batch, g->stride_u, AT_R, AT_UP);
        a.use_tma = ok ? 1 : 0;
    };
    const unsigned long long nthreads = (unsigned long long)rows * a.ngroups;
    dim3 grid((unsigned)((nthreads + 255) / 256), g->batch);
    if (proj) {
        if (!p || !vout || vout == v || proj != 1 || rows != g->h + 1 || !advect_can_fuse_project(g))
            return fail(SMK_EINVAL, "launch_advect: the fused gradient subtract is for the u advection on the tiled kernel, and needs p and a separate array for the projected v");
        ProfScope prof_(SMK_PH_PROJECT_ADVECT_U, s);
        dim3 tgrid((unsigned)((pitch + AT_C - 1) / AT_C), (unsigned)((rows + AT_R - 1) / AT_R), g->batch);
        const bool slab_ = g->gh != 0 && (g->gh != g->h || g->row0 != 0);
        make_maps();
        if (slab_) launch_chain(k_advect_tiled<true, 1>, tgrid, dim3(256), 0, s, a, mF, mU, mV, mP);
        else       launch_chain(k_advect_tiled<false, 1>, tgrid, dim3(256), 0, s, a, mF, mU, mV, mP);
        return check_launch("k_advect_tiled (fused gradient subtract)");
    }
    ProfScope prof_(rows == g->h + 1 ? SMK_PH_ADVECT_U : (cols == g->w + 1 ? SMK_PH_ADVECT_V : SMK_PH_ADVECT_D), s);
    // the tiled kernel wins on big fields (8192^2: 182 against 229 us), the direct one on small ones (1024^2: 10.0
    // against 10.7 us; equal at 2048^2): -1 picks by size, SMK_ADVECT_TILED = 0 / 1 forces one of them
    int tiled = -1;
    if (env().advect_tiled != SMK_ENV_UNSET) tiled = env().advect_tiled;
    const bool big = (int64_t)rows * cols * g->batch >= (int64_t)6 << 20;
    if ((tiled == 1 || (tiled == -1 && big)) && (rows + AT_R - 1) / AT_R <= 65535) {
        dim3 tgrid((unsigned)((pitch + AT_C - 1) / AT_C), (unsigned)((rows + AT_R - 1) / AT_R), g->batch);
        if (part) {
            // a band of tile rows, or everything but up to two bands
            int ny = (int)tgrid.y;
            if (part->band_n > 0) { a.ty0 = part->band_lo; ny = part->band_n; }
            else
                for (int k = 0; k < 2; ++k)
                    if (part->skip_n[k] > 0) { a.skip_lo[k] = part->skip_lo[k]; a.skip_n[k] = part->skip_n[k]; ny -= part->skip_n[k]; }
            if (ny <= 0) return SMK_OK;
            tgrid.y = (unsigned)ny;
        }
        make_maps();
        if (slab) launch_chain(k_advect_tiled<true, 0>, tgrid, dim3(256), 0, s, a, mF, mU, mV, mP);
        else      launch_chain(k_advect_tiled<false, 0>, tgrid, dim3(256), 0, s, a, mF, mU, mV, mP);
        return check_launch("k_advect_tiled");
    }
    if (part) return fail(SMK_EUNSUPPORTED, "launch_advect: a part of the rows needs the tiled kernel (advect_is_tiled)");
    if (slab) launch_chain(k_advect<true>, grid, dim3(256), 0, s, a);
    else      launch_chain(k_advect<false>, grid, dim3(256), 0, s, a);
    return check_launch("k_advect");
}

// ---- a2: add_smoke_source, batched ---------------------------------------------------------------------
// Cell-centric so that overlapping emitters are added in list order (fp32 addition is order dependent,
// and the reference applies them one call after another).  A CTA owns a 32 x 8 tile; it first culls the
// simulation's emitter list, 256 at a time, to those whose bounding box touches the tile (ordered
// compaction with ballots), then every cell walks the short list.  Large grids carry thousands of emitters.
__global__ void __launch_bounds__(256)
k_splat(float* __restrict__ Dn, const int h, const int w, const int pc, const long long sc_,
        const smk_source_t* __restrict__ src, const int32_t* __restrict__ off)
{
    __shared__ int list[256];
    __shared__ int wcount[8];
    const int tid = threadIdx.y * 32 + threadIdx.x, lane = threadIdx.x, wp = threadIdx.y;
    const int j0 = blockIdx.x * 32, i0 = blockIdx.y * 8;
    const int j = j0 + lane, i = i0 + wp;
    const int b = blockIdx.z;
    const int s0 = off[b], s1 = off[b + 1];
    if (s0 == s1) return;
    const bool in = i < h && j < w;
    float* cell = Dn + (size_t)b * sc_ + (size_t)i * pc + j;
    float acc = in ? *cell : 0.f;
    for (int base = s0; base < s1; base += 256) {
        const int k = base + tid;
        bool hit = false;
        if (k < s1) {
            const smk_source_t e = src[k];
            const long long r = e.radius;
            hit = (long long)j0 <= e.x + r && (long long)j0 + 31 >= e.x - r && (long long)i0 <= e.y + r && (long long)i0 + 7 >= e.y - r;
        }
        // most 256-emitter chunks of a long list miss the tile altogether: one barrier-with-vote, and on to the next chunk
        if (!__syncthreads_or(hit ? 1 : 0)) continue;
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) wcount[wp] = __popc(m);
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) { if (q < wp) before += wcount[q]; total += wcount[q]; }
        if (hit) list[before + __popc(m & ((1u << lane) - 1u))] = k;
        __syncthreads();
        for (int q = 0; q < total; ++q) acc = splat_add(acc, i, j, src[list[q]]);
        __syncthreads();
    }
    if (in) *cell = acc;
}

// The same for big grids with long emitter lists (8192 x 8192 carries 16 k emitters): every CTA of k_splat culls the WHOLE list, so
// its cost is (number of CTAs) x (list length) -- 10.2 ms at 8192^2, six steps' worth of kernels (profiles/r02q_launches_c4*).  Here
// a CTA owns 128 x 64 cells, 32 per thread, i.e. 32 x fewer passes over the list; a listed emitter is loaded once per thread and
// tested against the thread's 32 cells.  Every cell still adds its emitters in list order with the same operations: bit-identical.
constexpr int SPB_W = 128, SPB_H = 64;
__global__ void __launch_bounds__(256)
k_splat_big(float* __restrict__ Dn, const int h, const int w, const int pc, const long long sc_,
            const smk_source_t* __restrict__ src, const int32_t* __restrict__ off)
{
    __shared__ int list[256];
    __shared__ int wcount[8];
    const int tid = threadIdx.y * 32 + threadIdx.x, lane = threadIdx.x, wp = threadIdx.y;
    const int j0 = blockIdx.x * SPB_W, i0 = blockIdx.y * SPB_H;
    const int b = blockIdx.z;
    const int s0 = off[b], s1 = off[b + 1];
    if (s0 == s1) return;
    float* base_ = Dn + (size_t)b * sc_;
    float acc[SPB_H / 8][SPB_W / 32];
    bool any = false;
    for (int base = s0; base < s1; base += 256) {
        const int k = base + tid;
        bool hit = false;
        if (k < s1) {
            const smk_source_t e = src[k];
            const long long r = e.radius;
            hit = (long long)j0 <= e.x + r && (long long)j0 + (SPB_W - 1) >= e.x - r && (long long)i0 <= e.y + r && (long long)i0 + (SPB_H - 1) >= e.y - r;
        }
        // most 256-emitter chunks of a long list miss the tile altogether: one barrier-with-vote, and on to the next chunk
        if (!__syncthreads_or(hit ? 1 : 0)) continue;
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) wcount[wp] = __popc(m);
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) { if (q < wp) before += wcount[q]; total += wcount[q]; }
        if (hit) list[before + __popc(m & ((1u << lane) - 1u))] = k;
        __syncthreads();
        if (total > 0 && !any) {                                              // first emitter that touches the tile: load the cells
            any = true;
#pragma unroll
            for (int cy = 0; cy < SPB_H / 8; ++cy)
#pragma unroll
                for (int cx = 0; cx < SPB_W / 32; ++cx) {
                    const int i = i0 + wp + 8 * cy, j = j0 + lane + 32 * cx;
                    acc[cy][cx] = (i < h && j < w) ? base_[(size_t)i * pc + j] : 0.f;
                }
        }
        for (int q = 0; q < total; ++q) {
            const smk_source_t e = src[list[q]];
            const float rad = (float)e.radius;
            const double r3 = (double)e.radius / 3.0;
            const float denom = (float)(2.0 * (r3 * r3));
#pragma unroll
            for (int cy = 0; cy < SPB_H / 8; ++cy) {
                const long long dy = (long long)(i0 + wp + 8 * cy) - e.y;
#pragma unroll
                for (int cx = 0; cx < SPB_W / 32; ++cx) {
                    const long long dx = (long long)(j0 + lane + 32 * cx) - e.x;
                    const float dist = sqrtf((float)(dx * dx + dy * dy));    // navier_stokes.py:45
                    if (dist <= rad) {                                       // :46
                        const float d2 = dist * dist;
                        acc[cy][cx] = acc[cy][cx] + e.intensity * expf((-d2) / denom);      // :48
                    }
                }
            }
        }
        __syncthreads();
    }
    if (any) {
#pragma unroll
        for (int cy = 0; cy < SPB_H / 8; ++cy)
#pragma unroll
            for (int cx = 0; cx < SPB_W / 32; ++cx) {
                const int i = i0 + wp + 8 * cy, j = j0 + lane + 32 * cx;
                if (i < h && j < w) base_[(size_t)i * pc + j] = acc[cy][cx];
            }
    }
}

int launch_splat(const smk_grid_t* g, float* density, const smk_source_t* src, const int32_t* off, cudaStream_t s)
{
    ProfScope prof_(SMK_PH_SPLAT, s);
    // big grids (their lists are long: one emitter per 64 x 64 block in the benches) take the big-tile kernel; SMK_SPLAT_BIG = 0 / 1 forces
    const int forced = env().splat_big;
    const bool big = forced != SMK_ENV_UNSET ? forced != 0 : (int64_t)g->h * g->w >= ((int64_t)4 << 20);
    if (big) {
        dim3 grid((g->w + SPB_W - 1) / SPB_W, (g->h + SPB_H - 1) / SPB_H, g->batch), blk(32, 8);
        if (grid.y <= 65535) {
            k_splat_big<<<grid, blk, 0, s>>>(density, g->h, g->w, g->pitch_c, g->stride_c, src, off);
            return check_launch("k_splat_big");
        }
    }
    dim3 grid((g->w + 31) / 32, (g->h + 7) / 8, g->batch), blk(32, 8);
    k_splat<<<grid, blk, 0, s>>>(density, g->h, g->w, g->pitch_c, g->stride_c, src, off);
    return check_launch("k_splat");
}

// ---- velocity forcing: u = u + du, v = v + dv over the batch, one rounded add per cell ------------------------------------
// The head of a forced step on the phase kernels (after the emitters' splat, before k_forces_diffuse_div), and in reverse mode the
// accumulation of a constant forcing's gradient.  A thread adds one float4 of a row of u and the same float4 of v; only the cells
// inside rows x cols are read or written (a row's last group adds its cells one by one), so pads stay as they are.
__device__ __forceinline__ void add_row4(float* __restrict__ f, const float* __restrict__ df, const int c, const int cols)
{
    if (c + 4 <= cols) {
        float4 x = *reinterpret_cast<const float4*>(f + c);
        const float4 d = __ldg(reinterpret_cast<const float4*>(df + c));
        x.x = x.x + d.x; x.y = x.y + d.y; x.z = x.z + d.z; x.w = x.w + d.w;
        *reinterpret_cast<float4*>(f + c) = x;
    } else {
        for (int k = c; k < cols; ++k) f[k] = f[k] + __ldg(df + k);
    }
}

__global__ void __launch_bounds__(256)
k_add_forcing(float* __restrict__ U, float* __restrict__ V, const float* __restrict__ DU, const float* __restrict__ DV,
              const int h, const int w, const int pu, const int pv, const long long su_, const long long sv_)
{
    pdl_prologue();
    const int c = 4 * (int)(blockIdx.x * 32 + threadIdx.x), i = blockIdx.y * 8 + threadIdx.y;
    const size_t b = blockIdx.z;
    if (i <= h && c < w) add_row4(U + b * su_ + (size_t)i * pu, DU + b * su_ + (size_t)i * pu, c, w);
    if (i < h && c <= w) add_row4(V + b * sv_ + (size_t)i * pv, DV + b * sv_ + (size_t)i * pv, c, w + 1);
}

int launch_add_forcing(const smk_grid_t* g, float* u, float* v, const float* du, const float* dv, cudaStream_t s)
{
    const dim3 grid((g->w + 1 + 127) / 128, (g->h + 1 + 7) / 8, g->batch);
    ProfScope prof_(SMK_PH_OTHER, s);
    launch_chain(k_add_forcing, grid, dim3(32, 8), 0, s, u, v, du, dv, g->h, g->w, g->pitch_u, g->pitch_v,
                 (long long)g->stride_u, (long long)g->stride_v);
    return check_launch("k_add_forcing");
}

// ---- divergence norms: per simulation max|div| and sum div^2 (un-normalised u,v differences) -------------
__global__ void __launch_bounds__(256)
k_div_norms(const float* __restrict__ U, const float* __restrict__ V, float* __restrict__ out,
            const int h, const int w, const int pu, const int pv, const long long su_, const long long sv_)
{
    const size_t b = blockIdx.z;
    U += b * su_; V += b * sv_;
    float mx = 0.f, ss = 0.f;
    for (int i = blockIdx.y; i < h; i += gridDim.y)
        for (int j = blockIdx.x * 256 + threadIdx.x; j < w; j += gridDim.x * 256) {
            float s = U[(size_t)(i + 1) * pu + j] - U[(size_t)i * pu + j];
            s = s + V[(size_t)i * pv + j + 1];
            s = s - V[(size_t)i * pv + j];
            mx = fmaxf(mx, fabsf(s));
            ss += s * s;
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    __shared__ float smx[8], sss[8];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    if (lane == 0) { smx[wp] = mx; sss[wp] = ss; }
    __syncthreads();
    if (wp == 0) {
        mx = lane < 8 ? smx[lane] : 0.f; ss = lane < 8 ? sss[lane] : 0.f;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            ss += __shfl_xor_sync(0xffffffffu, ss, o);
        }
        if (lane == 0) {
            atomicMax(reinterpret_cast<int*>(out + 2 * b), __float_as_int(mx));   // mx >= 0: int order == float order
            atomicAdd(out + 2 * b + 1, ss);
        }
    }
}

int launch_div_norms(const smk_grid_t* g, const float* u, const float* v, float* out, cudaStream_t s)
{
    dim3 grid((g->w + 255) / 256, min(g->h, 64), g->batch);
    ProfScope prof_(SMK_PH_OTHER, s);
    k_div_norms<<<grid, 256, 0, s>>>(u, v, out, g->h, g->w, g->pitch_u, g->pitch_v, g->stride_u, g->stride_v);
    return check_launch("k_div_norms");
}

// ---- Jacobi residual: per simulation max|p' - p| and sum (p' - p)^2, p' = one more sweep of navier_stokes.py:139-145
// over (p, div) -- how far the K sweeps just done are from a fixed point.  Same warp-shuffle + atomic reduction as above.
__global__ void __launch_bounds__(256)
k_jacobi_residual(const float* __restrict__ P, const float* __restrict__ DIV, float* __restrict__ out,
                  const int h, const int w, const int pc, const long long sc_)
{
    const size_t b = blockIdx.z;
    P += b * sc_; DIV += b * sc_;
    float mx = 0.f, ss = 0.f;
    for (int i = blockIdx.y; i < h; i += gridDim.y)
        for (int j = blockIdx.x * 256 + threadIdx.x; j < w; j += gridDim.x * 256) {
            const float pc0 = P[(size_t)i * pc + j];
            float pn = 0.f;                                  // the ring is reset to zero by every sweep (:140-141)
            if (i >= 1 && i <= h - 2 && j >= 1 && j <= w - 2) {
                float s = P[(size_t)(i - 1) * pc + j] + P[(size_t)(i + 1) * pc + j];
                s = s + P[(size_t)i * pc + j - 1];
                s = s + P[(size_t)i * pc + j + 1];
                pn = 0.25f * (s - DIV[(size_t)i * pc + j]);
            }
            const float r = pn - pc0;
            mx = fmaxf(mx, fabsf(r));
            ss += r * r;
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    __shared__ float smx[8], sss[8];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    if (lane == 0) { smx[wp] = mx; sss[wp] = ss; }
    __syncthreads();
    if (wp == 0) {
        mx = lane < 8 ? smx[lane] : 0.f; ss = lane < 8 ? sss[lane] : 0.f;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            ss += __shfl_xor_sync(0xffffffffu, ss, o);
        }
        if (lane == 0) {
            atomicMax(reinterpret_cast<int*>(out + 2 * b), __float_as_int(mx));
            atomicAdd(out + 2 * b + 1, ss);
        }
    }
}

int launch_jacobi_residual(const smk_grid_t* g, const float* div, const float* p, float* out, cudaStream_t s)
{
    dim3 grid((g->w + 255) / 256, min(g->h, 64), g->batch);
    ProfScope prof_(SMK_PH_OTHER, s);
    k_jacobi_residual<<<grid, 256, 0, s>>>(p, div, out, g->h, g->w, g->pitch_c, g->stride_c);
    return check_launch("k_jacobi_residual");
}

// ---- a13: FractalGenerator fields (constant per grid shape; computed once and cached by the host) -------
// Output index [a][b] pairs px[a]/mx[a] with py[b]/my[b] (torch.meshgrid(x_w, y_h, indexing='ij'),
// fractal_generator.py:17-19,:38-42): shape (na=w, nb=h).  Any of perlin / mandel / mul may be NULL.
__global__ void k_fractal_fields(float* __restrict__ perlin, float* __restrict__ mandel, float* __restrict__ mul,
                                 const int na, const int nb, const int pitch, const float intensity, const int iterations,
                                 const float* __restrict__ px, const float* __restrict__ py,
                                 const float* __restrict__ mx, const float* __restrict__ my)
{
    const int bcol = blockIdx.x * 32 + threadIdx.x, a = blockIdx.y * 8 + threadIdx.y;
    if (a >= na || bcol >= nb) return;
    float P = 0.f, M = 0.f;
    if (perlin || mul) {
        // octaves: noise += (amp*sin(f*X))*cos(f*Y); (noise+1)/2                 fractal_generator.py:21-31
        const float X = px[a], Y = py[bcol];
        float noise = 0.f, amp = 1.f, freq = 1.f;
        for (int o = 0; o < 6; ++o) {
            float t = amp * sinf(freq * X);
            t = t * cosf(freq * Y);
            noise = noise + t;
            amp *= 0.5f; freq *= 2.0f;
        }
        P = (noise + 1.0f) / 2.0f;
        if (perlin) perlin[(size_t)a * pitch + bcol] = P;
    }
    if (mandel || mul) {
        // escape count of z <- z^2 + c while |z| <= 2, c = mx[a] + i*my[b]       fractal_generator.py:44-51
        // z^2 as ATen's vectorised complex square: re = a*a - b*b, im = a*b + b*a, each op rounded.
        const float cr = mx[a], ci = my[bcol];
        float zr = 0.f, zi = 0.f, cnt = 0.f;
        for (int it = 0; it < iterations; ++it) {
            // |z| <= 2 with |z| the fp32-rounded hypot  <=>  zr^2+zi^2 <= (2 + 2^-23)^2, evaluated in double
            const double s2 = (double)zr * (double)zr + (double)zi * (double)zi;
            if (!(s2 <= 4.0 + 0x1p-21 + 0x1p-46)) break;      // once outside, z is frozen: it stays outside
            const float aa = zr * zr, bb = zi * zi;
            const float re = aa - bb;
            const float im = zr * zi + zi * zr;
            zr = re + cr; zi = im + ci;
            cnt = (float)it;
        }
        M = cnt / (float)iterations;
        if (mandel) mandel[(size_t)a * pitch + bcol] = M;
    }
    if (mul) {
        const float F = 0.7f * P + 0.3f * M;                                      // :59
        mul[(size_t)a * pitch + bcol] = intensity * F;                            // :62
    }
}

int launch_fractal_fields(float* perlin, float* mandel, float* mul, int na, int nb, int pitch, float intensity, int iterations,
                          const float* px, const float* py, const float* mx, const float* my, cudaStream_t s)
{
    dim3 grid((nb + 31) / 32, (na + 7) / 8), blk(32, 8);
    ProfScope prof_(SMK_PH_OTHER, s);
    k_fractal_fields<<<grid, blk, 0, s>>>(perlin, mandel, mul, na, nb, pitch, intensity, iterations, px, py, mx, my);
    return check_launch("k_fractal_fields");
}

__global__ void k_apply_mul(const float* __restrict__ F, const float* __restrict__ M, float* __restrict__ O,
                            const int rows, const int cols, const int pitch, const long long stride)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= rows || j >= cols) return;
    const size_t o = (size_t)blockIdx.z * stride + (size_t)i * pitch + j;
    const float f = F[o];
    O[o] = f + M[(size_t)i * pitch + j] * f;
}

int launch_apply_mul(const float* f, const float* mul, float* out, int rows, int cols, int pitch, int batch, int64_t stride, cudaStream_t s)
{
    dim3 grid((cols + 31) / 32, (rows + 7) / 8, batch), blk(32, 8);
    ProfScope prof_(SMK_PH_OTHER, s);
    k_apply_mul<<<grid, blk, 0, s>>>(f, mul, out, rows, cols, pitch, stride);
    return check_launch("k_apply_mul");
}

// ---- solid obstacles (DESIGN.md s5.7); u_closed / v_closed are in common.cuh --------------------------------------------
// O1 (DIV != NULL): close the faces of the diffused u, v and rewrite the divergence from them; O4 (DIV == NULL): close the faces of
// the advected u, v.  Thread (i, j) owns u face (i, j), v face (i, j) and cell (i, j); it reads a neighbour's face only when that
// face is open, which no thread writes.
__global__ void __launch_bounds__(256)
k_obstacle_faces(float* __restrict__ U, float* __restrict__ V, float* __restrict__ DIV, const uint8_t* __restrict__ S,
                 const int h, const int w, const int pu, const int pv, const int pc,
                 const long long su_, const long long sv_, const long long sc_, const long long ss_, const float dt)
{
    pdl_prologue();
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    const size_t b = blockIdx.z;
    U += b * su_; V += b * sv_; S += b * ss_;
    const bool cu0 = i <= h && j < w && u_closed(S, h, pc, i, j);
    const bool cv0 = i < h && j <= w && v_closed(S, w, pc, i, j);
    if (cu0) U[(size_t)i * pu + j] = 0.0f;
    if (cv0) V[(size_t)i * pv + j] = 0.0f;
    if (DIV && i < h && j < w) {
        const float u0 = cu0 ? 0.0f : U[(size_t)i * pu + j];
        const float u1 = u_closed(S, h, pc, i + 1, j) ? 0.0f : U[(size_t)(i + 1) * pu + j];
        const float v0 = cv0 ? 0.0f : V[(size_t)i * pv + j];
        const float v1 = v_closed(S, w, pc, i, j + 1) ? 0.0f : V[(size_t)i * pv + j + 1];
        float s = u1 - u0;                                   // the divergence of navier_stokes.py:136
        s = s + v1;
        s = s - v0;
        DIV[b * sc_ + (size_t)i * pc + j] = s / dt;
    }
}

int launch_obstacle_faces(const smk_grid_t* g, float* u, float* v, float* div, const uint8_t* solid, int64_t solid_stride, float dt,
                          cudaStream_t s)
{
    const dim3 grid((g->w + 1 + 31) / 32, (g->h + 1 + 7) / 8, g->batch);
    ProfScope prof_(SMK_PH_OTHER, s);
    launch_chain(k_obstacle_faces, grid, dim3(32, 8), 0, s, u, v, div, solid, g->h, g->w, g->pitch_u, g->pitch_v, g->pitch_c,
                 (long long)g->stride_u, (long long)g->stride_v, (long long)g->stride_c, (long long)solid_stride, dt);
    return check_launch("k_obstacle_faces");
}

// O3: the density of solid cells, and their element of this step's frame (any SMK_FRAME_* format), := +0.0
__global__ void __launch_bounds__(256)
k_obstacle_cells(float* __restrict__ D, void* frame, const long long frame_stride, const int frame_format,
                 const uint8_t* __restrict__ S, const int h, const int w, const int pc, const long long sc_, const long long ss_)
{
    pdl_prologue();
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= h || j >= w) return;
    const size_t b = blockIdx.z;
    if (S[b * ss_ + (size_t)i * pc + j] == 0) return;
    D[b * sc_ + (size_t)i * pc + j] = 0.0f;
    if (frame) frame_st1(frame, b * frame_stride + (size_t)i * pc + j, 0.0f, frame_format);
}

int launch_obstacle_cells(const smk_grid_t* g, float* d, void* frame, int64_t frame_stride, int frame_format, const uint8_t* solid,
                          int64_t solid_stride, cudaStream_t s)
{
    const dim3 grid((g->w + 31) / 32, (g->h + 7) / 8, g->batch);
    ProfScope prof_(SMK_PH_OTHER, s);
    launch_chain(k_obstacle_cells, grid, dim3(32, 8), 0, s, d, frame, (long long)frame_stride, frame_format, solid, g->h, g->w,
                 g->pitch_c, (long long)g->stride_c, (long long)solid_stride);
    return check_launch("k_obstacle_cells");
}

// The gradient subtract of k_project on open faces only (u rows 1 .. h-1, v columns 1 .. w-1, as navier_stokes.py:148-149);
// closed faces keep the +0.0 of O1.  One thread per u face (i, j) and v face (i, j).
__global__ void __launch_bounds__(256)
k_project_obst(const float* __restrict__ P, float* __restrict__ U, float* __restrict__ V, const uint8_t* __restrict__ S,
               const int h, const int w, const int pu, const int pv, const int pc,
               const long long su_, const long long sv_, const long long sc_, const long long ss_, const float dt)
{
    pdl_prologue();
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= h) return;
    const size_t b = blockIdx.z;
    P += b * sc_; U += b * su_; V += b * sv_; S += b * ss_;
    if (i >= 1 && j < w && !u_closed(S, h, pc, i, j)) {
        const float g = P[(size_t)i * pc + j] - P[(size_t)(i - 1) * pc + j];
        const float t = dt * g;
        U[(size_t)i * pu + j] = U[(size_t)i * pu + j] - t;
    }
    if (j >= 1 && j < w && !v_closed(S, w, pc, i, j)) {
        const float g = P[(size_t)i * pc + j] - P[(size_t)i * pc + j - 1];
        const float t = dt * g;
        V[(size_t)i * pv + j] = V[(size_t)i * pv + j] - t;
    }
}

int launch_project_obst(const smk_grid_t* g, const float* p, float* u, float* v, const uint8_t* solid, int64_t solid_stride, float dt,
                        cudaStream_t s)
{
    const dim3 grid((g->w + 31) / 32, (g->h + 7) / 8, g->batch);
    ProfScope prof_(SMK_PH_PROJECT, s);
    launch_chain(k_project_obst, grid, dim3(32, 8), 0, s, p, u, v, solid, g->h, g->w, g->pitch_u, g->pitch_v, g->pitch_c,
                 (long long)g->stride_u, (long long)g->stride_v, (long long)g->stride_c, (long long)solid_stride, dt);
    return check_launch("k_project_obst");
}

// k_jacobi_residual with p' the masked sweep of k_jacobi_obst (Neumann ghost values at solid neighbours, 0 on solid cells)
__global__ void __launch_bounds__(256)
k_jacobi_residual_obst(const float* __restrict__ P, const float* __restrict__ DIV, const uint8_t* __restrict__ S, float* __restrict__ out,
                       const int h, const int w, const int pc, const long long sc_, const long long ss_)
{
    const size_t b = blockIdx.z;
    P += b * sc_; DIV += b * sc_; S += b * ss_;
    float mx = 0.f, ss = 0.f;
    for (int i = blockIdx.y; i < h; i += gridDim.y)
        for (int j = blockIdx.x * 256 + threadIdx.x; j < w; j += gridDim.x * 256) {
            const size_t c = (size_t)i * pc + j;
            const float pc0 = P[c];
            float pn = 0.f;
            if (i >= 1 && i <= h - 2 && j >= 1 && j <= w - 2 && S[c] == 0) {
                float s = (S[c - pc] ? pc0 : P[c - pc]) + (S[c + pc] ? pc0 : P[c + pc]);
                s = s + (S[c - 1] ? pc0 : P[c - 1]);
                s = s + (S[c + 1] ? pc0 : P[c + 1]);
                pn = 0.25f * (s - DIV[c]);
            }
            const float r = pn - pc0;
            mx = fmaxf(mx, fabsf(r));
            ss += r * r;
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    __shared__ float smx[8], sss[8];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    if (lane == 0) { smx[wp] = mx; sss[wp] = ss; }
    __syncthreads();
    if (wp == 0) {
        mx = lane < 8 ? smx[lane] : 0.f; ss = lane < 8 ? sss[lane] : 0.f;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            ss += __shfl_xor_sync(0xffffffffu, ss, o);
        }
        if (lane == 0) {
            atomicMax(reinterpret_cast<int*>(out + 2 * b), __float_as_int(mx));
            atomicAdd(out + 2 * b + 1, ss);
        }
    }
}

int launch_jacobi_residual_obst(const smk_grid_t* g, const float* div, const float* p, const uint8_t* solid, int64_t solid_stride,
                                float* out, cudaStream_t s)
{
    dim3 grid((g->w + 255) / 256, min(g->h, 64), g->batch);
    ProfScope prof_(SMK_PH_OTHER, s);
    k_jacobi_residual_obst<<<grid, 256, 0, s>>>(p, div, solid, out, g->h, g->w, g->pitch_c, g->stride_c, (long long)solid_stride);
    return check_launch("k_jacobi_residual_obst");
}

}  // namespace smk
