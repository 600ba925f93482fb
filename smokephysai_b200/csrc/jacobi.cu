// jacobi.cu -- a6: the Jacobi pressure sweeps of pressure_projection (navier_stokes.py:139-145).
//
//   K times:  p' = 0 ;  p'[i][j] = 0.25 * ((((p[i-1][j] + p[i+1][j]) + p[i][j-1]) + p[i][j+1]) - div[i][j])
//             for 1 <= i <= h-2, 1 <= j <= w-2 ;  p = p'
//
// Design (B200): the pressure tile lives in REGISTERS for T fused sweeps (temporal blocking).  A warp
// spans 128 columns (lane l owns columns 4l..4l+3 as a float4) and R consecutive rows; a CTA stacks NW
// warps, i.e. a (NW*R) x 128 tile.  Per sweep a thread needs, from outside its registers, only
//   - the column to its left / right: one __shfl_up / __shfl_down per row,
//   - the row above its first / below its last row: one float4 through a double-buffered shared-memory
//     halo line per warp, one __syncthreads per sweep.
// div is loop-invariant and stays in registers too.  HBM/L2 traffic per launch is one read of p and div
// and one write of p for T sweeps: 12/T B per cell-sweep (+ the overlap redundancy) instead of 12.
// Tiles overlap by T rows and HX = roundup4(T) columns (trapezoid scheme: the outer ring of a tile goes
// stale by one cell per sweep and is not stored); a grid that fits one tile needs no halo and does all K
// sweeps in a single launch.  The Dirichlet ring and everything outside the domain is handled with a
// per-cell multiplier (0.25 inside, 0 on the ring/outside), which costs no extra instruction.
//
// Bit-exactness: the association above is kept literally; 0.25*x == x*0.25 in IEEE; no FMA (-fmad=false).
//
// Kernels: k_jacobi (scalar strips), k_jacobi_packed (f32x2 row pairs, the default up to a few CTA waves) and
// k_jacobi_stream (persistent CTAs that prefetch their next tile with TMA tensor loads, the default from four CTA
// waves); launch_jacobi at the end of the file picks tile shape, sweeps per launch and kernel.
#include <cstdlib>
#include <cstring>
#include <cuda.h>
#include "common.cuh"
#include "jacobi_core.cuh"

namespace smk {

template <int R, int NW>
__global__ void __launch_bounds__(NW * 32, (NW * 32 <= 256) ? 2 : 1)
k_jacobi(const float* __restrict__ pin, float* __restrict__ pout, const float* __restrict__ div,
         const int h, const int w, const int pitch, const long long bstride,
         const int T, const int HX, const int ox, const int oy)
{
    pdl_prologue();
    __shared__ float4 halo[2][2][NW][32];          // [buffer][0: first row, 1: last row][warp][lane]

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * ox, y0 = blockIdx.y * oy;
    const int gj = x0 + lane * 4;
    const int gi0 = y0 + warp * R;
    const size_t boff = (size_t)blockIdx.z * (size_t)bstride;
    pin += boff; pout += boff; div += boff;

    float4 P[R], D[R];
    const bool colin = gj < pitch;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int gi = gi0 + r;
        if (colin && gi < h) {
            P[r] = *reinterpret_cast<const float4*>(pin + (size_t)gi * pitch + gj);
            D[r] = __ldg(reinterpret_cast<const float4*>(div + (size_t)gi * pitch + gj));
        } else {
            P[r] = make_float4(0.f, 0.f, 0.f, 0.f);
            D[r] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    const float cm0 = (gj + 0 >= 1 && gj + 0 <= w - 2) ? 0.25f : 0.f;
    const float cm1 = (gj + 1 >= 1 && gj + 1 <= w - 2) ? 0.25f : 0.f;
    const float cm2 = (gj + 2 >= 1 && gj + 2 <= w - 2) ? 0.25f : 0.f;
    const float cm3 = (gj + 3 >= 1 && gj + 3 <= w - 2) ? 0.25f : 0.f;
    const bool fast = (gi0 >= 1) && (gi0 + R - 1 <= h - 2);     // warp-uniform: no ring row in this warp
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);

    halo[0][0][warp][lane] = P[0];
    halo[0][1][warp][lane] = P[R - 1];
    __syncthreads();
    for (int s = 0; s < T; ++s) {
        const int buf = s & 1;
        const float4 up = warp > 0 ? halo[buf][1][warp - 1][lane] : zero4;
        const float4 dn = warp < NW - 1 ? halo[buf][0][warp + 1][lane] : zero4;
        float4* pf = (s + 1 < T) ? &halo[buf ^ 1][0][warp][lane] : nullptr;
        float4* pl = (s + 1 < T) ? &halo[buf ^ 1][1][warp][lane] : nullptr;
        if (fast) sweep_rows<R, true>(P, D, up, dn, cm0, cm1, cm2, cm3, gi0, h, pf, pl);
        else      sweep_rows<R, false>(P, D, up, dn, cm0, cm1, cm2, cm3, gi0, h, pf, pl);
        if (s + 1 < T) __syncthreads();
    }

    // store the part of the tile that is still exact after T sweeps
    const int vx0 = x0 + (blockIdx.x > 0 ? HX : 0);
    const int vx1 = (blockIdx.x + 1 < gridDim.x) ? x0 + 128 - HX : pitch;
    const int vy0 = y0 + (blockIdx.y > 0 ? T : 0);
    const int vy1 = (blockIdx.y + 1 < gridDim.y) ? y0 + NW * R - T : h;
    if (gj >= vx0 && gj < vx1 && gj < pitch) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int gi = gi0 + r;
            if (gi >= vy0 && gi < vy1 && gi < h)
                *reinterpret_cast<float4*>(pout + (size_t)gi * pitch + gj) = P[r];
        }
    }
}

// ---- masked variant: solid obstacles (DESIGN.md s5.7) -------------------------------------------------------------------
// The scalar strip of k_jacobi with a uint8 cell mask (non-zero = solid) of the pressure's pitch: per sweep a fluid interior cell
// computes 0.25 * ((((qN + qS) + qW) + qE) - div), qX the neighbour's p when that neighbour is fluid and the cell's own p when it
// is solid (Neumann ghost value); solid cells and the ring get +0.0.  With no solid cell this is the reference sweep bit for bit.
// The mask does not change between sweeps, so each lane reads it once (one 32-bit word = its four cells, per strip row and the
// rows above and below the strip, through L1) and folds it into 5 bits per cell: keep, and the four neighbours' solid flags.
// The tile, overlap and store are k_jacobi's, so every tile configuration and multi-launch chain of run_cfg applies unchanged.
__device__ __forceinline__ float4 stencil_row_obst(const float4 up, const float4 cur, const float4 dn, const float4 d, const unsigned f)
{
    const float left = __shfl_up_sync(0xffffffffu, cur.w, 1);
    const float right = __shfl_down_sync(0xffffffffu, cur.x, 1);
    const float c[4] = {cur.x, cur.y, cur.z, cur.w}, u[4] = {up.x, up.y, up.z, up.w}, dd[4] = {dn.x, dn.y, dn.z, dn.w};
    const float dv[4] = {d.x, d.y, d.z, d.w};
    float o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const unsigned bits = f >> (5 * k);
        const float qn = (bits & 2u) ? c[k] : u[k];
        const float qs = (bits & 4u) ? c[k] : dd[k];
        const float qw = (bits & 8u) ? c[k] : (k == 0 ? left : c[k - 1]);
        const float qe = (bits & 16u) ? c[k] : (k == 3 ? right : c[k + 1]);
        float s = qn + qs;
        s = s + qw;
        s = s + qe;
        s = s - dv[k];
        o[k] = (bits & 1u) ? 0.25f * s : 0.0f;
    }
    return make_float4(o[0], o[1], o[2], o[3]);
}

template <int R, int NW>
__global__ void __launch_bounds__(NW * 32, (NW * 32 <= 256) ? 2 : 1)
k_jacobi_obst(const float* __restrict__ pin, float* __restrict__ pout, const float* __restrict__ div,
              const uint8_t* __restrict__ solid, const long long sstride,
              const int h, const int w, const int pitch, const long long bstride,
              const int T, const int HX, const int ox, const int oy)
{
    pdl_prologue();
    __shared__ float4 halo[2][2][NW][32];          // [buffer][0: first row, 1: last row][warp][lane]

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * ox, y0 = blockIdx.y * oy;
    const int gj = x0 + lane * 4;
    const int gi0 = y0 + warp * R;
    const size_t boff = (size_t)blockIdx.z * (size_t)bstride;
    pin += boff; pout += boff; div += boff;
    solid += (size_t)blockIdx.z * (size_t)sstride;

    float4 P[R], D[R];
    const bool colin = gj < pitch;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int gi = gi0 + r;
        if (colin && gi < h) {
            P[r] = *reinterpret_cast<const float4*>(pin + (size_t)gi * pitch + gj);
            D[r] = __ldg(reinterpret_cast<const float4*>(div + (size_t)gi * pitch + gj));
        } else {
            P[r] = make_float4(0.f, 0.f, 0.f, 0.f);
            D[r] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    // cell flags: bit 5k keep (fluid and interior), 5k+1 .. 5k+4 the N, S, W, E neighbour is solid.  Cells outside the grid read
    // as fluid; they are never kept, and an interior cell's neighbours are all inside.
    unsigned F[R];
    {
        auto mrow = [&](const int gi) -> unsigned {
            return (colin && gi >= 0 && gi < h) ? __ldg(reinterpret_cast<const unsigned*>(solid + (size_t)gi * pitch + gj)) : 0u;
        };
        unsigned above = mrow(gi0 - 1), me = mrow(gi0);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const unsigned below = mrow(gi0 + r + 1);
            const unsigned lw = __shfl_up_sync(0xffffffffu, me, 1), rw = __shfl_down_sync(0xffffffffu, me, 1);
            const int gi = gi0 + r;
            const bool rowin = gi >= 1 && gi <= h - 2;
            unsigned f = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const bool keep = rowin && gj + k >= 1 && gj + k <= w - 2 && ((me >> (8 * k)) & 0xffu) == 0;
                const bool sn = ((above >> (8 * k)) & 0xffu) != 0, ss = ((below >> (8 * k)) & 0xffu) != 0;
                const bool sw = (k == 0 ? (lw >> 24) : (me >> (8 * (k - 1)))) & 0xffu;
                const bool se = (k == 3 ? rw : (me >> (8 * (k + 1)))) & 0xffu;
                f |= ((keep ? 1u : 0u) | (sn ? 2u : 0u) | (ss ? 4u : 0u) | (sw ? 8u : 0u) | (se ? 16u : 0u)) << (5 * k);
            }
            F[r] = f;
            above = me; me = below;
        }
    }
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);

    halo[0][0][warp][lane] = P[0];
    halo[0][1][warp][lane] = P[R - 1];
    __syncthreads();
    for (int s = 0; s < T; ++s) {
        const int buf = s & 1;
        float4 prev = warp > 0 ? halo[buf][1][warp - 1][lane] : zero4;
        const float4 dn = warp < NW - 1 ? halo[buf][0][warp + 1][lane] : zero4;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float4 cur = P[r];
            P[r] = stencil_row_obst(prev, cur, r + 1 < R ? P[r + 1] : dn, D[r], F[r]);
            prev = cur;
        }
        if (s + 1 < T) {
            halo[buf ^ 1][0][warp][lane] = P[0];
            halo[buf ^ 1][1][warp][lane] = P[R - 1];
            __syncthreads();
        }
    }

    const int vx0 = x0 + (blockIdx.x > 0 ? HX : 0);
    const int vx1 = (blockIdx.x + 1 < gridDim.x) ? x0 + 128 - HX : pitch;
    const int vy0 = y0 + (blockIdx.y > 0 ? T : 0);
    const int vy1 = (blockIdx.y + 1 < gridDim.y) ? y0 + NW * R - T : h;
    if (gj >= vx0 && gj < vx1 && gj < pitch) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int gi = gi0 + r;
            if (gi >= vy0 && gi < vy1 && gi < h)
                *reinterpret_cast<float4*>(pout + (size_t)gi * pitch + gj) = P[r];
        }
    }
}

// Packed variant (see jacobi_core.cuh): add.f32x2 / mul.f32x2 halve the FP32 issue slots of a sweep.  The strip is
// always 8 rows per thread (R == 8); sweeps ping-pong between two register sets, two sweeps per loop trip.
template <int R, int NW, int PMASK>
__global__ void __launch_bounds__(NW * 32, (NW * 32 <= 256) ? 2 : 1)
k_jacobi_packed(const float* __restrict__ pin, float* __restrict__ pout, const float* __restrict__ div,
                const int h, const int w, const int pitch, const long long bstride,
                const int T, const int HX, const int ox, const int oy)
{
    pdl_prologue();
    static_assert(R == 8, "the packed strip pairs row r with row r + 4");
    __shared__ float4 halo[2][2][NW][32];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * ox, y0 = blockIdx.y * oy;
    const int gj = x0 + lane * 4;
    const int gi0 = y0 + warp * R;
    const size_t boff = (size_t)blockIdx.z * (size_t)bstride;
    pin += boff; pout += boff; div += boff;

    PackedStrip A, B, ND;
    const bool colin = gj < pitch;
    unsigned ringmask = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int gi = gi0 + r;
        float4 p4 = make_float4(0.f, 0.f, 0.f, 0.f), d4 = p4;
        if (colin && gi < h) {
            p4 = *reinterpret_cast<const float4*>(pin + (size_t)gi * pitch + gj);
            d4 = __ldg(reinterpret_cast<const float4*>(div + (size_t)gi * pitch + gj));
        }
        if (gi < 1 || gi > h - 2) ringmask |= 1u << r;
        packed_set_row(A, r, p4);
        packed_set_row(ND, r, make_float4(-d4.x, -d4.y, -d4.z, -d4.w));
    }
    float2 M[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const float m = (gj + c >= 1 && gj + c <= w - 2) ? 0.25f : 0.f;
        M[c] = make_float2(m, m);
    }
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);

    halo[0][0][warp][lane] = packed_row(A, 0);
    halo[0][1][warp][lane] = packed_row(A, 7);
    __syncthreads();
    int s = 0;
    for (; s + 1 < T; s += 2) {            // s is even here: sweep s reads halo[0], sweep s+1 reads halo[1]
        {
            const float4 up = warp > 0 ? halo[0][1][warp - 1][lane] : zero4;
            const float4 dn = warp < NW - 1 ? halo[0][0][warp + 1][lane] : zero4;
            sweep_packed<PMASK, 0, false, 1>(A, B, ND, up, dn, M, ringmask, &halo[1][0][warp][lane], &halo[1][1][warp][lane]);
            __syncthreads();
        }
        {
            const float4 up = warp > 0 ? halo[1][1][warp - 1][lane] : zero4;
            const float4 dn = warp < NW - 1 ? halo[1][0][warp + 1][lane] : zero4;
            const bool more = s + 2 < T;
            sweep_packed<PMASK, 0, false, 1>(B, A, ND, up, dn, M, ringmask, more ? &halo[0][0][warp][lane] : nullptr, more ? &halo[0][1][warp][lane] : nullptr);
            if (more) __syncthreads();
        }
    }
    if (s < T) {                           // odd T: one more sweep, then move the result back into A
        const float4 up = warp > 0 ? halo[0][1][warp - 1][lane] : zero4;
        const float4 dn = warp < NW - 1 ? halo[0][0][warp + 1][lane] : zero4;
        sweep_packed<PMASK, 0, false, 1>(A, B, ND, up, dn, M, ringmask, nullptr, nullptr);
        A = B;
    }

    const int vx0 = x0 + (blockIdx.x > 0 ? HX : 0);
    const int vx1 = (blockIdx.x + 1 < gridDim.x) ? x0 + 128 - HX : pitch;
    const int vy0 = y0 + (blockIdx.y > 0 ? T : 0);
    const int vy1 = (blockIdx.y + 1 < gridDim.y) ? y0 + NW * R - T : h;
    if (gj >= vx0 && gj < vx1 && gj < pitch) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int gi = gi0 + r;
            if (gi >= vy0 && gi < vy1 && gi < h)
                *reinterpret_cast<float4*>(pout + (size_t)gi * pitch + gj) = packed_row(A, r);
        }
    }
}

// ---- streaming variant for grids of many tiles -------------------------------------------------------------------
// One persistent CTA per SM walks over 128 x 128 tiles; while it sweeps the tile it holds in registers, the next
// tile's pressure and divergence (128 KB) are already on their way into shared memory, so the tile load overlaps
// the arithmetic without needing a second resident CTA (k_jacobi_packed gets that overlap from two 64 x 128 CTAs
// per SM, at the price of keeping only 44 of 64 rows per launch of 10 sweeps; here 108 of 128 survive).
// Two staging engines (template parameter TMA):
//   TMA   -- two cp.async.bulk.tensor.3d loads per tile (pressure, divergence: a 128 x 128 x 1 box of a (pitch, h, batch)
//            tensor map, out-of-domain elements zero-filled by the TMA unit), issued by one thread after the CTA barrier
//            that follows the strip reads and completed on one mbarrier.  The staging costs the LSU / MIO pipe nothing
//            while the sweeps run.  (One cp.async.bulk per tile ROW -- 256 UBLKCP per tile -- was tried first: the issuing
//            lanes stall on every copy and the tile took 4.7 us of overhead against 3.1 us with LDGSTS.)
//   !TMA  -- 16-byte cp.async (LDGSTS) issued by every thread for exactly the 8 x 4 strip it will consume (no CTA
//            barrier needed, zero-fill by src-size 0); 8192 LDGSTS per tile go through the same pipe as the sweeps'
//            shuffles and halo LDS/STS.
// shared memory of a CTA of NW warps (tile = 8 NW x 128): staged pressure, staged divergence, halo lines, mbarrier, arguments
__host__ __device__ constexpr size_t js_bar_off(const int NW) { return (size_t)2 * 8 * NW * 128 * 4 + sizeof(float4) * 2 * 2 * NW * 32; }
__host__ __device__ constexpr size_t js_out_off(const int NW) { return js_bar_off(NW) + 128; }      // mbarrier (16 B), arguments (<= 112 B)
// TMA kernels also stage the rows and columns of a tile that survive the launch -- (8 NW - 2 T) x (128 - 2 HX), dense -- for one
// cp.async.bulk.tensor store per tile
__host__ __device__ constexpr size_t js_smem_bytes(const int NW, const int T = 0, const int HX = 0, const bool tma = false)
{
    return js_out_off(NW) + (tma ? (size_t)(8 * NW - 2 * T) * (128 - 2 * HX) * 4 : 0);
}

__device__ __forceinline__ void js_cp_async16_zfill(float* smem_dst, const float* gmem_src, const unsigned src_bytes)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void js_tma_tile(float* smem_dst, const CUtensorMap* map, const int x, const int y, const int z, unsigned long long* bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 :: "r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(map), "r"(x), "r"(y), "r"(z),
                    "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void js_mbar_wait(unsigned long long* bar, const unsigned parity)
{
    unsigned done = 0;
    while (!done)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}

#ifndef SMK_JS_ELEM
#define SMK_JS_ELEM unsigned long long
#endif
typedef SMK_JS_ELEM JsElem;        // strip element of the streaming kernel: a pinned 64-bit pair (see jacobi_core.cuh)

struct JsArgs {
    const float* pin; float* pout; const float* div;
    int h, w, pitch; long long bstride;
    int T, HX, ox, oy, nx, ny, ntot;
};
struct JsTile { int bx, by, bz; };
__device__ __forceinline__ JsTile js_coords(const JsArgs& a, const int t)
{
    JsTile c;
    c.bx = t % a.nx; c.by = (t / a.nx) % a.ny; c.bz = t / (a.nx * a.ny);
    return c;
}

// tile c -> shared memory (asynchronously)
template <bool TMA, int NW>
__device__ __forceinline__ void js_stage(const JsArgs& a, const CUtensorMap* mp, const CUtensorMap* md, float* js_smem, const JsTile c)
{
    constexpr int R = 8, TH = R * NW;
    float (*sp)[128] = reinterpret_cast<float (*)[128]>(js_smem);                       // staged pressure tile
    float (*sdv)[128] = reinterpret_cast<float (*)[128]>(js_smem + TH * 128);             // staged divergence tile
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(js_smem) + js_bar_off(NW));
    const int x0 = c.bx * a.ox, y0 = c.by * a.oy;
    if (TMA) {
        if (threadIdx.x == 0) {
            // the strip reads of the previous tile (generic proxy, ordered before this point by the CTA barrier) precede the
            // TMA writes (async proxy) into the same buffer
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                         :: "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(2u * (unsigned)TH * 128u * 4u) : "memory");
            js_tma_tile(&sp[0][0], mp, x0, y0, c.bz, bar);
            js_tma_tile(&sdv[0][0], md, x0, y0, c.bz, bar);
        }
    } else {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const size_t boff = (size_t)c.bz * (size_t)a.bstride;
        const int gj = x0 + lane * 4, gi0 = y0 + warp * R;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int gi = gi0 + r;
            const bool ok = gj < a.pitch && gi < a.h;
            const size_t off = ok ? boff + (size_t)gi * a.pitch + gj : 0;
            js_cp_async16_zfill(&sp[warp * R + r][4 * lane], a.pin + off, ok ? 16u : 0u);
            js_cp_async16_zfill(&sdv[warp * R + r][4 * lane], a.div + off, ok ? 16u : 0u);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
}

// One tile: wait for its staged copy, move the thread's strip to registers, start the copy of the next tile, T sweeps,
// store.  Deliberately NOT inlined into the tile loop, and with 64-bit strip elements: compiled inside the loop with
// float2 elements, ptxas kept the f32x2 operands in unpaired registers and predicated the ring rows with selects
// (52 MOV + 36 FSEL per sweep and warp, +37 % instructions: profiles/r01j_*).
template <int PMASK, bool TMA, bool RING, class E, int NW>
__device__ __noinline__ void js_tile(const JsArgs& a, const CUtensorMap* mp, const CUtensorMap* md, const CUtensorMap* mo, float* js_smem,
                                     const JsTile c, const JsTile cnext, const bool has_next, const unsigned parity)
{
    constexpr int R = 8, TH = R * NW;
    float (*sp)[128] = reinterpret_cast<float (*)[128]>(js_smem);
    float (*sdv)[128] = reinterpret_cast<float (*)[128]>(js_smem + TH * 128);
    float4 (*halo)[2][NW][32] = reinterpret_cast<float4 (*)[2][NW][32]>(js_smem + 2 * TH * 128);
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(js_smem) + js_bar_off(NW));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const int T = a.T;
    const int x0 = c.bx * a.ox, y0 = c.by * a.oy;
    const int gj = x0 + lane * 4, gi0 = y0 + warp * R;

    if (TMA) js_mbar_wait(bar, parity);
    else asm volatile("cp.async.wait_group 0;" ::: "memory");
    PackedStripT<E> A, B, ND;
    unsigned ringmask = 0;
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
        const float4 pl = *reinterpret_cast<const float4*>(&sp[warp * R + rr][4 * lane]);
        const float4 ph = *reinterpret_cast<const float4*>(&sp[warp * R + rr + 4][4 * lane]);
        const float4 dl = *reinterpret_cast<const float4*>(&sdv[warp * R + rr][4 * lane]);
        const float4 dh = *reinterpret_cast<const float4*>(&sdv[warp * R + rr + 4][4 * lane]);
        if (RING && (gi0 + rr < 1 || gi0 + rr > a.h - 2)) ringmask |= 1u << rr;
        if (RING && (gi0 + rr + 4 < 1 || gi0 + rr + 4 > a.h - 2)) ringmask |= 16u << rr;
        packed_set_rows(A, rr, pl, ph);
        packed_set_rows(ND, rr, make_float4(-dl.x, -dl.y, -dl.z, -dl.w), make_float4(-dh.x, -dh.y, -dh.z, -dh.w));
    }
    E M[4];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        const float m = (gj + cc >= 1 && gj + cc <= a.w - 2) ? 0.25f : 0.f;
        M[cc] = pe_make<E>(make_float2(m, m));
    }
    halo[0][0][warp][lane] = packed_row(A, 0);
    halo[0][1][warp][lane] = packed_row(A, 7);
    // the staged strip is in registers (the negations above consumed every load): refill the buffer with the next tile.
    // LDGSTS: a thread only overwrites its own strip, no barrier needed; the TMA loads overwrite the whole buffer, so they
    // are issued after the barrier that every thread passes once its strip is read.
    if (!TMA && has_next) js_stage<false, NW>(a, mp, md, js_smem, cnext);
    // the bulk store of the previous tile has read the output staging buffer before anybody passes the barrier below
    if (TMA && threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
    if (TMA && has_next) js_stage<true, NW>(a, mp, md, js_smem, cnext);
    int s = 0;
    for (; s + 1 < T; s += 2) {            // s is even here: sweep s reads halo[0], sweep s+1 reads halo[1]
        {
            const float4 up = warp > 0 ? halo[0][1][warp - 1][lane] : zero4;
            const float4 dn = warp < NW - 1 ? halo[0][0][warp + 1][lane] : zero4;
            sweep_packed<PMASK, 0, false, 1>(A, B, ND, up, dn, M, ringmask, &halo[1][0][warp][lane], &halo[1][1][warp][lane]);
            __syncthreads();
        }
        {
            const float4 up = warp > 0 ? halo[1][1][warp - 1][lane] : zero4;
            const float4 dn = warp < NW - 1 ? halo[1][0][warp + 1][lane] : zero4;
            const bool more = s + 2 < T;
            sweep_packed<PMASK, 0, false, 1>(B, A, ND, up, dn, M, ringmask, more ? &halo[0][0][warp][lane] : nullptr, more ? &halo[0][1][warp][lane] : nullptr);
            if (more) __syncthreads();
        }
    }
    if (s < T) {                           // odd T: one more sweep, then move the result back into A
        const float4 up = warp > 0 ? halo[0][1][warp - 1][lane] : zero4;
        const float4 dn = warp < NW - 1 ? halo[0][0][warp + 1][lane] : zero4;
        sweep_packed<PMASK, 0, false, 1>(A, B, ND, up, dn, M, ringmask, nullptr, nullptr);
        A = B;
    }

    // A tile with neighbours on all four sides keeps the box [T, TH - T) x [HX, 128 - HX): the TMA kernels write it to a dense
    // staging buffer (one STS.128 per surviving strip row) and ONE thread hands it to the TMA unit after the barrier that ends
    // the tile -- no address arithmetic, predicates or 16-byte global stores in the 512 threads.  Tiles on the rim of the
    // tiling keep more (up to the edge of the grid) and store their strips directly.
    const bool boxed = TMA && c.bx > 0 && c.bx + 1 < a.nx && c.by > 0 && c.by + 1 < a.ny;
    if (boxed) {
        const int bw = 128 - 2 * a.HX;                                                  // box width (floats), a multiple of 4
        float* so = reinterpret_cast<float*>(reinterpret_cast<char*>(js_smem) + js_out_off(NW));
        const int cx = 4 * lane - a.HX;
        if (cx >= 0 && cx < bw) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int ry = warp * R + r - T;
                if (ry >= 0 && ry < TH - 2 * T) *reinterpret_cast<float4*>(so + ry * bw + cx) = packed_row(A, r);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");               // generic-proxy writes -> visible to the TMA unit
    } else {
        const int vx0 = x0 + (c.bx > 0 ? a.HX : 0);
        const int vx1 = (c.bx + 1 < a.nx) ? x0 + 128 - a.HX : a.pitch;
        const int vy0 = y0 + (c.by > 0 ? T : 0);
        const int vy1 = (c.by + 1 < a.ny) ? y0 + NW * R - T : a.h;
        if (gj >= vx0 && gj < vx1 && gj < a.pitch) {
            float* out = a.pout + (size_t)c.bz * (size_t)a.bstride;
    #pragma unroll
            for (int r = 0; r < R; ++r) {
                const int gi = gi0 + r;
                if (gi >= vy0 && gi < vy1 && gi < a.h)
                    *reinterpret_cast<float4*>(out + (size_t)gi * a.pitch + gj) = packed_row(A, r);
            }
        }
    }
    __syncthreads();                       // the halo lines are reused by the next tile; the staged box is complete
    if (boxed && threadIdx.x == 0) {
        const float* so = reinterpret_cast<const float*>(reinterpret_cast<char*>(js_smem) + js_out_off(NW));
        asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];"
                     :: "l"(mo), "r"(x0 + a.HX), "r"(y0 + T), "r"(c.bz), "r"((unsigned)__cvta_generic_to_shared(so)) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
}

template <int PMASK, bool TMA, int NW>
__global__ void __launch_bounds__(NW * 32, (NW * 32 <= 256) ? 2 : 1)
k_jacobi_stream(const __grid_constant__ JsArgs ga, const __grid_constant__ CUtensorMap mp, const __grid_constant__ CUtensorMap md,
                const __grid_constant__ CUtensorMap mo)
{
    pdl_prologue();
    extern __shared__ __align__(128) float js_smem[];
    static_assert(sizeof(JsArgs) <= 96, "js_smem_bytes reserves 96 bytes for the argument copy");
    // js_tile is a separate function: it reads the arguments from shared memory (generic loads of the kernel parameters
    // cost it a long-scoreboard stall per field and tile: 14 % of the samples in profiles/r01k_*)
    JsArgs& a = *reinterpret_cast<JsArgs*>(reinterpret_cast<char*>(js_smem) + js_bar_off(NW) + 16);
    if (threadIdx.x == 0) {
        a = ga;
        if (TMA) {
            unsigned long long* bar = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(js_smem) + js_bar_off(NW));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    }
    __syncthreads();
    int t = blockIdx.x;
    unsigned parity = 0;
    if (t >= ga.ntot) return;
    JsTile c = js_coords(ga, t);
    js_stage<TMA, NW>(ga, &mp, &md, js_smem, c);
    // the next tile of this CTA is gridDim.x further along the (bx fastest, by, bz) order: stepped, not divided out per tile
    // (the three divisions by run-time values were 3.8 % of the kernel's instructions: profiles/r02j_*)
    const int step_y = (int)gridDim.x / ga.nx, step_x = (int)gridDim.x - step_y * ga.nx;
    for (; t < ga.ntot; t += gridDim.x, parity ^= 1u) {
        const bool has_next = t + (int)gridDim.x < ga.ntot;
        JsTile cnext = c;
        if (has_next) {
            cnext.bx += step_x; cnext.by += step_y;
            if (cnext.bx >= ga.nx) { cnext.bx -= ga.nx; ++cnext.by; }
            while (cnext.by >= ga.ny) { cnext.by -= ga.ny; ++cnext.bz; }
        }
        // tiles in the first / last tile row of a simulation hold rows of the Dirichlet ring (or rows outside the grid);
        // every other tile runs the sweeps without the ring-row tests
        const bool ring = c.by == 0 || c.by * ga.oy + 8 * NW > ga.h - 1;
        if (ring) js_tile<PMASK, TMA, true, JsElem, NW>(a, &mp, &md, &mo, js_smem, c, cnext, has_next, parity);
        else      js_tile<PMASK, TMA, false, JsElem, NW>(a, &mp, &md, &mo, js_smem, c, cnext, has_next, parity);
        c = cnext;
    }
    // the staging buffer must outlive the last bulk store's reads, and its writes complete before the grid counts as finished
    if (TMA && threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

static int ntiles(int n, int tile, int halo)
{
    // first tile starts at 0, tiles advance by tile-2*halo, last tile must reach n
    if (n <= tile) return 1;
    const int adv = tile - 2 * halo;
    return (n - tile + adv - 1) / adv + 1;
}

// Sweeps per launch for an overlapped-tile run, from a cost model fitted on a B200 (tools/tune_jacobi.py):
//   time = launches * 2.3 us  +  sum over launches of  waves * (3 us + T * 0.56 us)        (128 x 128 tiles, 1 CTA / SM)
// Small grids want the largest T that still fits one wave of CTAs; large grids settle near T = 12, where the
// halo redundancy ((128 / (128 - 2 HX)) * (128 / (128 - 2 T))) starts to outweigh the saved loads.
static int pick_T(const smk_grid_t* g, int K, int TH, int tmax, int sms)
{
    double best = 1e30; int bestT = 1;
    for (int nl = 1; nl <= K; ++nl) {
        const int T = (K + nl - 1) / nl;
        if (T > tmax) continue;
        double cost = 2.3 * nl;
        int left = K;
        for (int l = 0; l < nl; ++l) {
            const int t = (left + (nl - l) - 1) / (nl - l);       // balanced split
            left -= t;
            const int HX = (t + 3) & ~3;
            const long ctas = (long)ntiles(g->w, 128, HX) * ntiles(g->h, TH, t) * g->batch;
            const long waves = (ctas + sms - 1) / sms;
            cost += waves * (3.0 + 0.56 * t);
        }
        if (cost < best) { best = cost; bestT = T; }
        if (T == 1) break;
    }
    return bestT;
}

// 0: scalar in-place kernel (k_jacobi); else the ping-pong kernel (k_jacobi_packed) with this mask of row pairs
// (bit rr) on f32x2 arithmetic.  Default 6: measured fastest on B200 (tools/micro/jacobi_probe.cu: 886 cycles per
// sweep of a 128 x 128 tile against 928 all-scalar, 920 all-packed; the in-place k_jacobi needs ~1130).
static int use_packed()
{
    const int v = env().jacobi_packed;
    return v == SMK_ENV_UNSET ? 6 : v;
}

static int sm_count();

// Streaming kernel: SMK_JACOBI_STREAM = 0 (off) / 1 (LDGSTS staging) / 2 (TMA staging) forces, otherwise launch_jacobi picks it
// for grids of many CTA waves.  Measured on B200 (tools/tune_jacobi_stream.py, K = 20, T = 10, us per 20 sweeps):
//                      two CTAs per SM   128 x 128   stream LDGSTS   stream TMA   stream TMA, 64 x 128 x 2
//   8192 x 8192             644             711          669            576              635
//   4096 x 4096             178             195          193            168              177
//   1024 x 8192 (slab)       96             111          110             99               93
//   2048 x 2048              54              50           58             54               54
// A tile still costs 2.3 us on top of its sweeps (0.48 us each).
static int stream_env()
{
    const int v = env().jacobi_stream;
    if (v != SMK_ENV_UNSET) return use_packed() != 0 ? v : 0;
    return -1;
}

constexpr int SMK_ENOTMA = -1000;          // internal: no tensor map could be built, the caller falls back to k_jacobi_packed
// cuTensorMapEncodeTiled through the runtime's driver entry point (nothing of libcuda is linked)
typedef CUresult (*js_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static js_encode_fn js_encoder()
{
    static js_encode_fn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (js_encode_fn)p;
    }
    return fn;
}
// a (pitch, rows, batch) fp32 tensor accessed in box_cols x box_rows x 1 boxes; elements outside it are zero-filled on a load and
// dropped on a store.  false: no tensor map could be encoded (the caller keeps its non-TMA path).          (common.cuh)
bool tma_map_3d(void* map128, const float* base, int pitch, int rows, int batch, int64_t batch_stride, int box_rows, int box_cols)
{
    js_encode_fn enc = js_encoder();
    if (!enc || pitch < 4 || (pitch & 3) || rows < 1 || box_cols > 256 || box_rows > 256 || (box_cols & 3)) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)pitch, (cuuint64_t)rows, (cuuint64_t)(batch > 0 ? batch : 1)};
    // the stride of the batch dimension is not used when there is one simulation, but it has to be a valid one
    const cuuint64_t strides[2] = {(cuuint64_t)pitch * 4u, (batch > 1 ? (cuuint64_t)batch_stride : (cuuint64_t)pitch * (cuuint64_t)rows) * 4u};
    const cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1}, estr[3] = {1, 1, 1};
    const CUresult r = enc(reinterpret_cast<CUtensorMap*>(map128), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}
static int js_make_map(CUtensorMap* m, const smk_grid_t* g, const float* base, const int box_rows, const int box_cols = 128)
{
    return tma_map_3d(m, base, g->pitch_c, g->h, g->batch, g->stride_c, box_rows, box_cols) ? SMK_OK : SMK_ENOTMA;
}

template <int NW>
static int launch_stream(const smk_grid_t* g, const float* src, float* dst, const float* div, int t, int HX, int nx, int ny, int mode, cudaStream_t s)
{
    constexpr size_t SMEM_MAX = js_smem_bytes(NW, 1, 4, true);                      // the shallowest launch keeps the largest box
    const size_t SMEM = js_smem_bytes(NW, t, HX, mode != 1);
    constexpr int PER_SM = (NW * 32 <= 256) ? 2 : 1;
    static bool attr_set[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 63;
    if (!attr_set[dev] || dev == 63) {
        cudaError_t e = cudaFuncSetAttribute(k_jacobi_stream<6, false, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)js_smem_bytes(NW));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_jacobi_stream<6, true, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX);
        if (e != cudaSuccess) return fail((int)e, "k_jacobi_stream: cannot opt in to %zu B of shared memory: %s", SMEM_MAX, cudaGetErrorString(e));
        attr_set[dev] = true;
    }
    const long ntot = (long)nx * ny * g->batch;
    const long resident = (long)PER_SM * sm_count();
    const int ctas = (int)(ntot < resident ? ntot : resident);
    JsArgs a;
    a.pin = src; a.pout = dst; a.div = div; a.h = g->h; a.w = g->w; a.pitch = g->pitch_c; a.bstride = (long long)g->stride_c;
    a.T = t; a.HX = HX; a.ox = 128 - 2 * HX; a.oy = 8 * NW - 2 * t; a.nx = nx; a.ny = ny; a.ntot = (int)ntot;
    CUtensorMap mp, md, mo;
    memset(&mp, 0, sizeof mp); memset(&md, 0, sizeof md); memset(&mo, 0, sizeof mo);
    if (mode != 1) {
        int rc = js_make_map(&mp, g, src, 8 * NW);
        if (rc == SMK_OK) rc = js_make_map(&md, g, div, 8 * NW);
        if (rc == SMK_OK) rc = js_make_map(&mo, g, dst, 8 * NW - 2 * t, 128 - 2 * HX);
        if (rc != SMK_OK) return rc;
    }
    ProfScope prof_(SMK_PH_JACOBI, s);
    if (mode == 1) launch_chain(k_jacobi_stream<6, false, NW>, dim3(ctas), dim3(NW * 32), SMEM, s, a, mp, md, mo);
    else           launch_chain(k_jacobi_stream<6, true, NW>, dim3(ctas), dim3(NW * 32), SMEM, s, a, mp, md, mo);
    return check_launch("k_jacobi_stream");
}

// solid != NULL: every launch is k_jacobi_obst (the packed and streaming kernels have no masked variant)
template <int R, int NW>
static int run_cfg(const smk_grid_t* g, const float* div, float* a, float* b, int K, int T, int* in_scratch, cudaStream_t s, const int stream = 0,
                   const uint8_t* solid = nullptr, const int64_t solid_stride = 0)
{
    const int TH = R * NW;
    const bool whole = (g->h <= TH) && (g->w <= 128);
    float* src = a; float* dst = b;
    int left = K;
    int nl = whole ? 1 : (K + T - 1) / T;
    for (int l = 0; l < nl; ++l) {
        const int t = (left + (nl - l) - 1) / (nl - l);           // K sweeps split evenly over the launches
        left -= t;
        const int HX = (t + 3) & ~3;
        const int nx = ntiles(g->w, 128, HX), ny = ntiles(g->h, TH, t);
        dim3 grid(nx, ny, g->batch);
        int rc;
        int stream_mode = (R == 8 && (NW == 16 || NW == 8) && !solid) ? stream : 0;
        if (stream_mode == 2 && (g->pitch_c < 128 || g->h < TH)) stream_mode = 1;       // the TMA box is 128 x TH: keep it inside the tensor
        if (stream_mode) {
            rc = launch_stream<(R == 8 && NW == 8) ? 8 : 16>(g, src, dst, div, t, HX, nx, ny, stream_mode, s);
            if (rc == SMK_OK) {
                float* tmp = src; src = dst; dst = tmp;
                continue;
            }
            if (rc != SMK_ENOTMA) return rc;             // no tensor map for this grid: the non-streaming kernel below gives the same result
        }
        {
            ProfScope prof_(SMK_PH_JACOBI, s);
#define SMK_PACKED_CASE(M) case M: launch_chain(k_jacobi_packed<8, NW, M>, grid, dim3(NW * 32), 0, s, src, dst, div, g->h, g->w, g->pitch_c, \
                                                           (long long)g->stride_c, t, HX, 128 - 2 * HX, TH - 2 * t); break;
            if (solid)
                launch_chain(k_jacobi_obst<R, NW>, grid, dim3(NW * 32), 0, s, src, dst, div, solid, (long long)solid_stride, g->h, g->w,
                             g->pitch_c, (long long)g->stride_c, t, HX, 128 - 2 * HX, TH - 2 * t);
            else if (R == 8 && use_packed()) {
                switch (use_packed()) {
                    SMK_PACKED_CASE(6) SMK_PACKED_CASE(9) SMK_PACKED_CASE(2) SMK_PACKED_CASE(7) SMK_PACKED_CASE(16)
                    default: launch_chain(k_jacobi_packed<8, NW, 15>, grid, dim3(NW * 32), 0, s, src, dst, div, g->h, g->w, g->pitch_c,
                                                           (long long)g->stride_c, t, HX, 128 - 2 * HX, TH - 2 * t);
                }
            } else
                launch_chain(k_jacobi<R, NW>, grid, dim3(NW * 32), 0, s, src, dst, div, g->h, g->w, g->pitch_c, (long long)g->stride_c,
                                                         t, HX, 128 - 2 * HX, TH - 2 * t);
            rc = check_launch(solid ? "k_jacobi_obst" : "k_jacobi");
        }
        if (rc != SMK_OK) return rc;
        float* tmp = src; src = dst; dst = tmp;
    }
    *in_scratch = (src == b) ? 1 : 0;
    return SMK_OK;
}

static int sm_count()
{
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    }
    return n;
}

int launch_jacobi(const smk_grid_t* g, const float* div, float* p, float* scratch, int K, int T, int* in_scratch, cudaStream_t s,
                  const uint8_t* solid, int64_t solid_stride)
{
    *in_scratch = 0;
    if (K <= 0) return SMK_OK;
    if (g->batch > 65535) return fail(SMK_EUNSUPPORTED, "smk_jacobi: batch %d > 65535", g->batch);
    const uint8_t* S = solid;
    const int64_t ss = solid_stride;
    if (g->w <= 128 && g->h <= 32) return run_cfg<4, 8>(g, div, p, scratch, K, T > 0 ? T : 8, in_scratch, s, 0, S, ss);
    if (g->w <= 128 && g->h <= 64) return run_cfg<8, 8>(g, div, p, scratch, K, T > 0 ? T : 8, in_scratch, s, 0, S, ss);
    if (g->w <= 128 && g->h <= 128) return run_cfg<8, 16>(g, div, p, scratch, K, T > 0 ? T : 8, in_scratch, s, 0, S, ss);
    // large grids: overlapped tiles.  T must leave a positive advance in both directions.
    int tile = 0;                                   // 0 auto, 1: 64 x 128 (8 warps), 2: 128 x 128 (16 warps), 3: 64 x 128 (16 warps)
    if (env().jacobi_tile != SMK_ENV_UNSET) tile = env().jacobi_tile;
    int stream = S ? 0 : stream_env();              // -1 auto, 0 off, 1 LDGSTS, 2 TMA (k_jacobi_stream)
    if (tile == 0) {
        // Many waves of CTAs (>= 4 per SM: 4096^2, or a 1/8 slab of 8192^2): overlap one tile's load / store with another's sweeps.
        // Without the TMA kernel: 64 x 128 tiles at two CTAs per SM (7-8 % faster than 128 x 128 tiles at 4096^2 and 8192^2, equal
        // at 2048^2: tools/tune_jacobi.py).  With it: persistent CTAs on 128 x 128 tiles that prefetch their next tile and store by
        // TMA, from 8 tile rows on (tools/tune_jacobi_stream.py after the TMA store, us per 20 sweeps of an h x 8192 slab, streaming
        // 128 x 128 / streaming 64 x 128 x 2 / plain 64 x 128 x 2: h = 560: 51 / 59 / 48, 1072: 93 / 95 / 92, 1600: 129 / 131 / 135,
        // 2096: 155 / 168 / 174); shorter grids keep the plain two-CTAs-per-SM kernel.
        const long ctas128 = (long)ntiles(g->w, 128, 12) * ntiles(g->h, 128, 10) * g->batch;
        if (ctas128 >= 4L * sm_count()) {
            tile = 1;
            if (stream < 0 && use_packed() != 0 && g->pitch_c >= 128 && js_encoder() != nullptr && ntiles(g->h, 128, 10) >= 8) {
                stream = 2;
                tile = 2;
            }
        }
    }
    if (stream < 0) stream = 0;
    if (T <= 0) T = (tile == 1 || tile == 3 || stream != 0) ? 10 : pick_T(g, K, 128, 24, sm_count());
    if (tile == 1) return run_cfg<8, 8>(g, div, p, scratch, K, min(T, 12), in_scratch, s, stream, S, ss);
    if (tile == 3) return run_cfg<4, 16>(g, div, p, scratch, K, min(T, 12), in_scratch, s, 0, S, ss);
    return run_cfg<8, 16>(g, div, p, scratch, K, min(T, stream != 0 ? 12 : 24), in_scratch, s, stream, S, ss);
}

}  // namespace smk
