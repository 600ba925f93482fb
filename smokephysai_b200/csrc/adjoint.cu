// adjoint.cu -- reverse mode of one step() (navier_stokes.py:151-173): the adjoint (transpose) of every phase, for
// smokephysai_b200.autodiff.  The host composes a reverse step from these entries the way pressure_projection composes
// smk_divergence, smk_jacobi and smk_project (DESIGN.md "Reverse mode").
//
// Conventions of the gradients: those of torch autograd through the reference's own ops -- floor has no gradient,
// torch.clamp passes it where lo <= x <= hi (inclusive), bilinear weights come from the clamped integer corners.  The
// recomputed forward the host feeds in is bit-exact, so every mask below is the reference's mask.
//
// Determinism: no float atomics.  Every scatter of the forward (bilinear corners, stencil taps, emitter footprints) is
// written as a gather in a fixed order, so two calls on the same inputs give bitwise-equal gradients.  The one atomic is
// an integer max (the advection's reach), which is order independent.
#include "common.cuh"

namespace smk {
namespace {

// ---- a10 adjoint: advection_step (navier_stokes.py:74-95) -------------------------------------------------------------
// Pass 1 (k_adv_adj_trace), one thread per output cell (i, j): redo the back-trace exactly as k_advect does, then store
//   wg     = the four bilinear weights times the effective output gradient e = (g_out + (g_frame + fmul*g_frame)) * scale
//   corner = (x0, y0): the upper-left clamped corner (x1 = min(x0+1, cols-1), y1 likewise)
//   gvel   = (d/du_i, d/dv_i) = (-dt * d/dpx, -dt * d/dpy) where the clamp of px / py passed the gradient, else 0
// and fold the largest corner distance |corner - cell| per axis into reach[2] (integer atomicMax: order independent).
// Pass 2 (k_adv_adj_gather), one thread per source cell (a, b): the field gradient is the sum of the weights of every
// output cell whose corners include (a, b).  Those cells lie within reach of (a, b) (the clamp only moves a back-trace
// closer to its cell), so the thread walks that window in row-major order: a fixed-order gather, no scatter.
// Pass 3 (k_adv_adj_vel): u_i = 0.5*U[i][j] + 0.5*U[i][j+1] and v_i = 0.5*V[i][j] + 0.5*V[i+1][j] where defined (common.cuh
// interp_u_at / interp_v_at), so dU and dV are fixed two-tap gathers of gvel, added into g_u and g_v.
// Pass 2 writes g_field before pass 3 adds into g_u / g_v, so g_field may alias either (u advects u by u itself), and
// pass 1 reads all of g_out before anything is written, so g_out may alias any output too.
struct AdvWs {
    int* reach;          // [2]: x, y
    float4* wg;          // [n]
    int2* corner;        // [n]
    float2* gvel;        // [n]
};

__host__ __device__ inline AdvWs adv_ws(void* base, int64_t n)
{
    char* p = static_cast<char*>(base);
    AdvWs w;
    w.reach = reinterpret_cast<int*>(p);
    w.wg = reinterpret_cast<float4*>(p + 16);
    w.corner = reinterpret_cast<int2*>(p + 16 + 16 * n);
    w.gvel = reinterpret_cast<float2*>(p + 16 + 24 * n);
    return w;
}

__global__ void __launch_bounds__(256)
k_adv_adj_trace(const float* __restrict__ F, const int rows, const int cols, const int pitch, const long long stride,
                const float* __restrict__ U, const float* __restrict__ V, const int h, const int w, const int pu, const int pv,
                const long long su, const long long sv, const float dt, const float scale,
                const float* __restrict__ gout, const float* __restrict__ gframe, const long long fstride, const int pc,
                const float* __restrict__ fmul, AdvWs ws)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    const size_t b = blockIdx.z;
    int rx = 0, ry = 0;
    if (i < rows && j < cols) {
        const GlobalField Uf{U + b * su, pu}, Vf{V + b * sv, pv};
        const float ui = interp_u_at(Uf, h, w, i, j);                 // :84
        const float vi = interp_v_at(Vf, h, w, i, j);                 // :85
        const float X = (float)j, Y = (float)i;
        const float tx = dt * ui, ty = dt * vi;
        float px = X - tx, py = Y - ty;                               // :87-88
        const float xmax = (float)(cols - 1), ymax = (float)(rows - 1);
        const bool pass_x = px >= 0.0f && px <= xmax;                 // torch.clamp's gradient mask (:91-92)
        const bool pass_y = py >= 0.0f && py <= ymax;
        px = clampf(px, 0.0f, xmax);
        py = clampf(py, 0.0f, ymax);
        const int x0 = clampi((int)floorf(px), 0, cols - 1), y0 = clampi((int)floorf(py), 0, rows - 1);
        const int x1 = min(x0 + 1, cols - 1), y1 = min(y0 + 1, rows - 1);
        const float ax = (float)x1 - px, bx = px - (float)x0;
        const float ay = (float)y1 - py, by = py - (float)y0;
        const size_t k = b * (size_t)stride + (size_t)i * pitch + j;
        float e = gout ? gout[k] : 0.0f;
        if (gframe) {                                                  // frame = d + fmul*d (fractal_generator.py:62)
            const float gf = gframe[b * (size_t)fstride + (size_t)i * pc + j];
            const float gm = fmul ? fmul[(size_t)i * pc + j] * gf : 0.0f;
            e = e + (gf + gm);
        }
        e = e * scale;                                                 // the 0.995 decay of :171
        const float* Fb = F + b * (size_t)stride;
        const float f00 = Fb[(size_t)y0 * pitch + x0], f01 = Fb[(size_t)y0 * pitch + x1];
        const float f10 = Fb[(size_t)y1 * pitch + x0], f11 = Fb[(size_t)y1 * pitch + x1];
        const size_t n = (b * rows + i) * (size_t)cols + j;
        ws.wg[n] = make_float4((ax * ay) * e, (bx * ay) * e, (ax * by) * e, (bx * by) * e);
        ws.corner[n] = make_int2(x0, y0);
        const float gpx = e * (ay * (f01 - f00) + by * (f11 - f10));   // d/dpx of ((wa f00 + wb f01) + wc f10) + wd f11
        const float gpy = e * (ax * (f10 - f00) + bx * (f11 - f01));
        ws.gvel[n] = make_float2(pass_x ? -(dt * gpx) : 0.0f, pass_y ? -(dt * gpy) : 0.0f);
        rx = max(abs(x0 - j), abs(x1 - j));
        ry = max(abs(y0 - i), abs(y1 - i));
    }
    rx = __reduce_max_sync(0xffffffffu, rx);
    ry = __reduce_max_sync(0xffffffffu, ry);
    if (threadIdx.x == 0) {
        if (rx > 0) atomicMax(ws.reach, rx);
        if (ry > 0) atomicMax(ws.reach + 1, ry);
    }
}

__global__ void __launch_bounds__(256)
k_adv_adj_gather(const int rows, const int cols, const int pitch, const long long stride, float* __restrict__ gfield,
                 const int accumulate, const AdvWs ws)
{
    const int bc = blockIdx.x * 32 + threadIdx.x, a = blockIdx.y * 8 + threadIdx.y;
    if (a >= rows || bc >= cols) return;
    const size_t b = blockIdx.z;
    const int rx = ws.reach[0], ry = ws.reach[1];
    const int ilo = max(a - ry, 0), ihi = min(a + ry, rows - 1);
    const int jlo = max(bc - rx, 0), jhi = min(bc + rx, cols - 1);
    float s = 0.0f;
    for (int i = ilo; i <= ihi; ++i) {
        const size_t row = (b * rows + i) * (size_t)cols;
        for (int j = jlo; j <= jhi; ++j) {
            const int2 c = ws.corner[row + j];
            const int x1 = min(c.x + 1, cols - 1), y1 = min(c.y + 1, rows - 1);
            const bool hx0 = c.x == bc, hx1 = x1 == bc, hy0 = c.y == a, hy1 = y1 == a;
            if (!((hx0 || hx1) && (hy0 || hy1))) continue;
            const float4 q = ws.wg[row + j];
            if (hy0 && hx0) s = s + q.x;
            if (hy0 && hx1) s = s + q.y;
            if (hy1 && hx0) s = s + q.z;
            if (hy1 && hx1) s = s + q.w;
        }
    }
    float* o = gfield + b * (size_t)stride + (size_t)a * pitch + bc;
    *o = accumulate ? *o + s : s;
}

__global__ void __launch_bounds__(256)
k_adv_adj_vel(const int rows, const int cols, const int h, const int w, const int pu, const int pv,
              const long long su, const long long sv, float* __restrict__ gU, float* __restrict__ gV, const AdvWs ws)
{
    const int bc = blockIdx.x * 32 + threadIdx.x, a = blockIdx.y * 8 + threadIdx.y;
    const size_t b = blockIdx.z;
    const size_t row = (b * rows + a) * (size_t)cols;
    const bool in_field_row = a < rows;
    if (a <= h && bc <= w - 1) {                                  // u cell: taps u_i(a, bc) and u_i(a, bc - 1)
        const bool t0 = a <= h - 1 && bc <= w - 2 && in_field_row && bc < cols;
        const bool t1 = a <= h - 1 && bc >= 1 && bc - 1 <= w - 2 && in_field_row && bc - 1 < cols;
        if (t0 || t1) {
            const float g0 = t0 ? 0.5f * ws.gvel[row + bc].x : 0.0f;
            const float g1 = t1 ? 0.5f * ws.gvel[row + bc - 1].x : 0.0f;
            float* o = gU + b * (size_t)su + (size_t)a * pu + bc;
            *o = *o + (g0 + g1);
        }
    }
    if (a <= h - 1 && bc <= w) {                                  // v cell: taps v_i(a, bc) and v_i(a - 1, bc)
        const bool t0 = a <= h - 2 && bc <= w - 1 && in_field_row && bc < cols;
        const bool t1 = a >= 1 && a - 1 <= h - 2 && bc <= w - 1 && a - 1 < rows && bc < cols;
        if (t0 || t1) {
            const float g0 = t0 ? 0.5f * ws.gvel[row + bc].y : 0.0f;
            const float g1 = t1 ? 0.5f * ws.gvel[row - cols + bc].y : 0.0f;
            float* o = gV + b * (size_t)sv + (size_t)a * pv + bc;
            *o = *o + (g0 + g1);
        }
    }
}

// ---- a7 adjoint: gradient subtract (navier_stokes.py:148-149) ----------------------------------------------------------
// u[i][j] -= dt*(p[i][j] - p[i-1][j]) for 1 <= i <= h-1, v[i][j] -= dt*(p[i][j] - p[i][j-1]) for 1 <= j <= w-1:
// g_p = g_p_in + dt*((g_u[i+1][j] - g_u[i][j]) + (g_v[i][j+1] - g_v[i][j])) over the rows / columns that were updated.
__global__ void __launch_bounds__(256)
k_project_adj(const float* __restrict__ gU, const float* __restrict__ gV, const float* __restrict__ gPin, float* __restrict__ gP,
              const int h, const int w, const int pu, const int pv, const int pc,
              const long long su, const long long sv, const long long sc, const float dt)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= h || j >= w) return;
    const size_t b = blockIdx.z;
    gU += b * su; gV += b * sv;
    const float un = i + 1 <= h - 1 ? gU[(size_t)(i + 1) * pu + j] : 0.0f;
    const float uc = i >= 1 ? gU[(size_t)i * pu + j] : 0.0f;
    const float vn = j + 1 <= w - 1 ? gV[(size_t)i * pv + j + 1] : 0.0f;
    const float vc = j >= 1 ? gV[(size_t)i * pv + j] : 0.0f;
    const size_t k = b * sc + (size_t)i * pc + j;
    const float gp = gPin ? gPin[k] : 0.0f;
    gP[k] = gp + dt * ((un - uc) + (vn - vc));
}

// With solid cells (k_project_obst subtracts on open faces only): a closed face contributes nothing to g_p.
__global__ void __launch_bounds__(256)
k_project_adj_obst(const float* __restrict__ gU, const float* __restrict__ gV, const float* __restrict__ gPin, float* __restrict__ gP,
                   const uint8_t* __restrict__ S, const int h, const int w, const int pu, const int pv, const int pc,
                   const long long su, const long long sv, const long long sc, const long long ss, const float dt)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= h || j >= w) return;
    const size_t b = blockIdx.z;
    gU += b * su; gV += b * sv; S += b * ss;
    const float un = i + 1 <= h - 1 && !u_closed(S, h, pc, i + 1, j) ? gU[(size_t)(i + 1) * pu + j] : 0.0f;
    const float uc = i >= 1 && !u_closed(S, h, pc, i, j) ? gU[(size_t)i * pu + j] : 0.0f;
    const float vn = j + 1 <= w - 1 && !v_closed(S, w, pc, i, j + 1) ? gV[(size_t)i * pv + j + 1] : 0.0f;
    const float vc = j >= 1 && !v_closed(S, w, pc, i, j) ? gV[(size_t)i * pv + j] : 0.0f;
    const size_t k = b * sc + (size_t)i * pc + j;
    const float gp = gPin ? gPin[k] : 0.0f;
    gP[k] = gp + dt * ((un - uc) + (vn - vc));
}

// ---- a6 adjoint: K Jacobi sweeps (navier_stokes.py:139-145) ------------------------------------------------------------
// A sweep is p' = J0 p - 0.25*M*div with J0 = M*0.25*S (M: interior mask, S: 4-neighbour sum).  With r = M*g:
//   g_div = -0.25 * sum_{j<K} J0^j r          g_p = 0.25 * S * J0^(K-1) r   (ring cells of p included)
// Both powers run on the forward's own blocked kernel (launch_jacobi): K-1 sweeps from r with div = 0 give J0^(K-1) r, and
// K sweeps from 0 with div = -4r give sum_j J0^j r (a sweep computes J0 x - 0.25*M*div).  These two kernels do the rest.
__global__ void __launch_bounds__(256)
k_jacobi_adj_prep(const float* __restrict__ g, float* __restrict__ r, float* __restrict__ nd, const int h, const int w,
                  const int pc, const long long sc)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= h || j >= w) return;
    const size_t k = blockIdx.z * (size_t)sc + (size_t)i * pc + j;
    const bool interior = i >= 1 && i <= h - 2 && j >= 1 && j <= w - 2;
    const float x = interior ? g[k] : 0.0f;
    r[k] = x;
    if (nd) nd[k] = -4.0f * x;
}

__global__ void __launch_bounds__(256)
k_jacobi_adj_out(const float* __restrict__ y, const float* __restrict__ sum, float* __restrict__ gP, float* __restrict__ gDiv,
                 const int h, const int w, const int pc, const long long sc)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= h || j >= w) return;
    const size_t base = blockIdx.z * (size_t)sc, k = base + (size_t)i * pc + j;
    const float* Y = y + base;
    const float up = i >= 1 ? Y[(size_t)(i - 1) * pc + j] : 0.0f, dn = i + 1 < h ? Y[(size_t)(i + 1) * pc + j] : 0.0f;
    const float lf = j >= 1 ? Y[(size_t)i * pc + j - 1] : 0.0f, rt = j + 1 < w ? Y[(size_t)i * pc + j + 1] : 0.0f;
    float s = up + dn;
    s = s + lf;
    s = s + rt;
    gP[k] = 0.25f * s;
    gDiv[k] = -0.25f * sum[k];
}

// With solid cells (k_jacobi_obst, DESIGN.md s5.7).  A masked sweep is p' = J p - 0.25*M*div with M the fluid-interior mask and
// J = M*A, A[c][n] = 0.25 for each fluid neighbour n of c and A[c][c] = 0.25 * (the number of solid neighbours of c).  A restricted
// to fluid-interior cells is symmetric, so M J^T M = M J M and, with r = M*g, the two chains above carry over on k_jacobi_obst:
//   g_div = -0.25 * sum_{j<K} J^j r          g_p = J^T J^(K-1) r
// y = J^(K-1) r is 0 off the fluid interior, so J^T y at a fluid cell n is the forward's stencil read backwards: each neighbour
// slot takes y of a fluid neighbour, or y_n itself where the neighbour is solid (its Neumann ghost value); solid cells get 0.
__global__ void __launch_bounds__(256)
k_jacobi_adj_prep_obst(const float* __restrict__ g, float* __restrict__ r, float* __restrict__ nd, const uint8_t* __restrict__ S,
                       const int h, const int w, const int pc, const long long sc, const long long ss)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= h || j >= w) return;
    const size_t k = blockIdx.z * (size_t)sc + (size_t)i * pc + j;
    const bool keep = i >= 1 && i <= h - 2 && j >= 1 && j <= w - 2 && S[blockIdx.z * (size_t)ss + (size_t)i * pc + j] == 0;
    const float x = keep ? g[k] : 0.0f;
    r[k] = x;
    if (nd) nd[k] = -4.0f * x;
}

__global__ void __launch_bounds__(256)
k_jacobi_adj_out_obst(const float* __restrict__ y, const float* __restrict__ sum, float* __restrict__ gP, float* __restrict__ gDiv,
                      const uint8_t* __restrict__ S, const int h, const int w, const int pc, const long long sc, const long long ss)
{
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= h || j >= w) return;
    const size_t base = blockIdx.z * (size_t)sc, c = (size_t)i * pc + j, k = base + c;
    const float* Y = y + base;
    S += blockIdx.z * (size_t)ss;
    gDiv[k] = -0.25f * sum[k];
    if (S[c]) {
        gP[k] = 0.0f;
        return;
    }
    const float yc = Y[c];
    const float up = i >= 1 ? (S[c - pc] ? yc : Y[c - pc]) : 0.0f, dn = i + 1 < h ? (S[c + pc] ? yc : Y[c + pc]) : 0.0f;
    const float lf = j >= 1 ? (S[c - 1] ? yc : Y[c - 1]) : 0.0f, rt = j + 1 < w ? (S[c + 1] ? yc : Y[c + 1]) : 0.0f;
    float s = up + dn;
    s = s + lf;
    s = s + rt;
    gP[k] = 0.25f * s;
}

// ---- a3 + a4 + a5 adjoint: buoyancy (:154-155), the three diffusions (:158-160) and the divergence (:136) --------------
// Divergence: div[i][j] = (((u[i+1][j] - u[i][j]) + v[i][j+1]) - v[i][j]) / dt, so the u_diff / v_diff gradients gain the
// shifted differences of q = g_div / dt.  Diffusion f' = f + c*(S_clamped f - 4f) with replicate padding: its transpose
// sends t = c*g' back to each tap, and an edge cell receives its own clamped-neighbour taps.  Buoyancy v[:, :w] += dt*(d*0.1):
// g_d += (dt * g_v)*0.1 over the first w columns.  One thread per (row, col) of the (h+1) x (w+1) union of the domains.
struct DiffAdjIn {
    const float* gUd; const float* gVd; const float* gDd; const float* gDiv;
    int h, w, pu, pv, pc;
    float dt;
};

__device__ __forceinline__ float q_at(const DiffAdjIn& A, int i, int j) { return A.gDiv[(size_t)i * A.pc + j] / A.dt; }

// total gradient of u_diff / v_diff / d_diff at (a, b): the output gradient plus the divergence's transpose
__device__ __forceinline__ float gtot_u(const DiffAdjIn& A, int a, int b)
{
    const float lo = a >= 1 ? q_at(A, a - 1, b) : 0.0f, hi = a <= A.h - 1 ? q_at(A, a, b) : 0.0f;
    return A.gUd[(size_t)a * A.pu + b] + (lo - hi);
}
__device__ __forceinline__ float gtot_v(const DiffAdjIn& A, int a, int b)
{
    const float lo = b >= 1 ? q_at(A, a, b - 1) : 0.0f, hi = b <= A.w - 1 ? q_at(A, a, b) : 0.0f;
    return A.gVd[(size_t)a * A.pv + b] + (lo - hi);
}
__device__ __forceinline__ float gtot_d(const DiffAdjIn& A, int a, int b) { return A.gDd[(size_t)a * A.pc + b]; }

// OBST (solid cells S of this simulation): O1 set the closed faces of u_diff / v_diff to +0.0 before the divergence and the
// gradient subtract read them, so the total gradient of a closed face is +0.0 before the diffusion transpose gathers it
template <int KIND, bool OBST = false>
__device__ __forceinline__ float gtot(const DiffAdjIn& A, int a, int b, const uint8_t* S = nullptr)
{
    if (OBST && KIND == 0 && u_closed(S, A.h, A.pc, a, b)) return 0.0f;
    if (OBST && KIND == 1 && v_closed(S, A.w, A.pc, a, b)) return 0.0f;
    return KIND == 0 ? gtot_u(A, a, b) : (KIND == 1 ? gtot_v(A, a, b) : gtot_d(A, a, b));
}

// transpose of diffusion_step (navier_stokes.py:50-72) on a rows x cols field at (a, b)
template <int KIND, bool OBST = false>
__device__ __forceinline__ float diffuse_adj(const DiffAdjIn& A, int rows, int cols, int a, int b, float c,
                                             const uint8_t* S = nullptr)
{
    const float g = gtot<KIND, OBST>(A, a, b, S), t = c * g;
    float s = 0.0f;
    if (a + 1 < rows) s = s + c * gtot<KIND, OBST>(A, a + 1, b, S);          // (a, b) is the upper tap of (a+1, b)
    if (a == 0) s = s + t;                                           // ... and its own, clamped
    if (a >= 1) s = s + c * gtot<KIND, OBST>(A, a - 1, b, S);                 // lower tap of (a-1, b)
    if (a == rows - 1) s = s + t;
    if (b + 1 < cols) s = s + c * gtot<KIND, OBST>(A, a, b + 1, S);           // left tap of (a, b+1)
    if (b == 0) s = s + t;
    if (b >= 1) s = s + c * gtot<KIND, OBST>(A, a, b - 1, S);                 // right tap of (a, b-1)
    if (b == cols - 1) s = s + t;
    return g + (s - 4.0f * t);
}

__global__ void __launch_bounds__(256)
k_forces_diffuse_div_adj(DiffAdjIn A, float* __restrict__ gU, float* __restrict__ gV, float* __restrict__ gD,
                         const long long su, const long long sv, const long long sc, const float c_uv, const float c_d)
{
    const int b = blockIdx.x * 32 + threadIdx.x, a = blockIdx.y * 8 + threadIdx.y;
    const size_t n = blockIdx.z;
    const int h = A.h, w = A.w;
    if (a > h || b > w) return;
    A.gUd += n * su; A.gVd += n * sv; A.gDd += n * sc; A.gDiv += n * sc;
    if (b <= w - 1) gU[n * su + (size_t)a * A.pu + b] = diffuse_adj<0>(A, h + 1, w, a, b, c_uv);
    if (a <= h - 1) {
        const float gv = diffuse_adj<1>(A, h, w + 1, a, b, c_uv);
        gV[n * sv + (size_t)a * A.pv + b] = gv;
        if (b <= w - 1) {
            const float gd = diffuse_adj<2>(A, h, w, a, b, c_d);
            gD[n * sc + (size_t)a * A.pc + b] = gd + (A.dt * gv) * 0.1f;
        }
    }
}

// k_forces_diffuse_div_adj of a masked step (solid cells S, simulation n at S + n * ss); kept a separate kernel so that the one
// above, which runs on every unmasked reverse step, compiles exactly as it did
__global__ void __launch_bounds__(256)
k_forces_diffuse_div_adj_obst(DiffAdjIn A, float* __restrict__ gU, float* __restrict__ gV, float* __restrict__ gD,
                              const long long su, const long long sv, const long long sc, const float c_uv, const float c_d,
                              const uint8_t* __restrict__ S, const long long ss)
{
    const int b = blockIdx.x * 32 + threadIdx.x, a = blockIdx.y * 8 + threadIdx.y;
    const size_t n = blockIdx.z;
    const int h = A.h, w = A.w;
    if (a > h || b > w) return;
    A.gUd += n * su; A.gVd += n * sv; A.gDd += n * sc; A.gDiv += n * sc;
    S += n * ss;
    if (b <= w - 1) gU[n * su + (size_t)a * A.pu + b] = diffuse_adj<0, true>(A, h + 1, w, a, b, c_uv, S);
    if (a <= h - 1) {
        const float gv = diffuse_adj<1, true>(A, h, w + 1, a, b, c_uv, S);
        gV[n * sv + (size_t)a * A.pv + b] = gv;
        if (b <= w - 1) {
            const float gd = diffuse_adj<2, true>(A, h, w, a, b, c_d, S);
            gD[n * sc + (size_t)a * A.pc + b] = gd + (A.dt * gv) * 0.1f;
        }
    }
}

// ---- a2 adjoint: add_smoke_source (navier_stokes.py:37-48) -------------------------------------------------------------
// density += intensity * expf(-dist^2 / denom) over the footprint, so d/d(intensity) = sum g_d * expf(...), with the weight
// computed exactly as k_splat computes it.  One CTA per emitter; each thread sums a fixed, strided share of the bounding box,
// then a fixed-order shared-memory tree adds the 256 partial sums.  accumulate: gI[k] += the sum (one add per launch, so a
// sequence of launches sums in launch order), else gI[k] = the sum.
__global__ void __launch_bounds__(256)
k_splat_adj(const float* __restrict__ gD, const int h, const int w, const int pc, const long long sc, const int batch,
            const smk_source_t* __restrict__ src, const int32_t* __restrict__ off, float* __restrict__ gI, const int accumulate)
{
    __shared__ float part[256];
    const int k = blockIdx.x, tid = threadIdx.x;
    int lo = 0, hi = batch - 1;                                      // simulation b with off[b] <= k < off[b+1]
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= k) lo = mid; else hi = mid - 1;
    }
    const float* G = gD + (size_t)lo * sc;
    const smk_source_t e = src[k];
    const int r = max(e.radius, -1);
    const int ya = max(e.y - r, 0), yb = min(e.y + r, h - 1), xa = max(e.x - r, 0), xb = min(e.x + r, w - 1);
    const int bw = xb - xa + 1, bh = yb - ya + 1;
    const double r3 = (double)e.radius / 3.0;
    const float denom = (float)(2.0 * (r3 * r3));
    float acc = 0.0f;
    if (bw > 0 && bh > 0) {
        for (int q = tid; q < bw * bh; q += 256) {
            const int i = ya + q / bw, j = xa + q % bw;
            const long long dx = (long long)j - e.x, dy = (long long)i - e.y;
            const float dist = sqrtf((float)(dx * dx + dy * dy));
            if (dist <= (float)e.radius) {
                const float d2 = dist * dist;
                acc = acc + G[(size_t)i * pc + j] * expf((-d2) / denom);
            }
        }
    }
    part[tid] = acc;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (tid < s) part[tid] = part[tid] + part[tid + s];
        __syncthreads();
    }
    if (tid == 0) gI[k] = accumulate ? gI[k] + part[0] : part[0];
}

inline dim3 cells_grid(int rows, int cols, int batch) { return dim3((cols + 31) / 32, (rows + 7) / 8, batch); }

}  // namespace
}  // namespace smk

using namespace smk;

#define SMK_TRY(x) do { const int rc_ = (x); if (rc_ != SMK_OK) return rc_; } while (0)

static int adj_grid(const smk_grid_t* g, const char* who)
{
    SMK_TRY(check_grid(g, who));
    if (g->gh != 0) return fail(SMK_EUNSUPPORTED, "%s: not available on a slab grid (gh != 0)", who);
    return SMK_OK;
}

extern "C" {

int smk_advect_adjoint(const smk_grid_t* g, const float* field, int32_t rows, int32_t cols, int32_t pitch, int64_t stride,
                       const float* u, const float* v, float dt, float scale,
                       const float* g_out, const float* g_frame, int64_t frame_stride, const float* fmul,
                       float* g_field, int32_t accumulate, float* g_u, float* g_v, void* workspace, void* stream)
{
    SMK_TRY(adj_grid(g, "smk_advect_adjoint"));
    if (!field || !u || !v || !g_field || !g_u || !g_v || !workspace) return fail(SMK_EINVAL, "smk_advect_adjoint: NULL pointer");
    if (!aligned16(workspace)) return fail(SMK_EINVAL, "smk_advect_adjoint: workspace is not 16-byte aligned");
    if (rows < 1 || cols < 1 || pitch < cols) return fail(SMK_EINVAL, "smk_advect_adjoint: bad field shape %d x %d pitch %d", rows, cols, pitch);
    if (rows > g->h + 1 || cols > g->w + 1)
        return fail(SMK_EINVAL, "smk_advect_adjoint: a %d x %d field does not fit the %d x %d cell grid", rows, cols, g->h, g->w);
    if (g->batch > 1 && stride < (int64_t)rows * pitch) return fail(SMK_EINVAL, "smk_advect_adjoint: batch stride smaller than one field");
    if ((g_frame || fmul) && (rows != g->h || cols != g->w)) return fail(SMK_EINVAL, "smk_advect_adjoint: frame gradient needs a cell-centred field");
    if (fmul && !g_frame) return fail(SMK_EINVAL, "smk_advect_adjoint: fmul without g_frame");
    const float* writes[3] = {g_field, g_u, g_v};
    for (const float* p : writes)
        if (p == field || p == u || p == v) return fail(SMK_EINVAL, "smk_advect_adjoint: a gradient output aliases a forward input");
    if (g_u == g_v) return fail(SMK_EINVAL, "smk_advect_adjoint: g_u and g_v must differ");
    if ((int64_t)rows * cols * g->batch >= (1ll << 40)) return fail(SMK_EUNSUPPORTED, "smk_advect_adjoint: field too large");
    cudaStream_t s = (cudaStream_t)stream;
    const AdvWs ws = adv_ws(workspace, (int64_t)rows * cols * g->batch);
    ProfScope prof_(SMK_PH_OTHER, s);
    cudaError_t e = cudaMemsetAsync(ws.reach, 0, 2 * sizeof(int), s);
    if (e != cudaSuccess) return fail((int)e, "smk_advect_adjoint: %s", cudaGetErrorString(e));
    const dim3 blk(32, 8), grid = cells_grid(rows, cols, g->batch);
    k_adv_adj_trace<<<grid, blk, 0, s>>>(field, rows, cols, pitch, stride, u, v, g->h, g->w, g->pitch_u, g->pitch_v,
                                         g->stride_u, g->stride_v, dt, scale, g_out, g_frame, frame_stride, g->pitch_c, fmul, ws);
    SMK_TRY(check_launch("k_adv_adj_trace"));
    k_adv_adj_gather<<<grid, blk, 0, s>>>(rows, cols, pitch, stride, g_field, accumulate ? 1 : 0, ws);
    SMK_TRY(check_launch("k_adv_adj_gather"));
    k_adv_adj_vel<<<cells_grid(g->h + 1, g->w + 1, g->batch), blk, 0, s>>>(rows, cols, g->h, g->w, g->pitch_u, g->pitch_v,
                                                                         g->stride_u, g->stride_v, g_u, g_v, ws);
    return check_launch("k_adv_adj_vel");
}

int smk_project_adjoint(const smk_grid_t* g, const float* g_u, const float* g_v, const float* g_p_in, float* g_p, float dt, void* stream)
{
    return smk_project_adjoint_ex(g, g_u, g_v, g_p_in, g_p, dt, nullptr, 0, stream);
}

int smk_project_adjoint_ex(const smk_grid_t* g, const float* g_u, const float* g_v, const float* g_p_in, float* g_p, float dt,
                           const uint8_t* solid, int64_t solid_batch_stride, void* stream)
{
    SMK_TRY(adj_grid(g, "smk_project_adjoint"));
    if (!g_u || !g_v || !g_p) return fail(SMK_EINVAL, "smk_project_adjoint: NULL pointer");
    if (g_p == g_u || g_p == g_v) return fail(SMK_EINVAL, "smk_project_adjoint: g_p aliases g_u or g_v");
    SMK_TRY(check_solid(g, solid, solid_batch_stride, "smk_project_adjoint_ex"));
    cudaStream_t s = (cudaStream_t)stream;
    ProfScope prof_(SMK_PH_OTHER, s);
    const dim3 grid = cells_grid(g->h, g->w, g->batch), blk(32, 8);
    if (solid) {
        k_project_adj_obst<<<grid, blk, 0, s>>>(g_u, g_v, g_p_in, g_p, solid, g->h, g->w, g->pitch_u, g->pitch_v, g->pitch_c,
                                                g->stride_u, g->stride_v, g->stride_c, solid_batch_stride, dt);
        return check_launch("k_project_adj_obst");
    }
    k_project_adj<<<grid, blk, 0, s>>>(g_u, g_v, g_p_in, g_p, g->h, g->w, g->pitch_u, g->pitch_v, g->pitch_c, g->stride_u, g->stride_v,
                                       g->stride_c, dt);
    return check_launch("k_project_adj");
}

int smk_jacobi_adjoint(const smk_grid_t* g, const float* g_p_in, float* g_p, float* g_div, int32_t K, int32_t T,
                       float* workspace, void* stream)
{
    return smk_jacobi_adjoint_ex(g, g_p_in, g_p, g_div, K, T, workspace, nullptr, 0, stream);
}

// With solid cells: the prep and output kernels take the mask (k_jacobi_adj_*_obst) and both chains run on k_jacobi_obst.
int smk_jacobi_adjoint_ex(const smk_grid_t* g, const float* g_p_in, float* g_p, float* g_div, int32_t K, int32_t T,
                          float* workspace, const uint8_t* solid, int64_t solid_batch_stride, void* stream)
{
    SMK_TRY(adj_grid(g, "smk_jacobi_adjoint"));
    if (!g_p_in || !g_p || !g_div) return fail(SMK_EINVAL, "smk_jacobi_adjoint: NULL pointer");
    if (K < 0 || T < 0) return fail(SMK_EINVAL, "smk_jacobi_adjoint: negative K or T");
    if (g_p == g_p_in || g_div == g_p_in || g_p == g_div) return fail(SMK_EINVAL, "smk_jacobi_adjoint: outputs must not alias");
    if (K >= 1 && (!workspace || !aligned16(workspace))) return fail(SMK_EINVAL, "smk_jacobi_adjoint: workspace NULL or not 16-byte aligned");
    SMK_TRY(check_solid(g, solid, solid_batch_stride, "smk_jacobi_adjoint_ex"));
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t field = g->batch > 1 ? g->stride_c : (int64_t)g->h * g->pitch_c;
    const size_t bytes = sizeof(float) * (size_t)field * g->batch;
    const dim3 blk(32, 8), grid = cells_grid(g->h, g->w, g->batch);
    const long long ss = solid_batch_stride;
    cudaError_t e;
    if (K == 0) {                                    // no sweep: p passes through, the divergence has no effect
        e = cudaMemcpyAsync(g_p, g_p_in, bytes, cudaMemcpyDeviceToDevice, s);
        if (e == cudaSuccess) e = cudaMemsetAsync(g_div, 0, bytes, s);
        return e == cudaSuccess ? SMK_OK : fail((int)e, "smk_jacobi_adjoint: %s", cudaGetErrorString(e));
    }
    if (K == 1) {                                    // J0^0 r = sum_{j<1} J0^j r = r: no sweep
        ProfScope prof_(SMK_PH_OTHER, s);
        float* r = workspace;
        if (solid) {
            k_jacobi_adj_prep_obst<<<grid, blk, 0, s>>>(g_p_in, r, nullptr, solid, g->h, g->w, g->pitch_c, field, ss);
            SMK_TRY(check_launch("k_jacobi_adj_prep_obst"));
            k_jacobi_adj_out_obst<<<grid, blk, 0, s>>>(r, r, g_p, g_div, solid, g->h, g->w, g->pitch_c, field, ss);
            return check_launch("k_jacobi_adj_out_obst");
        }
        k_jacobi_adj_prep<<<grid, blk, 0, s>>>(g_p_in, r, nullptr, g->h, g->w, g->pitch_c, field);
        SMK_TRY(check_launch("k_jacobi_adj_prep"));
        k_jacobi_adj_out<<<grid, blk, 0, s>>>(r, r, g_p, g_div, g->h, g->w, g->pitch_c, field);
        return check_launch("k_jacobi_adj_out");
    }
    // workspace: A, B (J0^(K-1) r and its ping-pong), ND (-4r), Z, Z2 (the sum, from zero, and its ping-pong)
    float* A = workspace;
    float* B = A + field * g->batch;
    float* ND = B + field * g->batch;
    float* Z = ND + field * g->batch;
    float* Z2 = Z + field * g->batch;
    e = cudaMemsetAsync(A, 0, 5 * bytes, s);                       // pad columns of every buffer stay zero
    if (e == cudaSuccess) e = cudaMemsetAsync(g_div, 0, bytes, s);  // the zero divergence of the first chain
    if (e != cudaSuccess) return fail((int)e, "smk_jacobi_adjoint: %s", cudaGetErrorString(e));
    {
        ProfScope prof_(SMK_PH_OTHER, s);
        if (solid)
            k_jacobi_adj_prep_obst<<<grid, blk, 0, s>>>(g_p_in, A, ND, solid, g->h, g->w, g->pitch_c, field, ss);
        else
            k_jacobi_adj_prep<<<grid, blk, 0, s>>>(g_p_in, A, ND, g->h, g->w, g->pitch_c, field);
        SMK_TRY(check_launch(solid ? "k_jacobi_adj_prep_obst" : "k_jacobi_adj_prep"));
    }
    smk_grid_t gg = *g;
    gg.stride_c = field;
    int in_b = 0, in_z2 = 0;
    SMK_TRY(launch_jacobi(&gg, g_div, A, B, K - 1, T, &in_b, s, solid, ss));       // J0^(K-1) r
    SMK_TRY(launch_jacobi(&gg, ND, Z, Z2, K, T, &in_z2, s, solid, ss));            // sum_{j<K} J0^j r
    ProfScope prof_(SMK_PH_OTHER, s);
    if (solid) {
        k_jacobi_adj_out_obst<<<grid, blk, 0, s>>>(in_b ? B : A, in_z2 ? Z2 : Z, g_p, g_div, solid, g->h, g->w, g->pitch_c, field, ss);
        return check_launch("k_jacobi_adj_out_obst");
    }
    k_jacobi_adj_out<<<grid, blk, 0, s>>>(in_b ? B : A, in_z2 ? Z2 : Z, g_p, g_div, g->h, g->w, g->pitch_c, field);
    return check_launch("k_jacobi_adj_out");
}

int smk_forces_diffuse_div_adjoint(const smk_grid_t* g, const float* g_u_diff, const float* g_v_diff, const float* g_d_diff,
                                   const float* g_div, float* g_u, float* g_v, float* g_d, float dt, float c_uv, float c_d, void* stream)
{
    return smk_forces_diffuse_div_adjoint_ex(g, g_u_diff, g_v_diff, g_d_diff, g_div, g_u, g_v, g_d, dt, c_uv, c_d, nullptr, 0, stream);
}

int smk_forces_diffuse_div_adjoint_ex(const smk_grid_t* g, const float* g_u_diff, const float* g_v_diff, const float* g_d_diff,
                                      const float* g_div, float* g_u, float* g_v, float* g_d, float dt, float c_uv, float c_d,
                                      const uint8_t* solid, int64_t solid_batch_stride, void* stream)
{
    SMK_TRY(adj_grid(g, "smk_forces_diffuse_div_adjoint"));
    if (!g_u_diff || !g_v_diff || !g_d_diff || !g_div || !g_u || !g_v || !g_d)
        return fail(SMK_EINVAL, "smk_forces_diffuse_div_adjoint: NULL pointer");
    const float* ins[4] = {g_u_diff, g_v_diff, g_d_diff, g_div};
    for (const float* p : ins)
        if (p == g_u || p == g_v || p == g_d) return fail(SMK_EINVAL, "smk_forces_diffuse_div_adjoint: outputs must not alias inputs");
    if (!(dt != 0.0f)) return fail(SMK_EINVAL, "smk_forces_diffuse_div_adjoint: dt must be non-zero");
    SMK_TRY(check_solid(g, solid, solid_batch_stride, "smk_forces_diffuse_div_adjoint_ex"));
    cudaStream_t s = (cudaStream_t)stream;
    DiffAdjIn A{g_u_diff, g_v_diff, g_d_diff, g_div, g->h, g->w, g->pitch_u, g->pitch_v, g->pitch_c, dt};
    ProfScope prof_(SMK_PH_OTHER, s);
    const dim3 grid = cells_grid(g->h + 1, g->w + 1, g->batch), blk(32, 8);
    if (solid) {
        k_forces_diffuse_div_adj_obst<<<grid, blk, 0, s>>>(A, g_u, g_v, g_d, g->stride_u, g->stride_v, g->stride_c, c_uv, c_d, solid,
                                                           solid_batch_stride);
        return check_launch("k_forces_diffuse_div_adj_obst");
    }
    k_forces_diffuse_div_adj<<<grid, blk, 0, s>>>(A, g_u, g_v, g_d, g->stride_u, g->stride_v, g->stride_c, c_uv, c_d);
    return check_launch("k_forces_diffuse_div_adj");
}

int smk_splat_sources_adjoint(const smk_grid_t* g, const float* g_density, const smk_source_t* sources, const int32_t* offsets,
                              int32_t nsources, float* g_intensity, void* stream)
{
    return smk_splat_sources_adjoint_ex(g, g_density, sources, offsets, nsources, 0, g_intensity, stream);
}

int smk_splat_sources_adjoint_ex(const smk_grid_t* g, const float* g_density, const smk_source_t* sources, const int32_t* offsets,
                                 int32_t nsources, int32_t accumulate, float* g_intensity, void* stream)
{
    SMK_TRY(adj_grid(g, "smk_splat_sources_adjoint"));
    if (accumulate != 0 && accumulate != 1) return fail(SMK_EINVAL, "smk_splat_sources_adjoint_ex: accumulate must be 0 or 1");
    if (nsources < 0) return fail(SMK_EINVAL, "smk_splat_sources_adjoint: negative nsources");
    if (nsources == 0) return SMK_OK;
    if (!g_density || !sources || !offsets || !g_intensity) return fail(SMK_EINVAL, "smk_splat_sources_adjoint: NULL pointer");
    if (nsources > 0x7fffffff / 2) return fail(SMK_EUNSUPPORTED, "smk_splat_sources_adjoint: %d emitters", nsources);
    cudaStream_t s = (cudaStream_t)stream;
    ProfScope prof_(SMK_PH_OTHER, s);
    k_splat_adj<<<nsources, 256, 0, s>>>(g_density, g->h, g->w, g->pitch_c, g->stride_c, g->batch, sources, offsets, g_intensity, accumulate);
    return check_launch("k_splat_adj");
}

}  // extern "C"
