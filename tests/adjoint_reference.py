"""Float64 references of the adjoint entries of csrc/adjoint.cu, each with its absolute-value twin.

Every phase adjoint of the step is the transpose A^T of a linear map A; the velocity part of the advection is linear once the
fp32 back-trace is fixed.  For each entry this module gives
    adjoint(g)                 A^T g in float64
    adjoint(g, absolute=True)  |A|^T |g|: the same map with absolute coefficients applied to |g|, the running-error scale of an
                               fp32 evaluation of A^T g (a kernel's error at a cell is at most ~ m * 2^-24 times it, m the
                               number of roundings on the cell's longest path).
The linear phases go through float64 autograd of oracle/torch_step.py (those functions are dtype-generic); the Jacobi transpose is
written out (K float64 sweeps instead of a K-deep graph) and the advection's is formed from the fp32 back-trace positions, which
are bit-equal to the kernel's.  Constants are the fp32 values the kernels use.  tests/test_adjoint_reference_host.py checks
<A x, g> = <x, A^T g> against the forward functions of oracle/torch_step.py, and the advection against autograd of its
back-trace.  All fields are torch tensors with a leading batch dimension [B, rows, cols]."""
import numpy as np
import torch

from oracle import torch_step as ts

U = 2.0 ** -24           # unit roundoff of fp32


def f32(x):
    """The fp32 value of a Python scalar, as a float: the constant a kernel computes with."""
    return float(np.float32(x))


def _grad(outs, ins, gs):
    return torch.autograd.grad(outs, ins, gs, allow_unused=True)


def _leaf(shape):
    return torch.zeros(shape, dtype=torch.float64, requires_grad=True)


def _d(a):
    return a.detach().to(torch.float64) if torch.is_tensor(a) else torch.from_numpy(np.asarray(a, np.float64))


# --------------------------------------------------------------------------------------- a6: K Jacobi sweeps (navier_stokes.py:139-145)
def _sweep(x):
    """J0 x: 0.25 * 4-neighbour sum on the interior, zero ring (the div-free part of ts.jacobi)."""
    y = torch.zeros_like(x)
    y[..., 1:-1, 1:-1] = 0.25 * (x[..., :-2, 1:-1] + x[..., 2:, 1:-1] + x[..., 1:-1, :-2] + x[..., 1:-1, 2:])
    return y


def _nsum(x):
    """4-neighbour sum with zeros outside the grid."""
    s = torch.zeros_like(x)
    s[..., 1:, :] += x[..., :-1, :]
    s[..., :-1, :] += x[..., 1:, :]
    s[..., :, 1:] += x[..., :, :-1]
    s[..., :, :-1] += x[..., :, 1:]
    return s


def jacobi_adjoint(g, K, absolute=False):
    """Transpose of (p, div) -> ts.jacobi(p, div, K): (g_p, g_div) = (0.25 S J0^(K-1) r, -0.25 sum_{j<K} J0^j r), r = M g."""
    g = _d(g)
    if absolute:
        g = g.abs()
    if K == 0:
        return g.clone(), torch.zeros_like(g)
    r = torch.zeros_like(g)
    r[..., 1:-1, 1:-1] = g[..., 1:-1, 1:-1]
    y, acc = r, r.clone()
    for _ in range(K - 1):
        y = _sweep(y)
        acc += y
    return 0.25 * _nsum(y), (0.25 if absolute else -0.25) * acc


# --------------------------------------------------------------------------------- a7: gradient subtract (navier_stokes.py:148-149)
def _grad_subtract_abs(u, v, p, dt):
    dt = abs(dt)
    u = torch.cat([u[..., :1, :], u[..., 1:-1, :] + dt * (p[..., 1:, :] + p[..., :-1, :]), u[..., -1:, :]], dim=-2)
    v = torch.cat([v[..., :, :1], v[..., :, 1:-1] + dt * (p[..., :, 1:] + p[..., :, :-1]), v[..., :, -1:]], dim=-1)
    return u, v


def project_adjoint(g_u, g_v, g_p_in, dt, absolute=False):
    """g_p of smk_project_adjoint: g_p_in plus the transpose of ts.grad_subtract applied to (g_u, g_v)."""
    gu, gv, gp = _d(g_u), _d(g_v), _d(g_p_in)
    if absolute:
        gu, gv, gp = gu.abs(), gv.abs(), gp.abs()
    u, v, p = _leaf(gu.shape), _leaf(gv.shape), _leaf(gp.shape)
    u2, v2 = (_grad_subtract_abs if absolute else ts.grad_subtract)(u, v, p, f32(dt))
    (gP,) = _grad([u2, v2], [p], [gu, gv])
    return gp + gP


# ----------------------------------------------- a3 + a4 + a5: buoyancy, the three diffusions and the divergence (navier_stokes.py:136, :154-160)
def _diffuse_abs(f, c):
    H, W = f.shape[-2:]
    iu = torch.clamp(torch.arange(H) - 1, 0, H - 1)
    idn = torch.clamp(torch.arange(H) + 1, 0, H - 1)
    jl = torch.clamp(torch.arange(W) - 1, 0, W - 1)
    jr = torch.clamp(torch.arange(W) + 1, 0, W - 1)
    return f + abs(c) * (f.index_select(-2, iu) + f.index_select(-2, idn) + f.index_select(-1, jl) + f.index_select(-1, jr) + 4 * f)


def _forces_diffuse_div(u, v, d, dt, c_uv, c_d, absolute):
    if absolute:
        v = torch.cat([v[..., :-1] + abs(dt) * (d * f32(0.1)), v[..., -1:]], dim=-1)
        u2, v2, d2 = _diffuse_abs(u, c_uv), _diffuse_abs(v, c_uv), _diffuse_abs(d, c_d)
        div = (u2[..., 1:, :] + u2[..., :-1, :] + v2[..., :, 1:] + v2[..., :, :-1]) / abs(dt)
        return u2, v2, d2, div
    v = torch.cat([v[..., :-1] + dt * (d * f32(0.1)), v[..., -1:]], dim=-1)
    u2, v2, d2 = ts.diffusion_step(u, c_uv), ts.diffusion_step(v, c_uv), ts.diffusion_step(d, c_d)
    return u2, v2, d2, ts.divergence(u2, v2, dt)


def forces_diffuse_div_adjoint(g_u, g_v, g_d, g_div, dt, c_uv, c_d, absolute=False):
    """(g_u, g_v, g_d) of smk_forces_diffuse_div_adjoint: the transpose of (u, v, d) -> (u_diff, v_diff, d_diff, div)."""
    gs = [_d(a) for a in (g_u, g_v, g_d, g_div)]
    if absolute:
        gs = [a.abs() for a in gs]
    u, v, d = _leaf(gs[0].shape), _leaf(gs[1].shape), _leaf(gs[2].shape)
    outs = _forces_diffuse_div(u, v, d, f32(dt), f32(c_uv), f32(c_d), absolute)
    return _grad(outs, [u, v, d], gs)


# ----------------------------------------------------------------------------------------- a2: add_smoke_source (navier_stokes.py:37-48)
def splat_adjoint(g_d, emitters, absolute=False):
    """d/d(intensity) of ts.add_sources: one value per emitter, flattened in list order.  The footprint is torch's fp32 one."""
    g = _d(g_d)
    if absolute:
        g = g.abs()
    h, w = g.shape[-2:]
    out = []
    for b, lst in enumerate(emitters):
        for (x, y, r) in lst:
            out.append((g[b] * ts.splat_weight(h, w, x, y, r).to(torch.float64)).sum())
    return torch.stack(out) if out else torch.zeros(0, dtype=torch.float64)


def splat_footprint(h, w, emitters):
    """Cells each emitter's adjoint sums over (its clipped bounding box), flattened like splat_adjoint."""
    out = []
    for lst in emitters:
        for (x, y, r) in lst:
            out.append(max(0, min(y + r, h - 1) - max(y - r, 0) + 1) * max(0, min(x + r, w - 1) - max(x - r, 0) + 1))
    return np.array(out, np.int64)


# ---------------------------------------------------------------------------------------- a10: advection_step (navier_stokes.py:74-95)
def _mesh(rows, cols, dtype):
    return torch.meshgrid(torch.arange(rows, dtype=dtype), torch.arange(cols, dtype=dtype), indexing="ij")


def back_trace(rows, cols, u, v, dt):
    """The fp32 back-trace positions (px, py) of every cell of a rows x cols field, before the clamp, computed exactly as
    ts.advection_step computes them (bit-equal to k_advect and k_adv_adj_trace).  u [B, h+1, w], v [B, h, w+1] fp32."""
    Y, X = _mesh(rows, cols, torch.float32)
    with torch.no_grad():
        u_i = ts.interpolate_velocity_u(u, Y, X)
        v_i = ts.interpolate_velocity_v(v, Y, X)
        return X - dt * u_i, Y - dt * v_i


def advect_adjoint(field, u, v, dt, g_out, scale=1.0, g_frame=None, fmul=None, absolute=False):
    """(g_field, g_u, g_v, count) of smk_advect_adjoint with accumulate = 0 and zero initial g_u / g_v.

    out = scale * bilinear(field at the clamped back-trace), frame = out + fmul*out.  The weights, the clamp's inclusive pass masks,
    the corner scatter and d/dpx, d/dpy are formed in float64 from the fp32 positions of back_trace().  count[cell]: how many
    (output cell, corner) terms the scatter adds into a field cell, the length of the kernel's sum there."""
    field = field.to(torch.float32)
    B, rows, cols = field.shape
    px, py = back_trace(rows, cols, u, v, f32(dt))
    pass_x = (px >= 0) & (px <= cols - 1)                  # torch.clamp's gradient mask
    pass_y = (py >= 0) & (py <= rows - 1)
    px = torch.clamp(px, 0, cols - 1)
    py = torch.clamp(py, 0, rows - 1)
    x0 = torch.clamp(torch.floor(px).long(), 0, cols - 1)
    y0 = torch.clamp(torch.floor(py).long(), 0, rows - 1)
    x1 = torch.clamp(x0 + 1, 0, cols - 1)
    y1 = torch.clamp(y0 + 1, 0, rows - 1)
    P, Q = px.double(), py.double()
    ax, bx, ay, by = x1.double() - P, P - x0.double(), y1.double() - Q, Q - y0.double()
    F = _d(field)
    e = _d(g_out) if g_out is not None else torch.zeros(B, rows, cols, dtype=torch.float64)
    gf = _d(g_frame) if g_frame is not None else None
    fm = _d(fmul) if fmul is not None else None
    if absolute:
        e, F = e.abs(), F.abs()
        gf = gf.abs() if gf is not None else None
        fm = fm.abs() if fm is not None else None
    if gf is not None:
        e = e + (gf + (fm * gf if fm is not None else 0.0))
    e = e * (abs(f32(scale)) if absolute else f32(scale))
    corners = ((y0, x0, ax * ay), (y0, x1, bx * ay), (y1, x0, ax * by), (y1, x1, bx * by))
    g_field = torch.zeros(B, rows * cols, dtype=torch.float64)
    count = torch.zeros(B, rows * cols, dtype=torch.float64)
    for yy, xx, wt in corners:
        idx = (yy * cols + xx).reshape(B, -1)
        g_field.scatter_add_(1, idx, (wt * e).reshape(B, -1))
        count.scatter_add_(1, idx, torch.ones_like(wt).expand(B, rows, cols).reshape(B, -1))
    f00, f01 = ts._gather(F, y0, x0), ts._gather(F, y0, x1)
    f10, f11 = ts._gather(F, y1, x0), ts._gather(F, y1, x1)
    if absolute:
        gpx = e * (ay * (f01 + f00) + by * (f11 + f10))
        gpy = e * (ax * (f10 + f00) + bx * (f11 + f01))
    else:
        gpx = e * (ay * (f01 - f00) + by * (f11 - f10))
        gpy = e * (ax * (f10 - f00) + bx * (f11 - f01))
    dd = abs(f32(dt)) if absolute else -f32(dt)
    du_i = torch.where(pass_x, dd * gpx, torch.zeros_like(gpx))          # px = X - dt * u_i
    dv_i = torch.where(pass_y, dd * gpy, torch.zeros_like(gpy))
    Yd, Xd = _mesh(rows, cols, torch.float64)
    U, V = _leaf(tuple(u.shape)), _leaf(tuple(v.shape))
    g_u, g_v = _grad([ts.interpolate_velocity_u(U, Yd, Xd), ts.interpolate_velocity_v(V, Yd, Xd)], [U, V], [du_i, dv_i])
    return g_field.reshape(B, rows, cols), g_u, g_v, count.reshape(B, rows, cols)


def advect_forward(field, u, v, dt, scale=1.0, fmul=None):
    """(out, frame) of smk_advect in float64 at the fp32 back-trace positions (frame None without fmul)."""
    field = field.to(torch.float32)
    _, rows, cols = field.shape
    px, py = back_trace(rows, cols, u, v, f32(dt))
    px = torch.clamp(px, 0, cols - 1).double()
    py = torch.clamp(py, 0, rows - 1).double()
    out = ts.bilinear_interpolate(_d(field), py, px) * f32(scale)
    return out, (out + _d(fmul) * out if fmul is not None else None)
