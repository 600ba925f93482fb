"""Float64 references of the masked adjoint entries (smk_*_adjoint_ex with solid cells), each with its absolute-value twin, in the
style of tests/adjoint_reference.py:
    adjoint(..)                 A^T g in float64
    adjoint(.., absolute=True)  |A|^T |g|, the running-error scale of an fp32 evaluation of A^T g
The project and diffusion transposes go through float64 autograd of tests/obstacle_torch.py; the Jacobi transpose is written out
as DESIGN.md s5.7 derives it (float64 masked sweeps, then the output stencil), and tests/test_autodiff_obstacles_host.py checks it
against explicit matrices (J^T)^K.  S: bool tensor [h, w] or [B, h, w]; fields [B, rows, cols]."""
import torch

import adjoint_reference as ar
import obstacle_torch as ot
from oracle import torch_step as ts

f32 = ar.f32
_d, _leaf, _grad = ar._d, ar._leaf, ar._grad


def _S(S, like):
    return torch.as_tensor(S, dtype=torch.bool).expand(like.shape[:-2] + like.shape[-2:])


# ------------------------------------------------------------------------------------------------ masked Jacobi sweeps
def sweep(x, S):
    """J x: one masked sweep with div = 0 (a solid neighbour's slot takes the cell's own value; solid cells and the ring get 0)."""
    return ot.jacobi(x, torch.zeros_like(x), S, 1)


def jacobi_adjoint(g, S, K, absolute=False):
    """Transpose of (p, div) -> ot.jacobi(p, div, S, K):  with r = M g (M the fluid-interior mask), y = J^(K-1) r,
    g_p = J^T y (each neighbour slot of a fluid cell takes y of that neighbour, or y of the cell itself where the neighbour is
    solid; solid cells 0) and g_div = -0.25 sum_{j<K} J^j r.  J has no negative entry, so the absolute twin is the same map on |g|."""
    g = _d(g)
    if absolute:
        g = g.abs()
    S = _S(S, g)
    if K == 0:
        return g.clone(), torch.zeros_like(g)
    keep = ~S.clone()
    keep[..., 0, :] = keep[..., -1, :] = False
    keep[..., :, 0] = keep[..., :, -1] = False
    r = torch.where(keep, g, torch.zeros_like(g))
    y, acc = r, r.clone()
    for _ in range(K - 1):
        y = sweep(y, S)
        acc += y
    h, w = g.shape[-2:]
    gp = torch.zeros_like(g)
    for di, dj in ((-1, 0), (1, 0), (0, -1), (0, 1)):
        # slot (di, dj) of cell (i, j): neighbour n = (i + di, j + dj) inside the grid
        i0, i1 = max(0, -di), h - max(0, di)
        j0, j1 = max(0, -dj), w - max(0, dj)
        yc = y[..., i0:i1, j0:j1]
        yn = y[..., i0 + di:i1 + di, j0 + dj:j1 + dj]
        sn = S[..., i0 + di:i1 + di, j0 + dj:j1 + dj]
        gp[..., i0:i1, j0:j1] += torch.where(sn, yc, yn)
    gp = torch.where(S, torch.zeros_like(gp), 0.25 * gp)
    return gp, (0.25 if absolute else -0.25) * acc


def jacobi_matrix(S):
    """The explicit float64 matrix J [h*w, h*w] of one masked sweep with div = 0 (row c: what cell c's new value reads)."""
    S = torch.as_tensor(S, dtype=torch.bool)
    h, w = S.shape
    J = torch.zeros(h * w, h * w, dtype=torch.float64)
    for i in range(1, h - 1):
        for j in range(1, w - 1):
            if S[i, j]:
                continue
            c = i * w + j
            for a, b in ((i - 1, j), (i + 1, j), (i, j - 1), (i, j + 1)):
                if S[a, b]:
                    J[c, c] += 0.25
                else:
                    J[c, a * w + b] += 0.25
    return J


# ------------------------------------------------------------------------------------------ masked gradient subtract
def _grad_subtract_abs(u, v, p, S, dt):
    cu, cv = ot.faces(_S(S, p))
    dt = abs(dt)
    gu = u[..., 1:-1, :] + dt * (p[..., 1:, :] + p[..., :-1, :])
    gv = v[..., :, 1:-1] + dt * (p[..., :, 1:] + p[..., :, :-1])
    u = torch.cat([u[..., :1, :], torch.where(cu[..., 1:-1, :], u[..., 1:-1, :], gu), u[..., -1:, :]], dim=-2)
    v = torch.cat([v[..., :, :1], torch.where(cv[..., :, 1:-1], v[..., :, 1:-1], gv), v[..., :, -1:]], dim=-1)
    return u, v


def project_adjoint(g_u, g_v, g_p_in, S, dt, absolute=False):
    """g_p of smk_project_adjoint_ex: g_p_in plus the transpose of ot.grad_subtract applied to (g_u, g_v)."""
    gu, gv, gp = _d(g_u), _d(g_v), _d(g_p_in)
    if absolute:
        gu, gv, gp = gu.abs(), gv.abs(), gp.abs()
    u, v, p = _leaf(gu.shape), _leaf(gv.shape), _leaf(gp.shape)
    fwd = _grad_subtract_abs if absolute else (lambda u, v, p, S, dt: ot.grad_subtract(u, v, p, _S(S, p), dt))
    u2, v2 = fwd(u, v, p, S, f32(dt))
    (gP,) = _grad([u2, v2], [p], [gu, gv])
    return gp + gP


# -------------------------------------------------- buoyancy, the three diffusions, O1 and the divergence of the closed faces
def forces_diffuse_div(u, v, d, S, dt, c_uv, c_d, absolute=False):
    """(u_diff, v_diff, d_diff, div) of a masked step: the closed faces of the diffused u, v := 0 before the divergence."""
    cu, cv = ot.faces(_S(S, d))
    if absolute:
        u2, v2, d2, _ = ar._forces_diffuse_div(u, v, d, dt, c_uv, c_d, True)
        u2, v2 = ot.close(u2, cu), ot.close(v2, cv)
        return u2, v2, d2, (u2[..., 1:, :] + u2[..., :-1, :] + v2[..., :, 1:] + v2[..., :, :-1]) / abs(dt)
    v = torch.cat([v[..., :-1] + dt * (d * f32(0.1)), v[..., -1:]], dim=-1)
    u2, v2, d2 = ts.diffusion_step(u, c_uv), ts.diffusion_step(v, c_uv), ts.diffusion_step(d, c_d)
    u2, v2 = ot.close(u2, cu), ot.close(v2, cv)
    return u2, v2, d2, ts.divergence(u2, v2, dt)


def forces_diffuse_div_adjoint(g_u, g_v, g_d, g_div, S, dt, c_uv, c_d, absolute=False):
    """(g_u, g_v, g_d) of smk_forces_diffuse_div_adjoint_ex."""
    gs = [_d(a) for a in (g_u, g_v, g_d, g_div)]
    if absolute:
        gs = [a.abs() for a in gs]
    u, v, d = _leaf(gs[0].shape), _leaf(gs[1].shape), _leaf(gs[2].shape)
    outs = forces_diffuse_div(u, v, d, S, f32(dt), f32(c_uv), f32(c_d), absolute)
    return _grad(outs, [u, v, d], gs)
