"""Torch-eager restatement of the reference step (src/physics/navier_stokes.py:37-173, fractal_generator.py:62).

TEST INFRASTRUCTURE ONLY: the gradient oracle of smokephysai_b200.autodiff, never the product.

Written with the reference's ops in the reference's association (SURVEY.md s3.1, s8a), so on the CPU in fp32 its forward is
bit-equal to the C oracle (tests/test_autodiff_host.py) and torch autograd through it *is* the reference's gradient:
floor has no gradient, torch.clamp passes it where lo <= x <= hi, bilinear weights come from the clamped integer corners,
index gathers scatter-add their gradient.  Every function takes fields with any leading (batch) dimensions.
"""
import numpy as np
import torch
import torch.nn.functional as F


def coefs(dt, viscosity):
    """(c_uv, c_d): dt*viscosity and dt*(viscosity*0.1) formed in Python double, as navier_stokes.py:72 / :160."""
    return float(dt) * float(viscosity), float(dt) * (float(viscosity) * 0.1)


def _gather(field, y, x):
    """field[..., y, x] for integer index grids y, x [..., H', W'] (leading dims broadcast against the field's)."""
    Hg, Wg = field.shape[-2:]
    idx = y * Wg + x
    lead = torch.broadcast_shapes(field.shape[:-2], idx.shape[:-2])
    flat = field.reshape(field.shape[:-2] + (Hg * Wg,)).expand(lead + (Hg * Wg,))
    out = torch.gather(flat, -1, idx.expand(lead + tuple(idx.shape[-2:])).reshape(lead + (-1,)))
    return out.reshape(lead + tuple(idx.shape[-2:]))


def bilinear_interpolate(field, y, x):
    """navier_stokes.py:111-131: corners clamped after the +1, weights from the clamped corners."""
    Hg, Wg = field.shape[-2:]
    x0 = torch.floor(x).long()
    x1 = x0 + 1
    y0 = torch.floor(y).long()
    y1 = y0 + 1
    x0 = torch.clamp(x0, 0, Wg - 1)
    x1 = torch.clamp(x1, 0, Wg - 1)
    y0 = torch.clamp(y0, 0, Hg - 1)
    y1 = torch.clamp(y1, 0, Hg - 1)
    wa = (x1.float() - x) * (y1.float() - y)
    wb = (x - x0.float()) * (y1.float() - y)
    wc = (x1.float() - x) * (y - y0.float())
    wd = (x - x0.float()) * (y - y0.float())
    return wa * _gather(field, y0, x0) + wb * _gather(field, y0, x1) + wc * _gather(field, y1, x0) + wd * _gather(field, y1, x1)


def interpolate_velocity_u(u, Y, X):
    """navier_stokes.py:97-102"""
    w = u.shape[-1]
    return bilinear_interpolate(u, Y, torch.clamp(X + 0.5, 0, w - 1))


def interpolate_velocity_v(v, Y, X):
    """navier_stokes.py:104-109"""
    h = v.shape[-2]
    return bilinear_interpolate(v, torch.clamp(Y + 0.5, 0, h - 1), X)


def advection_step(field, u, v, dt):
    """navier_stokes.py:74-95: semi-Lagrangian back-trace of every cell of `field` by (u, v)."""
    H, W = field.shape[-2:]
    Y, X = torch.meshgrid(torch.arange(H, dtype=torch.float32, device=field.device),
                          torch.arange(W, dtype=torch.float32, device=field.device), indexing="ij")
    u_i = interpolate_velocity_u(u, Y, X)
    v_i = interpolate_velocity_v(v, Y, X)
    prev_x = X - dt * u_i
    prev_y = Y - dt * v_i
    prev_x = torch.clamp(prev_x, 0, W - 1)
    prev_y = torch.clamp(prev_y, 0, H - 1)
    return bilinear_interpolate(field, prev_y, prev_x)


def diffusion_step(field, c):
    """navier_stokes.py:50-72 with c = dt*viscosity: replicate padding, ((up + down) + left) + right - 4f."""
    H, W = field.shape[-2:]
    dev = field.device
    iu = torch.clamp(torch.arange(H, device=dev) - 1, 0, H - 1)
    idn = torch.clamp(torch.arange(H, device=dev) + 1, 0, H - 1)
    jl = torch.clamp(torch.arange(W, device=dev) - 1, 0, W - 1)
    jr = torch.clamp(torch.arange(W, device=dev) + 1, 0, W - 1)
    lap = field.index_select(-2, iu) + field.index_select(-2, idn) + field.index_select(-1, jl) + field.index_select(-1, jr) \
        - 4 * field
    return field + c * lap


def buoyancy(v, d, dt):
    """navier_stokes.py:154-155: v[:, :-1] += dt*(density*0.1) (column w untouched)."""
    return torch.cat([v[..., :-1] + dt * (d * 0.1), v[..., -1:]], dim=-1)


def forces_diffuse(u, v, d, dt, viscosity):
    """navier_stokes.py:154-160: buoyancy, then the three diffusions."""
    c_uv, c_d = coefs(dt, viscosity)
    v = buoyancy(v, d, dt)
    return diffusion_step(u, c_uv), diffusion_step(v, c_uv), diffusion_step(d, c_d)


def divergence(u, v, dt):
    """navier_stokes.py:136"""
    return (u[..., 1:, :] - u[..., :-1, :] + v[..., :, 1:] - v[..., :, :-1]) / dt


def jacobi(p, div, K):
    """navier_stokes.py:139-145: K sweeps, zero ring every sweep."""
    if K > 0 and (p.shape[-2] < 3 or p.shape[-1] < 3):
        return p * 0.0              # no interior: every cell is ring (padding an empty interior would not give p's shape)
    for _ in range(K):
        inner = 0.25 * (p[..., :-2, 1:-1] + p[..., 2:, 1:-1] + p[..., 1:-1, :-2] + p[..., 1:-1, 2:] - div[..., 1:-1, 1:-1])
        p = F.pad(inner, (1, 1, 1, 1))
    return p


def grad_subtract(u, v, p, dt):
    """navier_stokes.py:148-149: u[1:-1] -= dt*(p[1:] - p[:-1]); v[:, 1:-1] -= dt*(p[:, 1:] - p[:, :-1])."""
    u = torch.cat([u[..., :1, :], u[..., 1:-1, :] - dt * (p[..., 1:, :] - p[..., :-1, :]), u[..., -1:, :]], dim=-2)
    v = torch.cat([v[..., :, :1], v[..., :, 1:-1] - dt * (p[..., :, 1:] - p[..., :, :-1]), v[..., :, -1:]], dim=-1)
    return u, v


def step(u, v, p, d, dt=0.01, viscosity=0.001, K=20, fmul=None):
    """One NavierStokesSimulator.step() (navier_stokes.py:151-173) -> (frame, (u, v, p, d)).  fmul: the fractal multiply
    frame + fmul*frame of SmokeSimulator.simulate_step (fractal_generator.py:62), applied to the returned copy only."""
    u, v, d = forces_diffuse(u, v, d, dt, viscosity)
    div = divergence(u, v, dt)
    p = jacobi(p, div, K)
    u, v = grad_subtract(u, v, p, dt)
    u = advection_step(u, u, v, dt)
    v = advection_step(v, u, v, dt)
    d = advection_step(d, u, v, dt)
    d = d * 0.995
    frame = d if fmul is None else d + fmul * d
    return frame, (u, v, p, d)


def rollout(state, nsteps, dt=0.01, viscosity=0.001, K=20, fmul=None):
    """nsteps steps -> (frames [..., T, h, w], final state), as smokephysai_b200.autodiff.rollout."""
    u, v, p, d = state
    frames = []
    for _ in range(nsteps):
        fr, (u, v, p, d) = step(u, v, p, d, dt, viscosity, K, fmul)
        frames.append(fr)
    return torch.stack(frames, dim=-3), (u, v, p, d)


def splat_weight(h, w, x, y, radius):
    """The Gaussian footprint of add_smoke_source (navier_stokes.py:37-48) as an [h, w] fp32 tensor, zero outside."""
    i = torch.arange(h, dtype=torch.int64).view(-1, 1)
    j = torch.arange(w, dtype=torch.int64).view(1, -1)
    dist = torch.sqrt(((j - x) ** 2 + (i - y) ** 2).float())
    wgt = torch.exp(-(dist * dist) / np.float32(2.0 * ((radius / 3.0) ** 2)))
    return torch.where(dist <= radius, wgt, torch.zeros_like(wgt))


def add_sources(d, emitters, intensities):
    """d [B, h, w] plus emitters[b] = [(x, y, radius), ...] with the flattened intensities, in list order."""
    h, w = d.shape[-2:]
    out, k = [], 0
    for b, lst in enumerate(emitters):
        db = d[b]
        for (x, y, r) in lst:
            db = db + intensities[k] * splat_weight(h, w, x, y, r).to(d.device)
            k += 1
        out.append(db)
    return torch.stack(out)
