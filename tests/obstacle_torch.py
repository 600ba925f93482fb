"""Solid obstacles on the torch restatement of the step (oracle/torch_step.py) -- the gradient oracle of
smokephysai_b200.autodiff.rollout(..., obstacles=).

The masked step of DESIGN.md s5.7 written with torch.where on the reference's ops, in the association of tests/obstacle_oracle.py's
numpy restatement, so its fp32 CPU forward is bit-equal to smk_oracle_step_obst and autograd through it is the masked step's
gradient: torch.where passes the gradient to the branch it selected, so a face set to +0.0 passes none back.  Every function takes
fields with any leading (batch) dimensions; the mask S is a bool tensor [h, w] or [B, h, w].  The functions are dtype-generic, so
tests/test_autodiff_obstacles_host.py also runs them in float64 for the transpose identities."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import torch_step as ts
from schedule_oracle import add_row


def faces(S):
    """(closed u faces [.., h+1, w], closed v faces [.., h, w+1]) of the solid cells S [.., h, w] (bool tensors)."""
    cu = F.pad(S, (0, 0, 0, 1)) | F.pad(S, (0, 0, 1, 0))
    cv = F.pad(S, (0, 1)) | F.pad(S, (1, 0))
    return cu, cv


def close(f, closed):
    """O1 / O4: the closed entries of f := +0.0."""
    return torch.where(closed, torch.zeros((), dtype=f.dtype), f)


def jacobi(p, div, S, K):
    """K masked sweeps: a fluid interior cell takes its own p in place of a solid neighbour's; solid cells and the ring get +0.0."""
    if K > 0 and (p.shape[-2] < 3 or p.shape[-1] < 3):
        return p * 0.0
    Si = S[..., 1:-1, 1:-1]
    for _ in range(K):
        c = p[..., 1:-1, 1:-1]
        s = torch.where(S[..., :-2, 1:-1], c, p[..., :-2, 1:-1]) + torch.where(S[..., 2:, 1:-1], c, p[..., 2:, 1:-1])
        s = s + torch.where(S[..., 1:-1, :-2], c, p[..., 1:-1, :-2])
        s = s + torch.where(S[..., 1:-1, 2:], c, p[..., 1:-1, 2:])
        inner = torch.where(Si, torch.zeros((), dtype=p.dtype), 0.25 * (s - div[..., 1:-1, 1:-1]))
        p = F.pad(inner, (1, 1, 1, 1))
    return p


def grad_subtract(u, v, p, S, dt):
    """The gradient subtract on open faces only (rows 1 .. h-1 of u, columns 1 .. w-1 of v)."""
    cu, cv = faces(S)
    gu = u[..., 1:-1, :] - dt * (p[..., 1:, :] - p[..., :-1, :])
    gv = v[..., :, 1:-1] - dt * (p[..., :, 1:] - p[..., :, :-1])
    u = torch.cat([u[..., :1, :], torch.where(cu[..., 1:-1, :], u[..., 1:-1, :], gu), u[..., -1:, :]], dim=-2)
    v = torch.cat([v[..., :, :1], torch.where(cv[..., :, 1:-1], v[..., :, 1:-1], gv), v[..., :, -1:]], dim=-1)
    return u, v


def step(u, v, p, d, S, dt=0.01, viscosity=0.001, K=20, fmul=None):
    """One masked NavierStokesSimulator step -> (frame, (u, v, p, d)); fmul as ts.step."""
    cu, cv = faces(S)
    u, v, d = ts.forces_diffuse(u, v, d, dt, viscosity)
    u, v = close(u, cu), close(v, cv)                                                  # O1
    div = ts.divergence(u, v, dt)
    p = jacobi(p, div, S, K)
    u, v = grad_subtract(u, v, p, S, dt)
    u_adv = ts.advection_step(u, u, v, dt)
    v_adv = ts.advection_step(v, u_adv, v, dt)                                         # reads the u before O4
    u_adv, v_adv = close(u_adv, cu), close(v_adv, cv)                                  # O4
    d = ts.advection_step(d, u_adv, v_adv, dt) * 0.995
    d = close(d, S)                                                                    # O3
    frame = d if fmul is None else d + fmul * d
    return frame, (u_adv, v_adv, p, d)


def rollout(state, nsteps, S, dt=0.01, viscosity=0.001, K=20, fmul=None, sources=None, intensities=None, du=None, dv=None,
            xy=None, radius=None):
    """nsteps masked steps -> (frames [..., T, h, w], final state), as autodiff.rollout(..., obstacles=S).  At the head of each
    step: continuous sources (emitters[b] = [(x, y, r), ...] with the flattened intensities) or a schedule row (numpy xy / radius,
    intensities [T, B, E]), then the forcing (du / dv constant, or [T, ...] per step)."""
    u, v, p, d = state
    per_step = du is not None and du.dim() == u.dim() + 1
    frames = []
    for t in range(nsteps):
        if sources is not None:
            d = ts.add_sources(d, sources, intensities)
        if xy is not None:
            d = add_row(d, np.asarray(xy[t]), np.asarray(radius[t]), intensities[t])
        if du is not None:
            u = u + (du[t] if per_step else du)
            v = v + (dv[t] if per_step else dv)
        fr, (u, v, p, d) = step(u, v, p, d, S, dt, viscosity, K, fmul)
        frames.append(fr)
    return torch.stack(frames, dim=-3), (u, v, p, d)

