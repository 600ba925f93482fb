"""Velocity forcing on the torch restatement of the step (oracle/torch_step.py): du_t and dv_t are added to u and v at the head of
step t, after the emitters and before the buoyancy, as NavierStokesSimulator.run_steps(forcing=) does.  Autograd through it is the
gradient oracle of smokephysai_b200.autodiff.rollout(..., forcing=)."""
import numpy as np
import torch

from oracle import torch_step as ts
from schedule_oracle import add_row


def rollout(state, nsteps, dt=0.01, viscosity=0.001, K=20, fmul=None, du=None, dv=None, xy=None, radius=None, intensities=None):
    """ts.rollout with the forcing added before step t: du [B, h+1, w] / dv [B, h, w+1] at every step, or [T, B, ...] per step;
    an optional schedule (numpy xy / radius [T, B, E, ...], intensities [T, B, E]) splatted first."""
    u, v, p, d = state
    per_step = du is not None and du.dim() == 4
    frames = []
    for t in range(nsteps):
        if xy is not None:
            d = add_row(d, np.asarray(xy[t]), np.asarray(radius[t]), intensities[t])
        if du is not None:
            u = u + (du[t] if per_step else du)
            v = v + (dv[t] if per_step else dv)
        fr, (u, v, p, d) = ts.step(u, v, p, d, dt, viscosity, K, fmul)
        frames.append(fr)
    return torch.stack(frames, dim=-3), (u, v, p, d)


def wind(T, B, h, w, seed=0, strength=150.0):
    """A per-step forcing [T, B, h+1, w] / [T, B, h, w+1] (numpy float32): a smooth field that turns from step to step plus noise,
    scaled so that dt * |u| exceeds a cell within a few steps (dt = 0.01), and nonzero on u's row h and v's column w."""
    rng = np.random.default_rng(seed)
    yu, xu = np.meshgrid(np.arange(h + 1) / max(h, 1), np.arange(w) / max(w, 1), indexing="ij")
    yv, xv = np.meshgrid(np.arange(h) / max(h, 1), np.arange(w + 1) / max(w, 1), indexing="ij")
    du = np.empty((T, B, h + 1, w), np.float32)
    dv = np.empty((T, B, h, w + 1), np.float32)
    for b in range(B):
        ph = rng.uniform(0, 2 * np.pi, 2)
        for t in range(T):
            a = 0.6 * t + ph[0]
            du[t, b] = strength * (np.cos(a) * np.sin(np.pi * yu + ph[1]) + 0.3 * rng.standard_normal(yu.shape))
            dv[t, b] = strength * (np.sin(a) * np.cos(np.pi * xv + ph[1]) + 0.3 * rng.standard_normal(yv.shape))
    return du, dv
