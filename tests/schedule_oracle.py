"""Source schedules on the torch restatement of the step (oracle/torch_step.py): row t of the schedule is added to the density at
the head of step t, in list order, as NavierStokesSimulator.run_steps(schedule=) does; an entry with radius < 0 adds nothing.
Autograd through it is the gradient oracle of smokephysai_b200.autodiff.rollout(..., schedule=, intensities=)."""
import numpy as np
import torch

from oracle import torch_step as ts


def add_row(d, xy, radius, intensities, weight=ts.splat_weight):
    """d [B, h, w] plus row xy [B, E, 2], radius [B, E], intensities [B, E] (a tensor), in list order per simulation.
    weight(h, w, x, y, r) gives an emitter's footprint (default: torch's own expf; the host tests pass the C oracle's)."""
    h, w = d.shape[-2:]
    out = []
    for b in range(d.shape[0]):
        db = d[b]
        for e in range(radius.shape[1]):
            r = int(radius[b, e])
            if r >= 0:
                db = db + intensities[b, e] * weight(h, w, int(xy[b, e, 0]), int(xy[b, e, 1]), r).to(d.device)
        out.append(db)
    return torch.stack(out)


def rollout(state, nsteps, dt=0.01, viscosity=0.001, K=20, fmul=None, xy=None, radius=None, intensities=None,
            weight=ts.splat_weight):
    """ts.rollout with schedule row t applied before step t; [B, ...] fields, xy / radius numpy [T, B, E, ...]."""
    u, v, p, d = state
    frames = []
    for t in range(nsteps):
        if xy is not None:
            d = add_row(d, np.asarray(xy[t]), np.asarray(radius[t]), intensities[t], weight)
        fr, (u, v, p, d) = ts.step(u, v, p, d, dt, viscosity, K, fmul)
        frames.append(fr)
    return torch.stack(frames, dim=-3), (u, v, p, d)


def moving_schedule(T, B, h, w, seed=0, emax=3, pad=True):
    """A schedule whose emitters move by one cell and change intensity at every step: simulation b has 1 .. emax emitters
    (padded to emax with radius -1 entries when pad), starting at data-loader positions.  -> numpy (xy, radius, intensity)."""
    rng = np.random.default_rng(seed)
    E = emax
    xy = np.zeros((T, B, E, 2), np.int64)
    radius = np.full((T, B, E), -1, np.int32)
    inten = np.zeros((T, B, E), np.float32)
    for b in range(B):
        n = int(rng.integers(1, emax + 1)) if pad else emax
        x0 = rng.integers(20, max(21, w - 20), n)
        y0 = rng.integers(20, max(21, h - 20), n)
        dx = rng.choice([-1, 1], n)
        dy = rng.choice([-1, 0, 1], n)
        i0 = rng.uniform(0.5, 2.0, n)
        for t in range(T):
            xy[t, b, :n, 0] = x0 + dx * t
            xy[t, b, :n, 1] = y0 + dy * t
            radius[t, b, :n] = 8
            inten[t, b, :n] = i0 * (1.0 + 0.5 * np.sin(0.7 * t + np.arange(n)))
    return xy, radius, inten


def rows_as_lists(schedule, t):
    """Row t of a numpy schedule as add_sources' per-simulation lists, padded entries left out."""
    xy, radius, inten = schedule
    return [[(int(xy[t, b, e, 0]), int(xy[t, b, e, 1]), int(radius[t, b, e]), float(inten[t, b, e]))
             for e in range(radius.shape[2]) if radius[t, b, e] >= 0] for b in range(radius.shape[1])]
