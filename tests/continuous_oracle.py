"""Continuous sources on the torch restatement of the step (oracle/torch_step.py): the emitters are added to the density at the
head of every step, in list order, as NavierStokesSimulator.set_continuous_sources does.  Autograd through it is the gradient
oracle of smokephysai_b200.autodiff.rollout(..., sources=, intensities=)."""
import torch

from oracle import torch_step as ts


def add_sources(d, emitters, intensities, weight=ts.splat_weight):
    """d [B, h, w] plus emitters[b] = [(x, y, radius), ...] with the flattened intensities, in list order.  weight(h, w, x, y, r)
    gives an emitter's footprint (default: torch's own expf; the host tests pass the C oracle's for bit-equality)."""
    h, w = d.shape[-2:]
    out, k = [], 0
    for b, lst in enumerate(emitters):
        db = d[b]
        for (x, y, r) in lst:
            db = db + intensities[k] * weight(h, w, x, y, r).to(d.device)
            k += 1
        out.append(db)
    return torch.stack(out)


def rollout(state, nsteps, dt=0.01, viscosity=0.001, K=20, fmul=None, sources=None, intensities=None, weight=ts.splat_weight):
    """ts.rollout with the continuous sources applied before every step; [B, ...] fields."""
    u, v, p, d = state
    frames = []
    for _ in range(nsteps):
        if sources is not None:
            d = add_sources(d, sources, intensities, weight)
        fr, (u, v, p, d) = ts.step(u, v, p, d, dt, viscosity, K, fmul)
        frames.append(fr)
    return torch.stack(frames, dim=-3), (u, v, p, d)
