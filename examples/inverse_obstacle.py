"""Recover the emission rate of a source that sits below a wall with a gap, from observed frames (smokephysai_b200.autodiff).

    python examples/inverse_obstacle.py

A 64 x 64 box has a wall three cells thick across its middle rows, with a gap off centre (solid obstacles, DESIGN.md s5.7).  An
emitter below the wall injects smoke at every step, and a steady wind pushes it towards the wall, so the smoke piles up under the
wall and leaves through the gap.  The box is observed for 16 steps.  Starting from a guess of 0.3, L-BFGS fits the emission rate so
that the simulated frames match the observed ones.  Every loss evaluation is one differentiable rollout with obstacles=, sources=
and forcing=: the forward is set_obstacles + run_steps, and the backward runs through the masked step.  Needs a CUDA device.
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smokephysai_b200 import autodiff  # noqa: E402


def wall_with_gap(n):
    """Rows n/2 .. n/2 + 2 solid, except a gap of n/6 columns starting at column 5n/8."""
    S = np.zeros((n, n), bool)
    S[n // 2:n // 2 + 3, :] = True
    g0 = n // 2 + n // 8
    S[n // 2:n // 2 + 3, g0:g0 + max(2, n // 6)] = False
    return S


def problem(n=64, T=16, device="cuda"):
    """(rest state, emitters, forcing, wall mask, T) of the example."""
    zeros = lambda *s: torch.zeros(*s, device=device)
    rest = (zeros(n + 1, n), zeros(n, n + 1), zeros(n, n), zeros(n, n))               # u, v, p, d
    emitters = [(n // 3, n // 4, 6)]                                                  # (x, y, radius), below the wall
    wind = (zeros(n + 1, n), torch.full((n, n + 1), 20.0, device=device))             # dv > 0 moves smoke to higher rows
    return rest, emitters, wind, wall_with_gap(n), T


def fit(true_rate=1.3, guess=0.3, rounds=3, device="cuda", verbose=False):
    """-> (recovered rate, losses per round, relative change the wall makes to the observed frames)."""
    rest, emitters, wind, wall, T = problem(device=device)
    kw = dict(sources=emitters, forcing=wind, obstacles=wall)
    with torch.no_grad():                                                             # the observation
        observed, _ = autodiff.rollout(rest, T, intensities=torch.tensor([true_rate], device=device), **kw)
        open_box, _ = autodiff.rollout(rest, T, intensities=torch.tensor([true_rate], device=device), sources=emitters,
                                       forcing=wind)
    wall_effect = ((observed - open_box).norm() / open_box.norm()).item()

    x = torch.tensor([guess], device=device, requires_grad=True)
    opt = torch.optim.LBFGS([x], max_iter=50, tolerance_grad=1e-12, tolerance_change=1e-14, line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        frames, _ = autodiff.rollout(rest, T, intensities=x, **kw)
        loss = ((frames - observed) ** 2).sum()
        loss.backward()
        return loss

    losses = []
    for it in range(rounds):
        losses.append(opt.step(closure).item())
        if verbose:
            print("round %d: loss %.3e, rate %.6f" % (it, losses[-1], x.item()))
    return x.item(), losses, wall_effect


def main():
    rate, losses, wall_effect = fit(verbose=True)
    print("the wall changes the observed frames by %.1f%% (relative L2)" % (100 * wall_effect))
    print("true rate 1.3, recovered %.6f, relative error %.2e" % (rate, abs(rate - 1.3) / 1.3))


if __name__ == "__main__":
    main()
