"""Recover emitter intensities from observed frames by gradient descent through the simulator (smokephysai_b200.autodiff).

    python examples/inverse_sources.py

A 64 x 64 simulation at rest with three emitters of unknown intensity is observed for 10 steps.  Starting from intensities
of 1.0, L-BFGS fits the intensities so that the simulated frames match the observed ones; every loss evaluation is one
differentiable rollout (forward with checkpoints, backward on the adjoint kernels).  Needs a CUDA device.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smokephysai_b200 import autodiff  # noqa: E402


def main():
    n, T = 64, 10
    emitters = [(20, 24, 8), (40, 30, 8), (30, 44, 6)]               # (x, y, radius)
    true = torch.tensor([1.5, 0.7, 1.1], device="cuda")
    zeros = lambda *s: torch.zeros(*s, device="cuda")
    rest = (zeros(n + 1, n), zeros(n, n + 1), zeros(n, n))             # u, v, p

    with torch.no_grad():                                              # the observation
        observed, _ = autodiff.rollout(rest + (autodiff.add_sources(zeros(n, n), emitters, true),), T)

    x = torch.ones(3, device="cuda", requires_grad=True)
    opt = torch.optim.LBFGS([x], max_iter=100, tolerance_grad=1e-12, tolerance_change=1e-14, line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        frames, _ = autodiff.rollout(rest + (autodiff.add_sources(zeros(n, n), emitters, x),), T)
        loss = ((frames - observed) ** 2).sum()
        loss.backward()
        return loss

    for it in range(3):
        loss = opt.step(closure)
        print("round %d: loss %.3e, intensities %s" % (it, loss.item(), [round(v, 6) for v in x.tolist()]))
    rel = ((x.detach() - true).abs() / true).max().item()
    print("true %s, recovered %s, max relative error %.2e" % (true.tolist(), x.tolist(), rel))


if __name__ == "__main__":
    main()
