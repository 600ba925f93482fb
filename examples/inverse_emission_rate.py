"""Recover one emitter's emission history, one intensity per step, from observed frames (smokephysai_b200.autodiff).

    python examples/inverse_emission_rate.py

A 64 x 64 simulation at rest has one emitter that drifts by a cell per step and whose intensity changes at every step.  It is
observed for 10 steps.  Starting from a constant guess of 0.5, L-BFGS fits the 10 intensities so that the simulated frames match
the observed ones.  Every loss evaluation is one differentiable rollout with a source schedule: the forward is
run_steps(schedule=), and the backward gives each step's intensity its own gradient.  Needs a CUDA device.
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smokephysai_b200 import autodiff  # noqa: E402


def main():
    n, T = 64, 10
    xy = np.array([[[(32 + (t % 3) - 1, 40 - t)]] for t in range(T)], np.int64)    # [T, B = 1, E = 1, 2]: (x, y)
    radius = np.full((T, 1, 1), 8, np.int32)
    true = torch.tensor(1.0 + 0.5 * np.sin(np.arange(T)), dtype=torch.float32, device="cuda").view(T, 1, 1)
    zeros = lambda *s: torch.zeros(1, *s, device="cuda")
    rest = (zeros(n + 1, n), zeros(n, n + 1), zeros(n, n), zeros(n, n))            # u, v, p, d

    with torch.no_grad():                                                          # the observation
        observed, _ = autodiff.rollout(rest, T, schedule=(xy, radius), intensities=true)

    x = torch.full((T, 1, 1), 0.5, device="cuda", requires_grad=True)
    opt = torch.optim.LBFGS([x], max_iter=200, tolerance_grad=1e-12, tolerance_change=1e-14, line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        frames, _ = autodiff.rollout(rest, T, schedule=(xy, radius), intensities=x)
        loss = ((frames - observed) ** 2).sum()
        loss.backward()
        return loss

    for it in range(3):
        loss = opt.step(closure)
        print("round %d: loss %.3e" % (it, loss.item()))
    rel = ((x.detach() - true).norm() / true.norm()).item()
    print("true      %s" % [round(v, 6) for v in true.flatten().tolist()])
    print("recovered %s" % [round(v, 6) for v in x.detach().flatten().tolist()])
    print("relative error %.2e" % rel)


if __name__ == "__main__":
    main()
