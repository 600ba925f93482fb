"""Steer a plume: find a wind that pushes smoke sideways onto a target (smokephysai_b200.autodiff).

    python examples/steer_plume.py

A 64 x 64 simulation at rest holds a blob of smoke.  Left alone for 30 steps it rises straight up under the buoyancy; the target is
the same blob risen and shifted 12 cells to the right.  The control is a constant velocity forcing (du, dv) on a coarse 8 x 8 grid,
upsampled bilinearly by torch to the staggered shapes, so the parameterisation stays differentiable and smooth.  Adam fits the
coarse field so that the density after 30 steps matches the target.  Every loss evaluation is one differentiable rollout with
forcing=: the forward is run_steps(forcing=), and the backward gives the forcing's gradient.  Needs a CUDA device.
"""
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smokephysai_b200 import autodiff  # noqa: E402


def blob(n, x, y, r):
    i = torch.arange(n, device="cuda", dtype=torch.float32).view(-1, 1)
    j = torch.arange(n, device="cuda", dtype=torch.float32).view(1, -1)
    return torch.exp(-((j - x) ** 2 + (i - y) ** 2) / (2.0 * r * r))


def main():
    n, T, shift = 64, 30, 12
    torch.manual_seed(0)
    zeros = lambda *s: torch.zeros(1, *s, device="cuda")
    d0 = blob(n, 24, 20, 5.0)[None]
    rest = (zeros(n + 1, n), zeros(n, n + 1), zeros(n, n), d0)                     # u, v, p, d
    with torch.no_grad():
        _, (_, _, _, rise) = autodiff.rollout(rest, T)
    target = torch.roll(rise, shifts=shift, dims=-1)                               # the plume, pushed sideways

    coarse = torch.zeros(1, 2, 8, 8, device="cuda", requires_grad=True)            # (du, dv) on an 8 x 8 grid
    opt = torch.optim.Adam([coarse], lr=0.5)

    def forcing(c):
        du = F.interpolate(c[:, :1], size=(n + 1, n), mode="bilinear", align_corners=True)[:, 0]
        dv = F.interpolate(c[:, 1:], size=(n, n + 1), mode="bilinear", align_corners=True)[:, 0]
        return du, dv

    first = None
    for it in range(60):
        opt.zero_grad()
        _, (_, _, _, d) = autodiff.rollout(rest, T, forcing=forcing(coarse))
        loss = ((d - target) ** 2).sum()
        loss.backward()
        opt.step()
        first = loss.item() if first is None else first
        print("round %2d: loss %.4e" % (it, loss.item()))
    with torch.no_grad():
        _, (_, _, _, d) = autodiff.rollout(rest, T, forcing=forcing(coarse))
        final = ((d - target) ** 2).sum().item()
    print("loss %.4e -> %.4e (%.1fx lower)" % (first, final, first / final))


if __name__ == "__main__":
    main()
