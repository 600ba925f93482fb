"""A plume around a box: smoke rises from a burning stick, meets a solid box and splits around it (set_obstacles).

    python examples/obstacle_plume.py [--out obstacle_plume.npz] [--steps 200]

A 128 x 128 simulation with a continuous emitter at row 30 and a 16 x 40 box at rows 70-85.  The reference's buoyancy adds to v,
so the plume travels towards larger row indices, meets the box and flows around it.  The frames are written to an .npz file
(frames [steps, h, w] float32 and the mask) and a coarse text picture of the last frame is printed.  Needs a CUDA device.
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smokephysai_b200 import NavierStokesSimulator  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="obstacle_plume.npz")
    ap.add_argument("--steps", type=int, default=200)
    args = ap.parse_args()
    n = 128
    solid = np.zeros((n, n), bool)
    solid[70:86, 44:84] = True                                      # the box, across the plume's path
    sim = NavierStokesSimulator((n, n), dt=0.05, viscosity=0.001, device="cuda", jacobi_iters=100)
    sim.set_obstacles(solid)
    sim.set_continuous_sources([[(64, 30, 6, 0.5)]])                # a stick that keeps burning
    frames = sim.run_steps(args.steps).cpu().numpy()
    np.savez_compressed(args.out, frames=frames, solid=solid)
    last = frames[-1]
    assert not last[solid].any(), "no smoke inside the box"
    shades = " .:-=+*#%@"
    top = max(float(last.max()), 1e-6)
    for i in range(0, n, 4):
        print("".join("X" if solid[i, j] else shades[min(9, int(9 * last[i, j] / top))] for j in range(0, n, 2)))
    print("wrote %s: frames %s" % (args.out, frames.shape))


if __name__ == "__main__":
    main()
