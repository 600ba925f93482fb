"""Cost of solid obstacles (set_obstacles): the masked step always runs on the phase kernels.

    python tools/obstacle_bench.py [--out profiles/r10a_obstacles.json] [--repeats 5]

Workloads, each timed in one process with CUDA events around whole calls, the variants alternated `--repeats` times after a warm-up
of every variant (masks uploaded once, before the timing):
- c2: 256 x 128^2 simulations, K = 40, 20 steps, the data-loader emitter law splatted once after the reset
  (setup_grid(); add_sources(S); run_steps(20)):
  * none:       no mask (k_step_fused, one launch per call)
  * all_fluid:  an all-fluid mask (the phase path: the cost of leaving the fused kernel)
  * box:        a box, a partial wall and a single cell (DESIGN.md s5.7) in every simulation (phase path)
  * phases:     no mask with step_kernel="phases" (the same kernels without the four obstacle launches and the masked Jacobi)
- phase_1024: one 1024^2 simulation, K = 100, 5 steps, on the phase kernels: none / box;
- jacobi_share: the per-phase device time of the library's per-launch events (smk_profile_begin / _end) over one masked c2 call
  and one masked 1024^2 call, and of the same calls without a mask on the phase path: the Jacobi phase's milliseconds and share.
Prints one JSON object (and writes it to --out) with median ms, G cell-steps/s, launches per call, and the GPU's name, power
limit and maximum SM clock read in the same run.  Needs a GPU.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from smokephysai_b200 import NavierStokesSimulator, _lib  # noqa: E402
from continuous_sources_bench import gpu_info, loader_law, measure  # noqa: E402


def box_mask(h, w):
    """The box of rows 20-29 x columns 25-39 (scaled to the grid), a wall of rows h/2 .. h/2 + 2 over the first w/3 columns and the
    cell (5, 5)."""
    S = np.zeros((h, w), bool)
    S[20 * h // 64: 30 * h // 64, 25 * w // 64: 40 * w // 64] = True
    S[h // 2: h // 2 + 3, : w // 3] = True
    S[5, 5] = True
    return S


def variants(n, B, K, T, S, masks, **kw):
    out = {}
    for name, mask in masks.items():
        extra = {"step_kernel": "phases"} if name == "phases" else {}
        ns = NavierStokesSimulator((n, n), batch=B, jacobi_iters=K, **kw, **extra)
        if mask is not None:
            ns.set_obstacles(mask)

        def fn(ns=ns):
            ns.setup_grid()
            ns.add_sources(S)
            ns.run_steps(T, return_frames=False)
        out[name] = fn
    return out


def phase_share(fn):
    fn()
    torch.cuda.synchronize()
    _lib.profile_begin(1 << 16)
    fn()
    torch.cuda.synchronize()
    prof = _lib.profile_end()
    total = sum(ms for ms, _ in prof.values())
    return {"total_ms": total, "jacobi_ms": prof["jacobi"][0], "jacobi_launches": prof["jacobi"][1],
            "jacobi_share": prof["jacobi"][0] / total if total else None,
            "per_phase_ms": {k: ms for k, (ms, n) in prof.items() if n}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    res = {"gpu": gpu_info(torch.cuda.current_device()), "repeats": args.repeats}
    T = 20
    c2 = variants(128, 256, 40, T, loader_law(256, 128, 128, 1),
                {"none": None, "all_fluid": np.zeros((128, 128), bool), "box": box_mask(128, 128), "phases": None})
    res["c2"] = measure(c2, args.repeats, 256 * 128 * 128 * T)
    big = variants(1024, 1, 100, 5, [[(512, 512, 30, 1.0)]], {"none": None, "box": box_mask(1024, 1024)},
                  step_kernel="phases")
    res["phase_1024"] = measure(big, args.repeats, 1024 * 1024 * 5)
    res["jacobi_share"] = {"c2_box": phase_share(c2["box"]), "c2_phases": phase_share(c2["phases"]),
                           "phase_1024_box": phase_share(big["box"]), "phase_1024_none": phase_share(big["none"])}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
