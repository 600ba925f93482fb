"""Cost of reverse mode through solid obstacles: autodiff.rollout(..., obstacles=) forward and backward.

    python tools/autodiff_obstacle_bench.py [--out FILE] [--repeats 5]

Workloads (loss = sum of the frames squared, gradients of all four state fields):
- b64_128: 64 x 128^2 simulations, K = 40, T = 20;
- g1024: one 1024^2 simulation, K = 100, T = 20.
Variants of each: no mask (the step kernel the library picks), an all-fluid mask (the masked entries on the phase path), and the
box mask of tools/obstacle_bench.py (a box, a partial wall and a single cell).  Each call is timed with CUDA events: the forward
(the checkpointed rollout) and the backward separately; the variants are alternated `--repeats` times after a warm-up of each.  A
separate pass records the per-phase device time of one backward with the library's per-launch events (smk_profile_begin / _end):
the Jacobi adjoint chains run as the "jacobi" phase.  Prints one JSON object (and writes it to --out) with the GPU's name, power
limit and maximum SM clock read in the same run.  Needs a GPU.
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from smokephysai_b200 import _lib, autodiff  # noqa: E402
from continuous_sources_bench import gpu_info  # noqa: E402
from obstacle_bench import box_mask  # noqa: E402


def start_state(B, n, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s, scale=1.0: torch.randn(*s, generator=g, device="cuda") * scale
    return (r(B, n + 1, n, scale=20.0), r(B, n, n + 1, scale=20.0), torch.zeros(B, n, n, device="cuda"),
            torch.rand(B, n, n, generator=g, device="cuda"))


def make_call(B, n, K, T, mask):
    base = start_state(B, n)

    def run():
        st = tuple(t.clone().requires_grad_(True) for t in base)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        frames, final = autodiff.rollout(st, T, jacobi_iters=K, obstacles=mask)
        loss = frames.square().sum()
        e1.record()
        loss.backward()
        e2.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), e1.elapsed_time(e2)
    return run


def backward_phases(run):
    """Per-phase device ms of one backward (the forward runs outside the profiled window)."""
    torch.cuda.synchronize()
    holder = {}
    orig = autodiff._reverse

    def wrapped(*a, **k):
        torch.cuda.synchronize()
        _lib.profile_begin(1 << 18)
        out = orig(*a, **k)
        torch.cuda.synchronize()
        holder["prof"] = _lib.profile_end()
        return out
    autodiff._reverse = wrapped
    try:
        run()
    finally:
        autodiff._reverse = orig
    prof = holder["prof"]
    total = sum(ms for ms, _ in prof.values())
    return {"total_ms": total, "per_phase_ms": {k: ms for k, (ms, n) in prof.items() if n},
            "launches": sum(n for _, n in prof.values())}


def workload(B, n, K, T, repeats):
    calls = {"none": make_call(B, n, K, T, None), "all_fluid": make_call(B, n, K, T, np.zeros((n, n), bool)),
             "box": make_call(B, n, K, T, box_mask(n, n))}
    for run in calls.values():
        run()
        run()
    fw = {k: [] for k in calls}
    bw = {k: [] for k in calls}
    for _ in range(repeats):
        for k, run in calls.items():
            f, b = run()
            fw[k].append(f)
            bw[k].append(b)
    res = {"B": B, "n": n, "K": K, "T": T}
    for k in calls:
        res[k] = {"forward_ms": statistics.median(fw[k]), "backward_ms": statistics.median(bw[k]),
                  "forward_samples_ms": fw[k], "backward_samples_ms": bw[k]}
    res["backward_phases"] = {k: backward_phases(calls[k]) for k in calls}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    res = {"gpu": gpu_info(torch.cuda.current_device()), "repeats": args.repeats}
    res["b64_128"] = workload(64, 128, 40, 20, args.repeats)
    res["g1024"] = workload(1, 1024, 100, 20, args.repeats)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
