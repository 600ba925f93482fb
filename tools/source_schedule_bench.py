"""Cost of source schedules (run_steps(schedule=)): emitters that move and change intensity at every step.

    python tools/source_schedule_bench.py [--out profiles/r08a_source_schedule.json] [--repeats 5]

Workloads, each timed in one process with CUDA events around whole calls (a host clock for the packing), the variants alternated
`--repeats` times after a warm-up of every variant:
- c2: 256 x 128^2 simulations, K = 40, 20 steps, 1-3 emitters of radius 8 per simulation that move one cell per step and change
  intensity at every step:
  * schedule:       setup_grid(); run_steps(20, schedule=S) with S numpy arrays: the call with its packing and H2D upload
  * schedule_cuda:  the same with S already CUDA tensors (packing on the device, no upload)
  * continuous:     setup_grid(); run_steps(20) with set_continuous_sources(row 0): the same emitter counts, not moving
  * host_loop:      setup_grid(); 20 x [add_sources(S[t]); step()]  (what a user writes without the feature)
  and pack_ms: the host time of pack_schedule on the numpy S alone;
- single: one 128^2 simulation (k_step_cluster), K = 40, 20 steps, 3 moving emitters, the four variants;
- phase_1024: one 1024^2 simulation on the phase kernels, K = 100, 5 steps, 8 moving emitters of radius 30;
- autodiff_b64: rollout of 64 x 128^2, K = 40, T = 20 with 2 emitters per simulation, as a schedule against sources=: forward
  and backward.
Prints one JSON object (and writes it to --out) with median ms, G cell-steps/s, launches per call, and the GPU's name, power
limit and maximum SM clock read in the same run.  Needs a GPU.
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from smokephysai_b200 import NavierStokesSimulator, autodiff  # noqa: E402
from smokephysai_b200.navier_stokes import pack_schedule  # noqa: E402
from continuous_sources_bench import gpu_info, measure, timed  # noqa: E402


def moving(T, B, h, w, seed, emax=3, radius=8, fixed=None):
    """1 .. emax emitters per simulation (fixed: exactly that many), padded to emax with radius -1, starting at data-loader
    positions and moving one cell per step with an intensity that changes at every step.  -> numpy (xy, radius, intensity)."""
    rng = np.random.default_rng(seed)
    xy = np.zeros((T, B, emax, 2), np.int32)
    rad = np.full((T, B, emax), -1, np.int32)
    inten = np.zeros((T, B, emax), np.float32)
    t = np.arange(T)[:, None]
    for b in range(B):
        n = fixed or int(rng.integers(1, emax + 1))
        x0, y0 = rng.integers(20, w - 20, n), rng.integers(20, h - 20, n)
        dx, dy = rng.choice([-1, 1], n), rng.choice([-1, 0, 1], n)
        xy[:, b, :n, 0] = x0 + dx * t
        xy[:, b, :n, 1] = y0 + dy * t
        rad[:, b, :n] = radius
        inten[:, b, :n] = rng.uniform(0.5, 2.0, n) * (1.0 + 0.5 * np.sin(0.7 * t + np.arange(n)))
    return xy, rad, inten


def row(S, t):
    xy, rad, inten = S
    return [[(int(xy[t, b, e, 0]), int(xy[t, b, e, 1]), int(rad[t, b, e]), float(inten[t, b, e]))
             for e in range(rad.shape[2]) if rad[t, b, e] >= 0] for b in range(rad.shape[1])]


def variants(S, h, w, B, K, T, host_loop=True):
    sims = {k: NavierStokesSimulator((h, w), batch=B, jacobi_iters=K) for k in ("sched", "cuda", "cont", "loop")}
    sims["cont"].set_continuous_sources(row(S, 0))
    Sd = tuple(torch.from_numpy(a).cuda() for a in S)

    def schedule():
        sims["sched"].setup_grid()
        sims["sched"].run_steps(T, return_frames=False, schedule=S)

    def schedule_cuda():
        sims["cuda"].setup_grid()
        sims["cuda"].run_steps(T, return_frames=False, schedule=Sd)

    def continuous():
        sims["cont"].setup_grid()
        sims["cont"].run_steps(T, return_frames=False)

    def loop():
        ns = sims["loop"]
        ns.setup_grid()
        for t in range(T):
            ns.add_sources(row(S, t))
            ns.step()
    out = {"schedule": schedule, "schedule_cuda": schedule_cuda, "continuous": continuous}
    if host_loop:
        out["host_loop"] = loop
    return out


def pack_ms(S, T, B, repeats):
    pack_schedule(S, T, B)
    ms = []
    for _ in range(max(repeats, 5)):
        t0 = time.perf_counter()
        pack_schedule(S, T, B)
        ms.append((time.perf_counter() - t0) * 1e3)
    return {"median_ms": statistics.median(ms), "samples_ms": ms}


def workload(name, S, h, w, B, K, T, repeats, host_loop=True):
    res = measure(variants(S, h, w, B, K, T, host_loop), repeats, h * w * B * T)
    wl = {"grid": [h, w], "batch": B, "K": K, "T": T, "results": res, "host_pack": pack_ms(S, T, B, repeats),
          "schedule_over_continuous": res["schedule"]["median_ms"] / res["continuous"]["median_ms"],
          "schedule_cuda_over_continuous": res["schedule_cuda"]["median_ms"] / res["continuous"]["median_ms"]}
    if host_loop:
        wl["host_loop_over_schedule"] = res["host_loop"]["median_ms"] / res["schedule"]["median_ms"]
    print(name, json.dumps({k: v for k, v in wl.items() if k != "results"}), file=sys.stderr)
    return wl


def autodiff_case(B, K, T, repeats):
    h = w = 128
    sim = NavierStokesSimulator((h, w), batch=B, step_kernel="phases")
    sim.add_sources([[(w // 2, h // 3, 8, 1.5), (w // 3 + b % 7, h // 2, 8, 0.8)] for b in range(B)])
    st = [t.reshape(B, *t.shape[-2:]).clone() for t in (sim.u, sim.v, sim.p, sim.density)]
    em = [[(w // 2 + b % 5, h - 20, 8), (w // 3, h - 25, 8)] for b in range(B)]
    xy, rad, inten = moving(T, B, h, w, 3, emax=2, fixed=2)
    I_sched = torch.from_numpy(inten).cuda()
    I_src = torch.full((2 * B,), 1.0, device="cuda")
    cases = {"sources": lambda I: {"sources": em, "intensities": I}, "schedule": lambda I: {"schedule": (xy, rad), "intensities": I}}
    base = {"sources": I_src, "schedule": I_sched}
    res = {}

    def once(name):
        lv = [t.clone().requires_grad_(True) for t in st]
        kw = cases[name](base[name].clone().requires_grad_(True))
        box = [None]
        fwd = timed(lambda: box.__setitem__(0, autodiff.rollout(tuple(lv), T, jacobi_iters=K, **kw)))[0]
        frames, final = box[0]
        loss = frames.square().sum() + final[3].sum()
        bwd = timed(lambda: loss.backward())[0]
        return fwd, bwd
    for name in cases:
        once(name)
    f = {k: [] for k in cases}
    b = {k: [] for k in cases}
    for _ in range(repeats):
        for name in cases:
            x, y = once(name)
            f[name].append(x)
            b[name].append(y)
    for name in cases:
        res[name] = {"forward_median_ms": statistics.median(f[name]), "backward_median_ms": statistics.median(b[name]),
                     "forward_samples_ms": f[name], "backward_samples_ms": b[name]}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.cuda.current_device()
    out = {"gpu": gpu_info(dev), "workloads": {}}
    K, T = 40, 20
    out["workloads"]["c2"] = workload("c2", moving(T, 256, 128, 128, 0), 128, 128, 256, K, T, args.repeats)
    out["workloads"]["single"] = workload("single", moving(T, 1, 128, 128, 1, fixed=3), 128, 128, 1, K, T, args.repeats)
    out["workloads"]["phase_1024"] = workload("phase_1024", moving(5, 1, 1024, 1024, 2, emax=8, radius=30, fixed=8), 1024, 1024,
                                              1, 100, 5, args.repeats)
    out["workloads"]["autodiff_b64"] = {"batch": 64, "K": K, "T": T, "results": autodiff_case(64, K, T, args.repeats)}
    out["gpu_after"] = gpu_info(dev)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
