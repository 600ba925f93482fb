"""Cost of continuous sources (NavierStokesSimulator.set_continuous_sources): the splat at the head of every step.

    python tools/continuous_sources_bench.py [--out profiles/r07a_continuous_sources.json] [--repeats 5]

Workloads, each timed in one process with CUDA events around whole calls, the variants alternated `--repeats` times after a
warm-up of every variant:
- c2: 256 x 128^2 simulations, K = 40, 20 steps, the data-loader emitter law (1-3 emitters of radius 8 per simulation):
  * oneshot:    setup_grid(); add_sources(S); run_steps(20)          (today's puff: the reset and splat consumed on chip)
  * continuous: setup_grid(); run_steps(20) with set_continuous_sources(S)
  * host_loop:  setup_grid(); 20 x [add_sources(S); step()]            (what a user writes without the feature)
- c2_32: the same with a 32-emitter list per simulation (oneshot and continuous);
- single: one 128^2 simulation (k_step_cluster, clusters of four SMs), K = 40, 20 steps, the three variants;
- autodiff: rollout of 64 x 128^2, K = 40, T = 20 with and without 2 continuous emitters per simulation: forward and backward.
Prints one JSON object (and writes it to --out) with median ms, G cell-steps/s, launches per call, and the GPU's name, power
limit and maximum SM clock read in the same run.  Needs a GPU.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smokephysai_b200 import NavierStokesSimulator, _lib, autodiff  # noqa: E402


def gpu_info(index):
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"] = float(q[0])
        info["sm_max_mhz"] = float(q[1])
    except Exception as e:
        info["power_limit_w"] = None
        info["power_limit_error"] = repr(e)
    return info


def loader_law(B, h, w, seed):
    """data_loader.py:49-58: 1-3 emitters per sample, x, y in [20, size - 20), intensity in [0.5, 2), radius 8."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(B):
        n = int(rng.integers(1, 4))
        out.append([(int(rng.integers(20, w - 20)), int(rng.integers(20, h - 20)), 8, float(rng.uniform(0.5, 2.0))) for _ in range(n)])
    return out


def long_law(B, h, w, seed, n=32):
    rng = np.random.default_rng(seed)
    return [[(int(rng.integers(0, w)), int(rng.integers(0, h)), 8, float(rng.uniform(0.5, 2.0))) for _ in range(n)] for _ in range(B)]


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), _lib.launch_count() - n0


def variants(S, B, K, T):
    ns_once = NavierStokesSimulator((128, 128), batch=B, jacobi_iters=K)
    ns_cont = NavierStokesSimulator((128, 128), batch=B, jacobi_iters=K)
    ns_cont.set_continuous_sources(S)
    ns_loop = NavierStokesSimulator((128, 128), batch=B, jacobi_iters=K)
    out = {}

    def oneshot():
        ns_once.setup_grid()
        ns_once.add_sources(S)
        ns_once.run_steps(T, return_frames=False)

    def continuous():
        ns_cont.setup_grid()
        ns_cont.run_steps(T, return_frames=False)

    def host_loop():
        ns_loop.setup_grid()
        for _ in range(T):
            ns_loop.add_sources(S)
            ns_loop.step()
    out["oneshot"], out["continuous"], out["host_loop"] = oneshot, continuous, host_loop
    return out


def measure(fns, repeats, cells):
    for fn in fns.values():                     # warm-up: modules, schedules, allocator
        fn()
        fn()
    ms = {k: [] for k in fns}
    launches = {}
    for _ in range(repeats):
        for k, fn in fns.items():
            t, n = timed(fn)
            ms[k].append(t)
            launches[k] = n
    res = {}
    for k in fns:
        med = statistics.median(ms[k])
        res[k] = {"median_ms": med, "min_ms": min(ms[k]), "max_ms": max(ms[k]), "gcell_steps_per_s": cells / med / 1e6,
                  "launches_per_call": launches[k], "samples_ms": ms[k]}
    return res


def autodiff_case(B, K, T, repeats):
    h = w = 128
    sim = NavierStokesSimulator((h, w), batch=B, step_kernel="phases")
    sim.add_sources([[(w // 2, h // 3, 8, 1.5), (w // 3 + b % 7, h // 2, 8, 0.8)] for b in range(B)])
    st = [t.reshape(B, *t.shape[-2:]).clone() for t in (sim.u, sim.v, sim.p, sim.density)]
    em = [[(w // 2 + b % 5, h - 20, 8), (w // 3, h - 25, 8)] for b in range(B)]
    inten = torch.full((2 * B,), 1.0, device="cuda")
    res = {}
    for name, kw in (("no_sources", {}), ("continuous_2_per_sim", {"sources": em, "intensities": inten})):
        def once():
            lv = [t.clone().requires_grad_(True) for t in st]
            if kw:
                kw["intensities"] = inten.clone().requires_grad_(True)
            fwd = timed(lambda: once.out.__setitem__(0, autodiff.rollout(tuple(lv), T, jacobi_iters=K, **kw)))[0]
            frames, final = once.out[0]
            loss = frames.square().sum() + final[3].sum()
            bwd = timed(lambda: loss.backward())[0]
            return fwd, bwd
        once.out = [None]
        once()
        f, b = [], []
        for _ in range(repeats):
            x, y = once()
            f.append(x)
            b.append(y)
        res[name] = {"forward_median_ms": statistics.median(f), "backward_median_ms": statistics.median(b),
                     "forward_samples_ms": f, "backward_samples_ms": b}
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
    B, K, T = 256, 40, 20
    cells = 128 * 128 * B * T
    out["workloads"]["c2"] = {"batch": B, "K": K, "T": T, "emitters": "1-3 per simulation, radius 8 (data-loader law)",
                              "results": measure(variants(loader_law(B, 128, 128, 0), B, K, T), args.repeats, cells)}
    fns = variants(long_law(B, 128, 128, 1), B, K, T)
    del fns["host_loop"]
    out["workloads"]["c2_32"] = {"batch": B, "K": K, "T": T, "emitters": "32 per simulation, radius 8",
                                 "results": measure(fns, args.repeats, cells)}
    out["workloads"]["single"] = {"batch": 1, "K": K, "T": T, "emitters": "3, radius 8",
                                  "results": measure(variants([[(64, 100, 8, 1.0), (40, 110, 8, 0.5), (90, 105, 8, 0.75)]], 1, K, T),
                                                     args.repeats, 128 * 128 * T)}
    out["workloads"]["autodiff_b64"] = {"batch": 64, "K": K, "T": T, "results": autodiff_case(64, K, T, args.repeats)}
    for name, wl in out["workloads"].items():
        r = wl["results"]
        if "continuous" in r and "oneshot" in r:
            wl["continuous_over_oneshot"] = r["continuous"]["median_ms"] / r["oneshot"]["median_ms"]
        if "host_loop" in r:
            wl["host_loop_over_continuous"] = r["host_loop"]["median_ms"] / r["continuous"]["median_ms"]
    out["gpu_after"] = gpu_info(dev)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
