"""Cost of velocity forcing (run_steps(forcing=)): increments added to u and v at the head of every step.

    python tools/forcing_bench.py [--out profiles/r09a_forcing.json] [--repeats 5]

Workloads, each timed in one process with CUDA events around whole calls, the variants alternated `--repeats` times after a warm-up
of every variant (forcing buffers already staged on the device, so constant / per_step time the stepping, not the staging):
- c2: 256 x 128^2 simulations, K = 40, 20 steps, the data-loader emitter law (1-3 emitters of radius 8 per simulation splatted
  once after the reset):
  * none:      setup_grid(); add_sources(S); run_steps(20)
  * constant:  the same with forcing=(du, dv), one pair for every step (34 MB read per call)
  * per_step:  the same with a [20, 256, ...] forcing, a pair per step (680 MB read per call)
  * per_step_public: the same through the public run_steps(forcing=(du, dv)) with du, dv CUDA tensors: the per-call staging
    (pack_forcing's zero-padded copy into the simulator's layout) included
  * host_loop: setup_grid(); add_sources(S); 20 x [u += du[t]; v += dv[t]; step()]  (what a user writes without the feature)
- single: one 128^2 simulation (k_step_cluster), K = 40, 20 steps, the four variants;
- phase_1024: one 1024^2 simulation on the phase kernels, K = 100, 5 steps: none / constant / per_step / host_loop;
- autodiff_b64: rollout of 64 x 128^2, K = 40, T = 20, without and with a per-step forcing: forward and backward.
Prints one JSON object (and writes it to --out) with median ms, G cell-steps/s, launches per call, and the GPU's name, power
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

from smokephysai_b200 import NavierStokesSimulator, autodiff  # noqa: E402
from continuous_sources_bench import gpu_info, loader_law, measure, timed  # noqa: E402


def wind(T, B, h, w, seed, strength=50.0):
    """Per-step increments [T, B, h+1, w] / [T, B, h, w+1] on the device: a field that turns from step to step."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    du = strength * torch.randn(T, B, h + 1, w, device="cuda", generator=g)
    dv = strength * torch.randn(T, B, h, w + 1, device="cuda", generator=g)
    return du, dv


def variants(n, B, K, T, S, seed, **kw):
    du, dv = wind(T, B, n, n, seed)
    sims = {k: NavierStokesSimulator((n, n), batch=B, jacobi_iters=K, **kw)
            for k in ("none", "constant", "per_step", "per_step_public", "host_loop")}
    # staged once, in the simulator's layout: the calls below time the stepping only
    staged = {"constant": sims["constant"]._forcing((du[0], dv[0]), T), "per_step": sims["per_step"]._forcing((du, dv), T)}
    out = {}

    def call(name):
        def fn():
            ns = sims[name]
            ns.setup_grid()
            ns.add_sources(S)
            ns._run_steps(T, None, False, None, None, None, staged.get(name))
        return fn
    for name in ("none", "constant", "per_step"):
        out[name] = call(name)

    def public():
        ns = sims["per_step_public"]
        ns.setup_grid()
        ns.add_sources(S)
        ns.run_steps(T, return_frames=False, forcing=(du, dv))
    out["per_step_public"] = public

    def host_loop():
        ns = sims["host_loop"]
        ns.setup_grid()
        ns.add_sources(S)
        for t in range(T):
            ns.u += du[t].reshape(ns.u.shape)
            ns.v += dv[t].reshape(ns.v.shape)
            ns.step()
    out["host_loop"] = host_loop
    return out


def autodiff_case(B, K, T, repeats):
    h = w = 128
    sim = NavierStokesSimulator((h, w), batch=B, step_kernel="phases")
    sim.add_sources([[(w // 2, h // 3, 8, 1.5), (w // 3 + b % 7, h // 2, 8, 0.8)] for b in range(B)])
    st = [t.reshape(B, *t.shape[-2:]).clone() for t in (sim.u, sim.v, sim.p, sim.density)]
    du, dv = wind(T, B, h, w, 7, strength=5.0)
    res = {}
    for name, f in (("no_forcing", None), ("per_step_forcing", (du, dv))):
        def once():
            lv = [t.clone().requires_grad_(True) for t in st]
            kw = {} if f is None else {"forcing": tuple(a.clone().requires_grad_(True) for a in f)}
            fwd = timed(lambda: once.out.__setitem__(0, autodiff.rollout(tuple(lv), T, jacobi_iters=K, **kw)))[0]
            frames, final = once.out[0]
            loss = frames.square().sum() + final[3].sum()
            bwd = timed(lambda: loss.backward())[0]
            return fwd, bwd
        once.out = [None]
        once()
        fw, bw = [], []
        for _ in range(repeats):
            x, y = once()
            fw.append(x)
            bw.append(y)
        res[name] = {"forward_median_ms": statistics.median(fw), "backward_median_ms": statistics.median(bw),
                     "forward_samples_ms": fw, "backward_samples_ms": bw}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    res = {"gpu": gpu_info(torch.cuda.current_device()), "repeats": args.repeats}
    T = 20
    res["c2"] = measure(variants(128, 256, 40, T, loader_law(256, 128, 128, 1), 1), args.repeats, 256 * 128 * 128 * T)
    res["single"] = measure(variants(128, 1, 40, T, loader_law(1, 128, 128, 2), 2), args.repeats, 128 * 128 * T)
    res["phase_1024"] = measure(variants(1024, 1, 100, 5, [[(512, 512, 30, 1.0)]], 3), args.repeats, 1024 * 1024 * 5)
    res["autodiff_b64"] = autodiff_case(64, 40, 20, args.repeats)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
