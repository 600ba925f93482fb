"""Cost of reverse mode (smokephysai_b200.autodiff.rollout): checkpointed forward, backward, and plain run_steps.

    python tools/autodiff_bench.py [--out profiles/<name>.json] [--repeats 5]

Two sizes: 128^2 x 64 simulations (K = 40, T = 20) and 1024^2 x 1 (K = 100, T = 20), from a splatted state at rest, phase
kernels (step_kernel="phases") and the library's default selection ("auto").  Every piece is warmed up, then timed with CUDA
events around whole calls, `--repeats` times, interleaved:
- run_steps: NavierStokesSimulator.run_steps(T) (what rollout runs when no input requires grad);
- forward: rollout with inputs that require grad (one step at a time plus 4 checkpoint copies per step);
- backward: loss.backward() on the frames and the final density (the adjoint kernels, T reverse steps).
Prints one JSON object (and writes it to --out): median ms, G cell-steps/s (h * w * B * T / time), the backward / forward and
backward / run_steps ratios, checkpoint bytes, the kernel time of one backward by library phase (per-kernel CUDA events,
in a separate backward call), and the GPU's name and power limit read in the same run.  Needs a GPU.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smokephysai_b200 import NavierStokesSimulator, _lib, autodiff  # noqa: E402
from smokephysai_b200.navier_stokes import FieldLayout  # noqa: E402

SIZES = [{"name": "128x128_b64_k40", "h": 128, "w": 128, "B": 64, "K": 40, "T": 20},
         {"name": "1024x1024_b1_k100", "h": 1024, "w": 1024, "B": 1, "K": 100, "T": 20}]


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


def initial_state(cfg):
    """A state at rest with two emitters per simulation (the splat of add_smoke_source)."""
    h, w, B = cfg["h"], cfg["w"], cfg["B"]
    sim = NavierStokesSimulator((h, w), batch=B, step_kernel="phases")
    sim.add_sources([[(w // 2, h // 3, 8, 1.5), (w // 3 + b % 7, h // 2, 8, 0.8)] for b in range(B)])
    st = [sim.u, sim.v, sim.p, sim.density]
    return [t.reshape(B, *t.shape[-2:]).clone() for t in st]


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), out


def bench(cfg, kernel, repeats):
    h, w, B, K, T = cfg["h"], cfg["w"], cfg["B"], cfg["K"], cfg["T"]
    state = initial_state(cfg)
    sim = NavierStokesSimulator((h, w), batch=B, jacobi_iters=K, step_kernel=kernel)

    def run_steps():
        for k, t in zip(("u", "v", "p", "density"), state):
            setattr(sim, k, t if B > 1 else t[0])
        return sim.run_steps(T)

    def forward():
        lv = [t.clone().requires_grad_(True) for t in state]
        frames, final = autodiff.rollout(tuple(lv), T, jacobi_iters=K, step_kernel=kernel)
        return frames.sum() + final[3].sum()

    res = {"run_steps": [], "forward": [], "backward": []}
    for rep in range(repeats + 1):                      # repeat 0 warms every shape up
        t_rs, _ = timed(run_steps)
        t_fw, loss = timed(forward)
        t_bw, _ = timed(loss.backward)
        if rep:
            res["run_steps"].append(t_rs)
            res["forward"].append(t_fw)
            res["backward"].append(t_bw)
    # one more backward under the library's per-kernel event timing: where the reverse steps spend their kernel time
    # (recompute: forces_diffuse_div + project; the Jacobi adjoint's two sweep chains: jacobi; every adjoint kernel: other)
    loss = forward()
    torch.cuda.synchronize()
    _lib.profile_begin(16384)
    loss.backward()
    prof = {k: {"ms": ms, "launches": n} for k, (ms, n) in _lib.profile_end().items() if n}
    L = FieldLayout(h, w, B)
    cells = h * w * B * T
    out = {"kernel": kernel, "cell_steps": cells,
           "checkpoint_bytes": 4 * (T + 1) * B * ((h + 1) * L.pitch_u + h * L.pitch_v + 2 * h * L.pitch_c)}
    for k, v in res.items():
        med = statistics.median(v)
        out[k] = {"ms_median": med, "ms_all": v, "G_cell_steps_per_s": cells / (med * 1e-3) / 1e9}
    out["backward_kernel_ms_by_phase"] = prof
    out["backward_over_forward"] = out["backward"]["ms_median"] / out["forward"]["ms_median"]
    out["backward_over_run_steps"] = out["backward"]["ms_median"] / out["run_steps"]["ms_median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("autodiff_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    result = {"tool": "tools/autodiff_bench.py", "gpu": gpu_info(0), "repeats": a.repeats, "sizes": []}
    for cfg in SIZES:
        entry = dict(cfg)
        entry["results"] = [bench(cfg, kernel, a.repeats) for kernel in ("phases", "auto")]
        result["sizes"].append(entry)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
