"""End-to-end and device rates of the c2 configuration (256 x 128^2, K = 40, 20 steps per call) with fp32, fp16 and bf16 frames.

    python tools/frame_dtype_e2e.py [--out profiles/<name>.json] [--seconds 1.0] [--repeats 3]

- e2e: SmokeSimulator.generate_sequences(to_host=True, frame_dtype=...) -- host emitter lists in, pinned host frames out --
  for the three dtypes, interleaved call by call; every dtype is warmed up first, then timed for >= --seconds per repeat.
- device: ns.run_steps(T, out=<preallocated device buffer of that dtype>) after the reset and the splat (what bench.py's c2
  `value` times), CUDA events, interleaved the same way.
- ceiling: 4 back-to-back cudaMemcpyAsync (torch's copy_) of one contiguous block device -> pinned host, for the fp32 and
  the half frame size, in the same process (as bench.py's d2h_ceiling).

Prints one JSON object (and writes it to --out): G cell-steps/s, ms per call, D2H bytes per call and per step, the share of
the measured ceiling, plus the GPU's name and power limit read in the same run.  Needs a GPU; there is no CPU fallback.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smokephysai_b200 import SmokeSimulator, hostmem  # noqa: E402

DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}


def seeded_emitters(B, h, w, seed):
    """data_loader.py:49-58's emitter law (1-3 emitters, radius 8, intensity in [0.5, 2]) from one seeded generator."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(B):
        n = int(rng.integers(1, 4))
        out.append([((int(rng.integers(20, w - 20)), int(rng.integers(20, h - 20))), float(rng.uniform(0.5, 2.0))) for _ in range(n)])
    return out


def gpu_info(index):
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"] = float(q[0])
        info["sm_max_mhz"] = float(q[1])
    except Exception as e:                       # the rates stand without it, but say so
        info["power_limit_w"] = None
        info["power_limit_error"] = repr(e)
    return info


def d2h_ceiling(nbytes, dev_index, reps=4, rounds=3):
    """GB/s of `reps` back-to-back copies of one contiguous nbytes block device -> pinned host (NUMA-local), `rounds` times."""
    n = nbytes // 4
    dev = torch.empty(n, dtype=torch.float32, device=dev_index)
    host = hostmem.pinned_empty((n,), torch.float32, torch.device("cuda", dev_index))
    host.copy_(dev, non_blocking=True)
    torch.cuda.synchronize()
    out = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        for _ in range(reps):
            host.copy_(dev, non_blocking=True)
        torch.cuda.synchronize()
        out.append(reps * n * 4 / (time.perf_counter() - t0) / 1e9)
    del dev, host
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--grid", type=int, default=128)
    ap.add_argument("--K", type=int, default=40)
    ap.add_argument("--T", type=int, default=20)
    ap.add_argument("--seconds", type=float, default=1.0, help="timed seconds per dtype and repeat, at least")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("frame_dtype_e2e.py needs a CUDA device")
    torch.cuda.set_device(0)
    B, h, w, K, T = args.batch, args.grid, args.grid, args.K, args.T
    sim = SmokeSimulator((h, w), 0.01, 0.001, "cuda:0", jacobi_iters=K, batch=B)
    ns = sim.ns_solver
    L = ns._layout
    ems = seeded_emitters(B, h, w, args.seed)
    fmul = sim.fractal_gen.multiplier((h, w), 0.05)
    src, off, _ = ns.upload_sources([[(x, y, 8, i) for (x, y), i in lst] for lst in ems])
    cells_per_call = B * h * w * T

    # warm-up of every shape; one fp32 call sizes the timed loops
    for dt in DTYPES.values():
        for _ in range(2):
            sim.generate_sequences(ems, T, to_host=True, frame_dtype=dt)
    t0 = time.perf_counter()
    sim.generate_sequences(ems, T, to_host=True)
    calls = max(3, int(np.ceil(args.seconds / (time.perf_counter() - t0))))

    dev_bufs = {k: torch.empty(B, T, h, L.pitch_c, dtype=dt, device="cuda") for k, dt in DTYPES.items()}

    def device_call(k):
        ns.setup_grid()
        ns.splat_uploaded(src, off)
        ns.run_steps(T, fmul=fmul, out=dev_bufs[k])

    for k in DTYPES:
        device_call(k)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    device_call("f32")
    torch.cuda.synchronize()
    dcalls = max(5, int(np.ceil(args.seconds / (time.perf_counter() - t0))))

    e2e = {k: [] for k in DTYPES}
    dev = {k: [] for k in DTYPES}
    checks = {}
    for _ in range(args.repeats):
        acc = dict.fromkeys(DTYPES, 0.0)
        for _ in range(calls):
            for k, dt in DTYPES.items():
                t0 = time.perf_counter()
                fr = sim.generate_sequences(ems, T, to_host=True, frame_dtype=dt)      # returns after the last D2H copy
                acc[k] += time.perf_counter() - t0
                checks[k] = float(fr[:, -1].double().sum())
        for k in DTYPES:
            e2e[k].append(acc[k] / calls)
        acc = dict.fromkeys(DTYPES, 0.0)
        for _ in range(dcalls):
            for k in DTYPES:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                device_call(k)
                b.record()
                b.synchronize()
                acc[k] += a.elapsed_time(b) * 1e-3
        for k in DTYPES:
            dev[k].append(acc[k] / dcalls)

    bytes_per_call = {k: T * B * h * L.pitch_c * torch.empty(0, dtype=dt).element_size() for k, dt in DTYPES.items()}
    ceiling = {"f32": d2h_ceiling(bytes_per_call["f32"], 0), "half": d2h_ceiling(bytes_per_call["f16"], 0)}
    result = {
        "tool": "tools/frame_dtype_e2e.py",
        "gpu": gpu_info(0),
        "config": {"batch": B, "grid": [h, w], "K": K, "T": T, "emitter_seed": args.seed, "fractal": True,
                   "e2e_calls_per_repeat": calls, "device_calls_per_repeat": dcalls, "repeats": args.repeats},
        "d2h_ceiling_gbs": {k: {"median": statistics.median(v), "all": v} for k, v in ceiling.items()},
        "d2h_ceiling_how": "4 back-to-back cudaMemcpyAsync of one contiguous block (%d MB fp32, %d MB half) device -> pinned "
                           "NUMA-local host, 3 rounds" % (bytes_per_call["f32"] // 1000000, bytes_per_call["f16"] // 1000000),
        "dtypes": {},
    }
    for k in DTYPES:
        ceil = statistics.median(ceiling["f32" if k == "f32" else "half"])
        s = statistics.median(e2e[k])
        d = statistics.median(dev[k])
        result["dtypes"][k] = {
            "e2e_gcells_per_s": {"median": cells_per_call / s / 1e9, "all": [cells_per_call / x / 1e9 for x in e2e[k]]},
            "e2e_ms_per_call": {"median": 1e3 * s, "all": [1e3 * x for x in e2e[k]]},
            "device_gcells_per_s": {"median": cells_per_call / d / 1e9, "all": [cells_per_call / x / 1e9 for x in dev[k]]},
            "device_ms_per_call": {"median": 1e3 * d, "all": [1e3 * x for x in dev[k]]},
            "d2h_bytes_per_call": bytes_per_call[k],
            "d2h_bytes_per_step": bytes_per_call[k] // T,
            "d2h_gbs": bytes_per_call[k] / s / 1e9,
            "frac_of_d2h_ceiling": bytes_per_call[k] / s / 1e9 / ceil,
            "last_frame_checksum": checks[k],
        }
    f32 = result["dtypes"]["f32"]["e2e_gcells_per_s"]["median"]
    result["e2e_speedup_vs_f32"] = {k: v["e2e_gcells_per_s"]["median"] / f32 for k, v in result["dtypes"].items()}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
