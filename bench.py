#!/usr/bin/env python
"""bench.py -- throughput of the grid smoke step (BASELINE.json metric: grid cell-updates/s and % of the
HBM roofline) on N B200s, with the CPU restatement of the reference timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload all|c2|c2s|c3|c4] [--dump-outputs DIR]

The printed line is the c2 measurement (BASELINE.json configs[1], the configuration the metric is quoted on):
batched dataset generation, 256 independent 128x128 sequences per GPU, 40 Jacobi sweeps per time step, 20 time
steps per sequence, emitters drawn by the law of data_loader.py:49-58 with seed 1234 + global sequence index.
One bench "step" = one pass of the hot path over the rank's batch: reset the state, splat the emitters, run the
20 time steps and write the 20 returned (fractal-scaled) frames of every sequence.  Sequences are independent,
so ranks share nothing on the data path (no collective; weak scaling: 256 sequences per GPU).

With the default --workload all the same line carries, under "also", the other BASELINE configurations measured
in the same process right after c2:
    c2_strong  configs[1] as written: 256 sequences in TOTAL, 256 / N per GPU (strong scaling; N > 1 only)
    c3         configs[2]: one 1024x1024 grid, 100 sweeps per step (N = 1 only: it does not shard)
    c4         configs[3]: one 8192x8192 grid, 20 sweeps per step, row slabs over the N GPUs with halo exchange
               (strong scaling) -- and, at N > 1, a `parity` object: two steps of the slab run gathered and
               compared bit for bit with the undecomposed run on rank 0 (outside every timed region)
each with value, ms_per_step, clocks, e2e and a per-kernel roofline list.

`value` = cell-steps/s of the whole job with the emitter records already on the device and frames left in HBM;
`e2e` = the same through the public API from host emitter lists (pinned H2D) to frames in pinned host memory
(D2H), copies inside the timed region.  `roofline` is for the kernel with the largest share of the step, from
CUDA events the library records around every launch (smk_profile_begin/end) in a second pass over the same
steps; `kernels` lists every kernel of the step the same way, each with the bound that actually limits it.
`cpu_baseline` is the oracle (a C port of the reference step, NOT the product) on the host cores.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "grid_cell_updates_per_sec"
UNIT = "cell-steps/s"
L2_MB = 126

WORKLOADS = {
    # name: (h, w, sequences per GPU, jacobi sweeps, time steps per bench step)
    "c2": dict(h=128, w=128, batch=256, K=40, tsteps=20, scaling="weak",
               name="c2: batched dataset generation, 256 independent 128x128 sequences per GPU, 40 Jacobi sweeps/step, "
                    "20 steps/sequence (BASELINE.json configs[1])"),
    "c2s": dict(h=128, w=128, batch=256, K=40, tsteps=20, scaling="strong",
                name="c2 strong-scaled: 256 independent 128x128 sequences in total (256 / N per GPU), 40 Jacobi sweeps/step, "
                     "20 steps/sequence (BASELINE.json configs[1] as written)"),
    "c3": dict(h=1024, w=1024, batch=1, K=100, tsteps=20, scaling="weak",
               name="c3: single 1024x1024 grid, 100 Jacobi sweeps/step, 20 steps (BASELINE.json configs[2])"),
    "c4": dict(h=8192, w=8192, batch=1, K=20, tsteps=5, scaling="strong",
               name="c4: single 8192x8192 grid, 20 Jacobi sweeps/step, 5 steps per bench step, row slabs over the GPUs "
                    "(BASELINE.json configs[3]; strong scaling)"),
}

# algorithmic bytes per cell per launch of each kernel family (SURVEY.md s8d; fp32, each array touched once)
def phase_bytes_per_cell(K, sweeps_in_launch, steps_in_launch=1):
    return {
        "step_fused": (100 + 12 * K) * steps_in_launch,   # k_step_fused: whole steps, every phase of SURVEY s8d
        "forces_diffuse_div": 24 + 12,      # R(u,v,d) W(u,v,d)  +  divergence R(u,v) W(div), fused in one kernel
        "jacobi": 12 * sweeps_in_launch,    # per sweep R(p,div) W(p)
        "project": 20,                      # R(p,u,v) W(u,v)
        "advect_u": 12, "advect_v": 12,     # R(u,v) W(field)
        "project_advect_u": 20 + 12,        # k_project_advect_u: gradient subtract and the u advection in one kernel
        "advect_d": 16 + 4,                 # R(u,v,d) W(d) + the returned copy
        "splat": 8,
        "other": 0, "halo": 0, "halo_unpack": 0,
    }


# fp32 adds / multiplies / divides per cell per launch, counted from the reference's expressions (no FMA by the bit-parity
# contract, so one instruction = one flop): buoyancy 3, diffusion 3 x 7, divergence 4, Jacobi 5 per sweep, gradient
# subtract 6, advection 27 each, decay 1, fractal multiply 2.  Clamps, floors and index math are not counted.
def phase_flops_per_cell(K, sweeps_in_launch, steps_in_launch=1):
    return {
        "step_fused": (118 + 5 * K) * steps_in_launch,
        "forces_diffuse_div": 3 + 21 + 4, "jacobi": 5 * sweeps_in_launch, "project": 6,
        "advect_u": 27, "advect_v": 27, "project_advect_u": 33, "advect_d": 30, "splat": 0, "other": 0, "halo": 0, "halo_unpack": 0,
    }


KERNEL_NAMES = {"jacobi": "k_jacobi", "forces_diffuse_div": "k_forces_diffuse_div", "project": "k_project",
                "advect_u": "k_advect(u)", "advect_v": "k_advect(v)", "advect_d": "k_advect(density)", "splat": "k_splat",
                "project_advect_u": "k_advect_tiled<1>(u) with k_project fused in", "step_fused": "k_step_fused", "other": "other", "halo": "k_halo_push", "halo_unpack": "k_halo_unpack"}


def emitters_for_sequence(s, h, w):
    """data_loader.py:49-58 with fixed seeds (SURVEY.md s8d); larger grids get one emitter per 64x64 block."""
    rng = np.random.default_rng(1234 + s)
    out = []
    if h <= 128 and w <= 128:
        n = int(rng.integers(1, 4))
        for _ in range(n):
            x = int(rng.integers(20, w - 20)); y = int(rng.integers(20, h - 20))
            out.append((x, y, 8, float(rng.uniform(0.5, 2.0))))
    else:
        for by in range(h // 64):
            for bx in range(w // 64):
                out.append((int(bx * 64 + rng.integers(8, 56)), int(by * 64 + rng.integers(8, 56)), 8,
                            float(rng.uniform(0.5, 2.0))))
    return out


def config_for(key, world):
    """The `config` object of a workload: built from the workload table alone, so the GPU arm and the reference arm
    print the same keys and values for the same run."""
    wl = WORKLOADS[key]
    h, w, K, T = wl["h"], wl["w"], wl["K"], wl["tsteps"]
    B = wl["batch"] // world if key == "c2s" else wl["batch"]
    pitch_v = (w + 1 + 3) & ~3
    if key == "c4":
        rows = h // world
        fields = 2 * ((rows + 1) * w + rows * pitch_v + 2 * rows * w) * 4 + 2 * rows * w * 4
        par = "single GPU, undecomposed" if world == 1 else "row slabs over %d GPU(s) with halo exchange over NVLink" % world
        ws = fields
    else:
        fields = B * (2 * ((h + 1) * w + h * pitch_v + 2 * h * w) + 2 * h * w) * 4
        ws = fields + B * T * h * w * 4
        par = ("sequences sharded over %d GPU(s), no data-path collective" % world) if B > 1 or world > 1 else "single GPU"
    return {"workload": wl["name"], "grid": [h, w], "sequences_per_gpu": B, "jacobi_iters": K, "time_steps_per_bench_step": T,
            "parallelism": par,
            "l2": ("no flush: working set %.0f MB per GPU (fields + frames) > %d MB L2" % (ws / 1e6, L2_MB)) if ws > L2_MB * 1e6
                  else ("L2 flushed (a 256 MB buffer is written) before every bench step, outside the timed events: working set "
                        "%.0f MB per GPU fits the %d MB L2" % (ws / 1e6, L2_MB))}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def committed_traffic(phase, workload):
    """dram bytes per launch of the kernel of `phase` from the committed ncu --set full capture (profiles/traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return t.get(workload, {}).get(phase)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 25 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "25"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, power = [], [], set(), []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); power.append(float(c[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


# ------------------------------------------------------------------------------------------ CPU (oracle) arm
def cpu_run(wl, nseq, nthreads, seq0=0):
    """Time the oracle (C port of the reference step) on nseq sequences x tsteps steps with nthreads threads."""
    import oracle
    h, w, K, T = wl["h"], wl["w"], wl["K"], wl["tsteps"]
    u = np.zeros((nseq, h + 1, w), np.float32); v = np.zeros((nseq, h, w + 1), np.float32)
    p = np.zeros((nseq, h, w), np.float32); d = np.zeros((nseq, h, w), np.float32)
    for s in range(nseq):
        for x, y, r, i in emitters_for_sequence(seq0 + s, h, w):
            y0, y1, x0, x1 = max(0, y - r), min(h, y + r + 1), max(0, x - r), min(w, x + r + 1)
            sub = np.ascontiguousarray(d[s, y0:y1, x0:x1])          # the splat only touches the emitter's bounding box
            oracle.splat(sub, x - x0, y - y0, r, i)
            d[s, y0:y1, x0:x1] = sub
    fmul = oracle.fractal_mul(h, 0.05) if h == w else None
    t0 = time.perf_counter()
    oracle.run_batch(u, v, p, d, 0.01, 0.001, K, T, fmul=fmul, want_frames=True, nthreads=nthreads)
    dt = time.perf_counter() - t0
    return nseq * h * w * T / dt, dt


def reference_arm(args, key):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    import oracle
    oracle.build()
    wl = WORKLOADS[key]
    cores = os.cpu_count() or 1
    nseq = wl["batch"]
    wl_cpu = dict(wl)
    if wl["h"] >= 1024:
        wl_cpu["tsteps"] = 2 if wl["h"] < 4096 else 1
    for _ in range(args.warmup):
        cpu_run(wl_cpu, nseq, cores)
    t_tot, cells = 0.0, 0
    for _ in range(args.steps):
        thr, dt = cpu_run(wl_cpu, nseq, cores)
        t_tot += dt
        cells += nseq * wl["h"] * wl["w"] * wl_cpu["tsteps"]
    val = cells / t_tot
    sample = "%d sequences x %d steps of %dx%d, K=%d per bench step" % (nseq, wl_cpu["tsteps"], wl["h"], wl["w"], wl["K"])
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": wl["scaling"],
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_for(key, world),
        "host": "rank 0 only; oracle/ C port of the reference step (the reference is pure Python/PyTorch and publishes no number "
                "for this path), pthreads over sequences",
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": min(cores, nseq), "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))
    return 0


def reference_torch_numbers(dev, K):
    """Informational: the UNMODIFIED reference NavierStokesSimulator (installed in git-ignored baseline/_ref by
    `pip install --no-deps --target baseline/_ref <copy of /root/reference>`) stepped on the host CPU and, eagerly,
    on this GPU.  128x128, one sequence; with its hard-coded 20 Jacobi sweeps (navier_stokes.py:139) and with the literal
    overridden to this bench's K the way tests/golden/make_golden.py does.  None if the install is absent."""
    path = os.path.join(ROOT, "baseline", "_ref", "src", "physics", "navier_stokes.py")
    if not os.path.exists(path):
        return None
    try:
        import importlib.util
        import inspect
        import re
        import textwrap
        import torch
        spec = importlib.util.spec_from_file_location("_reference_navier_stokes", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)

        def with_iters(k):
            if k == 20:
                return mod.NavierStokesSimulator
            src = textwrap.dedent(inspect.getsource(mod.NavierStokesSimulator.pressure_projection))
            src, n = re.subn(r"range\(20\)", "range(%d)" % k, src)
            assert n == 1
            ns = {"torch": torch}
            exec(src, ns)
            return type("NavierStokesSimulatorK%d" % k, (mod.NavierStokesSimulator,), {"pressure_projection": ns["pressure_projection"]})

        out = {"config": "unmodified reference NavierStokesSimulator.step(), 128x128, 1 sequence; K=20 is its literal, K=%d the "
                         "literal overridden (range(20) -> range(%d)) to match this bench" % (K, K)}
        for k in sorted({20, K}):
            cls = with_iters(k)
            for name, device, nsteps in (("cpu", "cpu", 10), ("cuda_eager", str(dev), 20)):
                sim = cls((128, 128), 0.01, 0.001, device)
                sim.add_smoke_source(64, 64, radius=8, intensity=1.5)
                for _ in range(3):
                    sim.step()
                if device != "cpu":
                    torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(nsteps):
                    sim.step()
                if device != "cpu":
                    torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                out["%s_K%d" % (name, k)] = {"cell_steps_per_s": 128 * 128 * nsteps / dt, "ms_per_step": 1e3 * dt / nsteps,
                                             "threads": torch.get_num_threads() if device == "cpu" else None}
        return out
    except Exception as e:           # informational only
        return {"error": repr(e)[:200]}


# ------------------------------------------------------------------------------------------------ GPU arm
class Ctx:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the smoke step has no CPU path (use --impl reference for the CPU oracle)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peak, self.peak_src = peaks()
        self.sm_count = torch.cuda.get_device_properties(self.dev).multi_processor_count

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def min_over_ranks(self, x):
        return -self.max_over_ranks(-x)


DUMP_MAX_VALUES = 1 << 20          # per dumped array over all ranks (4 MB of fp32): --workload all dumps 14 arrays, 56 MB at most


def dump_sample(t, max_values=DUMP_MAX_VALUES):
    """A [..., cols] tensor on the host as fp32; above max_values values, the rows of a fixed seeded sample (sorted row
    indices of the [-1, cols] view, the same for the same shape in every run)."""
    import torch
    cols = t.shape[-1]
    if t.numel() <= max_values:
        return t.float().cpu().numpy()
    rows = t.flatten(0, -2)
    idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], max(1, max_values // cols), replace=False))
    return rows.index_select(0, torch.from_numpy(idx).to(rows.device)).float().cpu().numpy()


def dump_outputs(ctx, key, arrays):
    """--dump-outputs: DIR/<workload>_<name>.npy (<workload>_rank<r>_<name>.npy on several GPUs, each rank within an equal
    share of DUMP_MAX_VALUES) for every array."""
    os.makedirs(ctx.args.dump_outputs, exist_ok=True)
    prefix = key if ctx.world == 1 else "%s_rank%d" % (key, ctx.rank)
    for name, t in arrays.items():
        np.save(os.path.join(ctx.args.dump_outputs, "%s_%s.npy" % (prefix, name)), dump_sample(t, DUMP_MAX_VALUES // ctx.world))


def timed_passes(ctx, device_step, e2e_step, steps, warmup, count_launches, flush_l2=False, after_timed=None):
    """The three measurement passes of one workload: device-resident throughput (CUDA events, max over ranks), the same
    steps once more with an event pair around every launch, and the end-to-end pass through the public API.
    flush_l2: the working set fits the L2, so a 256 MB buffer is written before every bench step (outside the events /
    the clock: each step is then timed on its own and the times are added up).
    after_timed: called once right after the timed steps, before anything else runs on the state they left."""
    torch, _lib = ctx.torch, ctx._lib
    flush = torch.empty(64 << 20, dtype=torch.float32, device=ctx.dev) if flush_l2 else None
    for _ in range(warmup):
        device_step()
    ctx.barrier()
    clocks = ClockSampler(ctx.local)
    if ctx.rank == 0:
        clocks.start()
    n0 = count_launches()
    ctx.barrier()
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            device_step()
        e1.record()
        ctx.barrier()
        ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    else:
        evs = []
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            device_step()
            b.record()
            evs.append((a, b))
        ctx.barrier()
        ms = ctx.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs))
    launches = count_launches() - n0
    if after_timed is not None:
        after_timed()
    # per-kernel shares: events around every launch (cannot be recorded inside a replayed graph: always eager)
    ctx.barrier()
    _lib.profile_begin(max_records=launches + 64)
    for _ in range(steps):
        if flush is not None:
            flush.zero_()
        device_step(eager=True)
    torch.cuda.synchronize()
    prof = _lib.profile_end()
    # clocks / throttle reasons were sampled from before the timed region to here: the timed steps and the same
    # steps once more for the per-kernel events, i.e. only while the GPU runs the measured kernels
    clk = clocks.stop() if ctx.rank == 0 else None
    for _ in range(2):
        host = e2e_step()
    ctx.barrier()
    if flush is None:
        t0 = time.perf_counter()
        for _ in range(steps):
            host = e2e_step()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    else:
        e2e_s = 0.0
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            host = e2e_step()
            torch.cuda.synchronize()
            e2e_s += time.perf_counter() - t0
    e2e_s = ctx.max_over_ranks(e2e_s)
    ctx.barrier()
    return ms, launches, prof, clk, e2e_s, host


def kernel_rooflines(ctx, key, prof, K, T, steps, cells_per_launch, clk, fits_l2):
    """One entry per kernel of the step: algorithmic GB/s against the measured HBM peak (the contract's roofline), Tflop/s
    against the non-FMA fp32 issue peak, and which of the two actually limits the kernel."""
    sm_mhz = (clk or {}).get("sm_mhz") or 1965.0
    fp32_peak = ctx.sm_count * 128 * sm_mhz * 1e6 / 1e12
    total_ms = sum(v[0] for v in prof.values()) or 1.0
    out = []
    for ph, (ms, n) in sorted(prof.items(), key=lambda kv: -kv[1][0]):
        if not n or ph in ("other", "splat", "halo", "halo_unpack"):
            continue
        sweeps = K * T * steps / n if ph == "jacobi" else 0
        nsteps = T * steps / n if ph == "step_fused" else 1
        bpc, fpc = phase_bytes_per_cell(K, sweeps, nsteps)[ph], phase_flops_per_cell(K, sweeps, nsteps)[ph]
        if ph == "advect_v" and prof.get("project_advect_u", (0, 0))[1]:
            bpc, fpc = bpc + 4, fpc + 3                     # the v advection then re-reads p and projects v itself
        t = ms / n * 1e-3
        gbs, tfs = bpc * cells_per_launch / t / 1e9, fpc * cells_per_launch / t / 1e12
        traffic = committed_traffic(ph, key)
        on_chip = ph in ("step_fused", "jacobi")            # state / pressure tile resident on chip across sweeps or steps
        bound = "fp32_issue" if on_chip else ("l2" if fits_l2 else "hbm")
        e = {"kernel": KERNEL_NAMES[ph], "launches": int(n), "avg_launch_us": 1e3 * ms / n, "share_of_step": ms / total_ms,
             "algorithmic_gbs": gbs, "frac_hbm": gbs / ctx.peak, "fp32_tflops": tfs, "frac_fp32": tfs / fp32_peak,
             "bound": bound, "frac": (tfs / fp32_peak) if on_chip else gbs / ctx.peak, "traffic": traffic}
        if traffic:
            e["dram_gbs"] = traffic / t / 1e9
            e["frac_dram"] = traffic / t / 1e9 / ctx.peak
        out.append(e)
    return out, fp32_peak


def contract_roofline(ctx, key, prof, K, T, steps, cells_per_launch, kernels, rename=None):
    """The `roofline` object of the contract: dominant kernel, algorithmic bytes per launch / mean launch duration / HBM peak."""
    dom = max((k for k in prof if prof[k][1] > 0 and k not in ("other", "splat", "halo", "halo_unpack")), key=lambda k: prof[k][0])
    dom_ms, dom_n = prof[dom]
    total_ms = sum(v[0] for v in prof.values())
    sweeps = K * T * steps / dom_n if dom == "jacobi" else 0
    nsteps = T * steps / dom_n if dom == "step_fused" else 1
    alg = phase_bytes_per_cell(K, sweeps, nsteps)[dom] * cells_per_launch
    achieved = alg / (dom_ms / dom_n * 1e-3) / 1e9
    kname = rename if (rename and dom == "step_fused") else KERNEL_NAMES[dom]
    k = next(e for e in kernels if e["kernel"] == kname)
    if dom == "jacobi":
        note = ("achieved > peak is possible: %d sweeps are fused per launch with the pressure tile on-chip, so real DRAM "
                "traffic is below the algorithmic 12 B/cell-sweep (see `traffic`); `binding` names what limits the kernel" % round(sweeps))
    elif dom == "step_fused":
        note = ("achieved > peak is possible: %d whole steps run per launch with u, v, density in shared memory and the pressure "
                "in registers, so real DRAM traffic is one state read + write per launch and 4 B/cell-step of frames, far below "
                "the algorithmic %d B/cell-step (see `traffic`, `dram`); the kernel is bound by FP32 issue, not HBM: see `binding`"
                % (round(nsteps), 100 + 12 * K))
    else:
        note = ""
    r = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": ctx.peak, "unit": "GB/s", "frac": achieved / ctx.peak,
         "traffic": k["traffic"], "peak_source": ctx.peak_src, "algorithmic_bytes_per_launch": alg, "avg_launch_ms": dom_ms / dom_n,
         "launches_timed": int(dom_n), "share_of_step": dom_ms / total_ms,
         "binding": {"bound": k["bound"], "frac": k["frac"],
                     "what": "fraction of %s" % ("148 SMs x 128 fp32 lanes x SM clock, one non-FMA add or multiply per lane per clock"
                                                 if k["bound"] == "fp32_issue" else "the measured copy bandwidth")},
         "note": note}
    if k.get("dram_gbs") is not None:
        r["dram"] = {"gbs": k["dram_gbs"], "frac_of_peak": k["frac_dram"], "what": "ncu dram bytes per launch / measured launch time"}
    return r


def d2h_ceiling(ctx, nbytes):
    """What the box sustains when every rank copies device -> pinned host at once (one contiguous block per copy, four
    copies back to back): the bound of the e2e leg.  Returns (aggregate GB/s, slowest rank GB/s)."""
    torch = ctx.torch
    from smokephysai_b200 import hostmem
    n = max(1 << 20, int(nbytes)) // 4
    dev = torch.empty(n, dtype=torch.float32, device=ctx.dev)
    host = hostmem.pinned_empty((n,), torch.float32, ctx.dev)
    reps = 4
    host.copy_(dev, non_blocking=True)
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        host.copy_(dev, non_blocking=True)
    torch.cuda.synchronize()
    mine = time.perf_counter() - t0
    slowest = ctx.max_over_ranks(mine)
    ctx.barrier()
    del dev, host
    return ctx.world * reps * n * 4 / slowest / 1e9, reps * n * 4 / slowest / 1e9


def run_batched(ctx, key, steps, warmup):
    """c2 / c2s / c3: `batch` independent grids per GPU through SmokeSimulator (fused kernel or phase kernels, the library picks)."""
    torch, args = ctx.torch, ctx.args
    from smokephysai_b200 import SmokeSimulator, _lib
    ctx._lib = _lib
    wl = WORKLOADS[key]
    cfg = config_for(key, ctx.world)
    h, w, K, T, B = wl["h"], wl["w"], wl["K"], wl["tsteps"], cfg["sequences_per_gpu"]
    sim = SmokeSimulator((h, w), 0.01, 0.001, ctx.dev, jacobi_iters=K, batch=B, sweeps_per_launch=args.sweeps_per_launch,
                         step_kernel=args.step_kernel)
    ns = sim.ns_solver
    L = ns._layout
    ems = [emitters_for_sequence(ctx.rank * B + s, h, w) for s in range(B)]
    fmul = sim.fractal_gen.multiplier((h, w), 0.05)
    frames = torch.empty(B, T, h, L.pitch_c, dtype=torch.float32, device=ctx.dev)
    src, off, h2d_bytes = ns.upload_sources(ems)
    emitter_lists = [[((x, y), i) for x, y, _, i in lst] for lst in ems]

    def device_step(eager=False):
        ns.setup_grid()
        ns.splat_uploaded(src, off)
        ns.run_steps(T, fmul=fmul, out=frames)

    def e2e_step():
        return sim.generate_sequences(emitter_lists, T, to_host=True)      # returns after the last D2H copy

    def dump():
        dump_outputs(ctx, key, {"frames": frames[..., :w], "u": ns.u, "v": ns.v, "p": ns.p, "density": ns.density})

    ws = ns._arena.numel() * 4 + frames.numel() * 4
    fits_l2 = ws < L2_MB * 1e6
    ms, launches, prof, clk, e2e_s, host_frames = timed_passes(ctx, device_step, e2e_step, steps, warmup, _lib.launch_count, flush_l2=fits_l2,
                                                               after_timed=dump if args.dump_outputs else None)
    total_cells = ctx.world * B * h * w * T
    value = total_cells * steps / (ms * 1e-3)
    d2h_bytes = T * B * h * L.pitch_c * 4
    checksum = float(host_frames[:, -1].double().sum())

    # the f4 hand-off: frames stay on the GPU and are consumed there (a reduction standing in for the model's forward);
    # 8 bytes come back per bench step
    for _ in range(2):
        float(sim.generate_sequences(emitter_lists, T, to_host=False).sum().item())
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        dsum = float(sim.generate_sequences(emitter_lists, T, to_host=False).sum().item())
    e2e_dev_s = ctx.max_over_ranks(time.perf_counter() - t0)
    ctx.barrier()
    ceiling = d2h_ceiling(ctx, d2h_bytes) if key in ("c2", "c2s") else None

    fused = ns.step_is_fused(T)
    cells_per_launch = B * h * w
    clustered = key == "c2s" and fused and B * 4 <= ctx.sm_count - 16          # k_step_cluster runs these: its own traffic capture
    kernels, fp32_peak = kernel_rooflines(ctx, "c2_strong" if clustered else ("c2" if key == "c2s" else key), prof, K, T, steps,
                                          cells_per_launch, clk, fits_l2)
    if clustered:
        for e in kernels:
            if e["kernel"] == "k_step_fused":
                e["kernel"] = "k_step_cluster<4>"
    step_bytes, step_flops = 100 + 12 * K, 118 + 5 * K
    per_gpu = value / ctx.world
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": cfg, "step_kernel": "fused" if fused else "phases",
        "clocks": clk,
        "e2e": {"value": total_cells * steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": 1e3 * e2e_s / steps,
                "api": "SmokeSimulator.generate_sequences(host emitter lists, to_host=True) -> pinned host frames",
                "last_frame_checksum": checksum, "pinned_host_numa_node": getattr(sim, "_gen_host_node", None),
                "d2h_gbs_per_gpu": d2h_bytes / (e2e_s / steps) / 1e9},
        "e2e_device": {"value": total_cells * steps / e2e_dev_s, "unit": UNIT, "ms_per_step": 1e3 * e2e_dev_s / steps,
                       "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 8, "checksum": dsum,
                       "api": "SmokeSimulator.generate_sequences(host emitter lists, to_host=False) -> frames stay in HBM, consumed "
                              "by a device-side reduction (the simulator -> model hand-off of train.py:59-80)"},
        "gpu_launches": int(launches),
        "roofline": contract_roofline(ctx, key, prof, K, T, steps, cells_per_launch, kernels, "k_step_cluster<4>" if clustered else None),
        "kernels": kernels,
        "roofline_step": {"algorithmic_bytes_per_cell_step": step_bytes, "achieved": per_gpu * step_bytes / 1e9, "peak": ctx.peak,
                          "unit": "GB/s", "frac": per_gpu * step_bytes / 1e9 / ctx.peak, "per": "GPU"},
        "roofline_fp32": {"bound": "fp32 issue (what actually bounds the on-chip kernels; the HBM roofline above is the contract's)",
                          "flops_per_cell_step": step_flops, "achieved": per_gpu * step_flops / 1e12, "peak": fp32_peak,
                          "unit": "Tflop/s per GPU, non-FMA fp32", "frac": per_gpu * step_flops / 1e12 / fp32_peak,
                          "peak_source": "%d SMs x 128 lanes x %.0f MHz" % (ctx.sm_count, (clk or {}).get("sm_mhz") or 1965.0)},
        "phases_ms_per_step": {k: v[0] / steps for k, v in prof.items() if v[1]},
    }
    if ceiling is not None:
        agg, slow = ceiling
        out["e2e"]["d2h_ceiling_gbs"] = agg
        out["e2e"]["d2h_ceiling_gbs_per_gpu"] = slow
        out["e2e"]["frac_of_d2h_ceiling"] = out["e2e"]["d2h_gbs_per_gpu"] / slow
        out["e2e"]["d2h_ceiling_how"] = "all %d rank(s) at once: 4 back-to-back cudaMemcpyAsync of %d MB device -> pinned host" % (ctx.world, d2h_bytes // 1000000)
    del sim, ns, frames, host_frames
    torch.cuda.empty_cache()
    return out


def run_slab(ctx, key, steps, warmup):
    """c4: ONE grid in row slabs over the ranks (strong scaling), halo exchange between neighbours."""
    torch, args = ctx.torch, ctx.args
    from smokephysai_b200 import _lib
    from smokephysai_b200.slab import SlabNavierStokes
    ctx._lib = _lib
    wl = WORKLOADS[key]
    cfg = config_for(key, ctx.world)
    h, w, K, T = wl["h"], wl["w"], wl["K"], wl["tsteps"]
    world, rank = ctx.world, ctx.rank
    Tj = args.sweeps_per_launch or 10
    slab = SlabNavierStokes((h, w), 0.01, 0.001, ctx.dev, rank=rank, world=world, jacobi_iters=K, sweeps_per_launch=Tj,
                            halo=args.halo or (K + 4 if world > 1 else None), exchange=args.exchange)
    ems = emitters_for_sequence(0, h, w)
    slab.add_sources(ems)
    own_rows = slab.geom.R1 - slab.geom.R0
    # e2e: the owned density rows of a run go to pinned host memory through a device snapshot on a copy stream, so the read-back
    # of run k (268 MB at N = 1: 5 ms of PCIe) overlaps the steps of run k + 1; two snapshots / host buffers in rotation
    host_bufs = [torch.empty(own_rows, w, dtype=torch.float32).pin_memory() for _ in range(2)]
    snaps = [torch.empty(own_rows, w, dtype=torch.float32, device=ctx.dev) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=ctx.dev)
    copied = [torch.cuda.Event(), torch.cuda.Event()]
    for ev in copied:
        ev.record()
    host_d = host_bufs[0]
    run_no = [0]
    slab.step()                                   # eager once: NCCL / the peer mappings are set up on first use

    ahead = not args.no_push_ahead

    def device_step(eager=False):
        if ahead:
            slab.run_steps(T)               # every step but the last pushes the next step's ghost rows from its density advection
        else:
            for _ in range(T):
                slab.step()

    def e2e_step():
        slab.setup_grid()
        slab.add_sources(ems)
        device_step()
        k = run_no[0] & 1
        run_no[0] += 1
        main = torch.cuda.current_stream()
        main.wait_event(copied[k])                # the read-back that used this snapshot two runs ago is finished
        snaps[k].copy_(slab.owned("d"))
        ready = torch.cuda.Event()
        ready.record(main)
        copy_stream.wait_event(ready)
        with torch.cuda.stream(copy_stream):
            host_bufs[k].copy_(snaps[k], non_blocking=True)
            copied[k].record(copy_stream)
        return host_bufs[k].unsqueeze(0)          # complete after the synchronize that ends the timed region

    def dump():
        dump_outputs(ctx, key, {name: slab.owned(k) for k, name in (("u", "u"), ("v", "v"), ("p", "p"), ("d", "density"))})

    ms, launches, prof, clk, e2e_s, host = timed_passes(ctx, device_step, e2e_step, steps, warmup, _lib.launch_count,
                                                        after_timed=dump if args.dump_outputs else None)
    slab.check()
    total_cells = h * w * T
    value = total_cells * steps / (ms * 1e-3)
    cells_per_launch = slab.geom.hl * w
    kernels, fp32_peak = kernel_rooflines(ctx, key, prof, K, T, steps, cells_per_launch, clk, False)
    step_bytes = 100 + 12 * K
    per_gpu = value / world
    if world == 1:
        par = "single GPU, undecomposed; eager launches"
    else:
        par = "row slabs over %d GPU(s), halo %d rows; %s; %s; eager launches" % (
            world, slab.halo, slab.exchange_description(),
            "ghost rows of steps 2..%d pushed ahead from the previous step's density advection" % T if ahead else "every push at the head of its step")
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": cfg, "step_kernel": "phases", "exchange": par,
        "clocks": clk,
        "e2e": {"value": total_cells * steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 16 * len(ems) + 8,
                "d2h_bytes_per_step": host_d.numel() * 4, "ms_per_step": 1e3 * e2e_s / steps,
                "api": "SlabNavierStokes: setup_grid + add_sources(host list) + run_steps(%d) + owned density rows -> device snapshot -> pinned "
                       "host on a copy stream (the read-back of one run overlaps the steps of the next; all copies complete inside the timed region)" % T,
                "last_frame_checksum": float(host.double().sum())},
        "gpu_launches": int(launches),
        "roofline": contract_roofline(ctx, key, prof, K, T, steps, cells_per_launch, kernels),
        "kernels": kernels,
        "roofline_step": {"algorithmic_bytes_per_cell_step": step_bytes, "achieved": per_gpu * step_bytes / 1e9, "peak": ctx.peak,
                          "unit": "GB/s", "frac": per_gpu * step_bytes / 1e9 / ctx.peak,
                          "per": "GPU (owned cells only; ghost-row recompute not counted)"},
        "phases_ms_per_step": {k: v[0] / steps for k, v in prof.items() if v[1]},
        "ghost_rows_per_side": slab.halo if world > 1 else 0, "owned_rows_per_gpu": own_rows,
    }
    if world > 1:
        out["parity"] = slab_parity(ctx, slab, ems, h, w, K, Tj)
    if slab.exchanger is not None and hasattr(slab.exchanger, "close"):
        slab.exchanger.close()
    torch.cuda.synchronize()
    del slab, host_d, host_bufs, snaps
    torch.cuda.empty_cache()
    return out


def slab_parity(ctx, slab, ems, h, w, K, Tj, nsteps=2):
    """Outside every timed region: reset, run `nsteps` steps in slabs WITH the halo exchange the bench just timed, gather the owned
    rows of every field on every rank and compare them, on rank 0, bit for bit with the undecomposed run of the same grid."""
    torch = ctx.torch
    from smokephysai_b200 import NavierStokesSimulator
    slab.setup_grid()
    slab.add_sources(ems)
    if ctx.args.no_push_ahead:
        for _ in range(nsteps):
            slab.step()
    else:
        slab.run_steps(nsteps)
    slab.check()
    got = {k: slab.gather(k) for k in ("u", "v", "p", "d")}
    res = None
    if ctx.rank == 0:
        ref = NavierStokesSimulator((h, w), 0.01, 0.001, ctx.dev, jacobi_iters=K, sweeps_per_launch=Tj, step_kernel="phases")
        ref.add_sources([list(ems)])
        for _ in range(nsteps):
            ref.step()
        torch.cuda.synchronize()
        res = {"vs": "undecomposed %dx%d run on rank 0, %d steps, same emitters; owned rows of every rank gathered over NCCL" % (h, w, nsteps)}
        ok = True
        for k, name in (("u", "u"), ("v", "v"), ("p", "p"), ("d", "density")):
            a, b = got[k], getattr(ref, name)
            same = bool(a.shape == b.shape and torch.equal(a, b))
            ok &= same
            res[name] = "bit-equal" if same else "DIFFERS (max abs %.3e)" % float((a - b).abs().max())
        res["ok"] = ok
        res["sha256_density"] = hashlib.sha256(got["d"].cpu().numpy().tobytes()).hexdigest()
        res["max_abs_density"] = float(got["d"].abs().max())
        del ref
    del got
    ctx.barrier()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all"] + sorted(WORKLOADS),
                    help="all: the c2 line with c2_strong / c3 / c4 under `also`; a name: that workload alone as the printed line")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sweeps-per-launch", type=int, default=0)
    ap.add_argument("--halo", type=int, default=0, help="c4: ghost rows per slab side (0: K + 4, one halo exchange per step; "
                    "sweeps-per-launch + 4 is the minimum and exchanges p after every Jacobi launch)")
    ap.add_argument("--no-push-ahead", action="store_true", help="c4: every step pushes its ghost rows at its head (default: all but "
                    "the first step of a bench step push them from the previous step's density advection: SlabNavierStokes.run_steps)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="c4 halo exchange: peer = direct stores into the neighbour's arena over NVLink (CUDA IPC), nccl = "
                         "ncclSend/ncclRecv groups issued from C, auto = peer when every neighbour is peer-accessible")
    ap.add_argument("--step-kernel", default="auto", choices=["auto", "phases", "fused"],
                    help="auto: whole simulation on one SM for grids <= 128x128 (k_step_fused), else one kernel per phase")
    ap.add_argument("--dump-outputs", metavar="DIR", help="right after the timed steps of each workload, write what its last timed "
                    "step left as DIR/<workload>_<name>.npy in fp32: c2 / c3 the frames and the u, v, p, density state of every "
                    "sequence, c4 the u, v, p, density rows of the grid; an array of more than %d values as a fixed seeded sample "
                    "of its rows (on N GPUs every rank writes its own files, within 1/N of that).  The inputs are seeded, so two builds run with the same arguments can be compared file by file"
                    % DUMP_MAX_VALUES)
    args = ap.parse_args()
    main_key = "c2" if args.workload == "all" else args.workload
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes what the GPU path computed; --impl reference has none")
    if args.impl == "reference":
        return reference_arm(args, main_key)
    if args.warmup < 3:
        args.warmup = 3

    ctx = Ctx(args)
    world, rank = ctx.world, ctx.rank
    if main_key == "c4":
        out = run_slab(ctx, "c4", args.steps, args.warmup)
    elif main_key == "c2s" and world == 1:
        out = run_batched(ctx, "c2", args.steps, args.warmup)
    else:
        out = run_batched(ctx, main_key, args.steps, args.warmup)
    if args.workload == "all":
        also = {}
        if world > 1:
            also["c2_strong"] = run_batched(ctx, "c2s", args.steps, args.warmup)
        else:
            also["c2_strong"] = {"same_as": "the main line: at N = 1 the 256 sequences of configs[1] are the 256 sequences per GPU"}
            also["c3"] = run_batched(ctx, "c3", args.steps, args.warmup)
        also["c4"] = run_slab(ctx, "c4", args.steps, args.warmup)
        if world > 1:
            also["c3"] = {"skipped": "one 1024x1024 grid does not shard: measured at N = 1 only"}
        out["also"] = also

    if world > 1:
        ctx.dist.destroy_process_group()
    if rank != 0:
        return 0

    if not args.no_cpu_baseline:
        wl = WORKLOADS[main_key]
        out["reference_torch"] = reference_torch_numbers(ctx.dev, wl["K"]) if wl["h"] <= 128 else None
        import oracle
        oracle.build()
        cores = os.cpu_count() or 1
        nseq = wl["batch"]
        wl_cpu = dict(wl)
        if wl["h"] >= 1024:
            wl_cpu["tsteps"] = 2 if wl["h"] < 4096 else 1
        cpu_run(wl_cpu, min(nseq, cores), cores)                 # warm the threads / page in
        cval, cdt = cpu_run(wl_cpu, nseq, cores)
        out["cpu_baseline"] = {"value": cval, "unit": UNIT, "cores": min(cores, nseq), "kind": "port", "seconds": cdt,
                               "sample": "%d sequences x %d steps of %dx%d, K=%d (oracle C port, pthreads over sequences)"
                                         % (nseq, wl_cpu["tsteps"], wl["h"], wl["w"], wl["K"])}
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
