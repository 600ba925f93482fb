"""SmokeSimulator -- the reference's simulator facade (src/physics/smoke_simulator.py:8-140) on the
sm_100a solver: same constructor, attributes (ns_solver, fractal_gen, device, history, max_history) and
methods (add_incense_source, simulate_step, get_chaos_features, compute_*).

simulate_step() is ONE pass of the CUDA step with the fractal multiply fused into the returned copy
(the reference: ns.step() + ~960 eager launches of fractal recompute, SURVEY.md s2.2).
Keyword-only extensions: jacobi_iters, batch, sweeps_per_launch, step_kernel (forwarded to NavierStokesSimulator), and
generate_sequences() -- the batched back-end of data_loader.py:37-99.
"""
import numpy as np
import torch
import torch.nn as nn

from . import _lib, chaos, hostmem
from .fractal_generator import FractalGenerator
from .navier_stokes import NavierStokesSimulator


class SmokeSimulator(nn.Module):
    """Complete smoke physics simulation system (reference: smoke_simulator.py:8)."""

    def __init__(self, grid_size=(128, 128), dt=0.01, viscosity=0.001, device="cuda", *,
                 jacobi_iters=20, batch=1, sweeps_per_launch=0, step_kernel="auto"):
        super().__init__()
        self.ns_solver = NavierStokesSimulator(grid_size, dt, viscosity, device, jacobi_iters=jacobi_iters,
                                               batch=batch, sweeps_per_launch=sweeps_per_launch, step_kernel=step_kernel)
        self.fractal_gen = FractalGenerator(device)
        self.device = device
        self.history = []          # smoke_simulator.py:23
        self.max_history = 100     # :24

    def add_incense_source(self, positions, intensities, *, continuous=False):
        """Add incense smoke sources: radius is fixed to 8 (smoke_simulator.py:26-29).

        continuous=True: sticks that keep burning -- the emitters are appended to every simulation's continuous sources
        (NavierStokesSimulator.set_continuous_sources) and inject at the head of every later step instead of once."""
        if not continuous:
            for (x, y), intensity in zip(positions, intensities):
                self.ns_solver.add_smoke_source(x, y, radius=8, intensity=intensity)
            return
        ns = self.ns_solver
        new = [(int(x), int(y), 8, float(i)) for (x, y), i in zip(positions, intensities)]
        lists = ns.continuous_sources or [[] for _ in range(ns.batch)]
        ns.set_continuous_sources([lst + new for lst in lists])

    def set_obstacles(self, mask):
        """Solid obstacles of every later step: NavierStokesSimulator.set_obstacles (None clears them)."""
        self.ns_solver.set_obstacles(mask)

    def simulate_step(self, add_fractal=True):
        """One simulation step; returns the (fractal-scaled) density frame (smoke_simulator.py:31-45)."""
        ns = self.ns_solver
        fmul = self.fractal_gen.multiplier((ns.h, ns.w), 0.05) if add_fractal else None     # intensity=0.05 (:38)
        density = ns.step(fmul=fmul)
        self.history.append(density.clone())                                               # :41
        if len(self.history) > self.max_history:
            self.history.pop(0)                                                            # :42-43
        return density

    # -------------------------------------------------------------- batched generation (data_loader.py:37-99)
    def generate_sequences(self, emitters, sequence_length=20, add_fractal=True, to_host=False, steps_per_copy=None,
                           frame_dtype=torch.float32, continuous=False, schedule=None, forcing=None, obstacles=None):
        """Reset, splat one emitter list per simulation, run sequence_length steps.

        emitters[b] = [((x, y), intensity), ...] for simulation b (len == batch).  Returns frames
        [batch, sequence_length, h, w] -- each [b] is what the reference's per-sample loop stacks into
        sample['sequence'] (data_loader.py:66-68, :91).  History/chaos features are not touched.

        to_host=True hands the frames back in pinned host memory (the dataset is pickled from the host,
        data_loader.py:33-34): the frames of a chunk of steps are copied device->host on a second stream
        while the next chunk computes, from a time-major [sequence_length, batch, h, w] device buffer so every
        copy is one contiguous block.  steps_per_copy is the chunk length (default: 1 for the phase-per-kernel
        step, 2 when the fused kernel keeps the state on chip across the steps of a launch).  The returned
        tensor is the [batch, sequence_length, h, w] view of the pinned time-major buffer, which this
        simulator owns and reuses on the next call of the same frame_dtype.

        frame_dtype torch.float16 / torch.bfloat16: the frames are rounded once (to nearest even) by the kernels that
        write them -- equal to the float32 frames' .to(frame_dtype) -- so half the bytes cross PCIe; the simulation
        itself is the same whatever the dtype.

        continuous=True: every sample's emitters inject at the head of every step (a sustained plume) instead of once; frame 0
        is the same as with continuous=False.  The simulator's own continuous sources are set aside for the call and restored.

        schedule = (xy, radius, intensity), [T, B, E, ...] with T = sequence_length (NavierStokesSimulator.run_steps): emitters
        that move or change intensity, row t added at the head of step t after the samples' emitters were splatted once at the
        reset.  The records are uploaded once per call (through pinned memory when to_host); the chunks of the to_host path read
        their rows of the same records.  It does not combine with continuous sources (continuous=True or the simulator's own):
        fold constant emitters into the schedule.

        forcing = (du, dv), constant or [T, B, ...] per step (NavierStokesSimulator.run_steps): velocity increments added at the
        head of every step.  Uploaded once per call (through pinned memory when to_host); the chunks of the to_host path read their
        rows of the same upload.  It combines with continuous sources and schedules.

        obstacles: a solid mask for this call ([h, w] or [batch, h, w], NavierStokesSimulator.set_obstacles); the simulator's own
        obstacles (if any) apply when it is None, and are restored after the call.  With obstacles the steps run on the phase
        kernels, and steps_per_copy defaults to 1."""
        ns = self.ns_solver
        if obstacles is None:
            return self._generate(emitters, sequence_length, add_fractal, to_host, steps_per_copy, frame_dtype, continuous, schedule,
                                  forcing)
        saved = ns._solid
        ns.set_obstacles(obstacles)                        # ValueError for a bad mask, before any work
        try:
            return self._generate(emitters, sequence_length, add_fractal, to_host, steps_per_copy, frame_dtype, continuous, schedule,
                                  forcing)
        finally:
            ns._solid = saved

    def _generate(self, emitters, sequence_length, add_fractal, to_host, steps_per_copy, frame_dtype, continuous, schedule, forcing):
        ns = self.ns_solver
        B, T = ns.batch, int(sequence_length)
        _lib.frame_format(frame_dtype)                     # ValueError for an unsupported dtype, before any work
        if schedule is not None and (continuous or ns._csrc is not None):
            raise ValueError("a source schedule and continuous sources do not combine: fold the constant emitters into "
                             "the schedule")
        ns._check_forcing(forcing, T)                      # both inputs are checked before either is uploaded
        sched = None
        if schedule is not None:
            up = ns.upload_schedule(schedule, T, pin=to_host)
            sched = None if up is None else up + (0,)
        force = ns._forcing(forcing, T, pin=to_host)
        lists = [[(x, y, 8, inten) for (x, y), inten in lst] for lst in emitters]
        ns.setup_grid()
        src, off, _ = ns.upload_sources(lists, pin=to_host)
        fmul = self.fractal_gen.multiplier((ns.h, ns.w), 0.05) if add_fractal else None
        if not continuous:
            ns.splat_uploaded(src, off)
            return self._run_sequences(T, fmul, to_host, steps_per_copy, frame_dtype, sched, force)
        saved = ns._csrc
        ns._csrc = (lists, src, off)
        try:
            return self._run_sequences(T, fmul, to_host, steps_per_copy, frame_dtype, None, force)
        finally:
            ns._csrc = saved

    def _run_sequences(self, T, fmul, to_host, steps_per_copy, frame_dtype, sched=None, force=None):
        ns = self.ns_solver
        L = ns._layout
        B = ns.batch
        if not to_host:
            fr = ns._run_steps(T, fmul, True, None, frame_dtype, sched, force)
            return fr if B > 1 else fr.unsqueeze(0)
        # one (device, pinned host) buffer pair per frame dtype, keyed (T, dtype): calls that alternate dtypes each keep
        # their own buffers instead of reallocating pinned memory every call or handing one call's frames to the other
        if not hasattr(self, "_gen_bufs"):
            self._gen_bufs = {}
            self._gen_copy_stream = torch.cuda.Stream(device=ns._cuda)
        key = (T, frame_dtype)
        bufs = self._gen_bufs.get(frame_dtype)
        if bufs is None or bufs[0] != key:
            dev = torch.empty(T, B, L.h, L.pitch_c, dtype=frame_dtype, device=ns._cuda)
            # pinned pages on the NUMA node of this GPU's PCIe root: with several ranks copying at once a buffer on the far
            # socket costs most of the D2H bandwidth (hostmem.py)
            host = hostmem.pinned_empty((T, B, L.h, L.pitch_c), frame_dtype, ns._cuda)
            self._gen_host_node = hostmem.gpu_locality(ns._cuda)[0]
            bufs = self._gen_bufs[frame_dtype] = (key, dev, host)
        _, dev, host = bufs
        cs = self._gen_copy_stream
        main = torch.cuda.current_stream(ns._cuda)
        cs.wait_stream(main)                      # the previous call's consumer is done with the buffers
        n = int(steps_per_copy) if steps_per_copy else (2 if ns.step_is_fused(2) else 1)
        for t in range(0, T, n):
            m = min(n, T - t)
            # the chunk's steps t .. t + m - 1 are the schedule's and the forcing's rows t .. t + m - 1 (offsets from offsets[t * B]
            # on, forcing from element t * B * stride)
            ns._run_steps_time_major(m, dev[t:t + m], fmul, None if sched is None else sched[:2] + (t,),
                                     None if force is None else force[:3] + (t,))
            ev = torch.cuda.Event()
            ev.record(main)
            cs.wait_event(ev)
            with torch.cuda.stream(cs):
                host[t:t + m].copy_(dev[t:t + m], non_blocking=True)
        cs.synchronize()
        return host.permute(1, 0, 2, 3)[..., :L.w]

    # -------------------------------------------------------------- chaos features (smoke_simulator.py:47-140)
    def _staged_history(self, n):
        """The last n history frames as one contiguous padded [n, h, pitch] device tensor."""
        ns = self.ns_solver
        L = ns._layout
        buf = torch.zeros(n, L.h, L.pitch_c, dtype=torch.float32, device=ns._cuda)
        for k, f in enumerate(self.history[-n:]):
            if f.dim() != 2:
                raise ValueError("chaos features are defined for single simulations (batch == 1), as in the reference")
            buf[k, :, :L.w] = f.to(ns._cuda)
        return buf

    def get_chaos_features(self):
        if len(self.history) < 10:
            return {}
        return {
            "lyapunov_exponent": self.compute_lyapunov_exponent(),
            "fractal_dimension": self.compute_fractal_dimension(),
            "entropy": self.compute_entropy(),
        }

    def compute_lyapunov_exponent(self):
        """Mean log-growth of the distance between consecutive frames over the last 20 (smoke_simulator.py:67-87)."""
        if len(self.history) < 20:
            return 0.0
        return chaos.lyapunov_from_distances(chaos.frame_distances(self._staged_history(20), self.ns_solver.w))

    def compute_fractal_dimension(self):
        """Box-counting dimension of the above-mean mask at scales 2..32 (smoke_simulator.py:89-124)."""
        if not self.history:
            return 0.0
        box, _ = chaos.frame_counts(self._staged_history(1), self.ns_solver.w)
        return chaos.fractal_dimension_from_counts(box[0].cpu().numpy())

    def compute_entropy(self):
        """Shannon entropy of the 256-bin histogram of the last frame over [0, 1] (smoke_simulator.py:126-140)."""
        if not self.history:
            return 0.0
        _, hist = chaos.frame_counts(self._staged_history(1), self.ns_solver.w)
        return chaos.entropy_from_hist(hist[0])

    # -------------------------------------------------------------- dataset back-end (data_loader.py:37-99)
    def generate_dataset(self, num_samples, sequence_length=20, rng=None, to_cpu=False, progress=None):
        """Batched replacement of SyntheticSmokeDataset._generate_synthetic_data (data_loader.py:37-99).

        Draws the emitters of sample after sample with the same np.random call sequence as the reference
        (count in [1,3], then x, y, intensity per emitter, :49-58; `rng` defaults to the global np.random so a
        seeded run draws what the reference draws), simulates `batch` samples at a time, evaluates the chaos
        features of every frame t >= 10 on the device and averages them per sample (:71-88).  The history
        the reference never clears between samples (its Lyapunov feature of sample k sees the tail of sample
        k-1; SURVEY.md s3.3) is reproduced: distances run over the frames in sample-major order.
        Returns the reference's list of dicts: 'sequence' [T, h, w], 'chaos_features', 'source_config'."""
        rng = np.random if rng is None else rng
        ns = self.ns_solver
        L = ns._layout
        B, T, h, w = ns.batch, int(sequence_length), ns.h, ns.w
        if self.history:
            raise RuntimeError("generate_dataset starts from an empty history, like a freshly built reference simulator")
        fmul = self.fractal_gen.multiplier((h, w), 0.05)
        data, prev_last, all_dist = [], None, []          # all_dist[m] = ||frame m+1 - frame m|| over the flat sample-major order
        keep_cuda = ns._out_device.type == "cuda" and not to_cpu
        for first in range(0, num_samples, B):
            nb = min(B, num_samples - first)
            configs = []
            for _ in range(nb):
                n_src = rng.randint(1, 4)
                pos, inten = [], []
                for _ in range(n_src):
                    x = rng.randint(20, w - 20)
                    y = rng.randint(20, h - 20)
                    intensity = rng.uniform(0.5, 2.0)
                    pos.append((x, y))
                    inten.append(intensity)
                configs.append((pos, inten))
            ns.setup_grid()
            ns.add_sources([[(x, y, 8, i) for (x, y), i in zip(p, q)] for p, q in configs] + [[] for _ in range(B - nb)])
            padded = torch.empty(B, T, h, L.pitch_c, dtype=torch.float32, device=ns._cuda)
            ns.run_steps(T, fmul=fmul, out=padded)
            flat = padded.view(B * T, h, L.pitch_c)[: nb * T]
            box, hist = chaos.frame_counts(flat, w)
            if prev_last is not None:                                              # seam with the previous chunk
                all_dist.extend(chaos.frame_distances(torch.stack([prev_last, flat[0]]), w))
            all_dist.extend(chaos.frame_distances(flat, w))
            prev_last = flat[-1].clone()
            box_h, hist_h = box.cpu().numpy(), hist.cpu()
            seqs = padded[:nb, :, :, :w]
            seqs = seqs.contiguous() if keep_cuda else seqs.cpu()
            for s in range(nb):
                feats = []
                for t in range(10, T):                                             # data_loader.py:71 "wait for stabilization"
                    n = (first + s) * T + t                                        # flat index; the history holds frames <= n
                    lyap = chaos.lyapunov_from_distances(all_dist[n - 19: n]) if n + 1 >= 20 else 0.0
                    feats.append((lyap, chaos.fractal_dimension_from_counts(box_h[s * T + t]),
                                  chaos.entropy_from_hist(hist_h[s * T + t])))
                if feats:
                    avg = {"lyapunov_exponent": np.mean([f[0] for f in feats]), "fractal_dimension": np.mean([f[1] for f in feats]),
                           "entropy": np.mean([f[2] for f in feats])}
                else:
                    avg = {"lyapunov_exponent": 0.0, "fractal_dimension": 1.0, "entropy": 0.0}
                data.append({"sequence": seqs[s], "chaos_features": avg,
                             "source_config": {"positions": configs[s][0], "intensities": configs[s][1]}})
            if progress is not None:
                progress(nb)
        # leave the history as the reference's loop would: the last (up to) max_history frames
        frames = [d["sequence"][t] for d in data[-(self.max_history // max(T, 1) + 2):] for t in range(T)]
        self.history = frames[-self.max_history:]
        return data

    def forward(self, add_fractal=True):
        return self.simulate_step(add_fractal)
