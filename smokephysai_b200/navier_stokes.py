"""NavierStokesSimulator -- the reference's grid fluid solver surface (src/physics/navier_stokes.py:6-173)
on hand-written sm_100a kernels behind libsmoke_sm100.so.

Same constructor, attributes (grid_size, dt, viscosity, device, h, w, u, v, p, density, boundary) and
methods (setup_grid, add_smoke_source, diffusion_step, advection_step, interpolate_velocity_u/v,
bilinear_interpolate, pressure_projection, step) as the reference class, so callers written against
`src.physics.navier_stokes` run unchanged.  Keyword-only extensions (reference defaults):
`jacobi_iters=20` (the literal at navier_stokes.py:139), `batch=1` (independent simulations; fields gain
a leading dimension when batch > 1), `sweeps_per_launch=0` (temporal-blocking depth, 0 = library default),
`step_kernel="auto"` ("fused": whole simulation on one SM, all steps of a call in one launch, grids up to
128 x 128; "phases": one kernel per phase; "auto": fused when the grid qualifies and the call is run_steps(n >= 2)
or carries at least 32 simulations -- bit-identical results either way).

There is no CPU compute path.  `device='cpu'` (benchmark.py:260 passes it) only means "hand results back
as CPU tensors": the step always runs on the current CUDA device.

Host PyTorch is used for device memory and streams only; all arithmetic on the path is in csrc/*.cu.
"""
import ctypes as C

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._lib import Grid, Params, Source, State


SOURCE_DTYPE = np.dtype([("x", "<i4"), ("y", "<i4"), ("radius", "<i4"), ("intensity", "<f4")])     # smk_source_t


def _round4(n):
    return (int(n) + 3) & ~3


def check_source_lists(per_sim, batch):
    """per_sim[b] = [(x, y, radius, intensity), ...] for each of `batch` simulations -> the same as lists of
    (int, int, int, float) tuples; ValueError for anything else."""
    if isinstance(per_sim, (str, bytes)) or not hasattr(per_sim, "__len__") or len(per_sim) != batch:
        raise ValueError("need one emitter list per simulation (%d), got %r" % (batch, per_sim if not hasattr(per_sim, "__len__") else len(per_sim)))
    out = []
    for b, lst in enumerate(per_sim):
        if isinstance(lst, (str, bytes)) or not hasattr(lst, "__iter__"):
            raise ValueError("emitter list %d is not a list: %r" % (b, lst))
        recs = []
        for e in lst:
            if not hasattr(e, "__len__") or len(e) != 4:
                raise ValueError("an emitter is (x, y, radius, intensity), got %r in list %d" % (e, b))
            try:
                recs.append((int(e[0]), int(e[1]), int(e[2]), float(e[3])))
            except (TypeError, ValueError):
                raise ValueError("an emitter is (x, y, radius, intensity) of numbers, got %r in list %d" % (e, b)) from None
        out.append(recs)
    return out


def pack_sources(per_sim):
    """Per-simulation emitter lists -> (smk_source_t records as a SOURCE_DTYPE array of at least one record, int32 offsets
    [len(per_sim) + 1]): simulation b owns records offsets[b] .. offsets[b + 1] - 1, in list order."""
    flat, offs = [], [0]
    for lst in per_sim:
        flat.extend(lst)
        offs.append(len(flat))
    rec = np.zeros(max(len(flat), 1), dtype=SOURCE_DTYPE)          # smk_source_t records, 16 B each
    if flat:
        arr = np.asarray(flat, dtype=np.float64).reshape(len(flat), 4)
        rec["x"], rec["y"], rec["radius"] = arr[:, 0].astype(np.int32), arr[:, 1].astype(np.int32), arr[:, 2].astype(np.int32)
        rec["intensity"] = arr[:, 3].astype(np.float32)
    return rec, np.asarray(offs, dtype=np.int32)


def _as_tensor(name, a):
    if isinstance(a, np.ndarray):
        return torch.from_numpy(a)
    if torch.is_tensor(a):
        return a
    raise ValueError("schedule %s must be a numpy array or a torch tensor, got %r" % (name, type(a)))


def pack_schedule(schedule, nsteps, batch):
    """A source schedule (xy, radius, intensity) -> (int32 records [T * B * E, 4] in the smk_source_t layout with the intensity
    bits in column 3, E), or (None, 0) when E == 0.

    xy: integer [T, B, E, 2] (column x, row y); radius: integer [T, B, E]; intensity: float32 [T, B, E]; numpy arrays, CPU
    tensors or tensors on one CUDA device (the records are built where the inputs are).  Entry (t, b, e) is emitter e of
    simulation b at the head of step t; an entry with radius < 0 adds nothing, which pads lists of different lengths to E.
    The records are step-major, so the offsets of row (t, b) are arange(T * B + 1) * E (schedule_offsets).  Integer values
    must fit int32.  ValueError for anything else, before any work; T must be nsteps and B the batch."""
    if not isinstance(schedule, (tuple, list)) or len(schedule) != 3:
        raise ValueError("a schedule is a tuple (xy, radius, intensity)")
    xy, radius, inten = (_as_tensor(n, a) for n, a in zip(("xy", "radius", "intensity"), schedule))
    if xy.dim() != 4 or xy.shape[3] != 2:
        raise ValueError("schedule xy must be [T, B, E, 2], got shape %s" % (tuple(xy.shape),))
    T, B, E = (int(n) for n in xy.shape[:3])
    for name, t in (("radius", radius), ("intensity", inten)):
        if tuple(t.shape) != (T, B, E):
            raise ValueError("schedule %s must be [T, B, E] = %s like xy, got shape %s" % (name, (T, B, E), tuple(t.shape)))
    for name, t in (("xy", xy), ("radius", radius)):
        if t.dtype not in (torch.int32, torch.int64):
            raise ValueError("schedule %s must be int32 or int64, got %s" % (name, t.dtype))
    if inten.dtype != torch.float32:
        raise ValueError("schedule intensity must be float32, got %s" % (inten.dtype,))
    if len({t.device for t in (xy, radius, inten)}) != 1:
        raise ValueError("schedule xy, radius and intensity must be on one device, got %s"
                         % sorted({str(t.device) for t in (xy, radius, inten)}))
    if T != int(nsteps) or B != int(batch):
        raise ValueError("the schedule has %d steps of %d simulations; the call has %d steps of %d" % (T, B, nsteps, batch))
    if T * B * E > 0x7fffffff or T * B + 1 > 0x7fffffff:
        raise ValueError("a schedule of %d x %d x %d emitters does not fit int32 offsets" % (T, B, E))
    if xy.device.type == "cpu" and E:
        for name, t in (("xy", xy), ("radius", radius)):
            if t.dtype == torch.int64 and (int(t.min()) < -0x80000000 or int(t.max()) > 0x7fffffff):
                raise ValueError("schedule %s values must fit int32" % name)
    if E == 0:
        return None, 0
    rec = torch.empty(T * B * E, 4, dtype=torch.int32, device=xy.device)
    rec[:, 0:2] = xy.reshape(-1, 2)
    rec[:, 2] = radius.reshape(-1)
    rec[:, 3] = inten.reshape(-1).contiguous().view(torch.int32)
    return rec, E


def schedule_offsets(nsteps, batch, E, device):
    """Offsets of a packed schedule: int32 [nsteps * batch + 1], row (t, b) = records [(t * batch + b) * E, (t * batch + b + 1) * E).
    Step-major, so the steps t0 .. of a chunk read offsets[t0 * batch:] with the same records."""
    return torch.arange(0, (nsteps * batch + 1) * E, E, dtype=torch.int32, device=device)


class FieldLayout:
    """Where each field lives inside the single fp32 arena (pure host arithmetic, testable without a GPU).

    Every field is [batch][rows][pitch] with pitch = cols rounded up to 4 elements so each row starts
    16-byte aligned (float4 access); u, v, density and p have two copies (the step ping-pongs them).
    """
    FIELDS = ("u0", "u1", "v0", "v1", "d0", "d1", "p0", "p1", "div", "boundary")

    def __init__(self, h, w, batch=1, row0=0, gh=0):
        self.h, self.w, self.batch = int(h), int(w), int(batch)
        self.row0, self.gh = int(row0), int(gh)            # row-slab placement inside a gh-row grid (0 = not a slab)
        if self.h < 1 or self.w < 1 or self.batch < 1:
            raise ValueError("grid_size and batch must be positive, got %r x %r, batch %r" % (h, w, batch))
        self.pitch_u = _round4(self.w)
        self.pitch_v = _round4(self.w + 1)
        self.pitch_c = _round4(self.w)
        self.stride_u = (self.h + 1) * self.pitch_u
        self.stride_v = self.h * self.pitch_v
        self.stride_c = self.h * self.pitch_c
        self.offset = {}
        off = 0
        for name in self.FIELDS:
            self.offset[name] = off
            off += self.batch * self.stride_of(name)
        self.total = off

    def kind(self, name):
        return name[0] if name[0] in "uv" else "c"

    def stride_of(self, name):
        return {"u": self.stride_u, "v": self.stride_v, "c": self.stride_c}[self.kind(name)]

    def shape_of(self, name):
        """(rows, cols, pitch) of a field."""
        k = self.kind(name)
        if k == "u":
            return self.h + 1, self.w, self.pitch_u
        if k == "v":
            return self.h, self.w + 1, self.pitch_v
        return self.h, self.w, self.pitch_c

    def grid_struct(self):
        return Grid(self.h, self.w, self.batch, self.pitch_u, self.pitch_v, self.pitch_c,
                    self.stride_u, self.stride_v, self.stride_c, self.row0, self.gh)


def resolve_devices(device):
    """-> (compute cuda device, device results are returned on).  Raises when no GPU is visible."""
    out = torch.device(device) if not isinstance(device, torch.device) else device
    if not torch.cuda.is_available():
        raise RuntimeError("smokephysai_b200 needs a CUDA device (B200, sm_100a): the smoke step has no CPU fallback")
    if out.type == "cuda":
        idx = out.index if out.index is not None else torch.cuda.current_device()
        return torch.device("cuda", idx), torch.device("cuda", idx)
    return torch.device("cuda", torch.cuda.current_device()), out


class NavierStokesSimulator(nn.Module):
    """Simplified Navier-Stokes smoke solver (reference: navier_stokes.py:6)."""

    def __init__(self, grid_size=(128, 128), dt=0.01, viscosity=0.001, device="cuda", *,
                 jacobi_iters=20, batch=1, sweeps_per_launch=0, step_kernel="auto", _slab=None):
        super().__init__()
        self.grid_size = grid_size
        self.dt = dt
        self.viscosity = viscosity
        self.device = device
        self.h, self.w = grid_size
        self.jacobi_iters = int(jacobi_iters)
        self.batch = int(batch)
        self.sweeps_per_launch = int(sweeps_per_launch)
        if step_kernel not in _lib.STEP_KERNELS:
            raise ValueError("step_kernel must be one of %s, got %r" % (sorted(_lib.STEP_KERNELS), step_kernel))
        self.step_kernel = step_kernel
        self._cuda, self._out_device = resolve_devices(device)
        self._lib = _lib.load()
        row0, gh = _slab if _slab is not None else (0, 0)   # (global row of local row 0, global rows): slab.py
        self._layout = FieldLayout(self.h, self.w, self.batch, row0, gh)
        self._grid = self._layout.grid_struct()
        self._arena = None
        self._state = State()
        self._mirrors = {}
        # Deferred reset (see setup_grid): _pending is None, or the [(sources, offsets)] splats issued since a reset that is not
        # applied yet; _stale: a run that consumed a reset left the non-live copies, div and boundary as they were before it.
        self._pending = None
        self._stale = False
        # Continuous sources (set_continuous_sources): None, or (per-simulation lists, device records, device offsets), uploaded once
        # and splatted at the head of every step by the kernels.
        self._csrc = None
        self.setup_grid()

    # ------------------------------------------------------------------ state (navier_stokes.py:24-35)
    def setup_grid(self):
        """Reset u, v, p, density (and the unused boundary mask) to zero; drops the pressure warm start.

        On an existing state the reset is deferred: the next step()/run_steps that runs on the fused kernel builds the zero
        state (plus the density of a splat issued in between) on chip instead of reading it back from memory; anything else
        that reads or launches on the state applies the reset first.  What a caller can observe is the same either way."""
        L = self._layout
        if self._arena is None:
            self._arena = torch.zeros(L.total, dtype=torch.float32, device=self._cuda)
            base = self._arena.data_ptr()
            st = self._state
            for k, (a, b) in {"u": ("u0", "u1"), "v": ("v0", "v1"), "d": ("d0", "d1"), "p": ("p0", "p1")}.items():
                arr = getattr(st, k)
                arr[0] = base + 4 * L.offset[a]
                arr[1] = base + 4 * L.offset[b]
            st.div = base + 4 * L.offset["div"]
        else:
            self._mirrors.clear()
            if L.gh == 0:
                self._pending = []
            else:
                self._arena.zero_()                     # slabs are stepped phase by phase: never on the fused kernel
        self._state.cur_u = self._state.cur_v = self._state.cur_d = self._state.cur_p = 0

    def _materialize(self):
        """Apply a deferred reset and its splats (the eager memset + k_splat), or zero what a consumed reset left stale."""
        pending, self._pending = self._pending, None
        if pending is not None:
            self._arena.zero_()
            self._stale = False
            for src, off in pending:
                _lib.call("smk_splat_sources", C.byref(self._grid), self._ptr("d"), src.data_ptr(), off.data_ptr(),
                          _lib.stream_on(self._cuda))
        elif self._stale:
            L = self._layout
            for name in ("u1", "v1", "d1", "p1", "div", "boundary"):
                off = L.offset[name]
                self._arena[off: off + L.batch * L.stride_of(name)].zero_()
            self._stale = False

    def _field(self, name):
        """Strided view [batch, rows, cols] (or [rows, cols] when batch == 1) of a field in the arena."""
        self._materialize()
        L = self._layout
        rows, cols, pitch = L.shape_of(name)
        off = L.offset[name]
        v = self._arena[off: off + L.batch * rows * pitch].view(L.batch, rows, pitch)[:, :, :cols]
        return v[0] if L.batch == 1 else v

    def _live(self, k):
        cur = getattr(self._state, "cur_" + k)
        return self._field("%s%d" % (k, cur))

    def _get(self, k):
        v = self._live(k)
        if self._out_device.type == "cuda":
            return v
        # device='cpu' (benchmark.py:260): the caller gets a host copy.  The reference hands out its LIVE tensor, so
        # in-place edits (`sim.density[mask] += x`) must not be lost: remember the copy with its version counter and
        # write it back before the next launch if it was modified (_flush_mirrors).
        self._flush_mirrors()               # an earlier copy of this field may carry edits that are not on the device yet
        t = self._live(k).to(self._out_device)
        self._mirrors[k] = (t, t._version)
        return t

    def _flush_mirrors(self):
        """Write host copies that were edited in place since they were handed out back to the device state."""
        if not self._mirrors:
            return
        for k, (t, ver) in self._mirrors.items():
            if t._version != ver:
                self._live(k).copy_(t)
        self._mirrors.clear()

    def _set(self, k, value):
        mirror = self._mirrors.get(k)
        if mirror is not None and value is mirror[0]:        # `sim.density *= c` on the host copy re-assigns it
            self._mirrors.pop(k)
            self._live(k).copy_(value)
            return
        self._mirrors.pop(k, None)
        dst = self._live(k)
        if not torch.is_tensor(value):
            value = torch.as_tensor(value, dtype=torch.float32)
        if value.device == dst.device and value.data_ptr() == dst.data_ptr() and value.stride() == dst.stride():
            return                                      # `sim.density *= c` re-assigns the view to itself
        if tuple(value.shape) != tuple(dst.shape):
            raise ValueError("cannot assign a tensor of shape %s to a field of shape %s" % (tuple(value.shape), tuple(dst.shape)))
        dst.copy_(value)

    u = property(lambda self: self._get("u"), lambda self, t: self._set("u", t), doc="x-velocity, [h+1, w]")
    v = property(lambda self: self._get("v"), lambda self, t: self._set("v", t), doc="y-velocity, [h, w+1]")
    p = property(lambda self: self._get("p"), lambda self, t: self._set("p", t), doc="pressure, [h, w]")
    density = property(lambda self: self._get("d"), lambda self, t: self._set("d", t), doc="smoke density, [h, w]")

    @property
    def boundary(self):
        b = self._field("boundary")
        return b if self._out_device.type == "cuda" else b.to(self._out_device)

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        """The stream to launch on.  Also the one place every launch passes through: host copies edited in place are
        written back here, and the library's (statically linked) CUDA runtime is pointed at this simulator's device."""
        self._materialize()
        self._flush_mirrors()
        return _lib.stream_on(self._cuda)

    def _params(self):
        dt, nu = float(self.dt), float(self.viscosity)
        # c = float32(dt*viscosity): the Python-double product of navier_stokes.py:72; density uses viscosity*0.1 (:160)
        return Params(dt, dt * nu, dt * (nu * 0.1), 0.995, int(self.jacobi_iters), int(self.sweeps_per_launch),
                      _lib.STEP_KERNELS[self.step_kernel])

    def step_is_fused(self, nsteps=1):
        """True when a call of nsteps steps (step(): 1, run_steps(n): n) takes the single-launch on-chip path."""
        flag = C.c_int32(0)
        prm = self._params()
        _lib.call("smk_step_is_fused", C.byref(self._grid), C.byref(prm), int(nsteps), C.byref(flag))
        return bool(flag.value)

    def _to_out(self, t):
        return t if self._out_device.type == "cuda" else t.to(self._out_device)

    def _stage(self, t):
        """Any [.., rows, cols] tensor -> zero-padded contiguous cuda fp32 [B, rows, pitch]; returns (buf, B, rows, cols, pitch)."""
        t = torch.as_tensor(t)
        if t.dim() == 2:
            t = t.unsqueeze(0)
        if t.dim() != 3:
            raise ValueError("expected a 2-D field (or a [batch, rows, cols] stack), got shape %s" % (tuple(t.shape),))
        B, rows, cols = t.shape
        pitch = _round4(cols)
        buf = torch.zeros(B, rows, pitch, dtype=torch.float32, device=self._cuda)
        buf[:, :, :cols] = t.to(device=self._cuda, dtype=torch.float32)
        return buf, B, rows, cols, pitch

    def _unstage(self, buf, cols, like):
        out = buf[:, :, :cols]
        if torch.as_tensor(like).dim() == 2:
            out = out[0]
        return self._to_out(out.contiguous())

    # ------------------------------------------------------------------ a2 (navier_stokes.py:37-48)
    def add_smoke_source(self, x, y, radius=10, intensity=1.0, *, batch_index=None):
        """Add a Gaussian smoke source centred on column x, row y (to every simulation unless batch_index is given)."""
        targets = range(self.batch) if batch_index is None else [int(batch_index)]
        per_sim = [[] for _ in range(self.batch)]
        for b in targets:
            per_sim[b].append((int(x), int(y), int(radius), float(intensity)))
        self.add_sources(per_sim)

    def upload_sources(self, per_sim, pin=False):
        """Pack per-simulation emitter lists into (sources, offsets) device tensors for splat_uploaded().

        per_sim[b] is the ordered list [(x, y, radius, intensity), ...] of simulation b.  The records travel
        as one H2D copy of 16 B per emitter plus 4 B per simulation."""
        if len(per_sim) != self.batch:
            raise ValueError("need one emitter list per simulation (%d), got %d" % (self.batch, len(per_sim)))
        rec, offs = pack_sources(per_sim)
        src_h = torch.from_numpy(rec.view(np.uint8))
        off_h = torch.from_numpy(offs)
        if pin:
            # one cached pinned staging buffer (cudaHostAlloc per call costs more than the copy); the previous
            # call's H2D copy has long been consumed by the splat that followed it on the same stream
            need = src_h.numel() + 4 * off_h.numel()
            stage = self._pinned_stage("_pinned_sources", need)
            stage[:src_h.numel()].copy_(src_h)
            stage[src_h.numel():need].view(torch.int32).copy_(off_h)
            dev = stage[:need].to(self._cuda, non_blocking=True)
            return dev[:src_h.numel()], dev[src_h.numel():need].view(torch.int32), need
        return src_h.to(self._cuda), off_h.to(self._cuda), src_h.numel() + 4 * off_h.numel()

    def _pinned_stage(self, attr, need):
        """The cached pinned staging buffer `attr`, of at least `need` bytes (cudaHostAlloc per call costs more than the copy);
        the previous call's H2D copy has long been consumed by the launch that followed it on the same stream."""
        stage = getattr(self, attr, None)
        if stage is None or stage.numel() < need:
            stage = torch.empty(max(need, 4096), dtype=torch.uint8).pin_memory()
            setattr(self, attr, stage)
        else:
            torch.cuda.current_stream(self._cuda).synchronize()
        return stage

    def upload_schedule(self, schedule, nsteps, pin=False):
        """Pack a source schedule (pack_schedule) and put it on this simulator's device: (int32 records [T * B * E, 4], int32
        offsets [T * B + 1]), or None when it has no entries (E == 0).  Host inputs travel as one H2D copy of 16 B per entry,
        through pinned memory when pin; the offsets are built on the device."""
        rec, E = pack_schedule(schedule, nsteps, self.batch)
        if rec is None:
            return None
        if rec.device.type == "cpu":
            if pin:
                stage = self._pinned_stage("_pinned_schedule", rec.numel() * 4)
                stage[:rec.numel() * 4].view(torch.int32).view(rec.shape).copy_(rec)
                rec = stage[:rec.numel() * 4].to(self._cuda, non_blocking=True).view(torch.int32).view(rec.shape)
            else:
                rec = rec.to(self._cuda)
        elif rec.device != self._cuda:
            raise ValueError("the schedule is on %s; this simulator runs on %s" % (rec.device, self._cuda))
        return rec, schedule_offsets(int(nsteps), self.batch, E, self._cuda)

    def splat_uploaded(self, src, off):
        if self._pending == []:                         # right after a reset: the fused launch that consumes it splats
            self._pending.append((src, off))
            return
        _lib.call("smk_splat_sources", C.byref(self._grid), self._ptr("d"), src.data_ptr(), off.data_ptr(), self._stream())

    def set_continuous_sources(self, per_sim):
        """Emitters that keep injecting: per_sim[b] = [(x, y, radius, intensity), ...] is added to simulation b's density at the
        head of every later step (step, step_into, run_steps, run_steps_time_major), before the buoyancy, in list order -- the
        same cells and weights as add_smoke_source.  run_steps(n) then equals n rounds of add_sources(per_sim); step() bit for
        bit, on one launch per call.  A frame is the density after its step (before the next step's splat); the state a call
        leaves carries no trailing splat.  None clears the list.  The records are uploaded once, here; setup_grid() keeps them.
        The reference's per-phase methods (diffusion_step, advection_step, pressure_projection, ...) do not apply them."""
        if per_sim is None:
            self._csrc = None
            return
        lists = check_source_lists(per_sim, self.batch)
        if not any(lists):
            self._csrc = None
            return
        src, off, _ = self.upload_sources(lists)
        self._csrc = (lists, src, off)

    @property
    def continuous_sources(self):
        """The per-simulation lists of set_continuous_sources (a copy), or None when no simulation has one."""
        return None if self._csrc is None else [list(l) for l in self._csrc[0]]

    def add_sources(self, per_sim):
        """Batched splat: per_sim[b] is the ordered emitter list [(x, y, radius, intensity), ...] of simulation b."""
        if not any(len(l) for l in per_sim):
            if len(per_sim) != self.batch:
                raise ValueError("need one emitter list per simulation (%d), got %d" % (self.batch, len(per_sim)))
            return
        src, off, _ = self.upload_sources(per_sim)
        self.splat_uploaded(src, off)

    # ------------------------------------------------------------------ a4 (navier_stokes.py:50-72)
    def diffusion_step(self, field, viscosity):
        buf, B, rows, cols, pitch = self._stage(field)
        out = torch.zeros_like(buf)
        _lib.call("smk_diffuse", buf.data_ptr(), out.data_ptr(), rows, cols, pitch, B, rows * pitch,
                  float(self.dt) * float(viscosity), self._stream())
        return self._unstage(out, cols, field)

    # ------------------------------------------------------------------ a10 (navier_stokes.py:74-95)
    def advection_step(self, field, u, v):
        fb, B, rows, cols, pitch = self._stage(field)
        ub, Bu, hu, wu, pu = self._stage(u)
        vb, Bv, hv, wv, pv = self._stage(v)
        if Bu != B or Bv != B:
            raise ValueError("field, u and v must have the same batch size")
        # the staggered pair defines the cell grid: u [h+1, w], v [h, w+1] (navier_stokes.py:27-28).  The reference clamps
        # to whatever shapes it is given; the kernels index u and v by that grid, so anything else is refused, not guessed.
        if hu != hv + 1 or wv != wu + 1:
            raise ValueError("advection_step needs u of shape [h+1, w] and v of shape [h, w+1]; got u %s, v %s"
                             % ((hu, wu), (hv, wv)))
        if rows > hv + 1 or cols > wu + 1:
            raise ValueError("advection_step: a %d x %d field does not fit the %d x %d cell grid of u, v" % (rows, cols, hv, wu))
        g = Grid(hv, wu, B, pu, pv, _round4(wu), hu * pu, hv * pv, hv * _round4(wu))
        out = torch.zeros_like(fb)
        _lib.call("smk_advect", C.byref(g), fb.data_ptr(), out.data_ptr(), rows, cols, pitch, rows * pitch,
                  ub.data_ptr(), vb.data_ptr(), float(self.dt), 1.0, None, 0, None, self._stream())
        return self._unstage(out, cols, field)

    # ------------------------------------------------------------------ a8, a9 (navier_stokes.py:97-131)
    def _bilerp(self, field, y, x, mode):
        fb, B, rows, cols, pitch = self._stage(field)
        if B != 1:
            raise ValueError("bilinear_interpolate takes one 2-D field")
        y = torch.as_tensor(y)
        x = torch.as_tensor(x)
        shape = torch.broadcast_shapes(y.shape, x.shape)
        yc = y.to(device=self._cuda, dtype=torch.float32).expand(shape).contiguous()
        xc = x.to(device=self._cuda, dtype=torch.float32).expand(shape).contiguous()
        out = torch.empty(shape, dtype=torch.float32, device=self._cuda)
        _lib.call("smk_bilerp", fb.data_ptr(), rows, cols, pitch, yc.data_ptr(), xc.data_ptr(), out.data_ptr(),
                  out.numel(), mode, self._stream())
        return self._to_out(out)

    def interpolate_velocity_u(self, u, y, x):
        return self._bilerp(u, y, x, 1)

    def interpolate_velocity_v(self, v, y, x):
        return self._bilerp(v, y, x, 2)

    def bilinear_interpolate(self, field, y, x):
        return self._bilerp(field, y, x, 0)

    # ------------------------------------------------------------------ a5-a7 (navier_stokes.py:133-149)
    def _ptr(self, k, cur=None):
        cur = getattr(self._state, "cur_" + k) if cur is None else cur
        return getattr(self._state, k)[cur]

    def pressure_projection(self):
        """Divergence, jacobi_iters Jacobi sweeps (warm-started p, zero ring), gradient subtract -- in place."""
        st, s, g = self._state, self._stream(), C.byref(self._grid)
        _lib.call("smk_divergence", g, self._ptr("u"), self._ptr("v"), st.div, float(self.dt), s)
        flag = C.c_int32(0)
        _lib.call("smk_jacobi", g, st.div, self._ptr("p"), self._ptr("p", st.cur_p ^ 1), int(self.jacobi_iters),
                  int(self.sweeps_per_launch), C.byref(flag), s)
        st.cur_p ^= flag.value
        _lib.call("smk_project", g, self._ptr("p"), self._ptr("u"), self._ptr("v"), float(self.dt), s)

    # ------------------------------------------------------------------ a3-a11 (navier_stokes.py:151-173)
    def _new_frames(self, nsteps=None, dtype=torch.float32):
        L = self._layout
        shape = (L.batch, L.h, L.pitch_c) if nsteps is None else (L.batch, nsteps, L.h, L.pitch_c)
        return torch.empty(shape, dtype=dtype, device=self._cuda)

    def _check_frame_buffer(self, name, t, shape):
        """A caller-owned frame buffer: contiguous, `shape`, on this simulator's device, fp32 / fp16 / bf16 -> SMK_FRAME_*."""
        if (tuple(t.shape) != shape or not t.is_contiguous() or t.dtype not in _lib.FRAME_FORMATS or t.device != self._cuda):
            raise ValueError("%s must be a contiguous float32, float16 or bfloat16 %s tensor on %s"
                             % (name, list(shape), self._cuda))
        return _lib.frame_format(t.dtype)

    def _finish_frames(self, fr):
        L = self._layout
        if L.pitch_c != L.w:
            fr = fr[..., :L.w].contiguous()
        if L.batch == 1:
            fr = fr[0]
        return self._to_out(fr)

    def _offer_reset(self):
        """The pending reset to hand to the next step call, as (reset sources, offsets) device pointers, or None: a reset with
        at most one splat can be built on chip; anything else is applied eagerly by _materialize."""
        if self._pending is None or len(self._pending) > 1:
            return None
        return tuple(t.data_ptr() for t in self._pending[0]) if self._pending else (None, None)

    def _steps(self, nsteps, frames, step_stride, batch_stride, fmul, fmt, sched=None):
        """nsteps steps of the state, frames (a device pointer or None) at the given strides in elements of frame format fmt.

        One smk_run_steps_sched_ex call, with the continuous sources if any (offsets step stride 0) or the schedule `sched`:
        (device records, device offsets, t0), this call's step t reading the schedule's row t0 + t (offsets step stride batch).
        A pending reset is offered to it first (reset = 1, on the current stream without materializing anything); when the call
        does not consume it (not on k_step_fused), nothing was enqueued, and the reset is applied eagerly before the call is made
        again without it."""
        if nsteps == 0:
            return                                      # (a negative count goes on to the library, which refuses it)
        if sched is not None:
            src, off, stride = sched[0].data_ptr(), sched[1].data_ptr() + 4 * sched[2] * self.batch, self.batch
        elif self._csrc is not None:
            src, off, stride = self._csrc[1].data_ptr(), self._csrc[2].data_ptr(), 0
        else:
            src, off, stride = None, None, 0
        fm = fmul.data_ptr() if fmul is not None else None
        done = C.c_int32(0)
        offer = self._offer_reset()
        for reset in ((True, False) if offer is not None else (False,)):
            rsrc, roff = offer if reset else (None, None)
            _lib.call("smk_run_steps_sched_ex", C.byref(self._grid), C.byref(self._state), C.byref(self._params()), int(nsteps),
                      frames, step_stride, batch_stride, fm, fmt, src, off, stride, int(reset), rsrc, roff, C.byref(done),
                      _lib.stream_on(self._cuda) if reset else self._stream())
            if done.value:
                self._pending = None
                self._stale = True
                return

    def step(self, fmul=None, *, frame_dtype=torch.float32):
        """One time step; returns a copy of the new density ([h, w], or [batch, h, w]).

        fmul (optional, [h, pitch_c] device tensor) fuses the fractal multiply of SmokeSimulator.simulate_step
        into the returned copy: frame = d + fmul*d (fractal_generator.py:62); solver state is not perturbed.
        frame_dtype torch.float16 / torch.bfloat16 returns that copy rounded once (to nearest even) by the kernel that
        writes it, equal to the fp32 copy's .to(frame_dtype); the state is the same whatever the dtype.
        """
        fmt = _lib.frame_format(frame_dtype)
        fr = self._new_frames(dtype=frame_dtype)
        self._steps(1, fr.data_ptr(), 0, self._layout.h * self._layout.pitch_c, fmul, fmt)
        return self._finish_frames(fr)

    def step_into(self, frame, fmul=None):
        """One time step whose returned copy is written into `frame`, a contiguous [batch, h, pitch_c] float32, float16
        or bfloat16 device tensor owned by the caller (no allocation, no sync)."""
        L = self._layout
        fmt = self._check_frame_buffer("frame", frame, (L.batch, L.h, L.pitch_c))
        self._steps(1, frame.data_ptr(), 0, L.h * L.pitch_c, fmul, fmt)

    def _schedule(self, schedule, nsteps):
        """_steps' schedule argument for a run_steps* schedule, None for none; ValueError before any work."""
        if schedule is None:
            return None
        if self._csrc is not None:
            raise ValueError("a source schedule and continuous sources do not combine: fold the constant emitters into the "
                             "schedule (or set_continuous_sources(None))")
        up = self.upload_schedule(schedule, nsteps)
        return None if up is None else up + (0,)

    def run_steps(self, nsteps, fmul=None, return_frames=True, out=None, *, frame_dtype=None, schedule=None):
        """nsteps consecutive steps enqueued back to back; returns frames [batch, nsteps, h, w] ([nsteps, h, w] if batch == 1).

        out: optional preallocated [batch, nsteps, h, pitch_c] device buffer to write the frames into (float32, float16 or
        bfloat16).  frame_dtype: the frames' dtype (default float32; with `out`, out.dtype, and a different frame_dtype is
        an error); half-precision frames are the fp32 ones rounded once to nearest even, as in step().

        schedule = (xy, radius, intensity): emitters that move or change intensity from step to step (pack_schedule gives the
        format; T = nsteps, B = batch).  Row t is added to the density at the head of step t, before the buoyancy, exactly as
        add_sources of that row followed by step() would add it -- bit for bit, frames and state, in one launch on the fused
        and cluster kernels.  Frame t is the density after step t; the state left carries no trailing splat.  A schedule does
        not combine with continuous sources (ValueError)."""
        return self._run_steps(nsteps, fmul, return_frames, out, frame_dtype, self._schedule(schedule, nsteps))

    def _run_steps(self, nsteps, fmul, return_frames, out, frame_dtype, sched):
        L = self._layout
        if out is not None:
            fmt = self._check_frame_buffer("out", out, (L.batch, nsteps, L.h, L.pitch_c))
            if frame_dtype is not None and frame_dtype != out.dtype:
                raise ValueError("frame_dtype %s disagrees with out.dtype %s" % (frame_dtype, out.dtype))
            fr = out
        else:
            frame_dtype = torch.float32 if frame_dtype is None else frame_dtype
            fmt = _lib.frame_format(frame_dtype)
            fr = self._new_frames(nsteps, frame_dtype) if return_frames else None
        self._steps(nsteps, fr.data_ptr() if fr is not None else None, L.h * L.pitch_c, nsteps * L.h * L.pitch_c, fmul, fmt,
                    sched)
        return self._finish_frames(fr) if fr is not None else None

    def run_steps_time_major(self, nsteps, out, fmul=None, *, schedule=None):
        """nsteps consecutive steps whose frames go to `out`, a contiguous [nsteps, batch, h, pitch_c] float32, float16 or
        bfloat16 device buffer owned by the caller (time-major: the frames of one step are one contiguous block).
        schedule: as run_steps."""
        self._run_steps_time_major(nsteps, out, fmul, self._schedule(schedule, nsteps))

    def _run_steps_time_major(self, nsteps, out, fmul, sched):
        L = self._layout
        fmt = self._check_frame_buffer("out", out, (nsteps, L.batch, L.h, L.pitch_c))
        self._steps(nsteps, out.data_ptr(), L.batch * L.h * L.pitch_c, L.h * L.pitch_c, fmul, fmt, sched)

    def divergence_norms(self):
        """(max|div|, ||div||_2) of the un-normalised divergence of the live (u, v), per simulation: [batch, 2] on the host."""
        out = torch.zeros(self.batch, 2, dtype=torch.float32, device=self._cuda)
        _lib.call("smk_div_norms", C.byref(self._grid), self._ptr("u"), self._ptr("v"), out.data_ptr(), self._stream())
        out = out.cpu().double()
        out[:, 1] = out[:, 1].sqrt()
        return out

    def jacobi_residual_norms(self):
        """(max|p' - p|, ||p' - p||_2) per simulation, p' = one more Jacobi sweep (navier_stokes.py:139-145) over the live
        pressure and the divergence of the last projection: [batch, 2] on the host.  Meaningful right after
        pressure_projection() or a step() of the phase-per-kernel path (the fused kernel keeps the divergence in registers)."""
        out = torch.zeros(self.batch, 2, dtype=torch.float32, device=self._cuda)
        _lib.call("smk_jacobi_residual", C.byref(self._grid), self._state.div, self._ptr("p"), out.data_ptr(), self._stream())
        out = out.cpu().double()
        out[:, 1] = out[:, 1].sqrt()
        return out

    def forward(self):
        return self.step()


# every method that launches runs with the simulator's device current and restores the caller's afterwards
for _name in ("setup_grid", "_materialize", "add_sources", "set_continuous_sources", "splat_uploaded", "upload_sources",
              "upload_schedule", "diffusion_step", "advection_step", "_bilerp",
              "pressure_projection", "step", "step_into", "run_steps", "_run_steps", "run_steps_time_major", "_run_steps_time_major",
              "divergence_norms",
              "jacobi_residual_norms", "step_is_fused"):
    setattr(NavierStokesSimulator, _name, _lib.scoped(getattr(NavierStokesSimulator, _name)))
del _name
