"""Differentiable rollouts: reverse-mode gradients through the smoke step (navier_stokes.py:151-173) on sm_100a adjoint kernels.

    frames, (u, v, p, d) = autodiff.rollout((u0, v0, p0, d0), nsteps, dt=0.01, viscosity=0.001, jacobi_iters=20)
    d0 = autodiff.add_sources(d0, emitters, intensities)       # emitters[b] = [(x, y, radius), ...]
    frames, state = autodiff.rollout(state, nsteps, sources=emitters, intensities=intensities)   # emitters at every step
    frames, state = autodiff.rollout(state, nsteps, schedule=(xy, radius), intensities=I)       # an emission history, I [T, B, E]

The reference simulator is eager PyTorch, so autograd runs through it: a user can fit emitter intensities to observed frames,
optimise an initial state or train a model through the simulator.  This module gives the same capability on the CUDA path.

Forward: the simulator's own step (phase or fused kernels), one step at a time; after each step the state
S_t = (u, v, p, d) is copied into a [T+1, ...] checkpoint buffer, four plain device copies per step.  Frames and final state are
bit-identical to NavierStokesSimulator.run_steps.  Checkpoint memory, in bytes:

    4 * (T + 1) * B * ((h + 1) * pitch_u + h * pitch_v + 2 * h * pitch_c),    pitch_* = row length rounded up to 4

Backward, step t from T-1 down to 0: recompute the diffused fields and the projected velocities from S_t with the forward's own
bit-exact phase entries (smk_forces_diffuse_div, smk_project with p = S_{t+1}.p, which is the pressure the step projected with),
then apply the adjoint entries of csrc/adjoint.cu in reverse phase order (DESIGN.md "Reverse mode").  Torch only allocates, zeroes
and copies here; every gradient is computed by a CUDA kernel.  Gradients are deterministic (bitwise repeatable).

With grad disabled, or when no input requires grad, rollout is run_steps: no checkpoints, no extra copies.

Continuous sources (rollout(..., sources=, intensities=)): the emitters are added to the density at the head of every step, as
NavierStokesSimulator.set_continuous_sources does, and the forward is that call's run_steps bit for bit.  Checkpoints stay the
pre-splat states S_t; the backward re-applies the splat to a copy of S_t.d before the recompute.  The splat is an add, so the
gradient of the splatted density passes unchanged to S_t.d, and the intensity gradient is the sum over steps, t = T-1 down to 0
in that order, of the splat adjoint of that gradient (smk_splat_sources_adjoint_ex, accumulating): deterministic, no atomics.

Source schedules (rollout(..., schedule=(xy, radius), intensities=I)): row t of the schedule is added at the head of step t, as
NavierStokesSimulator.run_steps(schedule=) does, and the forward is that call bit for bit.  The backward splats a copy of S_t.d with
row t, and the gradient of step t's intensities is the splat adjoint of that step alone (smk_splat_sources_adjoint_ex on row t's
records, not accumulating), so I.grad[t] is exactly that of step t and padded entries (radius < 0) get exactly 0.
"""
import ctypes as C

import torch

from . import _lib
from .fractal_generator import FractalGenerator
from .navier_stokes import FieldLayout, NavierStokesSimulator, pack_schedule, schedule_offsets

__all__ = ["rollout", "add_sources"]

_FIELDS = ("u", "v", "p", "d")


def _check_state(state):
    """-> (batch or None for 2-D inputs, h, w, device).  ValueError for anything rollout cannot take."""
    if not isinstance(state, (tuple, list)) or len(state) != 4:
        raise ValueError("state must be a tuple (u, v, p, d)")
    for name, t in zip(_FIELDS, state):
        if not torch.is_tensor(t):
            raise ValueError("%s must be a torch.Tensor, got %r" % (name, type(t)))
        if t.dtype != torch.float32:
            raise ValueError("%s must be float32, got %s" % (name, t.dtype))
        if t.device.type != "cuda":
            raise ValueError("%s must be a CUDA tensor, got one on %s" % (name, t.device))
        if t.dim() not in (2, 3):
            raise ValueError("%s must be [rows, cols] or [batch, rows, cols], got shape %s" % (name, tuple(t.shape)))
    u, v, p, d = state
    if len({t.device for t in state}) != 1:
        raise ValueError("u, v, p and d must be on one device, got %s" % sorted({str(t.device) for t in state}))
    if len({t.dim() for t in state}) != 1:
        raise ValueError("u, v, p and d must all be 2-D or all be 3-D")
    h, w = d.shape[-2:]
    want = {"u": (h + 1, w), "v": (h, w + 1), "p": (h, w), "d": (h, w)}
    for name, t in zip(_FIELDS, state):
        if tuple(t.shape[-2:]) != want[name]:
            raise ValueError("inconsistent shapes: with d of %d x %d, %s must be %s, got %s"
                             % (h, w, name, want[name], tuple(t.shape[-2:])))
    batch = None
    if d.dim() == 3:
        if len({t.shape[0] for t in state}) != 1:
            raise ValueError("u, v, p and d must have the same batch size, got %s" % [t.shape[0] for t in state])
        batch = int(d.shape[0])
    if h < 1 or w < 1 or (batch is not None and batch < 1):
        raise ValueError("empty grid or batch")
    return batch, int(h), int(w), d.device


def _staged(layout, name, t, out=None):
    """[.., rows, cols] -> zero-padded [B, rows, pitch] in the simulator's FieldLayout (a copy)."""
    rows, cols, pitch = layout.shape_of(name)
    if out is None:
        out = torch.zeros(layout.batch, rows, pitch, dtype=torch.float32, device=t.device)
    out[:, :, :cols] = t.reshape(layout.batch, rows, cols)
    return out


class _Config:
    def __init__(self, batch, h, w, device, nsteps, dt, viscosity, jacobi_iters, add_fractal, step_kernel, sweeps_per_launch):
        self.batch, self.h, self.w, self.device = batch, h, w, device
        self.nsteps = int(nsteps)
        self.dt, self.viscosity, self.jacobi_iters = dt, viscosity, int(jacobi_iters)
        self.add_fractal, self.step_kernel, self.sweeps_per_launch = bool(add_fractal), step_kernel, int(sweeps_per_launch)
        self.B = 1 if batch is None else batch
        self.src = None                 # continuous sources: (int32 [n, 4] device records with the intensities, offsets, n)
        self.sched = None               # schedule: (int32 [T * B * E, 4] device records with the intensities, offsets [T * B + 1], E)

    def simulator(self, state):
        sim = NavierStokesSimulator((self.h, self.w), self.dt, self.viscosity, self.device, jacobi_iters=self.jacobi_iters,
                                    batch=self.B, sweeps_per_launch=self.sweeps_per_launch, step_kernel=self.step_kernel)
        for name, t in zip(_FIELDS, state):
            live = _arena_view(sim, name)
            rows, cols, _ = sim._layout.shape_of(_layout_name(name))
            live[:, :, :cols] = t.detach().reshape(self.B, rows, cols)
        if self.src is not None:
            sim._csrc = (None, self.src[0], self.src[1])          # set_continuous_sources with records already on the device
        return sim

    def step_sched(self, t0):
        """_steps' schedule argument for a call whose step 0 is step t0 of the rollout (None without a schedule)."""
        if self.sched is None:
            return None
        return self.sched[:2] + (t0,)

    def fmul(self):
        if not self.add_fractal:
            return None
        return FractalGenerator(self.device).multiplier((self.h, self.w), 0.05)      # smoke_simulator.py:38

    def shape_out(self, t):
        """[B, ...] -> the caller's shape ([...] for 2-D inputs)."""
        return t[0] if self.batch is None else t


def _layout_name(name):
    return {"u": "u0", "v": "v0", "p": "p0", "d": "d0"}[name]


def _arena_view(sim, name, cur=None):
    """The live copy of a field as a padded [B, rows, pitch] view of the simulator's arena."""
    L = sim._layout
    k = name
    cur = getattr(sim._state, "cur_" + k) if cur is None else cur
    off = L.offset["%s%d" % (k, cur)]
    rows, _, pitch = L.shape_of(_layout_name(name))
    return sim._arena[off: off + L.batch * rows * pitch].view(L.batch, rows, pitch)


def _first_order_only(what):
    """The adjoint kernels give first-order gradients: refuse a backward that would build a graph (create_graph=True, the
    first half of a double backward) instead of handing back gradients that silently carry no graph."""
    if torch.is_grad_enabled():
        raise RuntimeError("smokephysai_b200.autodiff.%s supports first-order gradients only: backward with create_graph=True "
                           "(double backward, higher-order gradients) is not supported" % what)


def _ptr(t):
    return t.data_ptr() if t is not None else None


class _Rollout(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cfg, u0, v0, p0, d0, intensities):
        with _lib.on_device(cfg.device):
            sim = cfg.simulator((u0, v0, p0, d0))
            L = sim._layout
            T = cfg.nsteps
            ck = {k: torch.empty((T + 1,) + tuple(_arena_view(sim, k).shape), dtype=torch.float32, device=cfg.device)
                  for k in _FIELDS}
            for k in _FIELDS:
                ck[k][0].copy_(_arena_view(sim, k))
            frames = torch.empty(L.batch, T, L.h, L.pitch_c, dtype=torch.float32, device=cfg.device)
            fmul = cfg.fmul()
            prm = sim._params()
            for t in range(T):
                sim._steps(1, frames.data_ptr() + 4 * t * L.h * L.pitch_c, 0, T * L.h * L.pitch_c, fmul, 0, cfg.step_sched(t))
                for k in _FIELDS:
                    ck[k][t + 1].copy_(_arena_view(sim, k))
            ctx.cfg, ctx.ck, ctx.fmul, ctx.layout, ctx.params = cfg, ck, fmul, L, prm
            out = [cfg.shape_out(frames[..., :L.w].contiguous())]
            for k in _FIELDS:
                rows, cols, _ = L.shape_of(_layout_name(k))
                out.append(cfg.shape_out(ck[k][T][:, :, :cols].clone()))
            return tuple(out)

    @staticmethod
    def backward(ctx, g_frames, g_u, g_v, g_p, g_d):
        _first_order_only("rollout")
        cfg, ck, L, prm = ctx.cfg, ctx.ck, ctx.layout, ctx.params
        with _lib.on_device(cfg.device):
            grads = _reverse(cfg, ck, L, prm, ctx.fmul, g_frames, {"u": g_u, "v": g_v, "p": g_p, "d": g_d})
        return (None,) + grads[:4] + (grads[4] if ctx.needs_input_grad[5] else None,)


def _reverse(cfg, ck, L, prm, fmul, g_frames, g_out):
    dev, T, B = cfg.device, cfg.nsteps, L.batch
    s = _lib.stream_on(dev)
    g = L.grid_struct()
    gp = C.byref(g)
    zeros = lambda k: torch.zeros_like(ck[k][0])
    G = {}
    for k in _FIELDS:
        G[k] = zeros(k)
        if g_out[k] is not None:
            _staged(L, _layout_name(k), g_out[k], G[k])
    gF = None
    if g_frames is not None:
        gF = torch.zeros(B, T, L.h, L.pitch_c, dtype=torch.float32, device=dev)
        gF[..., :L.w] = g_frames.reshape(B, T, L.h, L.w)
    Gn = {k: zeros(k) for k in _FIELDS}
    ud, vd, dd = zeros("u"), zeros("v"), zeros("d")          # recomputed u_diff -> u_proj, v_diff -> v_proj, d_diff
    gup, gvp, gdd, gpk, gdiv = zeros("u"), zeros("v"), zeros("d"), zeros("p"), zeros("p")
    ws_adv = torch.empty(16 + 32 * B * (L.h + 1) * (L.w + 1), dtype=torch.uint8, device=dev)
    ws_jac = torch.empty(5 * B * L.stride_c if cfg.jacobi_iters >= 1 else 4, dtype=torch.float32, device=dev)
    dt, c_uv, c_d = prm.dt, prm.c_uv, prm.c_d
    rows_u, rows_v, rows_c = L.h + 1, L.h, L.h
    g_int = None
    if cfg.src is not None:
        rec, off, n = cfg.src
        g_int = torch.zeros(n, dtype=torch.float32, device=dev)
        dsp = zeros("d")                                        # S_t.d with the step's splat, the density the step started from
    elif cfg.sched is not None:
        rec, off, E = cfg.sched
        g_int = torch.zeros(T, B, E, dtype=torch.float32, device=dev)
        row_off = schedule_offsets(1, B, E, dev)                # one row of B lists of E entries, for the per-step adjoint
        dsp = zeros("d")
    for t in range(T - 1, -1, -1):
        u0, v0, d0 = ck["u"][t], ck["v"][t], ck["d"][t]
        if g_int is not None:
            dsp.copy_(d0)
            _lib.call("smk_splat_sources", gp, dsp.data_ptr(), rec.data_ptr(), off.data_ptr() + (4 * t * B if cfg.sched else 0), s)
            d0 = dsp
        u1, v1, p1 = ck["u"][t + 1], ck["v"][t + 1], ck["p"][t + 1]
        # recompute: buoyancy + diffusions, then the gradient subtract with the pressure the step projected with
        _lib.call("smk_forces_diffuse_div", gp, u0.data_ptr(), v0.data_ptr(), d0.data_ptr(), ud.data_ptr(), vd.data_ptr(),
                  dd.data_ptr(), None, dt, c_uv, c_d, s)
        _lib.call("smk_project", gp, p1.data_ptr(), ud.data_ptr(), vd.data_ptr(), dt, s)
        gft = gF[:, t] if gF is not None else None
        # 1. density advection (+ decay, frame, fractal): field d_diff by (u_adv, v_adv) = (S_{t+1}.u, S_{t+1}.v)
        _lib.call("smk_advect_adjoint", gp, dd.data_ptr(), rows_c, L.w, L.pitch_c, L.stride_c, u1.data_ptr(), v1.data_ptr(),
                  dt, prm.decay, G["d"].data_ptr(), _ptr(gft), T * L.h * L.pitch_c, _ptr(fmul) if gft is not None else None,
                  gdd.data_ptr(), 0, G["u"].data_ptr(), G["v"].data_ptr(), ws_adv.data_ptr(), s)
        # 2. v advection: field v_proj by (u_adv, v_proj)
        _lib.call("smk_advect_adjoint", gp, vd.data_ptr(), rows_v, L.w + 1, L.pitch_v, L.stride_v, u1.data_ptr(), vd.data_ptr(),
                  dt, 1.0, G["v"].data_ptr(), None, 0, None, gvp.data_ptr(), 0, G["u"].data_ptr(), gvp.data_ptr(),
                  ws_adv.data_ptr(), s)
        # 3. u advection: field u_proj by (u_proj, v_proj); G.u is complete now
        _lib.call("smk_advect_adjoint", gp, ud.data_ptr(), rows_u, L.w, L.pitch_u, L.stride_u, ud.data_ptr(), vd.data_ptr(),
                  dt, 1.0, G["u"].data_ptr(), None, 0, None, gup.data_ptr(), 0, gup.data_ptr(), gvp.data_ptr(),
                  ws_adv.data_ptr(), s)
        # 4. gradient subtract, 5. Jacobi sweeps, 6. divergence + diffusions + buoyancy
        _lib.call("smk_project_adjoint", gp, gup.data_ptr(), gvp.data_ptr(), G["p"].data_ptr(), gpk.data_ptr(), dt, s)
        _lib.call("smk_jacobi_adjoint", gp, gpk.data_ptr(), Gn["p"].data_ptr(), gdiv.data_ptr(), cfg.jacobi_iters,
                  cfg.sweeps_per_launch, ws_jac.data_ptr(), s)
        _lib.call("smk_forces_diffuse_div_adjoint", gp, gup.data_ptr(), gvp.data_ptr(), gdd.data_ptr(), gdiv.data_ptr(),
                  Gn["u"].data_ptr(), Gn["v"].data_ptr(), Gn["d"].data_ptr(), dt, c_uv, c_d, s)
        G, Gn = Gn, G
        # G.d: the gradient of the splatted density, which is also that of S_t.d
        if cfg.src is not None:
            _lib.call("smk_splat_sources_adjoint_ex", gp, G["d"].data_ptr(), rec.data_ptr(), off.data_ptr(), n, 1, g_int.data_ptr(), s)
        elif cfg.sched is not None:
            _lib.call("smk_splat_sources_adjoint_ex", gp, G["d"].data_ptr(), rec.data_ptr() + 16 * t * B * E, row_off.data_ptr(),
                      B * E, 0, g_int[t].data_ptr(), s)
    out = []
    for k in _FIELDS:
        rows, cols, _ = L.shape_of(_layout_name(k))
        out.append(cfg.shape_out(G[k][:, :, :cols].contiguous()))
    return tuple(out) + (g_int,)


def rollout(state, nsteps, *, dt=0.01, viscosity=0.001, jacobi_iters=20, add_fractal=False, step_kernel="auto",
            sweeps_per_launch=0, sources=None, intensities=None, schedule=None):
    """nsteps steps of NavierStokesSimulator from state = (u, v, p, d); differentiable with respect to all four fields.

    u [.., h+1, w], v [.., h, w+1], p [.., h, w], d [.., h, w]: float32 CUDA tensors on one device, with an optional leading
    batch dimension.  Returns (frames, (u, v, p, d)): frames [B, T, h, w] ([T, h, w] for 2-D inputs) and the final state in
    the input shapes, bit-identical to NavierStokesSimulator.run_steps on the same state and parameters (any step_kernel).
    add_fractal multiplies the frames by 1 + 0.05*F as SmokeSimulator.simulate_step does (square grids only).  Gradients of
    outputs that are not used count as zero; higher-order gradients are not supported.

    sources / intensities: continuous emitters, added to the density at the head of every step (set_continuous_sources).
    sources[b] = [(x, y, radius), ...] for simulation b (for 2-D inputs one flat list is accepted too), intensities a 1-D float32
    tensor on the state's device with one value per emitter in flattened order; differentiable with respect to intensities.

    schedule = (xy, radius) / intensities: an emission history, row t added at the head of step t (run_steps(schedule=)).
    xy integer [T, B, E, 2], radius integer [T, B, E] (B = 1 for 2-D inputs; radius < 0 pads), intensities float32 [T, B, E]
    on the state's device, differentiable.  Exclusive with sources=."""
    batch, h, w, device = _check_state(state)
    if int(nsteps) < 1:
        raise ValueError("nsteps must be >= 1, got %r" % (nsteps,))
    if int(jacobi_iters) < 0:
        raise ValueError("jacobi_iters must be >= 0, got %r" % (jacobi_iters,))
    if step_kernel not in _lib.STEP_KERNELS:
        raise ValueError("step_kernel must be one of %s, got %r" % (sorted(_lib.STEP_KERNELS), step_kernel))
    cfg = _Config(batch, h, w, device, nsteps, dt, viscosity, jacobi_iters, add_fractal, step_kernel, sweeps_per_launch)
    if sources is not None and schedule is not None:
        raise ValueError("sources= and schedule= do not combine: fold the constant emitters into the schedule")
    if sources is None and schedule is None and intensities is not None:
        raise ValueError("intensities without sources or a schedule")
    if schedule is not None:
        cfg.sched = _schedule_records(schedule, intensities, cfg.nsteps, cfg.B, device)
    elif sources is not None:
        if intensities is None:
            raise ValueError("sources need intensities: a 1-D float32 tensor, one value per emitter")
        sources = _emitter_lists(sources, batch is None)
        rec, off, n = _source_records(sources, cfg.B, device)
        _check_intensities(intensities, n, device)
        if n:
            rec.view(torch.float32)[:n, 3].copy_(intensities.detach())           # smk_source_t.intensity
            cfg.src = (rec, off, n)
    differentiable = cfg.src is not None or cfg.sched is not None
    if torch.is_grad_enabled() and (any(t.requires_grad for t in state) or (differentiable and intensities.requires_grad)):
        frames, *final = _Rollout.apply(cfg, *state, intensities if differentiable else None)
        return frames, tuple(final)
    with _lib.on_device(device):
        sim = cfg.simulator(state)
        frames = sim._run_steps(cfg.nsteps, cfg.fmul(), True, None, None, cfg.step_sched(0))
        if batch is not None and cfg.B == 1:
            frames = frames.unsqueeze(0)
        final = []
        for k in _FIELDS:
            rows, cols, _ = sim._layout.shape_of(_layout_name(k))
            final.append(cfg.shape_out(_arena_view(sim, k)[:, :, :cols].clone()))
        return frames, tuple(final)


# ---------------------------------------------------------------------------------------------------------------- sources
def _source_records(emitters, batch, device):
    """emitters (per simulation lists of (x, y, radius)) -> (int32 [n, 4] device records, int32 [batch+1] offsets, n)."""
    if len(emitters) != batch:
        raise ValueError("need one emitter list per simulation (%d), got %d" % (batch, len(emitters)))
    flat, offs = [], [0]
    for lst in emitters:
        for e in lst:
            if not hasattr(e, "__len__") or len(e) != 3:
                raise ValueError("an emitter is (x, y, radius), got %r" % (e,))
            flat.append([int(e[0]), int(e[1]), int(e[2]), 0])
        offs.append(len(flat))
    rec = torch.tensor(flat if flat else [[0, 0, 0, 0]], dtype=torch.int32).to(device)
    return rec, torch.tensor(offs, dtype=torch.int32).to(device), len(flat)


def _schedule_records(schedule, intensities, T, B, device):
    """(xy, radius) and the intensities [T, B, E] -> (int32 [T * B * E, 4] device records with the intensities, offsets, E), or
    None for E == 0.  ValueError for anything pack_schedule refuses or intensities of another shape, dtype or device."""
    if not isinstance(schedule, (tuple, list)) or len(schedule) != 2:
        raise ValueError("rollout's schedule is (xy, radius); the intensities go in intensities=")
    if intensities is None:
        raise ValueError("a schedule needs intensities: a float32 [T, B, E] tensor")
    xy, radius = schedule
    shape = tuple(getattr(radius, "shape", ()))
    if not torch.is_tensor(intensities) or intensities.dtype != torch.float32 or intensities.device != device \
            or tuple(intensities.shape) != shape:
        raise ValueError("intensities must be a float32 tensor on %s shaped like radius %s" % (device, shape))
    rdev = radius.device if torch.is_tensor(radius) else torch.device("cpu")
    rec, E = pack_schedule((xy, radius, torch.zeros(shape, dtype=torch.float32, device=rdev)), T, B)
    if rec is None:
        return None
    rec = rec.to(device)
    rec[:, 3] = intensities.detach().reshape(-1).view(torch.int32)           # smk_source_t.intensity bits
    return rec, schedule_offsets(T, B, E, device), E


def _emitter_lists(emitters, two_d):
    """For a 2-D state or density, one flat list of (x, y, radius) stands for [that list]."""
    if two_d and len(emitters) and len(emitters[0]) and not isinstance(emitters[0][0], (list, tuple)):
        return [emitters]
    return emitters


def _check_intensities(intensities, n, device):
    if not torch.is_tensor(intensities) or intensities.dim() != 1 or intensities.dtype != torch.float32 \
            or intensities.device != device or intensities.numel() != n:
        raise ValueError("intensities must be a 1-D float32 tensor of %d values on %s" % (n, device))


class _AddSources(torch.autograd.Function):
    @staticmethod
    def forward(ctx, d0, rec, off, n, intensities, two_d):
        B, h, w = (1,) + tuple(d0.shape) if two_d else tuple(d0.shape)
        L = FieldLayout(h, w, B)
        dev = d0.device
        with _lib.on_device(dev):
            buf = _staged(L, "d0", d0.detach())
            rec = rec.clone()
            rec.view(torch.float32)[:n, 3].copy_(intensities.detach())          # smk_source_t.intensity
            g = L.grid_struct()
            if n:
                _lib.call("smk_splat_sources", C.byref(g), buf.data_ptr(), rec.data_ptr(), off.data_ptr(), _lib.stream_on(dev))
        ctx.layout, ctx.rec, ctx.off, ctx.n, ctx.two_d = L, rec, off, n, two_d
        out = buf[:, :, :w].contiguous()
        return out[0] if two_d else out

    @staticmethod
    def backward(ctx, g_d):
        _first_order_only("add_sources")
        L, n = ctx.layout, ctx.n
        g_int = None
        if ctx.needs_input_grad[4]:
            dev = g_d.device
            g_int = torch.zeros(n, dtype=torch.float32, device=dev)
            with _lib.on_device(dev):
                gbuf = _staged(L, "d0", g_d)
                g = L.grid_struct()
                _lib.call("smk_splat_sources_adjoint", C.byref(g), gbuf.data_ptr(), ctx.rec.data_ptr(), ctx.off.data_ptr(), n,
                          g_int.data_ptr(), _lib.stream_on(dev))
        return g_d, None, None, None, g_int, None


def add_sources(d0, emitters, intensities):
    """d0 plus Gaussian emitters (NavierStokesSimulator.add_smoke_source), differentiable with respect to d0 and intensities.

    d0: float32 CUDA density [h, w] or [B, h, w].  emitters[b] = [(x, y, radius), ...] for simulation b, applied in list order
    (for a 2-D d0, a single list of emitters is accepted too).  intensities: 1-D float32 tensor on d0's device, one per
    emitter, flattened in that order.  The result is bit-identical to add_smoke_source with the same intensities."""
    if not torch.is_tensor(d0) or d0.dtype != torch.float32 or d0.device.type != "cuda" or d0.dim() not in (2, 3):
        raise ValueError("d0 must be a float32 CUDA tensor [h, w] or [batch, h, w]")
    two_d = d0.dim() == 2
    emitters = _emitter_lists(emitters, two_d)
    batch = 1 if two_d else int(d0.shape[0])
    rec, off, n = _source_records(emitters, batch, d0.device)
    _check_intensities(intensities, n, d0.device)
    return _AddSources.apply(d0, rec, off, n, intensities, two_d)
