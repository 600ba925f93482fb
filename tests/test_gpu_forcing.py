"""Velocity forcing: per-step velocity increments added on chip by every step kernel.  Every case compares run_steps(forcing=F) with the
host loop [u += du[t]; v += dv[t]; step()] on the phase kernels, bit for bit on the frames and on u, v, p and density, on each kernel
that can run it: k_step_fused (FULL, one CTA per simulation and time-sliced with hand-overs; the generic instantiation on ragged
grids), k_step_cluster (clusters of 4 and 2 CTAs) and the phase path.  The forcing changes at every step and is strong enough that
dt * |u| exceeds a cell, so back-traces reach the far gathers of k_step_cluster and the global fallback of the tiled advection."""
import ctypes as C

import numpy as np
import pytest
import torch

from forcing_oracle import rollout as rollout_forced, wind
from helpers import emitters_for_sequence, nerr, smk_env
from schedule_oracle import moving_schedule, rows_as_lists

pytestmark = pytest.mark.gpu

DT, VISC = 0.01, 0.001
DEV = "cuda:0"
FIELDS = ("u", "v", "p", "density")


def N(t):
    return t.detach().float().cpu().numpy().copy()


def same(a, b, what):
    np.testing.assert_array_equal(np.asarray(a), np.asarray(b), err_msg=what)


def make(h, w, B, K, **kw):
    from smokephysai_b200 import NavierStokesSimulator
    return NavierStokesSimulator((h, w), DT, VISC, DEV, jacobi_iters=K, batch=B, **kw)


def forcing(T, B, h, w, per_step, seed, strength=150.0):
    du, dv = wind(T, B, h, w, seed=seed, strength=strength)
    return (du, dv) if per_step else (du[0], dv[0])


def host_loop(h, w, B, K, T, F, frame_dtype=torch.float32, init=None, fmul=None, sched=None, csrc=None):
    du, dv = (torch.from_numpy(a).to(DEV) for a in F)
    per_step = du.dim() == 4
    ns = make(h, w, B, K, step_kernel="phases")
    if csrc is not None:
        ns.set_continuous_sources(csrc)
    if init is not None:
        ns.add_sources(init)
    frames = []
    for t in range(T):
        if sched is not None:
            ns.add_sources(rows_as_lists(sched, t))
        a, b = (du[t], dv[t]) if per_step else (du, dv)
        ns.u += a.reshape(ns.u.shape)
        ns.v += b.reshape(ns.v.shape)
        frames.append(ns.step(fmul=fmul, frame_dtype=frame_dtype))
    return N(torch.stack(frames, dim=-3)), {k: N(getattr(ns, k)) for k in FIELDS}


def check(h, w, B, K, T, F, env=None, frame_dtype=torch.float32, fmul=None, as_tensors=None, sched=None, csrc=None, **kw):
    want_fr, want = host_loop(h, w, B, K, T, F, frame_dtype, fmul=fmul, sched=sched, csrc=csrc)
    G = F if as_tensors is None else tuple(torch.from_numpy(a).to(as_tensors) for a in F)
    with smk_env(**(env or {})):
        ns = make(h, w, B, K, **kw)
        if csrc is not None:
            ns.set_continuous_sources(csrc)
        fr = N(ns.run_steps(T, fmul=fmul, frame_dtype=frame_dtype, schedule=sched, forcing=G))
        got = {k: N(getattr(ns, k)) for k in FIELDS}
    same(fr, want_fr, "frames")
    for k in FIELDS:
        same(got[k], want[k], k)
    assert DT * max(np.abs(want["u"]).max(), np.abs(want["v"]).max()) > 1.0        # back-traces beyond a cell
    return ns


@pytest.mark.parametrize("per_step", [True, False])
def test_fused_full_one_cta_per_simulation(per_step):
    ns = check(128, 128, 40, 20, 6, forcing(6, 40, 128, 128, per_step, 1), env={"SMK_FUSED_SLICE": 0, "SMK_FUSED_CLUSTER": 0})
    assert ns.step_is_fused(6)


def test_fused_full_time_sliced_c2_size():
    """256 x 128^2, K = 40, 20 steps: the time-sliced schedule hands simulations from CTA to CTA, and an item that starts at
    t_begin > 0 must apply row t_begin.  One launch per call."""
    from smokephysai_b200 import _lib
    F = forcing(20, 256, 128, 128, True, 2)
    ns = check(128, 128, 256, 40, 20, F, as_tensors=DEV)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    ns.run_steps(20, return_frames=False, forcing=F)
    assert _lib.launch_count() - n0 == 1


@pytest.mark.parametrize("hw", [(100, 72), (128, 70), (70, 128), (97, 101)])
def test_fused_generic_ragged_grid(hw):
    """The generic instantiation: v's column w inside the strips (w < 128) or in the staggered extras (w == 128), u's row h likewise."""
    h, w = hw
    check(h, w, 150, 7, 5, forcing(5, 150, h, w, True, 3), step_kernel="fused", env={"SMK_FUSED_SLICE": 2})


@pytest.mark.parametrize("B", [1, 4])
@pytest.mark.parametrize("nc", [4, 2])
def test_cluster(B, nc):
    from smokephysai_b200 import _lib
    F = forcing(6, B, 128, 128, True, 4 + B)
    with smk_env(SMK_FUSED_CLUSTER=nc, SMK_FUSED_SLICE=0):
        ns = check(128, 128, B, 20, 6, F, step_kernel="fused")
        torch.cuda.synchronize()
        n0 = _lib.launch_count()
        ns.run_steps(6, return_frames=False, forcing=F)
        assert _lib.launch_count() - n0 == 1


def test_phase_path_1024():
    ns = check(1024, 1024, 1, 100, 3, forcing(3, 1, 1024, 1024, True, 5, strength=400.0))
    assert not ns.step_is_fused(3)


@pytest.mark.parametrize("kernel", ["fused", "phases"])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_frames(kernel, dtype):
    check(128, 128, 20, 20, 5, forcing(5, 20, 128, 128, True, 6), frame_dtype=dtype, step_kernel=kernel)


@pytest.mark.parametrize("kernel", ["fused", "phases"])
def test_fractal_multiplier(kernel):
    from smokephysai_b200.fractal_generator import FractalGenerator
    fmul = FractalGenerator(DEV).multiplier((128, 128), 0.05)
    check(128, 128, 20, 20, 5, forcing(5, 20, 128, 128, False, 7), fmul=fmul, step_kernel=kernel)


@pytest.mark.parametrize("kernel,B,env", [("fused", 20, {"SMK_FUSED_SLICE": 2}), ("fused", 2, {"SMK_FUSED_CLUSTER": 4}),
                                          ("phases", 3, {})])
def test_with_continuous_sources(kernel, B, env):
    csrc = [[(x, y, 8, i) for x, y, _, i in emitters_for_sequence(200 + b)] for b in range(B)]
    check(128, 128, B, 20, 5, forcing(5, B, 128, 128, True, 8), csrc=csrc, step_kernel=kernel, env=env)


@pytest.mark.parametrize("kernel,B,env", [("fused", 20, {"SMK_FUSED_SLICE": 2}), ("fused", 2, {"SMK_FUSED_CLUSTER": 2}),
                                          ("phases", 3, {})])
def test_with_schedule(kernel, B, env):
    S = moving_schedule(5, B, 128, 128, seed=9)
    check(128, 128, B, 20, 5, forcing(5, B, 128, 128, True, 9), sched=S, step_kernel=kernel, env=env)


def test_reset_oneshot_schedule_and_forcing_is_one_launch():
    from smokephysai_b200 import _lib
    h = w = 128
    B, K, T = 160, 20, 6
    A = [[(x, y, 8, i) for x, y, _, i in emitters_for_sequence(100 + b)] for b in range(B)]
    S = moving_schedule(T, B, h, w, seed=10)
    F = forcing(T, B, h, w, True, 10)
    ns = make(h, w, B, K)
    ns.add_sources(A)
    ns.run_steps(3, return_frames=False)            # leave a state for the reset to clear
    ns.setup_grid()
    ns.add_sources(A)
    up = tuple(torch.from_numpy(a).to(DEV) for a in S)
    G = tuple(torch.from_numpy(a).to(DEV) for a in F)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    fr = N(ns.run_steps(T, schedule=up, forcing=G))
    assert _lib.launch_count() - n0 == 1
    want_fr, want = host_loop(h, w, B, K, T, F, init=A, sched=S)
    same(fr, want_fr, "frames")
    for k in FIELDS:
        same(N(getattr(ns, k)), want[k], k)


@pytest.mark.parametrize("kernel", ["fused", "phases"])
def test_step_with_forcing(kernel):
    F = forcing(4, 20, 128, 128, True, 11)
    want_fr, want = host_loop(128, 128, 20, 20, 4, F)
    ns = make(128, 128, 20, 20, step_kernel=kernel)
    fr = [ns.step(forcing=(F[0][t], F[1][t])) for t in range(4)]
    same(N(torch.stack(fr, dim=1)), want_fr, "frames")
    for k in FIELDS:
        same(N(getattr(ns, k)), want[k], k)


def test_run_steps_time_major():
    F = forcing(5, 40, 128, 128, True, 12)
    want_fr, want = host_loop(128, 128, 40, 20, 5, F)
    ns = make(128, 128, 40, 20)
    out = torch.empty(5, 40, 128, 128, device=DEV)
    ns.run_steps_time_major(2, out[:2], forcing=tuple(a[:2] for a in F))
    ns.run_steps_time_major(3, out[2:], forcing=tuple(a[2:] for a in F))
    same(N(out).transpose(1, 0, 2, 3), want_fr, "frames")
    for k in FIELDS:
        same(N(getattr(ns, k)), want[k], k)


@pytest.mark.parametrize("steps_per_copy", [1, 2, 3])
@pytest.mark.parametrize("to_host", [True, False])
def test_generate_sequences(to_host, steps_per_copy):
    """The samples' emitters splatted once at the reset, then the forcing; the to_host chunks read their rows of one upload."""
    from smokephysai_b200 import SmokeSimulator
    B, T = 40, 7
    lists = [[((x, y), i) for x, y, _, i in emitters_for_sequence(s)] for s in range(B)]
    F = forcing(T, B, 128, 128, True, 13)
    sim = SmokeSimulator((128, 128), DT, VISC, DEV, jacobi_iters=20, batch=B)
    got = N(sim.generate_sequences(lists, T, add_fractal=False, to_host=to_host, steps_per_copy=steps_per_copy, forcing=F))
    want_fr, _ = host_loop(128, 128, B, 20, T, F, init=[[(x, y, 8, i) for (x, y), i in lst] for lst in lists])
    same(got, want_fr, "sequences")
    const = tuple(a[0] for a in F)
    got_c = N(sim.generate_sequences(lists, T, add_fractal=False, to_host=to_host, steps_per_copy=steps_per_copy, forcing=const))
    want_c, _ = host_loop(128, 128, B, 20, T, const, init=[[(x, y, 8, i) for (x, y), i in lst] for lst in lists])
    same(got_c, want_c, "constant forcing")


@pytest.mark.parametrize("kernel", ["fused", "phases"])
def test_zero_forcing_equals_no_forcing_by_value(kernel):
    """v + 0.0 turns -0 into +0, so zero forcing equals no forcing by value (==), not bit for bit."""
    B = 20
    z = (np.zeros((B, 129, 128), np.float32), np.zeros((B, 128, 129), np.float32))
    a, b = make(128, 128, B, 20, step_kernel=kernel), make(128, 128, B, 20, step_kernel=kernel)
    for ns in (a, b):
        ns.add_sources([[(60, 60, 8, 1.0)]] * B)
    same(N(a.run_steps(4, forcing=z)), N(b.run_steps(4)), "frames")
    for k in FIELDS:
        same(N(getattr(a, k)), N(getattr(b, k)), k)


# ----------------------------------------------------------------------------------------------------------- rejections
def test_value_errors_before_any_launch():
    from smokephysai_b200 import SmokeSimulator, _lib
    du, dv = forcing(3, 2, 64, 64, True, 14)
    ns = make(64, 64, 2, 20)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for bad in ((du,), (du, dv, dv), (du[:2], dv[:2]), (du[:, :1], dv[:, :1]), (du.astype(np.float64), dv),
                (du[..., :-1], dv), (du, dv[:, :, :-1]), (du[0], dv), (du.tolist(), dv)):
        with pytest.raises(ValueError):
            ns.run_steps(3, forcing=bad)
        with pytest.raises(ValueError):
            ns.run_steps_time_major(3, torch.empty(3, 2, 64, 64, device=DEV), forcing=bad)
    with pytest.raises(ValueError):
        ns.step(forcing=(du, dv))                          # step() takes a constant forcing only
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            ns.run_steps(3, forcing=(torch.from_numpy(du).to("cuda:1"), torch.from_numpy(dv).to("cuda:1")))
    assert _lib.launch_count() == n0
    sim = SmokeSimulator((64, 64), DT, VISC, DEV, jacobi_iters=20, batch=2)
    em = [[((30, 30), 1.0)], []]
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for bad in ((du[:2], dv[:2]), (du, dv[:, :, :, :-1])):
        with pytest.raises(ValueError):
            sim.generate_sequences(em, 3, add_fractal=False, forcing=bad)
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("kernel", ["phases", "fused"])
def test_malformed_calls_are_refused_before_any_launch(kernel):
    """Unpaired or misaligned forcing buffers, force_per_step outside {0, 1} or set without forcing: smk_run_steps_force_ex refuses
    each with nothing enqueued; the well-formed calls then run."""
    from smokephysai_b200 import _lib
    from smokephysai_b200._lib import SmokeLibraryError
    B = 48 if kernel == "fused" else 2
    ns = make(128, 128, B, 20, step_kernel=kernel)
    fu, fv, _, _ = ns._forcing(forcing(2, B, 128, 128, True, 15), 2)
    fr = torch.empty(B, 2, 128, 128, device=DEV)
    done = C.c_int32(0)

    def call(u=fu.data_ptr(), v=fv.data_ptr(), per_step=1, nsteps=2):
        _lib.call("smk_run_steps_force_ex", C.byref(ns._grid), C.byref(ns._state), C.byref(ns._params()), nsteps, fr.data_ptr(),
                  128 * 128, 2 * 128 * 128, None, 0, None, None, 0, u, v, per_step, 0, None, None, C.byref(done),
                  _lib.stream_on(ns._cuda))
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for kw in (dict(u=None), dict(v=None), dict(u=fu.data_ptr() + 4), dict(v=fv.data_ptr() + 8), dict(per_step=2),
               dict(per_step=-1), dict(u=None, v=None), dict(nsteps=0)):
        with pytest.raises(SmokeLibraryError):
            call(**kw)
    for bad in (dict(u=None), dict(dv=fv.data_ptr() + 4)):
        args = dict(u=fu.data_ptr(), v=fv.data_ptr(), du=fu.data_ptr(), dv=fv.data_ptr())
        args.update(bad)
        with pytest.raises(SmokeLibraryError):
            _lib.call("smk_add_forcing", C.byref(ns._grid), args["u"], args["v"], args["du"], args["dv"], _lib.stream_on(ns._cuda))
    assert _lib.launch_count() == n0
    call()                                          # the well-formed calls run
    call(per_step=0)
    call(u=None, v=None, per_step=0)
    torch.cuda.synchronize()
    assert _lib.launch_count() > n0


def test_add_forcing_touches_only_the_cells():
    """smk_add_forcing on a ragged grid adds inside u [h+1, w] and v [h, w+1] and leaves the pads alone (neither read nor written)."""
    from smokephysai_b200 import _lib
    from smokephysai_b200.navier_stokes import FieldLayout
    h, w, B = 13, 7, 3
    L = FieldLayout(h, w, B)
    g = L.grid_struct()
    rng = np.random.default_rng(16)
    u = torch.from_numpy(rng.standard_normal((B, h + 1, L.pitch_u)).astype(np.float32)).to(DEV)
    v = torch.from_numpy(rng.standard_normal((B, h, L.pitch_v)).astype(np.float32)).to(DEV)
    du = torch.from_numpy(rng.standard_normal(u.shape).astype(np.float32)).to(DEV)
    dv = torch.from_numpy(rng.standard_normal(v.shape).astype(np.float32)).to(DEV)
    du[..., w:] = float("nan")
    dv[..., w + 1:] = float("nan")
    want_u, want_v = u.clone(), v.clone()
    want_u[..., :w] += du[..., :w]
    want_v[..., :w + 1] += dv[..., :w + 1]
    _lib.call("smk_add_forcing", C.byref(g), u.data_ptr(), v.data_ptr(), du.data_ptr(), dv.data_ptr(), _lib.stream_on(u.device))
    assert N(u).tobytes() == N(want_u).tobytes() and N(v).tobytes() == N(want_v).tobytes()


# ------------------------------------------------------------------------------------------------------------ autodiff
def _state(B, n, seed, vel=30.0):
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    return [f(B, n + 1, n) * np.float32(vel), f(B, n, n + 1) * np.float32(vel), f(B, n, n) * np.float32(0.1),
            rng.random((B, n, n)).astype(np.float32)]


@pytest.mark.parametrize("per_step", [True, False])
@pytest.mark.parametrize("kernel", ["fused", "phases"])
@pytest.mark.parametrize("grad", [True, False])
def test_rollout_forward_bit_equal_to_run_steps(kernel, grad, per_step):
    from smokephysai_b200 import autodiff
    B, n, T = 3, 64, 6
    s = _state(B, n, 3, 60.0)
    F = forcing(T, B, n, n, per_step, 17)
    S = moving_schedule(T, B, n, n, seed=17)
    ns = make(n, n, B, 20, step_kernel=kernel)
    for k, a in zip(FIELDS, s):
        setattr(ns, k, torch.from_numpy(a).to(DEV))
    want = N(ns.run_steps(T, schedule=S, forcing=F))
    lv = [torch.from_numpy(a).to(DEV).requires_grad_(grad) for a in s]
    G = [torch.from_numpy(a).to(DEV).requires_grad_(grad) for a in F]
    frames, final = autodiff.rollout(tuple(lv), T, dt=DT, viscosity=VISC, jacobi_iters=20, step_kernel=kernel,
                                     schedule=S[:2], intensities=torch.from_numpy(S[2]).to(DEV), forcing=tuple(G))
    same(N(frames), want, "frames")
    for k, t in zip(FIELDS, final):
        same(N(t), N(getattr(ns, k)), k)


def _grads(B, n, T, K, per_step, sched=False, seed=1, two_d=False):
    from smokephysai_b200 import autodiff
    s = _state(B, n, seed)
    F = list(forcing(T, B, n, n, per_step, seed + 7, strength=30.0))
    S = moving_schedule(T, B, n, n, seed=seed + 3) if sched else None
    rng = np.random.default_rng(seed + 1)
    wf = rng.standard_normal((B, T, n, n)).astype(np.float32)
    wst = [rng.standard_normal(a.shape).astype(np.float32) for a in s]

    def loss(frames, final, to):
        return (frames * to(wf)).sum() + sum((a * to(wa)).sum() for a, wa in zip(final, wst))

    inputs = list(s) + F + ([S[2]] if sched else [])
    ref_lv = [torch.from_numpy(a).clone().requires_grad_(True) for a in inputs]
    frames, final = rollout_forced(tuple(ref_lv[:4]), T, DT, VISC, K, du=ref_lv[4], dv=ref_lv[5],
                                   xy=S[0] if sched else None, radius=S[1] if sched else None,
                                   intensities=ref_lv[6] if sched else None)
    loss(frames, final, torch.from_numpy).backward()
    ref = [a.grad.numpy() for a in ref_lv]

    def ours():
        lv = [torch.from_numpy(a).to(DEV).requires_grad_(True) for a in inputs]
        st, fu, fv = lv[:4], lv[4], lv[5]
        if two_d:                                                   # B == 1 given without the batch dimension
            st = [a[0] for a in st]
            fu, fv = (a.select(-3, 0) for a in (fu, fv))
        kw = dict(schedule=S[:2], intensities=lv[6]) if sched else {}
        frames, final = autodiff.rollout(tuple(st), T, dt=DT, viscosity=VISC, jacobi_iters=K, forcing=(fu, fv), **kw)
        if two_d:
            frames, final = frames[None], [a[None] for a in final]
        loss(frames, final, lambda a: torch.from_numpy(a).to(DEV)).backward()
        return [a.grad.cpu().numpy() for a in lv]
    return ours, ref


@pytest.mark.parametrize("per_step", [True, False])
@pytest.mark.parametrize("T", [1, 6])
@pytest.mark.parametrize("K", [0, 20])
def test_rollout_gradients_match_restatement(T, K, per_step):
    ours, ref = _grads(3, 48, T, K, per_step)
    got = ours()
    errs = {name: nerr(a, b) for name, a, b in zip(("u0", "v0", "p0", "d0", "du", "dv"), got, ref)}
    print("forcing rollout T=%d K=%d per_step=%s: %s" % (T, K, per_step, {k: "%.2e" % e for k, e in errs.items()}))
    assert max(errs.values()) <= 1e-4, errs


def test_rollout_gradients_with_schedule_and_2d():
    for per_step in (True, False):
        ours, ref = _grads(3, 48, 5, 20, per_step, sched=True, seed=3)
        got = ours()
        errs = {name: nerr(a, b) for name, a, b in zip(("u0", "v0", "p0", "d0", "du", "dv", "intensities"), got, ref)}
        print("forcing + schedule per_step=%s: %s" % (per_step, {k: "%.2e" % e for k, e in errs.items()}))
        assert max(errs.values()) <= 1e-4, errs
    ours, ref = _grads(1, 40, 4, 20, True, seed=4, two_d=True)
    errs = {name: nerr(a, b) for name, a, b in zip(("u0", "v0", "p0", "d0", "du", "dv"), ours(), ref)}
    assert max(errs.values()) <= 1e-4, errs


def test_per_step_gradient_is_the_gradient_at_the_head_of_each_step():
    """The per-step forcing gradient row 0 is the initial-state velocity gradient bit for bit (both are G.u / G.v after reverse step
    0), and the constant forcing's gradient is the per-step rows summed in fp32 in the order t = T-1 .. 0."""
    ours, _ = _grads(3, 48, 6, 20, True, seed=5)
    g = ours()
    assert g[4][0].tobytes() == g[0].tobytes() and g[5][0].tobytes() == g[1].tobytes()
    from smokephysai_b200 import autodiff
    B, n, T = 3, 48, 6
    s = [torch.from_numpy(a).to(DEV) for a in _state(B, n, 6)]
    du, dv = (torch.from_numpy(a).to(DEV) for a in forcing(T, B, n, n, False, 6, strength=30.0))
    w = torch.from_numpy(np.random.default_rng(7).standard_normal((B, T, n, n)).astype(np.float32)).to(DEV)
    cu, cv = du.clone().requires_grad_(True), dv.clone().requires_grad_(True)
    fr, _ = autodiff.rollout(tuple(s), T, jacobi_iters=20, forcing=(cu, cv))
    (fr * w).sum().backward()
    pu, pv = (a.unsqueeze(0).repeat(T, 1, 1, 1).requires_grad_(True) for a in (du, dv))
    fr2, _ = autodiff.rollout(tuple(s), T, jacobi_iters=20, forcing=(pu, pv))
    same(N(fr2), N(fr), "frames")
    (fr2 * w).sum().backward()
    for per, acc_grad in ((pu.grad, cu.grad), (pv.grad, cv.grad)):
        g = per.cpu().numpy()
        acc = np.zeros(g.shape[1:], np.float32)
        for t in range(T - 1, -1, -1):
            acc = (acc + g[t]).astype(np.float32)
        assert acc.tobytes() == acc_grad.cpu().numpy().tobytes()


def test_rollout_backward_is_deterministic():
    for per_step in (True, False):
        ours, _ = _grads(3, 48, 8, 20, per_step, sched=True, seed=8)
        a, b = ours(), ours()
        for x, y in zip(a, b):
            assert x.tobytes() == y.tobytes()


def test_rollout_rejections():
    from smokephysai_b200 import autodiff
    st = tuple(torch.zeros(2, *s, device=DEV) for s in ((33, 32), (32, 33), (32, 32), (32, 32)))
    du, dv = torch.zeros(2, 33, 32, device=DEV), torch.zeros(2, 32, 33, device=DEV)
    for f in ((du,), (du.cpu(), dv), (du.double(), dv), (du[:1], dv[:1]), (du[None].repeat(3, 1, 1, 1), dv[None].repeat(3, 1, 1, 1)),
              (du[0], dv[0]), (du, dv[None])):
        with pytest.raises(ValueError):
            autodiff.rollout(st, 2, forcing=f)
