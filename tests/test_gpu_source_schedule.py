"""Source schedules: emitters that move and change intensity from step to step.  Every case compares run_steps(schedule=S) with
the host loop [add_sources(S[t]); step()] on the phase kernels, bit for bit on the frames and on u, v, p and density, on each
kernel that can run it: k_step_fused (FULL, one CTA per simulation and time-sliced with hand-overs; the generic instantiation),
k_step_cluster (clusters of 4 and 2 CTAs) and the phase path.  The emitters move by a cell and change intensity at every step,
so reading any row but row t at step t changes the frames."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import emitters_for_sequence, nerr, smk_env
from schedule_oracle import moving_schedule, rollout as rollout_sched, rows_as_lists

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


def host_loop(h, w, B, K, sched, frame_dtype=torch.float32, init=None, fmul=None):
    T = sched[1].shape[0]
    ns = make(h, w, B, K, step_kernel="phases")
    if init is not None:
        ns.add_sources(init)
    frames = []
    for t in range(T):
        ns.add_sources(rows_as_lists(sched, t))
        frames.append(ns.step(fmul=fmul, frame_dtype=frame_dtype))
    return N(torch.stack(frames, dim=-3)), {k: N(getattr(ns, k)) for k in FIELDS}


def check(h, w, B, K, sched, env=None, frame_dtype=torch.float32, fmul=None, as_tensors=None, **kw):
    T = sched[1].shape[0]
    want_fr, want = host_loop(h, w, B, K, sched, frame_dtype, fmul=fmul)
    S = sched if as_tensors is None else tuple(torch.from_numpy(a).to(as_tensors) for a in sched)
    with smk_env(**(env or {})):
        ns = make(h, w, B, K, **kw)
        fr = N(ns.run_steps(T, fmul=fmul, frame_dtype=frame_dtype, schedule=S))
        got = {k: N(getattr(ns, k)) for k in FIELDS}
    same(fr, want_fr, "frames")
    for k in FIELDS:
        same(got[k], want[k], k)
    return ns


def test_fused_full_one_cta_per_simulation():
    ns = check(128, 128, 40, 20, moving_schedule(6, 40, 128, 128, seed=1), env={"SMK_FUSED_SLICE": 0, "SMK_FUSED_CLUSTER": 0})
    assert ns.step_is_fused(6)


def test_fused_full_time_sliced_c2_size():
    """256 x 128^2, K = 40, 20 steps: the time-sliced schedule hands simulations from CTA to CTA, and an item that starts at
    t_begin > 0 must splat row t_begin.  One launch per call."""
    from smokephysai_b200 import _lib
    S = moving_schedule(20, 256, 128, 128, seed=2)
    ns = check(128, 128, 256, 40, S, as_tensors=DEV)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    ns.run_steps(20, return_frames=False, schedule=S)
    assert _lib.launch_count() - n0 == 1


def test_fused_generic_ragged_grid():
    check(100, 72, 150, 7, moving_schedule(5, 150, 100, 72, seed=3), step_kernel="fused", env={"SMK_FUSED_SLICE": 2})


@pytest.mark.parametrize("B", [1, 4])
@pytest.mark.parametrize("nc", [4, 2])
def test_cluster(B, nc):
    from smokephysai_b200 import _lib
    S = moving_schedule(6, B, 128, 128, seed=4 + B)
    with smk_env(SMK_FUSED_CLUSTER=nc, SMK_FUSED_SLICE=0):
        ns = check(128, 128, B, 20, S, step_kernel="fused")
        torch.cuda.synchronize()
        n0 = _lib.launch_count()
        ns.run_steps(6, return_frames=False, schedule=S)
        assert _lib.launch_count() - n0 == 1


def test_phase_path_1024():
    S = moving_schedule(3, 1, 1024, 1024, seed=5)
    S[0][:, 0, 1] = [[0, 0], [1, 1], [2, 3]]          # one emitter clipped at the corner
    S[1][:, 0, 1] = 40
    ns = check(1024, 1024, 1, 100, S)
    assert not ns.step_is_fused(3)


@pytest.mark.parametrize("kernel", ["fused", "phases"])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_frames(kernel, dtype):
    check(128, 128, 20, 20, moving_schedule(5, 20, 128, 128, seed=6), frame_dtype=dtype, step_kernel=kernel)


@pytest.mark.parametrize("kernel", ["fused", "phases"])
def test_fractal_multiplier(kernel):
    from smokephysai_b200.fractal_generator import FractalGenerator
    fmul = FractalGenerator(DEV).multiplier((128, 128), 0.05)
    check(128, 128, 20, 20, moving_schedule(5, 20, 128, 128, seed=7), fmul=fmul, step_kernel=kernel)


def test_reset_oneshot_and_schedule_is_one_launch():
    from smokephysai_b200 import _lib
    h = w = 128
    B, K, T = 160, 20, 6
    A = [[(x, y, 8, i) for x, y, _, i in emitters_for_sequence(100 + b)] for b in range(B)]
    S = moving_schedule(T, B, h, w, seed=8)
    ns = make(h, w, B, K)
    ns.add_sources(A)
    ns.run_steps(3, return_frames=False)            # leave a state for the reset to clear
    ns.setup_grid()
    ns.add_sources(A)
    up = tuple(torch.from_numpy(a).to(DEV) for a in S)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    fr = N(ns.run_steps(T, schedule=up))
    assert _lib.launch_count() - n0 == 1
    want_fr, want = host_loop(h, w, B, K, S, init=A)
    same(fr, want_fr, "frames")
    for k in FIELDS:
        same(N(getattr(ns, k)), want[k], k)


def test_run_steps_time_major():
    S = moving_schedule(5, 40, 128, 128, seed=9)
    want_fr, want = host_loop(128, 128, 40, 20, S)
    ns = make(128, 128, 40, 20)
    out = torch.empty(5, 40, 128, 128, device=DEV)
    ns.run_steps_time_major(2, out[:2], schedule=tuple(a[:2] for a in S))
    ns.run_steps_time_major(3, out[2:], schedule=tuple(a[2:] for a in S))
    same(N(out).transpose(1, 0, 2, 3), want_fr, "frames")
    for k in FIELDS:
        same(N(getattr(ns, k)), want[k], k)


@pytest.mark.parametrize("steps_per_copy", [1, 2, 3])
@pytest.mark.parametrize("to_host", [True, False])
def test_generate_sequences(to_host, steps_per_copy):
    """The samples' emitters splatted once at the reset, then the schedule; the to_host chunks read their rows of one upload."""
    from smokephysai_b200 import SmokeSimulator
    B, T = 40, 7
    lists = [[((x, y), i) for x, y, _, i in emitters_for_sequence(s)] for s in range(B)]
    lists[3] = []
    S = moving_schedule(T, B, 128, 128, seed=10)
    sim = SmokeSimulator((128, 128), DT, VISC, DEV, jacobi_iters=20, batch=B)
    got = N(sim.generate_sequences(lists, T, add_fractal=False, to_host=to_host, steps_per_copy=steps_per_copy, schedule=S))
    want_fr, _ = host_loop(128, 128, B, 20, S, init=[[(x, y, 8, i) for (x, y), i in lst] for lst in lists])
    same(got, want_fr, "sequences")
    half = N(sim.generate_sequences(lists, T, add_fractal=False, to_host=to_host, steps_per_copy=steps_per_copy, schedule=S,
                                    frame_dtype=torch.float16))
    same(half, N(torch.from_numpy(got).to(torch.float16)), "fp16 sequences")


@pytest.mark.parametrize("kernel", ["fused", "phases"])
def test_padded_entries_equal_the_unpadded_lists(kernel):
    """Entries with radius < 0 anywhere in a row, and rows of very different lengths, against the host loop over the lists
    without them."""
    T, B = 5, 12
    xy, radius, inten = moving_schedule(T, B, 128, 128, seed=11, emax=3, pad=False)
    E = 9
    pxy = np.zeros((T, B, E, 2), np.int64)
    prad = np.full((T, B, E), -1, np.int32)
    pint = np.full((T, B, E), np.nan, np.float32)      # a padded entry's intensity is never read
    rng = np.random.default_rng(12)
    for b in range(B):
        slots = np.sort(rng.choice(E, 3, replace=False)) if b % 3 else np.array([0, 1, 2])
        n = b % 4                                      # 0 .. 3 real entries per row
        for t in range(T):
            pxy[t, b, slots[:n]] = xy[t, b, :n]
            prad[t, b, slots[:n]] = radius[t, b, :n]
            pint[t, b, slots[:n]] = inten[t, b, :n]
            prad[t, b, 8] = -7
            pxy[t, b, 8] = (64, 64)
    check(128, 128, B, 20, (pxy, prad, pint), step_kernel=kernel)


@pytest.mark.parametrize("kernel", ["fused", "phases"])
def test_equal_rows_are_continuous_sources(kernel):
    T, B = 6, 20
    one = moving_schedule(1, B, 128, 128, seed=13, pad=False)
    S = tuple(np.repeat(a, T, axis=0) for a in one)
    a, b = make(128, 128, B, 20, step_kernel=kernel), make(128, 128, B, 20, step_kernel=kernel)
    a.set_continuous_sources(rows_as_lists(one, 0))
    same(N(b.run_steps(T, schedule=S)), N(a.run_steps(T)), "frames")
    for k in FIELDS:
        same(N(getattr(b, k)), N(getattr(a, k)), k)


def test_empty_schedule_is_a_plain_call():
    S = (np.zeros((4, 8, 0, 2), np.int32), np.zeros((4, 8, 0), np.int32), np.zeros((4, 8, 0), np.float32))
    a, b = make(128, 128, 8, 20), make(128, 128, 8, 20)
    for ns in (a, b):
        ns.add_sources([[(60, 60, 8, 1.0)]] * 8)
    same(N(a.run_steps(4, schedule=S)), N(b.run_steps(4)), "frames")


# ----------------------------------------------------------------------------------------------------------- rejections
def test_value_errors_before_any_launch():
    from smokephysai_b200 import SmokeSimulator, _lib
    S = moving_schedule(3, 2, 64, 64)
    ns = make(64, 64, 2, 20)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for bad in ((S[0], S[1]), tuple(a[:2] for a in S), (S[0], S[1], S[2].astype(np.float64)),
                (S[0].astype(np.float32), S[1], S[2]), (S[0][:, :1], S[1], S[2]),
                (torch.from_numpy(S[0]).to(DEV), S[1], S[2])):
        with pytest.raises(ValueError):
            ns.run_steps(3, schedule=bad)
    ns.set_continuous_sources([[(5, 5, 3, 1.0)], []])
    with pytest.raises(ValueError):
        ns.run_steps(3, schedule=S)
    with pytest.raises(ValueError):
        ns.run_steps_time_major(3, torch.empty(3, 2, 64, 64, device=DEV), schedule=S)
    assert _lib.launch_count() == n0
    sim = SmokeSimulator((64, 64), DT, VISC, DEV, jacobi_iters=20, batch=2)
    em = [[((30, 30), 1.0)], []]
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for kw in (dict(continuous=True, schedule=S), dict(schedule=tuple(a[:2] for a in S))):
        with pytest.raises(ValueError):
            sim.generate_sequences(em, 3, add_fractal=False, **kw)
    sim.ns_solver.set_continuous_sources([[(5, 5, 3, 1.0)], []])
    with pytest.raises(ValueError):
        sim.generate_sequences(em, 3, add_fractal=False, schedule=S)
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("kernel", ["phases", "fused"])
def test_malformed_calls_and_bad_strides_are_refused_before_any_launch(kernel):
    """The malformed calls test_gpu_continuous_sources sends to smk_run_steps_src_ex, plus offsets step strides other than 0 and
    the batch, and a non-zero stride without sources: smk_run_steps_sched_ex refuses each with nothing enqueued."""
    from smokephysai_b200 import _lib
    from smokephysai_b200._lib import SmokeLibraryError
    B = 48 if kernel == "fused" else 2
    ns = make(128, 128, B, 20, step_kernel=kernel)
    up = ns.upload_schedule(moving_schedule(2, B, 128, 128), 2)
    src, off = up
    fr = torch.empty(B, 2, 128, 128, device=DEV)
    done = C.c_int32(0)

    def call(nsteps=2, s=src.data_ptr(), o=off.data_ptr(), stride=B, reset=0, rs=None, ro=None, consumed=C.byref(done)):
        _lib.call("smk_run_steps_sched_ex", C.byref(ns._grid), C.byref(ns._state), C.byref(ns._params()), nsteps, fr.data_ptr(),
                  128 * 128, 2 * 128 * 128, None, 0, s, o, stride, reset, rs, ro, consumed, _lib.stream_on(ns._cuda))
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for kw in (dict(nsteps=0), dict(o=None), dict(s=None), dict(rs=src.data_ptr()), dict(reset=1, rs=src.data_ptr()),
               dict(reset=2), dict(consumed=None), dict(stride=1 if B > 1 else 2), dict(stride=B + 1), dict(stride=-B),
               dict(s=None, o=None)):
        with pytest.raises(SmokeLibraryError):
            call(**kw)
    assert _lib.launch_count() == n0
    call()                                          # the well-formed calls run
    call(stride=0)
    call(s=None, o=None, stride=0)
    torch.cuda.synchronize()
    assert _lib.launch_count() > n0


# ------------------------------------------------------------------------------------------------------------ autodiff
def _state(B, n, seed, vel=30.0):
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    return [f(B, n + 1, n) * np.float32(vel), f(B, n, n + 1) * np.float32(vel), f(B, n, n) * np.float32(0.1),
            rng.random((B, n, n)).astype(np.float32)]


@pytest.mark.parametrize("kernel", ["fused", "phases"])
@pytest.mark.parametrize("grad", [True, False])
def test_rollout_forward_bit_equal_to_run_steps(kernel, grad):
    from smokephysai_b200 import autodiff
    B, n, T = 3, 64, 6
    s = _state(B, n, 3, 60.0)
    S = moving_schedule(T, B, n, n, seed=14)
    ns = make(n, n, B, 20, step_kernel=kernel)
    for k, a in zip(FIELDS, s):
        setattr(ns, k, torch.from_numpy(a).to(DEV))
    want = N(ns.run_steps(T, schedule=S))
    lv = [torch.from_numpy(a).to(DEV).requires_grad_(grad) for a in s]
    frames, final = autodiff.rollout(tuple(lv), T, dt=DT, viscosity=VISC, jacobi_iters=20, step_kernel=kernel,
                                     schedule=S[:2], intensities=torch.from_numpy(S[2]).to(DEV).requires_grad_(grad))
    same(N(frames), want, "frames")
    for k, t in zip(FIELDS, final):
        same(N(t), N(getattr(ns, k)), k)


def _grads(B, n, T, K, S, seed=1):
    from smokephysai_b200 import autodiff
    s = _state(B, n, seed)
    rng = np.random.default_rng(seed + 1)
    wf = rng.standard_normal((B, T, n, n)).astype(np.float32)
    wst = [rng.standard_normal(a.shape).astype(np.float32) for a in s]

    def loss(frames, final, to):
        return (frames * to(wf)).sum() + sum((a * to(wa)).sum() for a, wa in zip(final, wst))

    ref_lv = [torch.from_numpy(a).clone().requires_grad_(True) for a in list(s) + [S[2]]]
    frames, final = rollout_sched(tuple(ref_lv[:4]), T, DT, VISC, K, xy=S[0], radius=S[1], intensities=ref_lv[4])
    loss(frames, final, torch.from_numpy).backward()
    ref = [a.grad.numpy() for a in ref_lv]

    def ours():
        lv = [torch.from_numpy(a).to(DEV).requires_grad_(True) for a in list(s) + [S[2]]]
        frames, final = autodiff.rollout(tuple(lv[:4]), T, dt=DT, viscosity=VISC, jacobi_iters=K, schedule=S[:2],
                                         intensities=lv[4])
        loss(frames, final, lambda a: torch.from_numpy(a).to(DEV)).backward()
        return [a.grad.cpu().numpy() for a in lv]
    return ours, ref


@pytest.mark.parametrize("T", [1, 5, 12])
@pytest.mark.parametrize("K", [0, 20])
def test_rollout_gradients_match_restatement(T, K):
    S = moving_schedule(T, 3, 48, 48, seed=15)
    ours, ref = _grads(3, 48, T, K, S)
    got = ours()
    errs = {name: nerr(a, b) for name, a, b in zip(("u0", "v0", "p0", "d0", "intensities"), got, ref)}
    print("schedule rollout T=%d K=%d: %s" % (T, K, {k: "%.2e" % e for k, e in errs.items()}))
    assert max(errs.values()) <= 1e-4, errs
    pad = S[1] < 0
    assert pad.any() and np.all(got[4][pad] == 0)
    assert np.abs(got[4][~pad]).min() > 0


def test_rollout_backward_is_deterministic():
    ours, _ = _grads(3, 48, 8, 20, moving_schedule(8, 3, 48, 48, seed=16), seed=5)
    a, b = ours(), ours()
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


def test_equal_rows_gradient_sums_to_the_sources_gradient():
    """For a schedule whose rows are all equal, the per-step intensity gradients summed in fp32 in the order t = T-1 .. 0 are the
    gradient rollout(sources=) accumulates, bit for bit."""
    from smokephysai_b200 import autodiff
    B, n, T = 3, 48, 7
    one = moving_schedule(1, B, n, n, seed=17, pad=False)
    xy, radius = (np.repeat(a, T, axis=0) for a in one[:2])
    I0 = torch.from_numpy(one[2][0]).to(DEV)
    s = [torch.from_numpy(a).to(DEV) for a in _state(B, n, 18)]
    w = torch.from_numpy(np.random.default_rng(19).standard_normal((B, T, n, n)).astype(np.float32)).to(DEV)
    Is = I0.reshape(-1).clone().requires_grad_(True)
    em = [[(int(xy[0, b, e, 0]), int(xy[0, b, e, 1]), int(radius[0, b, e])) for e in range(radius.shape[2])] for b in range(B)]
    fr, _ = autodiff.rollout(tuple(s), T, jacobi_iters=20, sources=em, intensities=Is)
    (fr * w).sum().backward()
    It = I0.unsqueeze(0).repeat(T, 1, 1).requires_grad_(True)
    fr2, _ = autodiff.rollout(tuple(s), T, jacobi_iters=20, schedule=(xy, radius), intensities=It)
    same(N(fr2), N(fr), "frames")
    (fr2 * w).sum().backward()
    g = It.grad.cpu().numpy()
    acc = np.zeros(g.shape[1:], np.float32)
    for t in range(T - 1, -1, -1):
        acc = (acc + g[t]).astype(np.float32)
    assert acc.reshape(-1).tobytes() == Is.grad.cpu().numpy().tobytes()


def test_rollout_rejections():
    from smokephysai_b200 import autodiff
    st = tuple(torch.zeros(2, *s, device=DEV) for s in ((33, 32), (32, 33), (32, 32), (32, 32)))
    S = moving_schedule(2, 2, 32, 32)
    I = torch.from_numpy(S[2]).to(DEV)
    for kw in (dict(schedule=S, intensities=I),                         # (xy, radius, intensity): rollout takes two
               dict(schedule=S[:2]),                                    # no intensities
               dict(schedule=S[:2], intensities=I[:1]),                 # T = 1
               dict(schedule=S[:2], intensities=I.cpu()),               # wrong device
               dict(schedule=S[:2], intensities=I.double()),
               dict(schedule=tuple(a[:1] for a in S[:2]), intensities=I[:1]),     # T != nsteps
               dict(schedule=S[:2], intensities=I, sources=[[(1, 2, 3)], []])):
        with pytest.raises(ValueError):
            autodiff.rollout(st, 2, **kw)


def test_lbfgs_recovers_an_emission_history():
    """One emitter on 64^2 whose intensity changes at every step: LBFGS through rollout(schedule=) recovers the 10 intensities
    from the observed frames."""
    from smokephysai_b200 import autodiff
    n, T = 64, 10
    xy = np.zeros((T, 1, 1, 2), np.int64)
    xy[:, 0, 0] = [(32 + (t % 3) - 1, 40 - t) for t in range(T)]
    radius = np.full((T, 1, 1), 8, np.int32)
    true = torch.tensor(1.0 + 0.5 * np.sin(np.arange(T)), dtype=torch.float32, device=DEV).view(T, 1, 1)
    st = tuple(torch.zeros(1, *s, device=DEV) for s in ((n + 1, n), (n, n + 1), (n, n), (n, n)))
    with torch.no_grad():
        obs, _ = autodiff.rollout(st, T, jacobi_iters=20, schedule=(xy, radius), intensities=true)
    I = torch.full((T, 1, 1), 0.5, device=DEV, requires_grad=True)
    opt = torch.optim.LBFGS([I], lr=1, max_iter=200, tolerance_grad=1e-12, tolerance_change=1e-14,
                            line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        fr, _ = autodiff.rollout(st, T, jacobi_iters=20, schedule=(xy, radius), intensities=I)
        loss = ((fr - obs) ** 2).sum()
        loss.backward()
        return loss
    for _ in range(3):
        opt.step(closure)
    rel = float((I.detach() - true).norm() / true.norm())
    print("LBFGS emission history: relative error %.2e" % rel)
    assert rel < 1e-3
