"""Continuous sources: emitters that inject at the head of every step.  Every case compares a run with
set_continuous_sources(S) against the host loop [add_sources(S); step()] on the phase kernels, bit for bit on the frames and
on u, v, p and density, for each kernel that can run it: k_step_fused (FULL, one CTA per simulation and time-sliced with
hand-overs; the generic instantiation), k_step_cluster (clusters of 4 and 2 CTAs) and the phase path."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle
from continuous_oracle import rollout as rollout_src
from helpers import emitters_for_sequence, nerr, smk_env

pytestmark = pytest.mark.gpu

DT, VISC = 0.01, 0.001
DEV = "cuda:0"
FIELDS = ("u", "v", "p", "density")


def N(t):
    """A host copy (generate_sequences(to_host=True) hands out a buffer that its next call overwrites)."""
    return t.detach().float().cpu().numpy().copy()


def same(a, b, what):
    """Bit for bit, NaN-aware (a radius-0 emitter makes 0 / 0 in its own weight, as in the reference)."""
    np.testing.assert_array_equal(np.asarray(a), np.asarray(b), err_msg=what)


def make(h, w, B, K, **kw):
    from smokephysai_b200 import NavierStokesSimulator
    return NavierStokesSimulator((h, w), DT, VISC, DEV, jacobi_iters=K, batch=B, **kw)


def long_list(h, w, n=32):
    """n emitters over the whole grid, several overlapping, some clipped at the edges."""
    rng = np.random.default_rng(n)
    return [(int(rng.integers(-4, w + 4)), int(rng.integers(-4, h + 4)), int(rng.integers(1, 12)), float(rng.uniform(0.2, 1.5)))
            for _ in range(n)]


def lists_for(B, h, w, seed=0, radius0=True):
    """Per-simulation lists: the data-loader law, empty lists, overlapping and edge-clipped emitters, a 32-emitter list and
    (radius0) a radius-0 emitter."""
    out = []
    for b in range(B):
        base = [(x % w, y % h, r, i) for x, y, r, i in emitters_for_sequence(seed + b, h, w)]
        kind = b % 6
        if kind == 1:
            base = []
        elif kind == 2:
            base = base + [(w // 2, h // 2, 8, 1.0), (w // 2 + 3, h // 2 - 2, 6, 0.5), (0, h - 2, 8, 1.25), (w - 1, 1, 9, 0.75)]
        elif kind == 3 and radius0:
            base = base + [(w // 3, h // 3, 0, 1.0)]
        elif kind == 4 or B == 1:
            base = long_list(h, w)
        out.append(base)
    return out


def host_loop(h, w, B, K, T, S, frame_dtype=torch.float32, init=None):
    ns = make(h, w, B, K, step_kernel="phases")
    if init is not None:
        ns.add_sources(init)
    frames = []
    for _ in range(T):
        ns.add_sources(S)
        frames.append(ns.step(frame_dtype=frame_dtype))
    return N(torch.stack(frames, dim=-3)), {k: N(getattr(ns, k)) for k in FIELDS}


def check(h, w, B, K, T, S, env=None, frame_dtype=torch.float32, **kw):
    want_fr, want = host_loop(h, w, B, K, T, S, frame_dtype)
    with smk_env(**(env or {})):
        ns = make(h, w, B, K, **kw)
        ns.set_continuous_sources(S)
        fr = N(ns.run_steps(T, frame_dtype=frame_dtype))
        got = {k: N(getattr(ns, k)) for k in FIELDS}
    same(fr, want_fr, "frames")
    for k in FIELDS:
        same(got[k], want[k], k)
    return ns


def test_fused_full_one_cta_per_simulation():
    ns = check(128, 128, 40, 20, 6, lists_for(40, 128, 128), env={"SMK_FUSED_SLICE": 0, "SMK_FUSED_CLUSTER": 0})
    assert ns.step_is_fused(6)


def test_fused_full_time_sliced_c2_size():
    """256 x 128^2, K = 40, 20 steps: the time-sliced schedule hands simulations from CTA to CTA; still one launch per call."""
    from smokephysai_b200 import _lib
    S = lists_for(256, 128, 128, seed=50)
    ns = check(128, 128, 256, 40, 20, S)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    ns.run_steps(20, return_frames=False)
    assert _lib.launch_count() - n0 == 1


def test_fused_generic_ragged_grid_odd_k():
    check(100, 72, 14, 7, 6, lists_for(14, 100, 72, seed=3), step_kernel="fused", env={"SMK_FUSED_SLICE": 0})
    check(100, 72, 150, 7, 5, lists_for(150, 100, 72, seed=4), step_kernel="fused", env={"SMK_FUSED_SLICE": 2})


@pytest.mark.parametrize("B", [1, 4])
@pytest.mark.parametrize("nc", [4, 2])
def test_cluster(B, nc):
    """Finite states only: k_step_cluster's Jacobi masks the Dirichlet ring by a multiply by 0, which keeps a NaN there where the
    other kernels store 0, so a simulation that a radius-0 emitter turns into NaN differs in where its NaNs sit -- with or
    without continuous sources (DESIGN.md 5.5).  The radius-0 emitter is covered on k_step_fused and the phase kernels."""
    check(128, 128, B, 20, 6, lists_for(B, 128, 128, seed=7, radius0=False), env={"SMK_FUSED_CLUSTER": nc, "SMK_FUSED_SLICE": 0},
          step_kernel="fused")


def test_cluster_is_the_default_for_one_simulation():
    from smokephysai_b200 import _lib
    ns = check(128, 128, 1, 40, 8, lists_for(1, 128, 128, seed=8))
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    ns.run_steps(5, return_frames=False)
    assert _lib.launch_count() - n0 == 1


def test_phase_path_1024():
    S = [long_list(1024, 1024, 32) + [(512, 900, 30, 2.0), (0, 0, 40, 1.0)]]
    ns = check(1024, 1024, 1, 100, 3, S)
    assert not ns.step_is_fused(3)


def test_single_step_calls_and_step_into():
    S = lists_for(40, 128, 128, seed=11)
    want_fr, want = host_loop(128, 128, 40, 20, 4, S)
    for kernel in ("fused", "phases"):
        ns = make(128, 128, 40, 20, step_kernel=kernel)
        ns.set_continuous_sources(S)
        fr = [N(ns.step()) for _ in range(2)]
        buf = torch.empty(40, 128, 128, device=DEV)
        for _ in range(2):
            ns.step_into(buf)
            fr.append(N(buf))
        same(np.stack(fr, axis=1), want_fr, kernel + " frames")
        for k in FIELDS:
            same(N(getattr(ns, k)), want[k], kernel + " " + k)


def test_run_steps_time_major():
    S = lists_for(40, 128, 128, seed=12)
    want_fr, want = host_loop(128, 128, 40, 20, 5, S)
    ns = make(128, 128, 40, 20)
    ns.set_continuous_sources(S)
    out = torch.empty(5, 40, 128, 128, device=DEV)
    ns.run_steps_time_major(2, out[:2])
    ns.run_steps_time_major(3, out[2:])
    same(N(out).transpose(1, 0, 2, 3), want_fr, "frames")
    for k in FIELDS:
        same(N(getattr(ns, k)), want[k], k)


def test_against_c_oracle():
    """The C oracle's add_smoke_source + step per step; its expf is held to ulps, not bits, so within a tolerance."""
    h, w, K, T = 37, 53, 20, 4
    S = [[(20, 15, 8, 1.5), (24, 17, 6, 0.75), (2, 35, 5, 2.0), (50, 1, 4, 1.25)], [], [(30, 20, 8, 0.9)]]
    for kernel in ("fused", "phases"):
        ns = make(h, w, 3, K, step_kernel=kernel)
        ns.set_continuous_sources(S)
        fr = N(ns.run_steps(T))
        for b in range(3):
            o = oracle.OracleSolver((h, w), DT, VISC, K)
            ofr = []
            for _ in range(T):
                for x, y, r, i in S[b]:
                    o.add_smoke_source(x, y, r, i)
                ofr.append(o.step())
            assert nerr(fr[b], np.stack(ofr)) <= 1e-4, (kernel, b)
            for k, want in zip(FIELDS, (o.u, o.v, o.p, o.density)):
                assert nerr(N(getattr(ns, k))[b], want) <= 1e-4, (kernel, b, k)


def test_reset_oneshot_and_continuous_is_one_launch():
    from smokephysai_b200 import _lib
    h = w = 128
    B, K, T = 160, 20, 6
    A = lists_for(B, h, w, seed=20, radius0=False)
    S = lists_for(B, h, w, seed=30)
    ns = make(h, w, B, K)
    ns.add_sources(lists_for(B, h, w, seed=40))
    ns.run_steps(3, return_frames=False)            # leave a state for the reset to clear
    ns.set_continuous_sources(S)
    ns.setup_grid()                                 # keeps the continuous sources
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    ns.add_sources(A)
    fr = N(ns.run_steps(T))
    assert _lib.launch_count() - n0 == 1
    want_fr, want = host_loop(h, w, B, K, T, S, init=A)
    same(fr, want_fr, "frames")
    for k in FIELDS:
        same(N(getattr(ns, k)), want[k], k)


@pytest.mark.parametrize("kernel", ["fused", "phases"])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_frames(kernel, dtype):
    S = lists_for(20, 128, 128, seed=60)
    ns = make(128, 128, 20, 20, step_kernel=kernel)
    ns.set_continuous_sources(S)
    f32 = ns.run_steps(5)
    ns = make(128, 128, 20, 20, step_kernel=kernel)
    ns.set_continuous_sources(S)
    half = ns.run_steps(5, frame_dtype=dtype)
    assert half.dtype == dtype
    same(N(half), N(f32.to(dtype)), "half frames")


@pytest.mark.parametrize("to_host", [False, True])
def test_generate_sequences(to_host):
    from smokephysai_b200 import SmokeSimulator
    B, T = 40, 6
    lists = [[((x, y), i) for x, y, _, i in emitters_for_sequence(s)] for s in range(B)]
    lists[3] = []
    sim = SmokeSimulator((128, 128), DT, VISC, DEV, jacobi_iters=20, batch=B)
    once = N(sim.generate_sequences(lists, T, add_fractal=False, to_host=to_host))
    cont = N(sim.generate_sequences(lists, T, add_fractal=False, to_host=to_host, continuous=True))
    same(cont[:, 0], once[:, 0], "frame 0")
    assert sim.ns_solver.continuous_sources is None
    S = [[(x, y, 8, i) for (x, y), i in lst] for lst in lists]
    want_fr, _ = host_loop(128, 128, B, 20, T, S)
    same(cont, want_fr, "continuous sequences")
    assert not np.array_equal(cont, once)
    # half frames through the same path
    half = N(sim.generate_sequences(lists, T, add_fractal=False, to_host=to_host, continuous=True, frame_dtype=torch.bfloat16))
    same(half, N(torch.from_numpy(cont).to(torch.bfloat16)), "bf16 sequences")


def test_add_incense_source_continuous():
    from smokephysai_b200 import SmokeSimulator
    sim = SmokeSimulator((128, 128), DT, VISC, DEV, jacobi_iters=20)
    sim.add_incense_source([(64, 100)], [1.0], continuous=True)
    sim.add_incense_source([(40, 110), (90, 105)], [0.5, 0.75], continuous=True)
    assert sim.ns_solver.continuous_sources == [[(64, 100, 8, 1.0), (40, 110, 8, 0.5), (90, 105, 8, 0.75)]]
    fr = [N(sim.simulate_step(add_fractal=False)) for _ in range(4)]
    want_fr, _ = host_loop(128, 128, 1, 20, 4, sim.ns_solver.continuous_sources)
    same(np.stack(fr), want_fr, "incense frames")


def test_clearing_restores_todays_results():
    S = lists_for(40, 128, 128, seed=70)
    for kernel in ("fused", "phases"):
        a, b = make(128, 128, 40, 20, step_kernel=kernel), make(128, 128, 40, 20, step_kernel=kernel)
        for ns in (a, b):
            ns.add_sources(lists_for(40, 128, 128, seed=71, radius0=False))
        a.set_continuous_sources(S)
        a.set_continuous_sources(None)
        assert a.continuous_sources is None
        same(N(a.run_steps(4)), N(b.run_steps(4)), kernel + " frames")
        for k in FIELDS:
            same(N(getattr(a, k)), N(getattr(b, k)), kernel + " " + k)


# ------------------------------------------------------------------------------------------------------------ autodiff
def _state(B, n, seed, vel=30.0):
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    return [f(B, n + 1, n) * np.float32(vel), f(B, n, n + 1) * np.float32(vel), f(B, n, n) * np.float32(0.1),
            rng.random((B, n, n)).astype(np.float32)]


def _emitters(B, n):
    return [[(n // 2 + b, n // 3, 6), (n // 2 + b + 2, n // 3 + 1, 5), (0, n - 2, 6)] if b != 1 else [] for b in range(B)]


@pytest.mark.parametrize("kernel", ["fused", "phases"])
@pytest.mark.parametrize("grad", [True, False])
def test_rollout_forward_bit_equal_to_run_steps(kernel, grad):
    from smokephysai_b200 import autodiff
    B, n, T = 3, 64, 6
    s = _state(B, n, 3, 60.0)
    em = _emitters(B, n)
    inten = torch.tensor([1.5, 0.5, 0.25, 1.0, 0.75, 2.0], device=DEV)
    ns = make(n, n, B, 20, step_kernel=kernel)
    for k, a in zip(FIELDS, s):
        setattr(ns, k, torch.from_numpy(a).to(DEV))
    ns.set_continuous_sources([[(x, y, r, float(inten[k])) for k, (x, y, r) in enumerate(em[b], sum(len(l) for l in em[:b]))]
                               for b in range(B)])
    want = N(ns.run_steps(T))
    lv = [torch.from_numpy(a).to(DEV).requires_grad_(grad) for a in s]
    frames, final = autodiff.rollout(tuple(lv), T, dt=DT, viscosity=VISC, jacobi_iters=20, step_kernel=kernel,
                                     sources=em, intensities=inten.clone().requires_grad_(grad))
    same(N(frames), want, "frames")
    for k, t in zip(FIELDS, final):
        same(N(t), N(getattr(ns, k)), k)


def _grads(B, n, T, K, seed=1):
    from smokephysai_b200 import autodiff
    s = _state(B, n, seed)
    em = _emitters(B, n)
    inten = np.linspace(0.5, 1.5, sum(len(l) for l in em)).astype(np.float32)
    rng = np.random.default_rng(seed + 1)
    wf = rng.standard_normal((B, T, n, n)).astype(np.float32)
    wst = [rng.standard_normal(a.shape).astype(np.float32) for a in s]

    def loss(frames, final, to):
        return (frames * to(wf)).sum() + sum((a * to(wa)).sum() for a, wa in zip(final, wst))

    ref_lv = [torch.from_numpy(a).clone().requires_grad_(True) for a in list(s) + [inten]]
    frames, final = rollout_src(tuple(ref_lv[:4]), T, DT, VISC, K, sources=em, intensities=ref_lv[4])
    loss(frames, final, torch.from_numpy).backward()
    ref = [a.grad.numpy() for a in ref_lv]

    def ours():
        lv = [torch.from_numpy(a).to(DEV).requires_grad_(True) for a in list(s) + [inten]]
        frames, final = autodiff.rollout(tuple(lv[:4]), T, dt=DT, viscosity=VISC, jacobi_iters=K, sources=em, intensities=lv[4])
        loss(frames, final, lambda a: torch.from_numpy(a).to(DEV)).backward()
        return [a.grad.cpu().numpy() for a in lv]
    return ours, ref


@pytest.mark.parametrize("T", [1, 5, 20])
@pytest.mark.parametrize("K", [0, 1, 20])
def test_rollout_gradients_match_restatement(T, K):
    ours, ref = _grads(3, 32, T, K)
    got = ours()
    errs = {name: nerr(a, b) for name, a, b in zip(("u0", "v0", "p0", "d0", "intensities"), got, ref)}
    print("continuous rollout T=%d K=%d: %s" % (T, K, {k: "%.2e" % e for k, e in errs.items()}))
    assert max(errs.values()) <= 1e-4, errs
    assert np.abs(got[4]).max() > 0


def test_rollout_backward_is_deterministic():
    ours, _ = _grads(3, 48, 8, 20, seed=5)
    a, b = ours(), ours()
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


def test_intensities_only_require_grad():
    from smokephysai_b200 import autodiff
    s = [torch.from_numpy(a).to(DEV) for a in _state(3, 32, 9)]
    inten = torch.ones(6, device=DEV, requires_grad=True)
    frames, _ = autodiff.rollout(tuple(s), 4, jacobi_iters=20, sources=_emitters(3, 32), intensities=inten)
    frames.sum().backward()
    assert inten.grad is not None and torch.all(inten.grad > 0)


# ----------------------------------------------------------------------------------------------------------- rejections
def test_rejections_before_any_launch():
    from smokephysai_b200 import _lib, autodiff
    from smokephysai_b200._lib import SmokeLibraryError
    ns = make(128, 128, 2, 20)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for bad in ([[(1, 2, 3, 4)]], [[(1, 2, 3)], []], [[("x", 2, 3, 4)], []]):
        with pytest.raises(ValueError):
            ns.set_continuous_sources(bad)
    assert ns.continuous_sources is None
    src, off, _ = ns.upload_sources([[(5, 5, 3, 1.0)], []])
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    fr = torch.empty(2, 2, 128, 128, device=DEV)
    done = C.c_int32(0)

    def call(nsteps=2, s=src.data_ptr(), o=off.data_ptr(), reset=0, rs=None, ro=None, consumed=C.byref(done)):
        _lib.call("smk_run_steps_src_ex", C.byref(ns._grid), C.byref(ns._state), C.byref(ns._params()), nsteps, fr.data_ptr(),
                  128 * 128, 2 * 128 * 128, None, 0, s, o, reset, rs, ro, consumed, _lib.stream_on(ns._cuda))
    for kw in (dict(nsteps=0), dict(o=None), dict(s=None), dict(rs=src.data_ptr()), dict(reset=1, rs=src.data_ptr()),
               dict(reset=2), dict(consumed=None)):
        with pytest.raises(SmokeLibraryError):
            call(**kw)
    assert _lib.launch_count() == n0
    call()                                          # the well-formed call runs
    assert _lib.launch_count() > n0
    st = [torch.zeros(2, 33, 32, device=DEV), torch.zeros(2, 32, 33, device=DEV), torch.zeros(2, 32, 32, device=DEV),
          torch.zeros(2, 32, 32, device=DEV)]
    for kw in (dict(sources=[[(1, 2, 3)], []]), dict(intensities=torch.ones(1, device=DEV)),
               dict(sources=[[(1, 2, 3)], []], intensities=torch.ones(2, device=DEV)),
               dict(sources=[[(1, 2, 3)], []], intensities=torch.ones(1, device=DEV, dtype=torch.float64)),
               dict(sources=[[(1, 2, 3)]], intensities=torch.ones(1, device=DEV)),
               dict(sources=[[(1, 2)], []], intensities=torch.ones(1, device=DEV))):
        with pytest.raises(ValueError):
            autodiff.rollout(tuple(st), 2, **kw)


@pytest.mark.parametrize("kernel", ["phases", "fused"])
def test_every_step_entry_refuses_the_same_malformed_calls_before_any_launch(kernel):
    """smk_step, smk_step_ex, smk_run_steps, smk_run_steps_ex, smk_run_steps_reset_ex and smk_run_steps_src_ex check a call the
    same way, whichever kernel it would run on: each malformed grid, state, params or frame below is refused by every one of
    them with nothing enqueued, and the well-formed calls then run."""
    from smokephysai_b200 import _lib
    h, w, B = (128, 128, 48) if kernel == "fused" else (32, 32, 2)      # 48 full-size simulations: k_step_fused, not clusters
    ns = make(h, w, B, 20, step_kernel=kernel)
    assert ns.step_is_fused(1) == ns.step_is_fused(2) == (kernel == "fused")
    L, lib = ns._layout, _lib.load()
    fr = torch.empty(B, 2, L.h, L.pitch_c, device=DEV)
    src, off, _ = ns.upload_sources([[(5, 5, 3, 1.0)] for _ in range(B)])
    s = _lib.stream_on(ns._cuda)
    step, batch = L.h * L.pitch_c, 2 * L.h * L.pitch_c
    done = C.c_int32(0)
    entries = {
        "smk_step": lambda g, st, prm, f: lib.smk_step(g, st, prm, f, batch, None, s),
        "smk_step_ex": lambda g, st, prm, f: lib.smk_step_ex(g, st, prm, f, batch, None, 0, s),
        "smk_run_steps": lambda g, st, prm, f: lib.smk_run_steps(g, st, prm, 2, f, step, batch, None, s),
        "smk_run_steps_ex": lambda g, st, prm, f: lib.smk_run_steps_ex(g, st, prm, 2, f, step, batch, None, 0, s),
        "smk_run_steps_reset_ex": lambda g, st, prm, f: lib.smk_run_steps_reset_ex(g, st, prm, 2, f, step, batch, None, 0,
                                                                                   src.data_ptr(), off.data_ptr(), C.byref(done), s),
        "smk_run_steps_src_ex": lambda g, st, prm, f: lib.smk_run_steps_src_ex(g, st, prm, 2, f, step, batch, None, 0, src.data_ptr(),
                                                                               off.data_ptr(), 0, None, None, C.byref(done), s),
    }

    def edit(x, **fields):
        y = type(x).from_buffer_copy(x)
        for k, v in fields.items():
            if isinstance(v, tuple):                # (copy index, pointer) of a ping-pong pair
                getattr(y, k)[v[0]] = v[1]
            else:
                setattr(y, k, v)
        return y
    G, S, P, F = ns._grid, ns._state, ns._params(), fr.data_ptr()
    bad = {
        "NULL grid": (None, S, P, F),
        "NULL state": (G, None, P, F),
        "NULL params": (G, S, None, F),
        "batch 0": (edit(G, batch=0), S, P, F),
        "slab grid": (edit(G, gh=G.h + 8, row0=4), S, P, F),
        "NULL div": (G, edit(S, div=None), P, F),
        "NULL spare u": (G, edit(S, u=(S.cur_u ^ 1, None)), P, F),
        "misaligned spare density": (G, edit(S, d=(S.cur_d ^ 1, S.d[S.cur_d ^ 1] + 4)), P, F),
        "cur_v 2": (G, edit(S, cur_v=2), P, F),
        "negative jacobi_iters": (G, S, edit(P, jacobi_iters=-1), F),
        "dt 0": (G, S, edit(P, dt=0.0), F),
        "unknown step_kernel": (G, S, edit(P, step_kernel=7), F),
        "misaligned frames": (G, S, P, F + 4),
    }
    ref = lambda x: C.byref(x) if x is not None else None
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for name, call in entries.items():
        for what, (g, st, prm, f) in bad.items():
            assert call(ref(g), ref(st), ref(prm), f) != 0, "%s accepted a call with %s" % (name, what)
            assert _lib.launch_count() == n0, "%s launched on a call with %s" % (name, what)
    for name, call in entries.items():
        assert call(ref(G), ref(S), ref(P), F) == 0, "%s: %s" % (name, lib.smk_last_error_string())
    torch.cuda.synchronize()
    assert _lib.launch_count() > n0
