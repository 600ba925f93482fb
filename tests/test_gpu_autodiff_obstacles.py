"""Reverse mode through solid obstacles on the GPU: autodiff.rollout(..., obstacles=) and the masked adjoint entries.

- Forward: rollout(obstacles=) is set_obstacles + run_steps bit for bit, with grad and without, with shared and per-simulation
  masks, sources, schedules, forcing and the fractal multiplier.
- Per entry: smk_project_adjoint_ex, smk_jacobi_adjoint_ex (every Jacobi tile configuration, sweeps per launch, sweep counts, 1 x 1
  to 1024^2, per-simulation masks) and smk_forces_diffuse_div_adjoint_ex against the float64 references of
  tests/obstacle_adjoint_reference.py, elementwise: |gpu - ref| <= 2 m 2^-24 |A|^T |g|, and exactly 0 where that bound is 0.
- Whole rollouts against fp32 CPU autograd of the masked torch restatement (tests/obstacle_torch.py).
- Exact zeros, the all-fluid mask, determinism, the example's fit, and rejections before any launch."""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
import torch

import obstacle_adjoint_reference as oar
import obstacle_oracle as O
import obstacle_torch as ot
from helpers import assert_same, nerr, smk_env
from oracle import torch_step as ts
from smokephysai_b200 import FractalGenerator, NavierStokesSimulator, _lib, autodiff
from smokephysai_b200.navier_stokes import FieldLayout
from test_gpu_adjoint_paths import check, dev, host, rel_l2, rnd

pytestmark = pytest.mark.gpu

DT, VISC = 0.01, 0.001
C_UV, C_D = ts.coefs(DT, VISC)
DEV = "cuda"


@pytest.fixture
def rec(record_property):
    worst = {}

    def put(what, ratio):
        worst[what] = max(worst.get(what, 0.0), ratio)
    yield put
    record_property("ratio", {k: float("%.3g" % v) for k, v in worst.items()})


def stream():
    return torch.cuda.current_stream().cuda_stream


def masks(B, h, w, seed, shared=False):
    """bool [B, h, w] (or [h, w] shared): random solids (about 15%), the demo box and wall where they fit, a solid ring cell."""
    rng = np.random.default_rng(seed)
    out = []
    for b in range(1 if shared else B):
        S = O.demo_mask(h, w) if h >= 40 and w >= 40 else np.zeros((h, w), bool)
        S |= rng.random((h, w)) < 0.15
        S[0, min(w - 1, b)] = True
        out.append(S)
    return out[0] if shared else np.stack(out)


def solid_buf(L, S):
    """uint8 [n, h, pitch_c] device copy of S, and the batch stride."""
    S = np.asarray(S)
    n = 1 if S.ndim == 2 else S.shape[0]
    buf = torch.zeros(n, L.h, L.pitch_c, dtype=torch.uint8, device=DEV)
    buf[:, :, :L.w] = torch.from_numpy(S.reshape(n, L.h, L.w).astype(np.uint8)).to(DEV)
    return buf, (0 if S.ndim == 2 else L.h * L.pitch_c)


# ------------------------------------------------------------------------------------------------------------- per entry
def jacobi_case(shape, B, K, T, rec, seed=1, shared=False):
    h, w = shape
    L = FieldLayout(h, w, B)
    S = masks(B, h, w, seed, shared)
    sb, ss = solid_buf(L, S)
    G = rnd((B, h, w), seed)
    gp, gdiv = (torch.zeros(B, h, L.pitch_c, device=DEV) for _ in range(2))
    ws = torch.empty(5 * B * L.stride_c + 4, device=DEV)
    Gt = dev(L, "p0", G)
    _lib.call("smk_jacobi_adjoint_ex", C.byref(L.grid_struct()), Gt.data_ptr(), gp.data_ptr(), gdiv.data_ptr(), K, T, ws.data_ptr(),
              sb.data_ptr(), ss, stream())
    St = torch.from_numpy(S)
    rp, rdiv = oar.jacobi_adjoint(G, St, K)
    bp, bdiv = oar.jacobi_adjoint(G, St, K, absolute=True)
    m = 5 * K + 4
    check("jacobi_obst g_p", host(L, "p0", gp), rp, bp, m, rec)
    check("jacobi_obst g_div", host(L, "p0", gdiv), rdiv, bdiv, m, rec)


JACOBI_SHAPES = [((1, 1), 1), ((2, 2), 1), ((3, 3), 2), ((7, 1), 1), ((5, 131), 2), ((33, 128), 3), ((128, 129), 2),
                 ((257, 383), 2), ((1030, 260), 1), ((1024, 1024), 1)]


@pytest.mark.parametrize("shape,B", JACOBI_SHAPES, ids=["%dx%dx%d" % (b, s[0], s[1]) for s, b in JACOBI_SHAPES])
def test_jacobi_adjoint_obst_shapes(shape, B, rec):
    jacobi_case(shape, B, 30, 0, rec)


TILES = [{}, {"SMK_JACOBI_TILE": 1}, {"SMK_JACOBI_TILE": 2}, {"SMK_JACOBI_TILE": 3}]
JACOBI_RUNS = [(env, T, K) for env in TILES for T in (0, 1, 5, 12, 24) for K in (0, 1, 2, 40, 100)]


@pytest.mark.parametrize("env,T,K", JACOBI_RUNS,
                         ids=["%s-T%d-K%d" % (",".join("tile=%s" % v for v in e.values()) or "auto", T, K) for e, T, K in JACOBI_RUNS])
def test_jacobi_adjoint_obst_paths(env, T, K, rec):
    """300 x 260 x 2 with per-simulation masks: both chains run on k_jacobi_obst over overlapped tiles, for K > T > 0 over several
    launches that end in different ping-pong buffers."""
    with smk_env(**env):
        jacobi_case((300, 260), 2, K, T, rec, seed=K + 7 * T)


def test_jacobi_adjoint_obst_shared_mask_many_simulations(rec):
    jacobi_case((128, 128), 40, 20, 5, rec, shared=True)


PROJ_SHAPES = [((1, 1), 1), ((3, 3), 2), ((1, 40), 2), ((40, 1), 1), ((129, 128), 3), ((300, 200), 2), ((1024, 1024), 1)]


@pytest.mark.parametrize("shape,B", PROJ_SHAPES, ids=["%dx%dx%d" % (b, s[0], s[1]) for s, b in PROJ_SHAPES])
def test_project_and_diffuse_adjoints_obst(shape, B, rec):
    h, w = shape
    L = FieldLayout(h, w, B)
    S = masks(B, h, w, h + w)
    sb, ss = solid_buf(L, S)
    St = torch.from_numpy(S)
    g = L.grid_struct()
    gu, gv, gp = rnd((B, h + 1, w), 1), rnd((B, h, w + 1), 2), rnd((B, h, w), 3)
    ins = [dev(L, "u0", gu), dev(L, "v0", gv), dev(L, "p0", gp)]
    out = torch.zeros(B, h, L.pitch_c, device=DEV)
    _lib.call("smk_project_adjoint_ex", C.byref(g), ins[0].data_ptr(), ins[1].data_ptr(), ins[2].data_ptr(), out.data_ptr(), DT,
              sb.data_ptr(), ss, stream())
    check("project_obst g_p", host(L, "p0", out), oar.project_adjoint(gu, gv, gp, St, DT),
          oar.project_adjoint(gu, gv, gp, St, DT, absolute=True), 6, rec)

    gs = [gu, gv, gp, rnd((B, h, w), 4)]
    ins = [dev(L, n, a) for n, a in zip(("u0", "v0", "d0", "p0"), gs)]
    outs = [torch.zeros(B, r, pch, device=DEV) for r, pch in ((h + 1, L.pitch_u), (h, L.pitch_v), (h, L.pitch_c))]
    _lib.call("smk_forces_diffuse_div_adjoint_ex", C.byref(g), *[t.data_ptr() for t in ins], *[t.data_ptr() for t in outs],
              DT, C_UV, C_D, sb.data_ptr(), ss, stream())
    ref = oar.forces_diffuse_div_adjoint(*gs, St, DT, C_UV, C_D)
    bnd = oar.forces_diffuse_div_adjoint(*gs, St, DT, C_UV, C_D, absolute=True)
    for name, t, r, b in zip(("g_u", "g_v", "g_d"), outs, ref, bnd):
        check("forces_diffuse_div_obst " + name, host(L, {"g_u": "u0", "g_v": "v0", "g_d": "d0"}[name], t), r, b, 16, rec)


def test_entries_reject_bad_masks_before_any_launch():
    h, w, B = 20, 24, 2
    L = FieldLayout(h, w, B)
    g = L.grid_struct()
    sb, _ = solid_buf(L, masks(B, h, w, 0))
    a = torch.zeros(B, h + 1, L.pitch_u, device=DEV)
    b = torch.zeros(B, h, L.pitch_v, device=DEV)
    c, d, e = (torch.zeros(B, h, L.pitch_c, device=DEV) for _ in range(3))
    ws = torch.empty(5 * B * L.stride_c + 4, device=DEV)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for ptr, ss in ((sb.data_ptr() + 1, 0), (sb.data_ptr(), 7), (sb.data_ptr(), L.h * L.pitch_c + 4), (None, L.h * L.pitch_c)):
        with pytest.raises(_lib.SmokeLibraryError):
            _lib.call("smk_project_adjoint_ex", C.byref(g), a.data_ptr(), b.data_ptr(), None, c.data_ptr(), DT, ptr, ss, stream())
        with pytest.raises(_lib.SmokeLibraryError):
            _lib.call("smk_jacobi_adjoint_ex", C.byref(g), c.data_ptr(), d.data_ptr(), e.data_ptr(), 5, 0, ws.data_ptr(), ptr, ss,
                      stream())
        with pytest.raises(_lib.SmokeLibraryError):
            _lib.call("smk_project_ex", C.byref(g), c.data_ptr(), a.data_ptr(), b.data_ptr(), DT, ptr, ss, stream())
    with pytest.raises(_lib.SmokeLibraryError):
        _lib.call("smk_obstacle_faces", C.byref(g), a.data_ptr(), b.data_ptr(), None, None, 0, DT, stream())
    with pytest.raises(_lib.SmokeLibraryError):
        _lib.call("smk_obstacle_cells", C.byref(g), c.data_ptr(), None, 0, 3, sb.data_ptr(), 0, stream())
    assert _lib.launch_count() == n0


# ------------------------------------------------------------------------------------------------------- rollouts
def state(B, h, w, seed, vel):
    rng = np.random.default_rng(seed)
    return [rnd((B, h + 1, w), seed, vel), rnd((B, h, w + 1), seed + 1, vel), rnd((B, h, w), seed + 2, 0.1),
            rng.random((B, h, w)).astype(np.float32)]


def reference_sim(B, h, w, K, s, S, spl=0, sources=None, inten=None, force=None, kernel="auto"):
    sim = NavierStokesSimulator((h, w), DT, VISC, DEV, jacobi_iters=K, batch=B, sweeps_per_launch=spl, step_kernel=kernel)
    for k, a in zip(("u", "v", "p", "density"), s):
        a = torch.as_tensor(a).to(DEV)
        setattr(sim, k, a if B > 1 else a[0])
    sim.set_obstacles(S)
    if sources:
        k = 0
        lists = []
        for lst in sources:
            lists.append([(x, y, r, float(inten[k + i])) for i, (x, y, r) in enumerate(lst)])
            k += len(lst)
        sim.set_continuous_sources(lists)
    return sim


def rollout_case(B, shape, T, K, S, record_property, *, vel=30.0, fractal=False, sources=None, force=False, spl=0, seed=1,
                 tol=1e-4):
    """autodiff.rollout(obstacles=S) against fp32 CPU autograd of ot.rollout; loss on frames and final state; the forward is
    set_obstacles + run_steps bit for bit.  -> the GPU gradients (u0, v0, p0, d0[, intensities][, du, dv])."""
    h, w = shape
    s = state(B, h, w, seed, vel)
    n = sum(len(l) for l in sources) if sources else 0
    inten = np.linspace(0.5, 1.5, max(n, 1)).astype(np.float32)[:n]
    F = [rnd((B, h + 1, w), seed + 20, 40.0), rnd((B, h, w + 1), seed + 21, 40.0)] if force else []
    wf = rnd((B, T, h, w), seed + 3)
    wst = [rnd(a.shape, seed + 4 + k) for k, a in enumerate(s)]
    fm = FractalGenerator(DEV).multiplier((h, w), 0.05) if fractal else None

    def loss(frames, final, to):
        return (frames * to(wf)).sum() + sum((a * to(wa)).sum() for a, wa in zip(final, wst))

    St = torch.from_numpy(np.asarray(S))
    lv = [torch.from_numpy(a).clone().requires_grad_(True) for a in s + ([inten] if n else []) + F]
    fr, fin = ot.rollout(tuple(lv[:4]), T, St, DT, VISC, K, fm[:, :w].cpu() if fractal else None,
                         sources=sources, intensities=lv[4] if n else None,
                         du=lv[-2] if force else None, dv=lv[-1] if force else None)
    loss(fr, fin, torch.from_numpy).backward()
    ref = [a.grad.numpy() if a.grad is not None else np.zeros(a.shape, np.float32) for a in lv]

    gv = [torch.from_numpy(a).to(DEV).requires_grad_(True) for a in s + ([inten] if n else []) + F]
    kw = dict(dt=DT, viscosity=VISC, jacobi_iters=K, add_fractal=fractal, sweeps_per_launch=spl, obstacles=S)
    if n:
        kw.update(sources=sources, intensities=gv[4])
    if force:
        kw.update(forcing=(gv[-2], gv[-1]))
    frames, final = autodiff.rollout(tuple(gv[:4]), T, **kw)
    sim = reference_sim(B, h, w, K, s, S, spl, sources, inten)
    want = sim.run_steps(T, fmul=fm, forcing=tuple(torch.from_numpy(a).to(DEV) for a in F) if force else None)
    assert_same(frames.detach().cpu().numpy().reshape(B, T, h, w), want.cpu().numpy().reshape(B, T, h, w), "frames")
    for name, got in zip(("u", "v", "p", "density"), final):
        assert_same(got.detach().cpu().numpy(), getattr(sim, name).cpu().numpy().reshape(got.shape), name)
    loss(frames, final, lambda a: torch.from_numpy(a).to(DEV)).backward()
    got = [a.grad.cpu().numpy() for a in gv]
    names = ["u0", "v0", "p0", "d0"] + (["intensities"] if n else []) + (["du", "dv"] if force else [])
    errs = {k: nerr(a, b) for k, a, b in zip(names, got, ref)}
    l2 = {k: rel_l2(a, b) for k, a, b in zip(names, got, ref)}
    record_property("nerr", errs)
    record_property("rel_l2", l2)
    print("rollout obst %dx%dx%d T=%d K=%d: nerr %s" % (B, h, w, T, K, {k: "%.2e" % e for k, e in errs.items()}))
    assert max(errs.values()) <= tol, errs
    assert max(l2.values()) <= tol, l2
    return got


@pytest.mark.parametrize("shared", [True, False], ids=["shared", "per_sim"])
def test_rollout_128_batch(shared, record_property):
    B, h, w = 4, 128, 128
    rollout_case(B, (h, w), 4, 40, masks(B, h, w, 3, shared), record_property, vel=100.0)


@pytest.mark.parametrize("spl", [0, 5])
def test_rollout_tiled_300x260(spl, record_property):
    rollout_case(2, (300, 260), 3, 24, masks(2, 300, 260, 5), record_property, vel=300.0, spl=spl)


def test_rollout_1024_demo_mask(record_property):
    """1024^2, K = 100, T = 2 with demo_mask, fractal frames."""
    rollout_case(1, (1024, 1024), 2, 100, O.demo_mask(1024, 1024), record_property, fractal=True)


@pytest.mark.parametrize("shape", [(3, 3), (1, 40)])
def test_rollout_degenerate_grids(shape, record_property):
    h, w = shape
    S = np.zeros((h, w), bool)
    S[h // 2, w // 2] = True
    rollout_case(2, shape, 3, 20, S, record_property, vel=100.0)


def test_rollout_sources_and_forcing_with_a_mask(record_property):
    B, h, w = 2, 96, 80
    rollout_case(B, (h, w), 4, 30, masks(B, h, w, 8), record_property, vel=50.0, force=True,
                 sources=[[(30, 20, 6), (60, 70, 5)], [(45, 40, 8)]])


def test_p0_gradient_is_exactly_zero_on_solid_cells(record_property):
    B, h, w = 2, 64, 72
    S = masks(B, h, w, 11)
    got = rollout_case(B, (h, w), 3, 20, S, record_property, vel=60.0)
    assert not got[2][S].any(), "g_p0 on solid cells"


def _grads(state_np, T, K, **kw):
    gv = [torch.from_numpy(a).to(DEV).requires_grad_(True) for a in state_np]
    frames, final = autodiff.rollout(tuple(gv), T, dt=DT, viscosity=VISC, jacobi_iters=K, **kw)
    (frames.square().sum() + sum(f.sum() for f in final)).backward()
    return [a.grad.cpu().numpy() for a in gv]


def test_all_fluid_mask_gives_the_unmasked_gradients():
    B, h, w = 2, 128, 128
    s = state(B, h, w, 4, 80.0)
    a = _grads(s, 5, 30, obstacles=np.zeros((h, w), bool))
    b = _grads(s, 5, 30)
    for x, y, name in zip(a, b, ("u0", "v0", "p0", "d0")):
        assert np.array_equal(x, y), name


def test_backward_is_deterministic():
    B, h, w = 2, 200, 170
    s = state(B, h, w, 6, 150.0)
    S = masks(B, h, w, 6)
    a = _grads(s, 4, 40, obstacles=S)
    b = _grads(s, 4, 40, obstacles=S)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


def test_forward_with_schedule_forcing_fractal_and_no_grad():
    """With grad and without: set_obstacles + run_steps(schedule=, forcing=) bit for bit, fractal frames."""
    B, h, w, T = 2, 128, 128, 5
    s = state(B, h, w, 2, 40.0)
    S = masks(B, h, w, 2)
    rng = np.random.default_rng(0)
    xy = rng.integers(10, 118, (T, B, 2, 2))
    radius = np.full((T, B, 2), 6, np.int32)
    I = torch.from_numpy(rng.uniform(0.5, 1.5, (T, B, 2)).astype(np.float32)).to(DEV)
    F = (torch.from_numpy(rnd((T, B, h + 1, w), 9, 30.0)).to(DEV), torch.from_numpy(rnd((T, B, h, w + 1), 10, 30.0)).to(DEV))
    fm = FractalGenerator(DEV).multiplier((h, w), 0.05)
    sim = reference_sim(B, h, w, 20, s, S)
    want = sim.run_steps(T, fmul=fm, schedule=(xy, radius, I.cpu().numpy()), forcing=F).cpu().numpy()
    for grad in (False, True):
        st = tuple(torch.from_numpy(a).to(DEV).requires_grad_(grad) for a in s)
        frames, final = autodiff.rollout(st, T, dt=DT, viscosity=VISC, jacobi_iters=20, add_fractal=True, schedule=(xy, radius),
                                         intensities=I, forcing=F, obstacles=torch.from_numpy(S).to(DEV))
        assert_same(frames.detach().cpu().numpy(), want, "frames, grad %s" % grad)
        for name, got in zip(("u", "v", "p", "density"), final):
            assert_same(got.detach().cpu().numpy(), getattr(sim, name).cpu().numpy(), "%s, grad %s" % (name, grad))


def test_rejections_before_any_launch():
    h = w = 32
    st = tuple(torch.zeros(s, device=DEV, requires_grad=True) for s in ((h + 1, w), (h, w + 1), (h, w), (h, w)))
    m = np.zeros((h, w), bool)
    m[5, 7] = True
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with pytest.raises(ValueError):
        autodiff.rollout(st, 3, obstacles=m, step_kernel="fused")
    for bad in (m.astype(np.float32), m[:-1], np.stack([m] * 2), m.astype(np.int8) * 3, m.tolist()):
        with pytest.raises(ValueError):
            autodiff.rollout(st, 3, obstacles=bad)
    assert _lib.launch_count() == n0


def test_example_fit_converges():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "examples", "inverse_obstacle.py")
    spec = importlib.util.spec_from_file_location("inverse_obstacle", path)
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    rate, losses, wall_effect = ex.fit()
    print("example: rate %.6f, losses %s, wall effect %.3f" % (rate, losses, wall_effect))
    assert wall_effect > 0.05, "the wall shapes the observed frames"
    assert abs(rate - 1.3) / 1.3 < 1e-3, rate
    assert losses[-1] < 1e-6 * losses[0]
