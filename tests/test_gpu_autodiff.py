"""Reverse mode on the GPU (smokephysai_b200.autodiff, csrc/adjoint.cu): the checkpointed forward is bit-equal to run_steps,
every adjoint entry matches torch autograd of the matching function of oracle/torch_step.py (fp32, CPU), whole rollouts match
autograd of the restated step, gradients are bitwise repeatable, and an inverse problem converges."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import torch_step as ts
from helpers import assert_same, nerr
from smokephysai_b200 import FractalGenerator, NavierStokesSimulator, _lib, autodiff
from smokephysai_b200.navier_stokes import FieldLayout

pytestmark = pytest.mark.gpu

DT, VISC = 0.01, 0.001
DEV = "cuda"


def state_np(B, h, w, seed, vel):
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    return [f(B, h + 1, w) * np.float32(vel), f(B, h, w + 1) * np.float32(vel), f(B, h, w) * np.float32(0.1),
            rng.random((B, h, w)).astype(np.float32)]


def rnd(shape, seed):
    return np.random.default_rng(seed).standard_normal(shape).astype(np.float32)


def staged(L, name, a):
    """numpy [B, rows, cols] -> zero-padded cuda [B, rows, pitch].  Keep the result referenced while a launch may read it:
    a temporary's memory goes back to torch's caching allocator (and to the next allocation) as soon as it is dropped."""
    rows, cols, pitch = L.shape_of(name)
    t = torch.zeros(L.batch, rows, pitch, dtype=torch.float32, device=DEV)
    t[:, :, :cols] = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t


def unstaged(L, name, t):
    return t[:, :, :L.shape_of(name)[1]].cpu().numpy()


def leaves(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).clone().requires_grad_(True) for a in arrays]


def stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("B", [None, 3])
@pytest.mark.parametrize("kernel", ["phases", "fused"])
@pytest.mark.parametrize("fractal", [False, True])
@pytest.mark.parametrize("grad", [True, False])
def test_rollout_forward_bit_equal_to_run_steps(B, kernel, fractal, grad):
    n, T = 64, 6
    s = state_np(B or 1, n, n, 3, 60.0)
    sim = NavierStokesSimulator((n, n), DT, VISC, DEV, batch=B or 1, step_kernel=kernel)
    for k, a in zip(("u", "v", "p", "density"), s):
        setattr(sim, k, torch.from_numpy(a if B else a[0]).to(DEV))
    fmul = FractalGenerator(DEV).multiplier((n, n), 0.05) if fractal else None
    want = sim.run_steps(T, fmul=fmul)
    state = [torch.from_numpy(a if B else a[0]).to(DEV).requires_grad_(grad) for a in s]
    frames, final = autodiff.rollout(tuple(state), T, dt=DT, viscosity=VISC, add_fractal=fractal, step_kernel=kernel)
    assert frames.requires_grad == grad
    assert_same(frames.detach().cpu().numpy(), want.cpu().numpy(), "frames")
    for name, got in zip(("u", "v", "p", "density"), final):
        assert_same(got.detach().cpu().numpy(), getattr(sim, name).cpu().numpy(), name)


def test_add_sources_forward_bit_equal_to_add_smoke_source():
    sim = NavierStokesSimulator((48, 40), DT, VISC, DEV, batch=2)
    emitters = [[(10, 12, 8), (14, 15, 5)], [(30, 30, 6)]]
    inten = [1.25, 0.5, 2.0]
    sim.add_sources([[(10, 12, 8, inten[0]), (14, 15, 5, inten[1])], [(30, 30, 6, inten[2])]])
    d0 = torch.zeros(2, 48, 40, device=DEV)
    got = autodiff.add_sources(d0, emitters, torch.tensor(inten, device=DEV))
    assert_same(got.cpu().numpy(), sim.density.cpu().numpy(), "density")


# ---------------------------------------------------------------------------------------------------------- per phase
SHAPES = [(128, 128), (37, 53)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("vel", [0.0, 150.0])
@pytest.mark.parametrize("which", ["d", "v_alias", "u_alias", "d_accumulate"])
def test_advect_adjoint_matches_autograd(shape, vel, which, record_property):
    h, w = shape
    B = 2
    u, v, _, d = state_np(B, h, w, 17, vel)
    L = FieldLayout(h, w, B)
    g = L.grid_struct()
    gout_name = {"d": "d0", "d_accumulate": "d0", "v_alias": "v0", "u_alias": "u0"}[which]
    rows, cols, pitch = L.shape_of(gout_name)
    G = rnd((B, rows, cols), 5)
    U, V, D = leaves(u, v, d)
    gu = torch.zeros(B, h + 1, L.pitch_u, device=DEV)
    gv = torch.zeros(B, h, L.pitch_v, device=DEV)
    ws = torch.empty(16 + 32 * B * (h + 1) * (w + 1), dtype=torch.uint8, device=DEV)
    Ut, Vt = staged(L, "u0", u), staged(L, "v0", v)
    gout = staged(L, gout_name, G)
    if which in ("d", "d_accumulate"):
        GF = rnd((B, h, w), 6)
        fmul = torch.from_numpy((np.random.default_rng(2).random((h, w)) * 0.05).astype(np.float32))
        out = ts.advection_step(D, U, V, DT) * 0.995
        frame = out + fmul * out
        ((out * torch.from_numpy(G)).sum() + (frame * torch.from_numpy(GF)).sum()).backward()
        gd = torch.ones(B, h, L.pitch_c, device=DEV) if which == "d_accumulate" else torch.zeros(B, h, L.pitch_c, device=DEV)
        fm = torch.zeros(h, L.pitch_c, device=DEV)
        fm[:, :w] = fmul.to(DEV)
        Dt, GFt = staged(L, "d0", d), staged(L, "d0", GF)
        _lib.call("smk_advect_adjoint", C.byref(g), Dt.data_ptr(), h, w, L.pitch_c, L.stride_c, Ut.data_ptr(),
                  Vt.data_ptr(), DT, 0.995, gout.data_ptr(), GFt.data_ptr(), L.stride_c, fm.data_ptr(),
                  gd.data_ptr(), int(which == "d_accumulate"), gu.data_ptr(), gv.data_ptr(), ws.data_ptr(), stream())
        want_d = D.grad.numpy() + (1.0 if which == "d_accumulate" else 0.0)
        errs = {"d": nerr(unstaged(L, "d0", gd), want_d)}
    elif which == "v_alias":                                # v advects v: g_field is g_v
        (ts.advection_step(V, U, V, DT) * torch.from_numpy(G)).sum().backward()
        _lib.call("smk_advect_adjoint", C.byref(g), Vt.data_ptr(), h, w + 1, L.pitch_v, L.stride_v, Ut.data_ptr(), Vt.data_ptr(),
                  DT, 1.0, gout.data_ptr(), None, 0, None, gv.data_ptr(), 0, gu.data_ptr(), gv.data_ptr(), ws.data_ptr(), stream())
        errs = {}
    else:                                                   # u advects u by u: g_field is g_u, g_out aliases it too
        (ts.advection_step(U, U, V, DT) * torch.from_numpy(G)).sum().backward()
        errs = {}
        gu.copy_(gout)
        _lib.call("smk_advect_adjoint", C.byref(g), Ut.data_ptr(), h + 1, w, L.pitch_u, L.stride_u, Ut.data_ptr(), Vt.data_ptr(),
                  DT, 1.0, gu.data_ptr(), None, 0, None, gu.data_ptr(), 0, gu.data_ptr(), gv.data_ptr(), ws.data_ptr(), stream())
    errs["u"] = nerr(unstaged(L, "u0", gu), U.grad.numpy())
    errs["v"] = nerr(unstaged(L, "v0", gv), V.grad.numpy())
    record_property("nerr", errs)
    print("advect adjoint %s %s vel %g: %s" % (which, shape, vel, errs))
    assert max(errs.values()) <= 1e-5, errs


@pytest.mark.parametrize("shape", SHAPES)
def test_project_adjoint_matches_autograd(shape):
    h, w = shape
    B = 2
    u, v, p, _ = state_np(B, h, w, 4, 1.0)
    L = FieldLayout(h, w, B)
    U, V, P = leaves(u, v, p)
    gu_np, gv_np, gp_np = rnd((B, h + 1, w), 1), rnd((B, h, w + 1), 2), rnd((B, h, w), 3)
    u2, v2 = ts.grad_subtract(U, V, P, DT)
    ((u2 * torch.from_numpy(gu_np)).sum() + (v2 * torch.from_numpy(gv_np)).sum() + (P * torch.from_numpy(gp_np)).sum()).backward()
    out = torch.zeros(B, h, L.pitch_c, device=DEV)
    gut, gvt, gpt = staged(L, "u0", gu_np), staged(L, "v0", gv_np), staged(L, "p0", gp_np)
    _lib.call("smk_project_adjoint", C.byref(L.grid_struct()), gut.data_ptr(), gvt.data_ptr(), gpt.data_ptr(), out.data_ptr(), DT,
              stream())
    assert nerr(unstaged(L, "p0", out), P.grad.numpy()) <= 1e-5
    assert nerr(gu_np, U.grad.numpy()) == 0 and nerr(gv_np, V.grad.numpy()) == 0     # u, v gradients pass through


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("K", [0, 1, 2, 20, 40])
def test_jacobi_adjoint_matches_autograd(shape, K):
    h, w = shape
    B = 2
    L = FieldLayout(h, w, B)
    p, div, G = rnd((B, h, w), 1), rnd((B, h, w), 2), rnd((B, h, w), 3)
    P, DV = leaves(p, div)
    (ts.jacobi(P, DV, K) * torch.from_numpy(G)).sum().backward()
    gp, gdiv = torch.zeros(B, h, L.pitch_c, device=DEV), torch.zeros(B, h, L.pitch_c, device=DEV)
    ws = torch.empty(5 * B * L.stride_c, device=DEV)
    Gt = staged(L, "p0", G)
    _lib.call("smk_jacobi_adjoint", C.byref(L.grid_struct()), Gt.data_ptr(), gp.data_ptr(), gdiv.data_ptr(), K, 0,
              ws.data_ptr(), stream())
    want_div = DV.grad.numpy() if DV.grad is not None else np.zeros_like(div)
    assert nerr(unstaged(L, "p0", gp), P.grad.numpy()) <= 1e-5
    assert nerr(unstaged(L, "p0", gdiv), want_div) <= 1e-5


@pytest.mark.parametrize("shape", SHAPES)
def test_forces_diffuse_div_adjoint_matches_autograd(shape):
    h, w = shape
    B = 2
    u, v, _, d = state_np(B, h, w, 9, 1.0)
    L = FieldLayout(h, w, B)
    U, V, D = leaves(u, v, d)
    gu, gv, gd, gdv = rnd((B, h + 1, w), 1), rnd((B, h, w + 1), 2), rnd((B, h, w), 3), rnd((B, h, w), 4)
    u2, v2, d2 = ts.forces_diffuse(U, V, D, DT, VISC)
    div = ts.divergence(u2, v2, DT)
    T = torch.from_numpy
    ((u2 * T(gu)).sum() + (v2 * T(gv)).sum() + (d2 * T(gd)).sum() + (div * T(gdv)).sum()).backward()
    ou, ov, od = (torch.zeros(B, r, pch, device=DEV) for r, pch in ((h + 1, L.pitch_u), (h, L.pitch_v), (h, L.pitch_c)))
    c_uv, c_d = ts.coefs(DT, VISC)
    ins = [staged(L, "u0", gu), staged(L, "v0", gv), staged(L, "d0", gd), staged(L, "p0", gdv)]     # kept alive over the call
    _lib.call("smk_forces_diffuse_div_adjoint", C.byref(L.grid_struct()), *[t.data_ptr() for t in ins], ou.data_ptr(), ov.data_ptr(),
              od.data_ptr(),
              DT, c_uv, c_d, stream())
    for name, got, want in (("u0", ou, U.grad), ("v0", ov, V.grad), ("d0", od, D.grad)):
        assert nerr(unstaged(L, name, got), want.numpy()) <= 1e-5, name


def test_splat_adjoint_matches_autograd():
    h, w = 37, 53
    emitters = [[(10, 12, 8), (14, 15, 5), (50, 2, 9)], [], [(30, 30, 6)]]
    inten = np.array([1.25, 0.5, 2.0, 0.75], np.float32)
    G = rnd((3, h, w), 8)
    I = torch.from_numpy(inten).clone().requires_grad_(True)
    (ts.add_sources(torch.zeros(3, h, w), emitters, I) * torch.from_numpy(G)).sum().backward()
    Ig = torch.from_numpy(inten).to(DEV).requires_grad_(True)
    d0 = torch.zeros(3, h, w, device=DEV, requires_grad=True)
    (autodiff.add_sources(d0, emitters, Ig) * torch.from_numpy(G).to(DEV)).sum().backward()
    assert nerr(Ig.grad.cpu().numpy(), I.grad.numpy()) <= 1e-5
    assert_same(d0.grad.cpu().numpy(), G, "d0 gradient passes through")


# ------------------------------------------------------------------------------------------------------ whole rollouts
def _rollout_grads(B, n, T, K, fractal, loss_kind, seed=1, vel=30.0):
    s = state_np(B, n, n, seed, vel)
    emitters = [[(n // 2 + b, n // 3, 6), (n // 4, n // 2, 5)] for b in range(B)]
    inten = np.linspace(0.5, 1.5, 2 * B).astype(np.float32)
    wf = rnd((B, T, n, n), seed + 1)
    wst = [rnd(a.shape, seed + 2 + k) for k, a in enumerate(s)]
    fmul = FractalGenerator(DEV).multiplier((n, n), 0.05)[:, :n].cpu() if fractal else None

    def loss(frames, final, to):
        l = 0.0
        if loss_kind in ("frames", "both"):
            l = l + (frames * to(wf)).sum()
        if loss_kind in ("final", "both"):
            l = l + sum((a * to(wa)).sum() for a, wa in zip(final, wst))
        return l

    # restated step, fp32 on the CPU
    ref_leaves = leaves(*s, inten)
    d_src = ts.add_sources(ref_leaves[3], emitters, ref_leaves[4])
    frames, final = ts.rollout((ref_leaves[0], ref_leaves[1], ref_leaves[2], d_src), T, DT, VISC, K, fmul=fmul)
    loss(frames, final, torch.from_numpy).backward()
    ref = [a.grad.numpy() for a in ref_leaves]

    def ours():
        lv = [torch.from_numpy(a).to(DEV).requires_grad_(True) for a in list(s) + [inten]]
        d = autodiff.add_sources(lv[3], emitters, lv[4])
        frames, final = autodiff.rollout((lv[0], lv[1], lv[2], d), T, dt=DT, viscosity=VISC, jacobi_iters=K, add_fractal=fractal)
        loss(frames, final, lambda a: torch.from_numpy(a).to(DEV)).backward()
        return [a.grad.cpu().numpy() for a in lv]
    return ours, ref


@pytest.mark.parametrize("T", [1, 5, 20])
@pytest.mark.parametrize("K", [0, 1, 20, 40])
def test_rollout_gradients_match_restatement(T, K, record_property):
    ours, ref = _rollout_grads(3, 32, T, K, fractal=(T == 5), loss_kind="both")
    got = ours()
    errs = {name: nerr(a, b) for name, a, b in zip(("u0", "v0", "p0", "d0", "intensities"), got, ref)}
    record_property("nerr", errs)
    print("rollout T=%d K=%d: %s" % (T, K, {k: "%.2e" % e for k, e in errs.items()}))
    assert max(errs.values()) <= 1e-4, errs


@pytest.mark.parametrize("loss_kind", ["frames", "final", "both"])
@pytest.mark.parametrize("fractal", [False, True])
def test_rollout_gradients_loss_kinds(loss_kind, fractal, record_property):
    ours, ref = _rollout_grads(3, 48, 5, 20, fractal, loss_kind, seed=7, vel=60.0)
    got = ours()
    errs = {name: nerr(a, b) for name, a, b in zip(("u0", "v0", "p0", "d0", "intensities"), got, ref)}
    record_property("nerr", errs)
    print("rollout loss=%s fractal=%s: %s" % (loss_kind, fractal, {k: "%.2e" % e for k, e in errs.items()}))
    assert max(errs.values()) <= 1e-4, errs


def test_rollout_gradients_2d_and_ragged():
    h, w, T = 37, 53, 4
    s = [a[0] for a in state_np(1, h, w, 12, 100.0)]
    wf = rnd((T, h, w), 3)
    lv = leaves(*s)
    frames, _ = ts.rollout(tuple(lv), T, DT, VISC, 20)
    (frames * torch.from_numpy(wf)).sum().backward()
    lg = [torch.from_numpy(a).to(DEV).requires_grad_(True) for a in s]
    frames, _ = autodiff.rollout(tuple(lg), T)
    assert frames.shape == (T, h, w)
    (frames * torch.from_numpy(wf).to(DEV)).sum().backward()
    for name, a, b in zip("uvpd", lg, lv):
        assert a.grad.shape == b.grad.shape
        assert nerr(a.grad.cpu().numpy(), b.grad.numpy()) <= 1e-4, name


def test_backward_is_deterministic():
    ours, _ = _rollout_grads(2, 64, 5, 20, fractal=True, loss_kind="both", seed=4, vel=150.0)
    a, b = ours(), ours()
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


def test_inverse_problem_recovers_intensities():
    n, T = 64, 10
    emitters = [(20, 24, 8), (40, 30, 8), (30, 44, 6)]
    true = torch.tensor([1.5, 0.7, 1.1], device=DEV)
    z = lambda *s: torch.zeros(*s, device=DEV)
    state = (z(n + 1, n), z(n, n + 1), z(n, n))
    with torch.no_grad():
        target, _ = autodiff.rollout(state + (autodiff.add_sources(z(n, n), emitters, true),), T)
    x = torch.ones(3, device=DEV, requires_grad=True)
    opt = torch.optim.LBFGS([x], lr=1.0, max_iter=100, tolerance_grad=1e-12, tolerance_change=1e-14,
                            line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        frames, _ = autodiff.rollout(state + (autodiff.add_sources(z(n, n), emitters, x),), T)
        loss = ((frames - target) ** 2).sum()
        loss.backward()
        return loss
    for _ in range(3):
        opt.step(closure)
    rel = ((x.detach() - true).abs() / true).max().item()
    print("inverse problem: recovered %s, true %s, max relative error %.2e" % (x.detach().tolist(), true.tolist(), rel))
    assert rel < 1e-3


# ---------------------------------------------------------------------------------------------------------- rejections
def test_rejections():
    n = 16
    ok = [torch.zeros(n + 1, n, device=DEV), torch.zeros(n, n + 1, device=DEV), torch.zeros(n, n, device=DEV),
          torch.zeros(n, n, device=DEV)]
    bad_dtype = list(ok); bad_dtype[3] = ok[3].double()
    bad_dev = list(ok); bad_dev[0] = ok[0].cpu()
    bad_shape = list(ok); bad_shape[1] = torch.zeros(n, n, device=DEV)
    bad_batch = [t.unsqueeze(0).expand(2, *t.shape).contiguous() for t in ok]; bad_batch[2] = bad_batch[2][:1]
    mixed_dims = list(ok); mixed_dims[3] = ok[3].unsqueeze(0)
    for st in (bad_dtype, bad_dev, bad_shape, bad_batch, mixed_dims):
        with pytest.raises(ValueError):
            autodiff.rollout(tuple(st), 2)
    with pytest.raises(ValueError):
        autodiff.add_sources(ok[3], [(4, 4, 3)], torch.ones(2, device=DEV))
    with pytest.raises(ValueError):
        autodiff.add_sources(ok[3], [(4, 4, 3)], torch.ones(1, dtype=torch.float64, device=DEV))
    with pytest.raises(RuntimeError):            # the fractal multiplier needs a square grid, as in the reference
        autodiff.rollout((torch.zeros(9, 12, device=DEV), torch.zeros(8, 13, device=DEV), torch.zeros(8, 12, device=DEV),
                          torch.zeros(8, 12, device=DEV)), 1, add_fractal=True)
    # slab grids are refused by every adjoint entry
    L = FieldLayout(n, n, 1, row0=0, gh=2 * n)
    buf = torch.zeros(4 * n * n, device=DEV)
    with pytest.raises(_lib.SmokeLibraryError, match="slab"):
        _lib.call("smk_project_adjoint", C.byref(L.grid_struct()), buf.data_ptr(), buf.data_ptr(), None, buf[8:].data_ptr(), DT,
                  stream())
    with pytest.raises(_lib.SmokeLibraryError, match="slab"):
        _lib.call("smk_jacobi_adjoint", C.byref(L.grid_struct()), buf.data_ptr(), buf[8:].data_ptr(), buf[16:].data_ptr(), 0, 0,
                  None, stream())
    # double backward
    lv = [t.clone().requires_grad_(True) for t in ok]
    lv3 = lv[3] + 1.0
    frames, _ = autodiff.rollout((lv[0], lv[1], lv[2], lv3), 2)
    with pytest.raises(RuntimeError, match="first-order gradients only"):
        torch.autograd.grad(frames.sum(), lv[3], create_graph=True)
    d = autodiff.add_sources(lv[3], [(4, 4, 3)], torch.ones(1, device=DEV, requires_grad=True))
    with pytest.raises(RuntimeError, match="first-order gradients only"):
        torch.autograd.grad(d.sum(), lv[3], create_graph=True)
