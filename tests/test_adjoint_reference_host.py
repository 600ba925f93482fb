"""CPU checks of the float64 adjoint references (tests/adjoint_reference.py), no GPU: every helper is the transpose of the matching
forward of oracle/torch_step.py run in float64, <A x, g> = <x, A^T g> to about 1e-12; its absolute twin bounds it elementwise; and
the advection transpose equals float64 autograd through the advection at the same fixed fp32 back-trace."""
import numpy as np
import pytest
import torch

import adjoint_reference as ar
import continuous_oracle
import oracle
from oracle import torch_step as ts
from helpers import assert_same

DT, VISC = 0.01, 0.001
SHAPES = [(1, 1), (1, 7), (7, 1), (2, 2), (3, 3), (5, 13), (37, 53)]


def rnd(shape, seed, scale=1.0):
    return torch.from_numpy(np.random.default_rng(seed).standard_normal(shape) * scale)


def dot(a, b):
    return float((a.double() * b.double()).sum())


def close(lhs, rhs, scale):
    assert abs(lhs - rhs) <= 1e-12 * scale, (lhs, rhs, scale)


def dominated(ref, bound):
    """|A^T g| <= |A|^T |g| everywhere (with a float64 rounding margin)."""
    assert torch.all(ref.abs() <= bound * (1 + 1e-12) + 1e-300)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("K", [0, 1, 2, 7])
def test_jacobi_transpose(shape, K):
    h, w = shape
    p, div, g = rnd((2, h, w), 1), rnd((2, h, w), 2), rnd((2, h, w), 3)
    gp, gdiv = ar.jacobi_adjoint(g, K)
    assert ts.jacobi(p, div, K).shape == p.shape
    close(dot(ts.jacobi(p, div, K), g), dot(p, gp) + dot(div, gdiv), dot(p.abs(), gp.abs()) + dot(div.abs(), gdiv.abs()) + 1.0)
    bp, bdiv = ar.jacobi_adjoint(g, K, absolute=True)
    dominated(gp, bp)
    dominated(gdiv, bdiv)
    if h <= 2 or w <= 2:                          # no interior: p passes through K = 0 only, the divergence never acts
        assert torch.all(gdiv == 0)
    # against float64 autograd of the restated sweeps
    P, D = p.clone().requires_grad_(True), div.clone().requires_grad_(True)
    (ts.jacobi(P, D, K) * g).sum().backward()
    assert torch.allclose(gp, P.grad, rtol=1e-12, atol=1e-14)
    assert torch.allclose(gdiv, D.grad if D.grad is not None else torch.zeros_like(div), rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize("shape", SHAPES)
def test_project_transpose(shape):
    h, w = shape
    u, v, p = rnd((2, h + 1, w), 1), rnd((2, h, w + 1), 2), rnd((2, h, w), 3)
    gu, gv, gp = rnd((2, h + 1, w), 4), rnd((2, h, w + 1), 5), rnd((2, h, w), 6)
    gP = ar.project_adjoint(gu, gv, gp, DT)
    u2, v2 = ts.grad_subtract(u, v, p, ar.f32(DT))
    lhs = dot(u2, gu) + dot(v2, gv) + dot(p, gp)
    close(lhs, dot(u, gu) + dot(v, gv) + dot(p, gP), 10.0 * u.numel())
    dominated(gP, ar.project_adjoint(gu, gv, gp, DT, absolute=True))


@pytest.mark.parametrize("shape", SHAPES)
def test_forces_diffuse_div_transpose(shape):
    h, w = shape
    c_uv, c_d = ts.coefs(DT, VISC)
    x = [rnd((2, h + 1, w), 1), rnd((2, h, w + 1), 2), rnd((2, h, w), 3)]
    g = [rnd((2, h + 1, w), 4), rnd((2, h, w + 1), 5), rnd((2, h, w), 6), rnd((2, h, w), 7)]
    gx = ar.forces_diffuse_div_adjoint(*g, DT, c_uv, c_d)
    outs = ar._forces_diffuse_div(*x, ar.f32(DT), ar.f32(c_uv), ar.f32(c_d), False)
    scale = sum(dot(a.abs(), b.abs()) for a, b in zip(x, gx)) + 1.0
    close(sum(dot(o, gg) for o, gg in zip(outs, g)), sum(dot(a, b) for a, b in zip(x, gx)), scale)
    for a, b in zip(gx, ar.forces_diffuse_div_adjoint(*g, DT, c_uv, c_d, absolute=True)):
        dominated(a, b)
    # the restated step's own forces + diffusions (Python-double constants) give the same transpose to fp32 rounding
    X = [a.clone().requires_grad_(True) for a in x]
    u2, v2, d2 = ts.forces_diffuse(*X, DT, VISC)
    sum((o * gg).sum() for o, gg in zip((u2, v2, d2, ts.divergence(u2, v2, DT)), g)).backward()
    for a, b in zip(gx, X):
        assert torch.allclose(a, b.grad, rtol=1e-6, atol=1e-6 * float(b.grad.abs().max()))


def test_splat_transpose():
    h, w = 37, 53
    emitters = [[(10, 12, 8), (14, 15, 5), (50, 2, 9)], [], [(30, 30, 6), (0, 0, 1)]]
    g = rnd((3, h, w), 8)
    I = torch.tensor([1.25, 0.5, 2.0, 0.75, -1.5], dtype=torch.float64)
    gI = ar.splat_adjoint(g, emitters)
    weight64 = lambda *a: ts.splat_weight(*a).double()      # a 0-dim intensity would not promote an fp32 footprint
    lhs = dot(continuous_oracle.add_sources(torch.zeros(3, h, w, dtype=torch.float64), emitters, I, weight64), g)
    close(lhs, dot(I, gI), dot(I.abs(), gI.abs()) + 1.0)
    dominated(gI, ar.splat_adjoint(g, emitters, absolute=True))
    assert list(ar.splat_footprint(h, w, emitters)) == [17 * 17, 11 * 11, 12 * 12, 13 * 13, 2 * 2]


def _velocity(B, h, w, seed, vel):
    return (torch.from_numpy((np.random.default_rng(seed).standard_normal((B, h + 1, w)) * vel).astype(np.float32)),
            torch.from_numpy((np.random.default_rng(seed + 1).standard_normal((B, h, w + 1)) * vel).astype(np.float32)))


def _autograd_advect(field, u, v, dt, e):
    """float64 autograd through ts.advection_step with the back-trace pinned to its fp32 value: the position carries the fp32
    value forward and the float64 derivative backward (the advection's velocity part is linear once the back-trace is fixed)."""
    B, rows, cols = field.shape
    px32, py32 = ar.back_trace(rows, cols, u, v, ar.f32(dt))
    F, U, V = (a.double().clone().requires_grad_(True) for a in (field, u, v))
    Y, X = ar._mesh(rows, cols, torch.float64)
    px = X - ar.f32(dt) * ts.interpolate_velocity_u(U, Y, X)
    py = Y - ar.f32(dt) * ts.interpolate_velocity_v(V, Y, X)
    px = px + (px32.double() - px).detach()
    py = py + (py32.double() - py).detach()
    out = ts.bilinear_interpolate(F, torch.clamp(py, 0, rows - 1), torch.clamp(px, 0, cols - 1))
    (out * e).sum().backward()
    return F.grad, U.grad, V.grad


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("kind", ["d", "u", "v"])
@pytest.mark.parametrize("vel", [0.0, 40.0, 300.0, 2000.0])
def test_advect_transpose_and_autograd(shape, kind, vel):
    h, w = shape
    B = 2
    u, v = _velocity(B, h, w, 3, vel)
    rows, cols = {"d": (h, w), "u": (h + 1, w), "v": (h, w + 1)}[kind]
    field = torch.from_numpy(np.random.default_rng(5).standard_normal((B, rows, cols)).astype(np.float32))
    g = rnd((B, rows, cols), 6)
    gf, gu, gv, count = ar.advect_adjoint(field, u, v, DT, g)
    out, _ = ar.advect_forward(field, u, v, DT)
    close(dot(out, g), dot(field, gf), dot(field.abs(), gf.abs()) + 1.0)
    assert float(count.sum()) == 4 * B * rows * cols
    want = _autograd_advect(field, u, v, DT, g)
    for got, ref in zip((gf, gu, gv), want):
        assert torch.allclose(got, ref, rtol=1e-12, atol=1e-12 * float(ref.abs().max() + 1))
    bf, bu, bv, _ = ar.advect_adjoint(field, u, v, DT, g, absolute=True)
    for a, b in zip((gf, gu, gv), (bf, bu, bv)):
        dominated(a, b)


def test_advect_frame_and_fmul():
    h, w, B = 9, 9, 2
    u, v = _velocity(B, h, w, 8, 150.0)
    field = torch.from_numpy(np.random.default_rng(1).random((B, h, w)).astype(np.float32))
    g, gfr = rnd((B, h, w), 2), rnd((B, h, w), 3)
    fmul = torch.from_numpy((np.random.default_rng(4).random((h, w)) * 0.05).astype(np.float32))
    gf, _, _, _ = ar.advect_adjoint(field, u, v, DT, g, scale=0.995, g_frame=gfr, fmul=fmul)
    out, frame = ar.advect_forward(field, u, v, DT, scale=0.995, fmul=fmul)
    close(dot(out, g) + dot(frame, gfr), dot(field, gf), dot(field.abs(), gf.abs()) + 1.0)


def test_advect_dyadic_back_traces_hit_integers_and_the_clamp_bounds():
    """dt = 2^-6 and velocities k * 2^7: every back-trace is an exact integer, some exactly 0 or xmax (the clamp passes there)."""
    h, w, B = 6, 7, 1
    dt = 2.0 ** -6
    rng = np.random.default_rng(0)
    u = torch.from_numpy((rng.integers(-3, 4, (B, h + 1, w)) * 128.0).astype(np.float32))
    v = torch.from_numpy((rng.integers(-3, 4, (B, h, w + 1)) * 128.0).astype(np.float32))
    px, py = ar.back_trace(h, w, u, v, dt)
    assert torch.all(px == torch.round(px)) and torch.all(py == torch.round(py))
    assert bool(((px == 0) | (px == w - 1)).any()) and bool(((py == 0) | (py == h - 1)).any())
    field = torch.from_numpy(rng.standard_normal((B, h, w)).astype(np.float32))
    g = rnd((B, h, w), 1)
    gf, gu, gv, _ = ar.advect_adjoint(field, u, v, dt, g)
    want = _autograd_advect(field, u, v, dt, g)
    for got, ref in zip((gf, gu, gv), want):
        assert torch.allclose(got, ref, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("shape", [(1, 40), (40, 1), (2, 5), (3, 3)])
def test_restatement_forward_on_degenerate_grids_bit_equal_to_c_oracle(shape):
    """Grids without a Jacobi interior: the restated sweeps keep the pressure's shape and zero it, as the reference does."""
    h, w = shape
    rng = np.random.default_rng(2)
    f = lambda *s: (rng.standard_normal(s) * 100.0).astype(np.float32)
    state = [f(2, h + 1, w), f(2, h, w + 1), f(2, h, w), np.abs(f(2, h, w))]
    ref = [a.copy() for a in state]
    frames_ref = oracle.run_batch(*ref, DT, VISC, 20, 3)
    with torch.no_grad():
        frames, final = ts.rollout(tuple(torch.from_numpy(a) for a in state), 3, DT, VISC, 20)
    assert_same(frames.numpy(), frames_ref, "frames")
    for name, got, want in zip("uvpd", final, ref):
        assert_same(got.numpy(), want, name)
