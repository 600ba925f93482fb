"""The adjoint entries of csrc/adjoint.cu on the paths the forward really takes.

Every phase adjoint is the transpose of a linear map A whose forward entry is bit-exact to the oracle, so each entry is checked
two ways, elementwise rather than against the global maximum:
  * transpose identity against its own forward kernel: |<A x, g> - <x, A^T g>| <= C m 2^-24 <|x|, |A|^T |g|>, both inner products
    in float64 from the two kernels' fp32 outputs;
  * against the float64 restatement of tests/adjoint_reference.py: |gpu - ref64| <= C m 2^-24 (|A|^T |g|) at every cell, and exactly
    0 where |A|^T |g| is 0 (the pressure ring of g_div, velocity gradients of clamped back-traces, cells no term reaches).
m is the number of roundings on the longest path of a cell (about 5K for K Jacobi sweeps).  Shapes run from 1 x 1 to 1500 x 1900
and batch strides at c2 size; the Jacobi adjoint runs through every forward Jacobi kernel (tile shapes, streaming kernels, packed
masks) with sweeps per launch and sweep counts that split its two chains over different numbers of launches.  Whole rollouts at
the sizes users run are compared with fp32 CPU autograd of oracle/torch_step.py.  The worst error-to-bound ratio of each case
goes to record_property("ratio").

Cost note: k_adv_adj_gather walks a (2 rx + 1) x (2 ry + 1) window per cell, rx / ry the largest back-trace reach anywhere, so
the back-traces that reach the clamps are kept to grids of at most 300 x 300 here."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import adjoint_reference as ar
import continuous_oracle
import oracle
from oracle import torch_step as ts
from helpers import assert_same, nerr, smk_env
from smokephysai_b200 import FractalGenerator, NavierStokesSimulator, _lib, autodiff
from smokephysai_b200.navier_stokes import FieldLayout

pytestmark = pytest.mark.gpu

DT, VISC = 0.01, 0.001
C_UV, C_D = ts.coefs(DT, VISC)
DEV = "cuda"
SLACK = 2.0                     # C of the bounds above


# ------------------------------------------------------------------------------------------------------------ helpers
def stream():
    return torch.cuda.current_stream().cuda_stream


def rnd(shape, seed, scale=1.0):
    return (np.random.default_rng(seed).standard_normal(shape) * scale).astype(np.float32)


def dev(L, name, a):
    """numpy / torch [B, rows, cols] -> zero-padded cuda [B, rows, pitch] (keep it referenced while a launch may read it)."""
    rows, cols, pitch = L.shape_of(name)
    t = torch.zeros(L.batch, rows, pitch, dtype=torch.float32, device=DEV)
    t[:, :, :cols] = torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    return t


def host(L, name, t):
    """padded cuda [B, rows, pitch] -> float64 CPU [B, rows, cols]"""
    return t[:, :, :L.shape_of(name)[1]].double().cpu()


def dot(a, b):
    return float((torch.as_tensor(a).double() * torch.as_tensor(b).double()).sum())


def seam_lines(n):
    """Indices on the outer two lines and next to the forward Jacobi's tile seams (row advances TH - 2t, column advances
    128 - 2 HX for the sweep counts per launch the tests use)."""
    out = {0, 1, n - 2, n - 1}
    for t in (1, 5, 8, 10, 12, 24):
        hx = (t + 3) & ~3
        for adv in (128 - 2 * t, 64 - 2 * t, 128 - 2 * hx):
            for k in range(adv, n, adv):
                out.update((k - 1, k, k + 1))
    return sorted(i for i in out if 0 <= i < n)


def g_field(kind, B, rows, cols, seed):
    g = rnd((B, rows, cols), seed)
    if kind == "seams":
        m = np.zeros((rows, cols), bool)
        m[seam_lines(rows), :] = True
        m[:, seam_lines(cols)] = True
        g = g * m
    return g


def check(what, got, ref, bound, m, record):
    """|got - ref| <= SLACK * m * 2^-24 * bound elementwise (m a scalar or per-cell tensor); exact 0 where bound is 0.
    -> the worst ratio of error to bound."""
    got, ref, bound = (torch.as_tensor(a).double() for a in (got, ref, bound))
    assert got.shape == ref.shape == bound.shape, (what, got.shape, ref.shape)
    tol = SLACK * torch.as_tensor(m, dtype=torch.float64) * ar.U * bound
    zero = bound == 0
    if bool(zero.any()):
        bad = zero & (got != 0)
        assert not bool(bad.any()), "%s: %d structurally zero cells are not 0, first at %s: %r" % (
            what, int(bad.sum()), tuple(torch.nonzero(bad)[0].tolist()), float(got[bad][0]))
    err = (got - ref).abs()
    ratio = float((err[~zero] / tol.expand_as(err)[~zero]).max()) if bool((~zero).any()) else 0.0
    record(what, ratio)
    if ratio > 1.0:
        k = tuple(torch.nonzero((err > tol) & ~zero)[0].tolist())
        raise AssertionError("%s: error / bound %.3g, first at %s: gpu %r, ref %r, bound %r" % (
            what, ratio, k, float(got[k]), float(ref[k]), float(tol.expand_as(err)[k])))
    return ratio


def identity(what, lhs, rhs, scale, m, record):
    tol = SLACK * m * ar.U * scale
    ratio = abs(lhs - rhs) / tol if tol > 0 else (0.0 if lhs == rhs else math.inf)
    record(what + " <Ax,g>", ratio)
    assert ratio <= 1.0, "%s: <Ax, g> = %r, <x, A^T g> = %r, bound %r" % (what, lhs, rhs, tol)


@pytest.fixture
def rec(record_property):
    worst = {}

    def put(what, ratio):
        worst[what] = max(worst.get(what, 0.0), ratio)
    yield put
    record_property("ratio", {k: float("%.3g" % v) for k, v in worst.items()})


SHAPES = [(1, 1), (1, 7), (7, 1), (2, 2), (3, 3), (2, 131), (5, 131), (131, 5), (33, 128), (127, 127), (128, 129), (129, 128),
          (257, 383), (300, 200), (1030, 260), (1500, 1900), (1024, 1024)]
CASES = [(s, b) for s in SHAPES for b in (1, 3) if b == 1 or s[0] * s[1] <= 300 * 383 or s == (1030, 260)] + \
        [((300, 260), 40), ((128, 128), 256)]
CASE_IDS = ["%dx%dx%d" % (b, s[0], s[1]) for s, b in CASES]


# --------------------------------------------------------------------------------------------------- Jacobi (a6)
def run_jacobi_adjoint(L, G, K, T):
    gp, gdiv = (torch.zeros(L.batch, L.h, L.pitch_c, device=DEV) for _ in range(2))
    ws = torch.empty(5 * L.batch * L.stride_c + 4, device=DEV)
    Gt = dev(L, "p0", G)
    _lib.call("smk_jacobi_adjoint", C.byref(L.grid_struct()), Gt.data_ptr(), gp.data_ptr(), gdiv.data_ptr(), K, T, ws.data_ptr(),
              stream())
    return host(L, "p0", gp), host(L, "p0", gdiv)


def run_jacobi(L, p, div, K, T):
    P, S, D = dev(L, "p0", p), torch.zeros(L.batch, L.h, L.pitch_c, device=DEV), dev(L, "p0", div)
    flag = C.c_int32(0)
    _lib.call("smk_jacobi", C.byref(L.grid_struct()), D.data_ptr(), P.data_ptr(), S.data_ptr(), K, T, C.byref(flag), stream())
    return host(L, "p0", S if flag.value else P)


def jacobi_case(shape, B, K, T, gkind, rec, seed=1):
    h, w = shape
    L = FieldLayout(h, w, B)
    G = g_field(gkind, B, h, w, seed)
    gp, gdiv = run_jacobi_adjoint(L, G, K, T)
    rp, rdiv = ar.jacobi_adjoint(G, K)
    bp, bdiv = ar.jacobi_adjoint(G, K, absolute=True)
    m = 5 * K + 4
    check("jacobi g_p", gp, rp, bp, m, rec)
    check("jacobi g_div", gdiv, rdiv, bdiv, m, rec)
    p, div = rnd((B, h, w), seed + 10), rnd((B, h, w), seed + 11)
    out = run_jacobi(L, p, div, K, T)
    identity("jacobi", dot(out, G), dot(p, gp) + dot(div, gdiv),
             dot(np.abs(p), bp) + dot(np.abs(div), bdiv), m, rec)


@pytest.mark.parametrize("gkind", ["dense", "seams"])
@pytest.mark.parametrize("shape,B", CASES, ids=CASE_IDS)
def test_jacobi_adjoint_shapes(shape, B, gkind, rec):
    jacobi_case(shape, B, 30, 0, gkind, rec)


JACOBI_PATHS = [{}, {"SMK_JACOBI_TILE": 1}, {"SMK_JACOBI_TILE": 2}, {"SMK_JACOBI_TILE": 3},
                {"SMK_JACOBI_STREAM": 1}, {"SMK_JACOBI_STREAM": 2}] + [{"SMK_JACOBI_PACKED": m} for m in (0, 2, 7, 9, 15, 16)]


def _k_list(T):
    return sorted({0, 1, 2, T, T + 1, 2 * T, 2 * T + 1, 100})


JACOBI_RUNS = [(env, T, K) for env in JACOBI_PATHS for T in ((0, 1, 5, 12, 24) if "SMK_JACOBI_PACKED" not in env else (0, 5))
               for K in _k_list(T)]


def _env_id(env):
    return ",".join("%s=%s" % (k[11:].lower(), v) for k, v in env.items()) or "auto"


@pytest.mark.parametrize("env,T,K", JACOBI_RUNS, ids=["%s-T%d-K%d" % (_env_id(e), T, K) for e, T, K in JACOBI_RUNS])
def test_jacobi_adjoint_paths(env, T, K, rec):
    """300 x 260 is beyond one tile, so both chains run on the overlapped-tile (or streaming) kernels and, for K > T > 0, over
    several launches that end in different ping-pong buffers."""
    with smk_env(**env):
        jacobi_case((300, 260), 2, K, T, "dense", rec, seed=K + 7 * T)


@pytest.mark.parametrize("env", [{"SMK_JACOBI_STREAM": 1}, {"SMK_JACOBI_STREAM": 2}, {}], ids=_env_id)
def test_jacobi_adjoint_streaming_crosses_simulations(env, rec):
    """40 x 300 x 260: the streaming kernels' flat tile index runs across simulation boundaries."""
    with smk_env(**env):
        jacobi_case((300, 260), 40, 25, 10, "dense", rec)


@pytest.mark.parametrize("packed", [0, 2, 6, 7, 9, 15, 16])
@pytest.mark.parametrize("shape", [(100, 120), (300, 260)], ids=["whole_tile", "overlapped"])
def test_jacobi_forward_bit_equal_to_oracle(packed, shape):
    h, w = shape
    B, K = 2, 23
    L = FieldLayout(h, w, B)
    p, div = rnd((B, h, w), 3, 0.1), rnd((B, h, w), 4)
    with smk_env(SMK_JACOBI_PACKED=packed):
        for T in (0, 5):
            got = run_jacobi(L, p, div, K, T).float().numpy()
            for b in range(B):
                assert_same(got[b], oracle.jacobi(p[b], div[b], K), "packed %d T %d sim %d" % (packed, T, b))


# ------------------------------------------------------------------------------------------- gradient subtract (a7)
@pytest.mark.parametrize("gkind", ["dense", "seams"])
@pytest.mark.parametrize("shape,B", CASES, ids=CASE_IDS)
def test_project_adjoint(shape, B, gkind, rec):
    h, w = shape
    L = FieldLayout(h, w, B)
    gu, gv, gp = g_field(gkind, B, h + 1, w, 1), g_field(gkind, B, h, w + 1, 2), g_field(gkind, B, h, w, 3)
    ins = [dev(L, "u0", gu), dev(L, "v0", gv), dev(L, "p0", gp)]
    out = torch.zeros(B, h, L.pitch_c, device=DEV)
    _lib.call("smk_project_adjoint", C.byref(L.grid_struct()), ins[0].data_ptr(), ins[1].data_ptr(), ins[2].data_ptr(), out.data_ptr(),
              DT, stream())
    got = host(L, "p0", out)
    bound = ar.project_adjoint(gu, gv, gp, DT, absolute=True)
    check("project g_p", got, ar.project_adjoint(gu, gv, gp, DT), bound, 6, rec)
    u, v, p = rnd((B, h + 1, w), 4), rnd((B, h, w + 1), 5), rnd((B, h, w), 6)
    U, V, P = dev(L, "u0", u), dev(L, "v0", v), dev(L, "p0", p)
    _lib.call("smk_project", C.byref(L.grid_struct()), P.data_ptr(), U.data_ptr(), V.data_ptr(), DT, stream())
    lhs = dot(host(L, "u0", U), gu) + dot(host(L, "v0", V), gv) + dot(p, gp)
    rhs = dot(u, gu) + dot(v, gv) + dot(p, got)
    scale = dot(np.abs(u), np.abs(gu)) + dot(np.abs(v), np.abs(gv)) + dot(np.abs(p), bound)
    identity("project", lhs, rhs, scale, 6, rec)


# ------------------------------------------------------------------------- buoyancy + diffusions + divergence (a3-a5)
@pytest.mark.parametrize("gkind", ["dense", "seams"])
@pytest.mark.parametrize("shape,B", CASES, ids=CASE_IDS)
def test_forces_diffuse_div_adjoint(shape, B, gkind, rec):
    h, w = shape
    L = FieldLayout(h, w, B)
    gs = [g_field(gkind, B, h + 1, w, 1), g_field(gkind, B, h, w + 1, 2), g_field(gkind, B, h, w, 3), g_field(gkind, B, h, w, 4)]
    ins = [dev(L, n, a) for n, a in zip(("u0", "v0", "d0", "p0"), gs)]
    outs = [torch.zeros(B, r, pch, device=DEV) for r, pch in ((h + 1, L.pitch_u), (h, L.pitch_v), (h, L.pitch_c))]
    _lib.call("smk_forces_diffuse_div_adjoint", C.byref(L.grid_struct()), *[t.data_ptr() for t in ins], *[t.data_ptr() for t in outs],
              DT, C_UV, C_D, stream())
    got = [host(L, n, t) for n, t in zip(("u0", "v0", "d0"), outs)]
    ref = ar.forces_diffuse_div_adjoint(*gs, DT, C_UV, C_D)
    bnd = ar.forces_diffuse_div_adjoint(*gs, DT, C_UV, C_D, absolute=True)
    for name, a, b, c in zip(("g_u", "g_v", "g_d"), got, ref, bnd):
        check("forces_diffuse_div " + name, a, b, c, 16, rec)
    x = [rnd((B, h + 1, w), 5), rnd((B, h, w + 1), 6), rnd((B, h, w), 7)]
    X = [dev(L, n, a) for n, a in zip(("u0", "v0", "d0"), x)]
    Y = [torch.zeros_like(t) for t in X] + [torch.zeros(B, h, L.pitch_c, device=DEV)]
    _lib.call("smk_forces_diffuse_div", C.byref(L.grid_struct()), *[t.data_ptr() for t in X], *[t.data_ptr() for t in Y], DT, C_UV, C_D,
              stream())
    lhs = sum(dot(host(L, n, t), g) for n, t, g in zip(("u0", "v0", "d0", "p0"), Y, gs))
    identity("forces_diffuse_div", lhs, sum(dot(a, b) for a, b in zip(x, got)), sum(dot(np.abs(a), b) for a, b in zip(x, bnd)), 16, rec)


# --------------------------------------------------------------------------------------------------- splat (a2)
def emitters_for(B, h, w, seed):
    rng = np.random.default_rng(seed)
    out = []
    for b in range(B):
        lst = []
        for _ in range(int(rng.integers(0, 4)) if b else 3):
            r = int(rng.integers(1, max(2, min(40, (h + w) // 4)) + 1))
            lst.append((int(rng.integers(-r // 2, w + r // 2)), int(rng.integers(-r // 2, h + r // 2)), r))
        out.append(lst)
    return out


def source_records(emitters, B, inten):
    rec_, off, n = autodiff._source_records(emitters, B, DEV)
    rec_.view(torch.float32)[:n, 3].copy_(torch.as_tensor(inten[:n]))
    return rec_, off, n


@pytest.mark.parametrize("gkind", ["dense", "seams"])
@pytest.mark.parametrize("shape,B", CASES, ids=CASE_IDS)
def test_splat_adjoint(shape, B, gkind, rec):
    h, w = shape
    L = FieldLayout(h, w, B)
    emitters = emitters_for(B, h, w, h * 7 + w)
    n = sum(len(l) for l in emitters)
    inten = np.linspace(-1.0, 2.0, max(n, 1)).astype(np.float32)
    R, off, _ = source_records(emitters, B, inten)
    G = g_field(gkind, B, h, w, 5)
    Gt = dev(L, "d0", G)
    gI = torch.zeros(max(n, 1), device=DEV)
    _lib.call("smk_splat_sources_adjoint", C.byref(L.grid_struct()), Gt.data_ptr(), R.data_ptr(), off.data_ptr(), n, gI.data_ptr(),
              stream())
    gacc = torch.ones(max(n, 1), device=DEV)
    _lib.call("smk_splat_sources_adjoint_ex", C.byref(L.grid_struct()), Gt.data_ptr(), R.data_ptr(), off.data_ptr(), n, 1,
              gacc.data_ptr(), stream())
    got = gI[:n].double().cpu()
    m = torch.from_numpy(np.ceil(ar.splat_footprint(h, w, emitters) / 256.0) + 12.0)
    bound = ar.splat_adjoint(G, emitters, absolute=True)
    check("splat g_intensity", got, ar.splat_adjoint(G, emitters), bound, m, rec)
    assert torch.equal(gacc[:n].cpu(), (gI[:n] + 1.0).cpu()), "accumulate adds the sum once"
    d = torch.zeros(B, h, L.pitch_c, device=DEV)
    _lib.call("smk_splat_sources", C.byref(L.grid_struct()), d.data_ptr(), R.data_ptr(), off.data_ptr(), stream())
    identity("splat", dot(host(L, "d0", d), G), dot(inten[:n], got), dot(np.abs(inten[:n]), bound), float(m.max()) if n else 1.0, rec)


# ---------------------------------------------------------------------------------------------------- advection (a10)
FIELD = {"d": "d0", "u": "u0", "v": "v0"}


def velocities(B, h, w, seed, vel, dyadic=False):
    if dyadic:
        rng = np.random.default_rng(seed)
        return (rng.integers(-2, 3, (B, h + 1, w)) * np.float32(vel)).astype(np.float32), \
               (rng.integers(-2, 3, (B, h, w + 1)) * np.float32(vel)).astype(np.float32)
    return rnd((B, h + 1, w), seed, vel), rnd((B, h, w + 1), seed + 1, vel)


def advect_case(shape, B, kind, vel, rec, *, gkind="dense", dt=DT, frame=False, fmul=False, accumulate=0, dyadic=False, seed=3):
    h, w = shape
    L = FieldLayout(h, w, B)
    g = L.grid_struct()
    name = FIELD[kind]
    rows, cols, pitch = L.shape_of(name)
    stride = L.stride_of(name)
    u, v = velocities(B, h, w, seed, vel, dyadic)
    field = rnd((B, rows, cols), seed + 2)
    gout = g_field(gkind, B, rows, cols, seed + 3)
    gfr = g_field(gkind, B, h, w, seed + 4) if frame else None
    fm = (np.random.default_rng(seed + 5).random((h, w)) * 0.05).astype(np.float32) if fmul else None
    scale = 0.995 if kind == "d" else 1.0
    Ut, Vt, Ft, Gt = dev(L, "u0", u), dev(L, "v0", v), dev(L, name, field), dev(L, name, gout)
    GFt = dev(L, "d0", gfr) if frame else None
    FMt = None
    if fmul:
        FMt = torch.zeros(h, L.pitch_c, device=DEV)
        FMt[:, :w] = torch.from_numpy(fm).to(DEV)
    init = [rnd((B, r, c), seed + 6 + k) if accumulate else np.zeros((B, r, c), np.float32)
            for k, (r, c) in enumerate(((rows, cols), (h + 1, w), (h, w + 1)))]
    gF, gU, gV = dev(L, name, init[0]), dev(L, "u0", init[1]), dev(L, "v0", init[2])
    ws = torch.empty(16 + 32 * B * (h + 1) * (w + 1), dtype=torch.uint8, device=DEV)
    _lib.call("smk_advect_adjoint", C.byref(g), Ft.data_ptr(), rows, cols, pitch, stride, Ut.data_ptr(), Vt.data_ptr(), dt, scale,
              Gt.data_ptr(), GFt.data_ptr() if frame else None, L.stride_c, FMt.data_ptr() if fmul else None,
              gF.data_ptr(), accumulate, gU.data_ptr(), gV.data_ptr(), ws.data_ptr(), stream())
    ut, vt = torch.from_numpy(u), torch.from_numpy(v)
    fmt = torch.from_numpy(fm) if fmul else None
    ref = ar.advect_adjoint(torch.from_numpy(field), ut, vt, dt, torch.from_numpy(gout), scale,
                            torch.from_numpy(gfr) if frame else None, fmt)
    bnd = ar.advect_adjoint(torch.from_numpy(field), ut, vt, dt, torch.from_numpy(gout), scale,
                            torch.from_numpy(gfr) if frame else None, fmt, absolute=True)
    count = ref[3]
    tag = "advect %s" % kind
    for what, got, r, b, m, i in (("g_field", host(L, name, gF), ref[0], bnd[0], count + 8, init[0]),
                                  ("g_u", host(L, "u0", gU), ref[1], bnd[1], 14, init[1]),
                                  ("g_v", host(L, "v0", gV), ref[2], bnd[2], 14, init[2])):
        if accumulate or what != "g_field":            # g_u / g_v always accumulate: a nonzero start adds one rounding
            got = got - torch.from_numpy(i).double()
            b = b + torch.from_numpy(np.abs(i)).double()
        check("%s %s" % (tag, what), got, r, b, m, rec)
    # the field part against the forward kernel
    out = torch.zeros(B, rows, pitch, device=DEV)
    fr = torch.zeros(B, h, L.pitch_c, device=DEV) if frame else None
    _lib.call("smk_advect", C.byref(g), Ft.data_ptr(), out.data_ptr(), rows, cols, pitch, stride, Ut.data_ptr(), Vt.data_ptr(), dt,
              scale, fr.data_ptr() if frame else None, L.stride_c, FMt.data_ptr() if fmul else None, stream())
    lhs = dot(host(L, name, out), gout) + (dot(host(L, "d0", fr), gfr) if frame else 0.0)
    got_f = host(L, name, gF) - (torch.from_numpy(init[0]).double() if accumulate else 0.0)
    identity(tag, lhs, dot(field, got_f), dot(np.abs(field), bnd[0]), float(count.max()) + 8, rec)
    return ref


@pytest.mark.parametrize("gkind", ["dense", "seams"])
@pytest.mark.parametrize("kind", ["d", "u", "v"])
@pytest.mark.parametrize("shape,B", CASES, ids=CASE_IDS)
def test_advect_adjoint_shapes(shape, B, kind, gkind, rec):
    """Back-traces of about 3 cells (|vel| ~ 300 at dt = 0.01)."""
    advect_case(shape, B, kind, 300.0, rec, gkind=gkind, frame=kind == "d", fmul=kind == "d")


VEL = {"rest": 0.0, "sub_cell": 30.0, "3_cell": 300.0, "12_cell": 1200.0, "clamped": 5000.0}


@pytest.mark.parametrize("accumulate", [0, 1])
@pytest.mark.parametrize("frame", ["none", "frame", "frame_fmul"])
@pytest.mark.parametrize("kind", ["d", "u", "v"])
@pytest.mark.parametrize("motion", list(VEL))
def test_advect_adjoint_cases(motion, kind, frame, accumulate, rec):
    if kind != "d" and frame != "none":
        pytest.skip("the frame and its fractal multiply belong to the density advection")
    shape = (150, 130) if motion == "clamped" else (129, 200)
    advect_case(shape, 2, kind, VEL[motion], rec, frame=frame != "none", fmul=frame == "frame_fmul", accumulate=accumulate)


@pytest.mark.parametrize("kind", ["d", "u", "v"])
@pytest.mark.parametrize("shape", [(33, 47), (40, 40), (7, 9)])
def test_advect_adjoint_dyadic(shape, kind, rec):
    """dt = 2^-6 and velocities in multiples of 2^7: every back-trace lands exactly on an integer, many exactly on 0 or xmax,
    where the clamp still passes the gradient and half of the corner weights are exactly zero."""
    h, w = shape
    ref = advect_case(shape, 2, kind, 128.0, rec, dt=2.0 ** -6, dyadic=True, frame=kind == "d", fmul=kind == "d")
    u, v = velocities(2, h, w, 3, 128.0, dyadic=True)
    rows, cols, _ = FieldLayout(h, w, 2).shape_of(FIELD[kind])
    px, py = ar.back_trace(rows, cols, torch.from_numpy(u), torch.from_numpy(v), 2.0 ** -6)
    assert torch.all(px == torch.round(px)) and torch.all(py == torch.round(py))
    Y, X = ar._mesh(rows, cols, torch.float32)
    for p, P, n in ((px, X, cols), (py, Y, rows)):        # on the clamp bounds by motion, not by a zero velocity on the edge
        assert bool(((p == 0) & (P > 0)).any()) and bool(((p == n - 1) & (P < n - 1)).any())
    assert bool((ref[1] != 0).any()) and bool((ref[2] != 0).any())


# ------------------------------------------------------------------------------------------------------ whole rollouts
def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    n = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / (n if n > 0 else 1.0))


def rollout_case(B, shape, T, K, record_property, *, vel=30.0, fractal=False, emitters=None, continuous=None, step_kernel="auto",
                 spl=0, seed=1):
    """autodiff.rollout against fp32 CPU autograd of the restated step, loss on the frames and the final state; the forward is
    bit-equal to run_steps.  emitters: one-shot add_sources before the rollout; continuous: emitters at every step."""
    h, w = shape
    rng = np.random.default_rng(seed)
    s = [rnd((B, h + 1, w), seed, vel), rnd((B, h, w + 1), seed + 1, vel), rnd((B, h, w), seed + 2, 0.1),
         rng.random((B, h, w)).astype(np.float32)]
    em = emitters or continuous
    n = sum(len(l) for l in em) if em else 0
    inten = np.linspace(0.5, 1.5, max(n, 1)).astype(np.float32)[:n]
    wf = rnd((B, T, h, w), seed + 3)
    wst = [rnd(a.shape, seed + 4 + k) for k, a in enumerate(s)]
    fmul = FractalGenerator(DEV).multiplier((h, w), 0.05)[:, :w].cpu() if fractal else None

    def loss(frames, final, to):
        return (frames * to(wf)).sum() + sum((a * to(wa)).sum() for a, wa in zip(final, wst))

    lv = [torch.from_numpy(a).clone().requires_grad_(True) for a in s + [inten]]
    d0 = ts.add_sources(lv[3], emitters, lv[4]) if emitters else lv[3]
    if continuous:
        frames, final = continuous_oracle.rollout((lv[0], lv[1], lv[2], d0), T, DT, VISC, K, fmul, continuous, lv[4])
    else:
        frames, final = ts.rollout((lv[0], lv[1], lv[2], d0), T, DT, VISC, K, fmul=fmul)
    loss(frames, final, torch.from_numpy).backward()
    ref = [a.grad.numpy() if a.grad is not None else np.zeros_like(a.detach().numpy()) for a in lv]

    gv = [torch.from_numpy(a).to(DEV).requires_grad_(True) for a in s + [inten]]
    d0 = autodiff.add_sources(gv[3], emitters, gv[4]) if emitters else gv[3]
    kw = dict(dt=DT, viscosity=VISC, jacobi_iters=K, add_fractal=fractal, step_kernel=step_kernel, sweeps_per_launch=spl)
    if continuous:
        kw.update(sources=continuous, intensities=gv[4])
    frames, final = autodiff.rollout((gv[0], gv[1], gv[2], d0), T, **kw)
    # the forward is run_steps bit for bit
    sim = NavierStokesSimulator((h, w), DT, VISC, DEV, jacobi_iters=K, batch=B, sweeps_per_launch=spl, step_kernel=step_kernel)
    for k, a in zip(("u", "v", "p", "density"), (gv[0], gv[1], gv[2], d0)):
        setattr(sim, k, (a if B > 1 else a[0]).detach().clone())
    if continuous:
        sim.set_continuous_sources([[(x, y, r, float(inten[i])) for i, (x, y, r) in
                                     enumerate(lst, sum(len(l) for l in continuous[:b]))] for b, lst in enumerate(continuous)])
    want = sim.run_steps(T, fmul=FractalGenerator(DEV).multiplier((h, w), 0.05) if fractal else None)
    assert_same(frames.detach().cpu().numpy().reshape(B, T, h, w), want.cpu().numpy().reshape(B, T, h, w), "frames")
    for name, got in zip(("u", "v", "p", "density"), final):
        assert_same(got.detach().cpu().numpy(), getattr(sim, name).cpu().numpy().reshape(got.shape), name)
    loss(frames, final, lambda a: torch.from_numpy(a).to(DEV)).backward()
    names = ("u0", "v0", "p0", "d0", "intensities")[:5 if n else 4]
    got = [a.grad.cpu().numpy() for a in gv[:len(names)]]
    errs = {k: nerr(a, b) for k, a, b in zip(names, got, ref)}
    l2 = {k: rel_l2(a, b) for k, a, b in zip(names, got, ref)}
    record_property("nerr", errs)
    record_property("rel_l2", l2)
    print("rollout %dx%dx%d T=%d K=%d: nerr %s rel_l2 %s" % (B, h, w, T, K, {k: "%.2e" % e for k, e in errs.items()},
                                                           {k: "%.2e" % e for k, e in l2.items()}))
    assert max(errs.values()) <= 1e-4, errs
    assert max(l2.values()) <= 1e-4, l2


def test_rollout_1024_benchmark_shape(record_property):
    """The autodiff benchmark's shape: 1024^2, K = 100, T = 2, emitters, fractal, loss on frames and final state."""
    rollout_case(1, (1024, 1024), 2, 100, record_property, fractal=True,
                 emitters=[[(512, 300, 8), (700, 520, 8), (300, 700, 12)]])


@pytest.mark.parametrize("spl", [0, 5])
def test_rollout_tiled_300x260(spl, record_property):
    """300 x 260: tiled advection, fused gradient subtract and overlapped Jacobi tiles; back-traces of about 3 cells."""
    rollout_case(2, (300, 260), 3, 24, record_property, vel=300.0, spl=spl, emitters=[[(100, 80, 8)], [(200, 150, 10)]])


@pytest.mark.parametrize("B", [1, 48])
def test_rollout_continuous_sources_auto_kernel(B, record_property):
    """128^2, step_kernel auto, continuous sources: B = 1 steps on k_step_cluster, B = 48 on k_step_fused."""
    cont = [[(40 + b % 7, 50, 8), (90, 80 - b % 5, 6)] for b in range(B)]
    rollout_case(B, (128, 128), 4, 40, record_property, continuous=cont)


@pytest.mark.parametrize("shape", [(3, 3), (1, 40)])
def test_rollout_degenerate_grids(shape, record_property):
    rollout_case(2, shape, 3, 20, record_property, vel=100.0)
