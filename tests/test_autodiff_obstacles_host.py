"""CPU checks of reverse mode through solid obstacles (no GPU): the torch restatement of the masked step (tests/obstacle_torch.py)
is bit-equal to the C oracle's smk_oracle_step_obst, so autograd through it is the gradient oracle; the float64 references of the
masked adjoint entries (tests/obstacle_adjoint_reference.py) are transposes of their forward maps and the masked Jacobi one equals
explicit (J^T)^K; and the new ABI entries are declared, exported and bound."""
import re
import subprocess

import numpy as np
import pytest
import torch

import adjoint_reference as ar
import obstacle_adjoint_reference as oar
import obstacle_oracle as O
import obstacle_torch as ot
from oracle import torch_step as ts

DT, VISC = 0.01, 0.001
C_UV, C_D = ts.coefs(DT, VISC)


def _state(h, w, seed, vel=60.0):
    rng = np.random.default_rng(seed)
    return [(rng.standard_normal((h + 1, w)) * vel).astype(np.float32), (rng.standard_normal((h, w + 1)) * vel).astype(np.float32),
            (rng.standard_normal((h, w)) * 0.1).astype(np.float32), rng.random((h, w)).astype(np.float32)]


def _mask(h, w, kind, seed=0):
    if kind == "demo":
        return O.demo_mask(h, w)
    S = np.random.default_rng(seed).random((h, w)) < 0.2
    if kind == "ring":
        S[0, :] = S[-1, :] = True
    return S


FWD_CASES = [((24, 24), "random"), ((17, 29), "random"), ((1, 40), "random"), ((3, 3), "random"), ((17, 29), "ring"),
             ((64, 64), "demo"), ((70, 48), "demo")]


@pytest.mark.parametrize("K", [0, 1, 20])
@pytest.mark.parametrize("hw,kind", FWD_CASES, ids=["%dx%d-%s" % (hw + (k,)) for hw, k in FWD_CASES])
def test_torch_restatement_bit_equal_to_c_oracle(hw, kind, K):
    h, w = hw
    S = _mask(h, w, kind, seed=h * w + K)
    a = _state(h, w, K + 3)
    b = [torch.from_numpy(x.copy()) for x in a]
    St = torch.from_numpy(S)
    for t in range(4):
        fa, _ = O.step_obst(*a, S, DT, VISC, K)
        fb, b = ot.step(*b, St, DT, VISC, K)
        np.testing.assert_array_equal(fb.numpy(), fa, err_msg="frame %d" % t)
    for x, y, name in zip(a, b, "uvpd"):
        np.testing.assert_array_equal(y.numpy(), x, err_msg=name)


def test_all_fluid_mask_is_the_unmasked_restatement():
    h, w = 20, 23
    s = [torch.from_numpy(x) for x in _state(h, w, 5)]
    fa, a = ot.step(*s, torch.zeros(h, w, dtype=torch.bool), DT, VISC, 20)
    fb, b = ts.step(*s, DT, VISC, 20)
    assert torch.equal(fa, fb) and all(torch.equal(x, y) for x, y in zip(a, b))


# ------------------------------------------------------------------------------------------------ float64 references
def _rnd(shape, seed):
    return torch.from_numpy(np.random.default_rng(seed).standard_normal(shape))


MASKS = [("random", 9, 11), ("ring", 12, 7), ("demo", 64, 48), ("box", 9, 9), ("single", 3, 3), ("strip", 1, 12)]


def _ref_mask(kind, h, w, B):
    if kind == "box":
        S = np.zeros((h, w), bool)
        S[3:6, 3:6] = True
        S[3:6, 4] = [True, False, True]
    elif kind == "single":
        S = np.zeros((h, w), bool)
        S[1, 1] = True
    elif kind == "strip":
        S = np.zeros((h, w), bool)
        S[0, 3:5] = True
    else:
        S = np.stack([_mask(h, w, kind, seed=b) for b in range(B)])
    return torch.from_numpy(S)


def _dot(a, b):
    return float((a * b).sum())


@pytest.mark.parametrize("kind,h,w", MASKS)
@pytest.mark.parametrize("K", [0, 1, 2, 5, 13])
def test_jacobi_reference_is_the_transpose(kind, h, w, K):
    B = 2
    S = _ref_mask(kind, h, w, B)
    g = _rnd((B, h, w), K)
    gp, gdiv = oar.jacobi_adjoint(g, S, K)
    p, div = _rnd((B, h, w), K + 1), _rnd((B, h, w), K + 2)
    Sb = S.expand(B, h, w)
    lhs = _dot(ot.jacobi(p, div, Sb, K), g)
    assert abs(lhs - (_dot(p, gp) + _dot(div, gdiv))) <= 1e-12 * max(1.0, abs(lhs))
    bp, bdiv = oar.jacobi_adjoint(g, S, K, absolute=True)
    assert torch.all(bp >= gp.abs() - 1e-12) and torch.all(bdiv >= gdiv.abs() - 1e-12)
    assert not bool(gp[Sb].any()) or K == 0, "solid cells get exactly 0"
    if K >= 1:
        assert not bool(gdiv[Sb].any())
    if h * w <= 200:                                        # against the explicit matrix
        for b in range(B):
            J = oar.jacobi_matrix(Sb[b])
            keep = (~Sb[b]).clone()
            keep[0, :] = keep[-1, :] = False
            keep[:, 0] = keep[:, -1] = False
            M = torch.diag(keep.reshape(-1).double())
            gb = g[b].reshape(-1)
            want_p = torch.linalg.matrix_power(J.T, K) @ gb
            want_div = -0.25 * M @ sum((torch.linalg.matrix_power(J.T, j) @ gb for j in range(K)), torch.zeros_like(gb))
            assert torch.allclose(gp[b].reshape(-1), want_p, atol=1e-12, rtol=0)
            assert torch.allclose(gdiv[b].reshape(-1), want_div, atol=1e-12, rtol=0)


def test_jacobi_matrix_is_symmetric_on_the_fluid_interior():
    """The fact the reverse rests on: M J^T M = M J M for every mask (DESIGN.md s5.7)."""
    for seed in range(20):
        rng = np.random.default_rng(seed)
        h, w = (int(x) for x in rng.integers(3, 10, 2))
        S = torch.from_numpy(rng.random((h, w)) < 0.3)
        J = oar.jacobi_matrix(S)
        keep = (~S).clone()
        keep[0, :] = keep[-1, :] = False
        keep[:, 0] = keep[:, -1] = False
        M = torch.diag(keep.reshape(-1).double())
        assert torch.equal(M @ J.T @ M, M @ J @ M)


@pytest.mark.parametrize("kind,h,w", MASKS)
def test_project_reference_is_the_transpose(kind, h, w):
    B = 2
    S = _ref_mask(kind, h, w, B)
    gu, gv, gp = _rnd((B, h + 1, w), 1), _rnd((B, h, w + 1), 2), _rnd((B, h, w), 3)
    got = oar.project_adjoint(gu, gv, gp, S, DT)
    u, v, p = _rnd((B, h + 1, w), 4), _rnd((B, h, w + 1), 5), _rnd((B, h, w), 6)
    u2, v2 = ot.grad_subtract(u, v, p, S.expand(B, h, w), ar.f32(DT))
    lhs = _dot(u2, gu) + _dot(v2, gv) + _dot(p, gp)
    rhs = _dot(u, gu) + _dot(v, gv) + _dot(p, got)
    assert abs(lhs - rhs) <= 1e-12 * max(1.0, abs(lhs))
    bound = oar.project_adjoint(gu, gv, gp, S, DT, absolute=True)
    assert torch.all(bound >= got.abs() - 1e-12)


@pytest.mark.parametrize("kind,h,w", MASKS)
def test_forces_diffuse_div_reference_is_the_transpose(kind, h, w):
    B = 2
    S = _ref_mask(kind, h, w, B)
    gs = [_rnd((B, h + 1, w), 1), _rnd((B, h, w + 1), 2), _rnd((B, h, w), 3), _rnd((B, h, w), 4)]
    got = oar.forces_diffuse_div_adjoint(*gs, S, DT, C_UV, C_D)
    x = [_rnd((B, h + 1, w), 5), _rnd((B, h, w + 1), 6), _rnd((B, h, w), 7)]
    outs = oar.forces_diffuse_div(*x, S, ar.f32(DT), ar.f32(C_UV), ar.f32(C_D))
    lhs = sum(_dot(a, b) for a, b in zip(outs, gs))
    rhs = sum(_dot(a, b) for a, b in zip(x, got))
    assert abs(lhs - rhs) <= 1e-12 * max(1.0, abs(lhs))
    bnd = oar.forces_diffuse_div_adjoint(*gs, S, DT, C_UV, C_D, absolute=True)
    for a, b in zip(got, bnd):
        assert torch.all(b >= a.abs() - 1e-12)


# ---------------------------------------------------------------------------------------------------------- the ABI
NEW = {"smk_project_ex": 8, "smk_obstacle_faces": 8, "smk_obstacle_cells": 8, "smk_project_adjoint_ex": 9,
       "smk_jacobi_adjoint_ex": 10, "smk_forces_diffuse_div_adjoint_ex": 14}


def test_new_entries_are_declared_exported_and_bound():
    from smokephysai_b200 import _lib, build
    so = build.build()
    syms = subprocess.check_output(["nm", "-D", "--defined-only", so]).decode()
    header = open(build.os.path.join(build.HERE, "..", "include", "smoke_b200.h")).read()
    for name, n in NEW.items():
        assert re.search(r" T %s\b" % name, syms), name
        m = re.search(r"SMK_API int %s\(([^;]*)\);" % name, header)
        assert m and len(m.group(1).split(",")) == n, name
        assert len(_lib.SIGNATURES[name]) == n, name
    # each _ex adjoint is its entry with (solid, solid_batch_stride) before the stream
    for base in ("smk_project_adjoint", "smk_jacobi_adjoint", "smk_forces_diffuse_div_adjoint", "smk_project"):
        a, b = list(_lib.SIGNATURES[base]), list(_lib.SIGNATURES[base + "_ex"])
        assert b[:-3] + b[-1:] == a and b[-3:-1] == [_lib.c_p, _lib.c_i64], base
    assert int(re.search(r"#define SMK_ABI_VERSION (\d+)", header).group(1)) == 7

