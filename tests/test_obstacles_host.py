"""CPU checks of solid obstacles (no GPU): the obstacle oracle (tests/obstacle_oracle.c) against the reference oracle with an
all-fluid mask and against its numpy restatement, the invariants after every step, the projection's physics (divergence,
enclosed pockets), the mask validation, and the new ABI entries declared, exported and bound."""
import re
import subprocess

import numpy as np
import pytest
import torch

import oracle
import obstacle_oracle as O

DT, VISC = 0.01, 0.001
SHAPES = [(24, 24), (17, 29), (1, 40)]


def _state(h, w, seed):
    rng = np.random.default_rng(seed)
    u = rng.standard_normal((h + 1, w)).astype(np.float32)
    v = rng.standard_normal((h, w + 1)).astype(np.float32)
    p = np.zeros((h, w), np.float32)
    d = np.zeros((h, w), np.float32)
    oracle.splat(d, w // 2, h // 2, max(1, min(h, w) // 3), 1.5)
    return u, v, p, d


def _random_mask(h, w, seed, frac=0.15):
    return np.random.default_rng(seed).random((h, w)) < frac


def _invariants(u, v, p, d, S, K):
    cu, cv = O.faces(S)
    for name, f, c in (("u", u, cu), ("v", v, cv)):
        assert not np.signbit(f[c]).any() and not f[c].any(), name + ": a closed face is not +0"
    S = np.asarray(S)
    assert not np.signbit(d[S]).any() and not d[S].any(), "solid density is not +0"
    if K >= 1:
        assert not np.signbit(p[S]).any() and not p[S].any(), "solid pressure is not +0"


@pytest.mark.parametrize("hw", SHAPES)
def test_all_fluid_mask_is_the_reference_step(hw):
    h, w = hw
    a = list(_state(h, w, 1))
    b = [x.copy() for x in a]
    S = np.zeros((h, w), bool)
    for _ in range(4):
        fa, _ = O.step_obst(*a, S, DT, VISC, 20)
        fb, _ = O.step_obst(*b, None, DT, VISC, 20)
        assert fa.tobytes() == fb.tobytes()
    for x, y, name in zip(a, b, "uvpd"):
        assert x.tobytes() == y.tobytes(), name


@pytest.mark.parametrize("hw", SHAPES + [(64, 64)])
@pytest.mark.parametrize("K", [0, 1, 20])
def test_numpy_restatement_equals_c_oracle(hw, K):
    h, w = hw
    S = O.demo_mask(h, w) if h >= 40 else _random_mask(h, w, h * w)
    a = list(_state(h, w, 2))
    b = tuple(x.copy() for x in a)
    for _ in range(3):
        O.step_obst(*a, S, DT, VISC, K)
        b = O.np_step_obst(*b, S, DT, VISC, K)
    for x, y, name in zip(a, b, "uvpd"):
        np.testing.assert_array_equal(x, y, err_msg=name)
    # the Jacobi sweeps alone, on a random pressure and divergence
    rng = np.random.default_rng(K)
    P, D = rng.standard_normal((2, h, w)).astype(np.float32)
    np.testing.assert_array_equal(O.jacobi_obst(P, D, S, K), O.np_jacobi_obst(P, D, S, K))


@pytest.mark.parametrize("hw", SHAPES + [(64, 48)])
@pytest.mark.parametrize("K", [0, 3, 20])
def test_invariants_after_every_step(hw, K):
    h, w = hw
    S = O.demo_mask(h, w) if h >= 40 else _random_mask(h, w, 7 + h)
    S[0, 0] = S[-1, -1] = True                          # solids on the ring too
    u, v, p, d = _state(h, w, 3)
    d += np.float32(0.5)                               # smoke everywhere, inside the solids too, before the first step
    for _ in range(5):
        fr, _ = O.step_obst(u, v, p, d, S, DT, VISC, K)
        _invariants(u, v, p, d, S, K)
        assert not np.signbit(fr[S]).any() and not fr[S].any()


@pytest.mark.parametrize("hw", [(64, 64), (96, 80)])
def test_projection_removes_divergence_around_walls(hw):
    """The box, the partial wall and the single cell: after K = 1000 masked sweeps the gradient subtract leaves an interior-fluid
    divergence more than 100x below K = 0, and exactly 0 on solid cells."""
    h, w = hw
    S = O.demo_mask(h, w)
    cu, cv = O.faces(S)
    rng = np.random.default_rng(0)
    U = np.where(cu, 0, rng.standard_normal((h + 1, w))).astype(np.float32)
    V = np.where(cv, 0, rng.standard_normal((h, w + 1))).astype(np.float32)
    D = O.np_div(U, V, DT)
    fl = O.interior_fluid(S)
    res = {}
    for K in (0, 1000):
        P = O.jacobi_obst(np.zeros((h, w), np.float32), D, S, K)
        g = (P[1:] - P[:-1]) * np.float32(DT)
        U2 = U.copy()
        U2[1:-1] = np.where(cu[1:-1], U2[1:-1], U2[1:-1] - g)
        g = (P[:, 1:] - P[:, :-1]) * np.float32(DT)
        V2 = V.copy()
        V2[:, 1:-1] = np.where(cv[:, 1:-1], V2[:, 1:-1], V2[:, 1:-1] - g)
        div = O.np_div(U2, V2, 1.0)
        res[K] = np.abs(div[fl]).max()
        assert not div[S].any()
    assert res[1000] * 100 < res[0], res


@pytest.mark.parametrize("shape", ["pocket", "wall_row"])
def test_enclosed_fluid_keeps_pressure_bounded(shape):
    """A fluid pocket cut off from the ring has a singular Laplacian; its divergence sums to 0 (all its boundary faces are
    closed), so p stays finite and bounded as K grows."""
    h = w = 48
    S = np.zeros((h, w), bool)
    if shape == "pocket":
        S[10:28, 10:28] = True
        S[11:27, 11:27] = False                        # a 16 x 16 fluid pocket inside a closed box
    else:
        S[h // 2, :] = True                            # a full-width wall row splits the box in two
    u, v, p, d = _state(h, w, 5)
    cu, cv = O.faces(S)
    u[cu] = 0
    v[cv] = 0
    D = O.np_div(u, v, DT)
    peaks = []
    for K in (100, 1000, 4000):
        P = O.jacobi_obst(np.zeros((h, w), np.float32), D, S, K)
        assert np.isfinite(P).all()
        peaks.append(float(np.abs(P).max()))
    assert max(peaks) < 2 * min(peaks), peaks
    # and the whole step keeps it finite
    for _ in range(3):
        O.step_obst(u, v, p, d, S, DT, VISC, 200)
    assert all(np.isfinite(x).all() for x in (u, v, p, d))


def test_check_obstacles_accepts_and_refuses():
    from smokephysai_b200.navier_stokes import FieldLayout, check_obstacles, obstacle_stride
    h, w, B = 6, 9, 3
    cpu = torch.device("cpu")
    L = FieldLayout(h, w, B)
    m = np.zeros((h, w), bool)
    m[2, 3] = True
    for ok in (m, m.astype(np.uint8), m.astype(np.int64), torch.from_numpy(m), torch.from_numpy(m.astype(np.int32)),
               np.stack([m] * B)):
        t = check_obstacles(ok, h, w, B, cpu)
        assert obstacle_stride(t, L) == (0 if t.dim() == 2 else h * L.pitch_c)
    bad = [
        m.tolist(),                                    # a list
        m.astype(np.float32),                          # float
        m.astype(np.complex64),
        m.astype(np.int32) * 2,                        # integers other than 0 / 1
        -m.astype(np.int32),
        m[:-1],                                        # wrong shape
        m[:, :-1],
        m.T,
        np.stack([m] * (B + 1)),                       # wrong batch
        m[None, None],                                 # 4-D
        m[0],                                          # 1-D
    ]
    for b in bad:
        with pytest.raises(ValueError):
            check_obstacles(b, h, w, B, cpu)
    with pytest.raises(ValueError):                    # a tensor on another device than the simulator's
        check_obstacles(torch.from_numpy(m).to("meta"), h, w, B, cpu)


def test_new_entries_are_declared_exported_and_bound():
    from smokephysai_b200 import _lib, build
    so = build.build()
    syms = subprocess.check_output(["nm", "-D", "--defined-only", so]).decode()
    header = open(build.os.path.join(build.HERE, "..", "include", "smoke_b200.h")).read()
    for name, n in (("smk_run_steps_obst_ex", 22), ("smk_jacobi_obst", 10), ("smk_jacobi_residual_ex", 7)):
        assert re.search(r" T %s\b" % name, syms), name
        m = re.search(r"SMK_API int %s\(([^;]*)\);" % name, header)
        assert m and len(m.group(1).split(",")) == n, name
        assert len(_lib.SIGNATURES[name]) == n, name
    # the mask pair sits right after force_per_step; everything else is smk_run_steps_force_ex's
    force = list(_lib.SIGNATURES["smk_run_steps_force_ex"])
    obst = list(_lib.SIGNATURES["smk_run_steps_obst_ex"])
    assert obst[:15] + obst[17:] == force
    assert obst[15:17] == [_lib.c_p, _lib.c_i64]
    # smk_jacobi_obst is smk_jacobi with the mask pair after p_scratch
    jac = list(_lib.SIGNATURES["smk_jacobi"])
    jo = list(_lib.SIGNATURES["smk_jacobi_obst"])
    assert jo[:4] + jo[6:] == jac and jo[4:6] == [_lib.c_p, _lib.c_i64]
    assert int(re.search(r"#define SMK_ABI_VERSION (\d+)", header).group(1)) == 7
