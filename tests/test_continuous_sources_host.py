"""CPU checks of continuous sources (no GPU): record packing and validation of NavierStokesSimulator.set_continuous_sources and
of autodiff.rollout(sources=...), the new ABI entries, and the torch restatement with per-step sources against the C oracle's
add_smoke_source + step loop, bit for bit."""
import re
import subprocess

import numpy as np
import pytest
import torch

import oracle
from continuous_oracle import rollout as rollout_src
from helpers import assert_same

DT, VISC = 0.01, 0.001


def test_source_lists_are_checked_and_normalised():
    from smokephysai_b200.navier_stokes import check_source_lists
    got = check_source_lists([[(1, 2.0, 3, 4)], [], [np.array([5, 6, 7, 0.5])]], 3)
    assert got == [[(1, 2, 3, 4.0)], [], [(5, 6, 7, 0.5)]]
    assert all(isinstance(v, int) for v in got[0][0][:3]) and isinstance(got[0][0][3], float)
    for bad in ([[(1, 2, 3, 4)]],                   # one list for two simulations
                [[(1, 2, 3)], []],                   # a 3-tuple
                [[(1, 2, 3, 4, 5)], []],             # a 5-tuple
                [[("a", 2, 3, 4)], []],              # not a number
                [5, []],                             # not a list
                "ab", None):
        with pytest.raises(ValueError):
            check_source_lists(bad, 2)


def test_pack_sources_layout():
    from smokephysai_b200.navier_stokes import SOURCE_DTYPE, pack_sources
    rec, off = pack_sources([[(1, 2, 3, 0.5), (4, 5, 6, 1.5)], [], [(7, 8, 0, -2.0)]])
    assert rec.dtype == SOURCE_DTYPE and rec.itemsize == 16 and off.dtype == np.int32
    assert off.tolist() == [0, 2, 2, 3]
    assert rec["x"].tolist() == [1, 4, 7] and rec["y"].tolist() == [2, 5, 8] and rec["radius"].tolist() == [3, 6, 0]
    assert rec["intensity"].tolist() == [0.5, 1.5, -2.0]
    rec, off = pack_sources([[], []])
    assert len(rec) == 1 and off.tolist() == [0, 0, 0]      # one dummy record keeps the device pointer valid


def test_rollout_source_records():
    from smokephysai_b200 import autodiff
    rec, off, n = autodiff._source_records([[(1, 2, 3), (4, 5, 6)], [(7, 8, 9)]], 2, torch.device("cpu"))
    assert n == 3 and off.tolist() == [0, 2, 3]
    assert rec.tolist() == [[1, 2, 3, 0], [4, 5, 6, 0], [7, 8, 9, 0]]
    assert autodiff._emitter_lists([(1, 2, 3)], True) == [[(1, 2, 3)]]
    assert autodiff._emitter_lists([[(1, 2, 3)]], True) == [[(1, 2, 3)]]
    for bad in ([[(1, 2, 3)]], [[(1, 2)], []], [[(1, 2, 3, 4)], []], [[5], []]):
        with pytest.raises(ValueError):
            autodiff._source_records(bad, 2, torch.device("cpu"))
    autodiff._check_intensities(torch.zeros(3), 3, torch.device("cpu"))
    for bad in (torch.zeros(2), torch.zeros(3, dtype=torch.float64), torch.zeros(1, 3), [0.0, 0.0, 0.0]):
        with pytest.raises(ValueError):
            autodiff._check_intensities(bad, 3, torch.device("cpu"))


def test_new_entries_are_declared_exported_and_bound():
    from smokephysai_b200 import _lib, build
    so = build.build()
    syms = subprocess.check_output(["nm", "-D", "--defined-only", so]).decode()
    header = open(build.os.path.join(build.HERE, "..", "include", "smoke_b200.h")).read()
    for name, nargs in (("smk_run_steps_src_ex", 16), ("smk_splat_sources_adjoint_ex", 8)):
        assert re.search(r" T %s\b" % name, syms), name
        assert re.search(r"SMK_API int %s\(" % name, header), name
        assert len(_lib.SIGNATURES[name]) == nargs
    assert int(re.search(r"#define SMK_ABI_VERSION (\d+)", header).group(1)) == 7


def c_weight(h, w, x, y, r):
    """An emitter's footprint as the C oracle's add_smoke_source computes it (intensity 1: the weight itself)."""
    a = np.zeros((h, w), np.float32)
    oracle.splat(a, x, y, r, 1.0)
    return torch.from_numpy(a)


@pytest.mark.parametrize("K", [0, 1, 20])
def test_restatement_with_per_step_sources_bit_equal_to_c_oracle_loop(K):
    h, w, T = 37, 53, 5
    emitters = [[(20, 15, 8), (24, 17, 6), (2, 35, 5), (50, 1, 4), (10, 10, 0)], [], [(30, 20, 8)]]
    inten = np.array([1.5, 0.75, 2.0, 1.25, 0.0, 0.9], np.float32)
    B = len(emitters)
    frames_ref, finals_ref = [], []
    k = 0
    for b in range(B):
        ns = oracle.OracleSolver((h, w), DT, VISC, K)
        mine = [(e, inten[k + q]) for q, e in enumerate(emitters[b])]
        k += len(emitters[b])
        fr = []
        for _ in range(T):
            for (x, y, r), i in mine:
                ns.add_smoke_source(x, y, r, i)
            fr.append(ns.step())
        frames_ref.append(np.stack(fr))
        finals_ref.append((ns.u, ns.v, ns.p, ns.density))
    z = lambda *s: torch.zeros(s, dtype=torch.float32)
    state = (z(B, h + 1, w), z(B, h, w + 1), z(B, h, w), z(B, h, w))
    with torch.no_grad():
        frames, final = rollout_src(state, T, DT, VISC, K, sources=emitters, intensities=torch.from_numpy(inten), weight=c_weight)
    finite = [b for b in range(B) if np.isfinite(frames_ref[b]).all()]
    assert finite == [1, 2]                           # the radius-0 emitter makes 0 / 0 in its weight, as in the reference
    for b in range(B):
        np.testing.assert_array_equal(frames[b].numpy(), frames_ref[b])       # NaN-aware bit check
        for name, got, want in zip("uvpd", final, finals_ref[b]):
            np.testing.assert_array_equal(got[b].numpy(), want, err_msg=name)
    assert_same(frames[1:].numpy(), np.stack(frames_ref[1:]), "frames")
