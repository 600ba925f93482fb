"""CPU checks of source schedules (no GPU): the vectorised packing (record order, intensity bits, offsets, chunk slicing) of
numpy arrays and CPU tensors, every ValueError of the packing and of autodiff.rollout(schedule=), the new ABI entry, and the
torch restatement with a per-step list against the C oracle's add_smoke_source + step loop, bit for bit."""
import re
import subprocess

import numpy as np
import pytest
import torch

import oracle
from schedule_oracle import moving_schedule, rollout as rollout_sched, rows_as_lists
from helpers import assert_same

DT, VISC = 0.01, 0.001


def _small():
    xy = np.arange(3 * 2 * 2 * 2).reshape(3, 2, 2, 2)
    radius = np.array([[[1, 2], [3, -1]], [[4, 5], [6, 7]], [[8, -2], [9, 10]]], np.int32)
    inten = np.linspace(-1.5, 2.5, 12, dtype=np.float32).reshape(3, 2, 2)
    return xy, radius, inten


@pytest.mark.parametrize("kind", ["numpy", "tensor"])
def test_pack_schedule_order_and_bits(kind):
    from smokephysai_b200.navier_stokes import SOURCE_DTYPE, pack_schedule, pack_sources
    s = _small()
    if kind == "tensor":
        s = tuple(torch.from_numpy(a) for a in s)
    rec, E = pack_schedule(s, 3, 2)
    assert E == 2 and rec.dtype == torch.int32 and tuple(rec.shape) == (12, 4)
    xy, radius, inten = _small()
    for t in range(3):
        for b in range(2):
            for e in range(2):
                k = (t * 2 + b) * 2 + e
                assert rec[k, :3].tolist() == [xy[t, b, e, 0], xy[t, b, e, 1], radius[t, b, e]]
    assert rec[:, 3].numpy().view(np.float32).tolist() == inten.reshape(-1).tolist()
    # the same bytes as pack_sources of the flattened lists (padded entries included)
    flat = [[(int(xy[t, b, e, 0]), int(xy[t, b, e, 1]), int(radius[t, b, e]), float(inten[t, b, e]))
             for t in range(3) for b in range(2) for e in range(2)]]
    want, _ = pack_sources(flat)
    assert want.dtype == SOURCE_DTYPE
    assert rec.numpy().tobytes() == want.tobytes()


def test_schedule_offsets_and_chunks():
    from smokephysai_b200.navier_stokes import schedule_offsets
    T, B, E = 7, 3, 2
    off = schedule_offsets(T, B, E, torch.device("cpu"))
    assert off.dtype == torch.int32 and off.tolist() == [k * E for k in range(T * B + 1)]
    for t in range(T):
        for b in range(B):
            assert (int(off[t * B + b]), int(off[t * B + b + 1])) == ((t * B + b) * E, (t * B + b + 1) * E)
    # a chunk of steps t0 .. t0 + m - 1 reads offsets[t0 * B:] with the same records: its row (t, b) is the call's (t0 + t, b)
    for n in (1, 2, 3):
        for t0 in range(0, T, n):
            m = min(n, T - t0)
            chunk = off[t0 * B:]
            for t in range(m):
                for b in range(B):
                    assert int(chunk[t * B + b]) == int(off[(t0 + t) * B + b])
            assert len(chunk) >= m * B + 1


def test_pack_schedule_empty_and_errors():
    from smokephysai_b200.navier_stokes import pack_schedule
    z = (np.zeros((2, 3, 0, 2), np.int32), np.zeros((2, 3, 0), np.int32), np.zeros((2, 3, 0), np.float32))
    assert pack_schedule(z, 2, 3) == (None, 0)
    xy, radius, inten = _small()
    bad = [
        ((xy, radius), 3, 2),                                          # two arrays
        ((xy, radius, inten), 2, 2),                                   # T != nsteps
        ((xy, radius, inten), 3, 3),                                   # B != batch
        ((xy[..., :1], radius, inten), 3, 2),                          # xy [.., 1]
        ((xy[0], radius, inten), 3, 2),                                # xy 3-D
        ((xy, radius[:, :, :1], inten), 3, 2),                         # radius shape
        ((xy, radius, inten[:2]), 3, 2),                               # intensity shape
        ((xy.astype(np.float32), radius, inten), 3, 2),                # float xy
        ((xy, radius.astype(np.float64), inten), 3, 2),                # float radius
        ((xy, radius, inten.astype(np.float64)), 3, 2),                # float64 intensity
        ((xy.tolist(), radius, inten), 3, 2),                          # a list
        ((xy + 2 ** 33, radius, inten), 3, 2),                         # beyond int32
        (None, 3, 2),
    ]
    for s, T, B in bad:
        with pytest.raises(ValueError):
            pack_schedule(s, T, B)


def test_rollout_schedule_records_and_errors():
    from smokephysai_b200 import autodiff
    xy, radius, inten = _small()
    cpu = torch.device("cpu")
    I = torch.from_numpy(inten)
    rec, off, E = autodiff._schedule_records((xy, radius), I, 3, 2, cpu)
    assert E == 2 and off.tolist() == [0, 2, 4, 6, 8, 10, 12]
    assert rec[:, 3].numpy().view(np.float32).tolist() == inten.reshape(-1).tolist()
    assert rec[:, 2].tolist() == radius.reshape(-1).tolist()
    for s, i in (((xy, radius, inten), I),                         # rollout takes (xy, radius)
                 ((xy, radius), None),                             # no intensities
                 ((xy, radius), I[:2]),                            # wrong shape
                 ((xy, radius), I.double()),                       # wrong dtype
                 ((xy, radius), inten),                            # not a tensor
                 ((xy[:, :1], radius), I)):                        # xy / radius mismatch
        with pytest.raises(ValueError):
            autodiff._schedule_records(s, i, 3, 2, cpu)


def test_new_entry_is_declared_exported_and_bound():
    from smokephysai_b200 import _lib, build
    so = build.build()
    syms = subprocess.check_output(["nm", "-D", "--defined-only", so]).decode()
    header = open(build.os.path.join(build.HERE, "..", "include", "smoke_b200.h")).read()
    assert re.search(r" T smk_run_steps_sched_ex\b", syms)
    m = re.search(r"SMK_API int smk_run_steps_sched_ex\(([^;]*)\);", header)
    assert m and len(m.group(1).split(",")) == 17
    assert len(_lib.SIGNATURES["smk_run_steps_sched_ex"]) == 17
    # the new stride sits right after the offsets; everything else is smk_run_steps_src_ex's
    src = list(_lib.SIGNATURES["smk_run_steps_src_ex"])
    assert list(_lib.SIGNATURES["smk_run_steps_sched_ex"]) == src[:11] + [_lib.SIGNATURES["smk_run_steps_sched_ex"][11]] + src[11:]
    assert int(re.search(r"#define SMK_ABI_VERSION (\d+)", header).group(1)) == 7


def c_weight(h, w, x, y, r):
    a = np.zeros((h, w), np.float32)
    oracle.splat(a, x, y, r, 1.0)
    return torch.from_numpy(a)


@pytest.mark.parametrize("K", [0, 20])
def test_restatement_with_schedule_bit_equal_to_c_oracle_loop(K):
    h, w, T, B = 45, 53, 6, 3
    sched = moving_schedule(T, B, h, w, seed=K)
    sched[1][2, 1, 0] = -1                            # a padded entry inside a row, not only at its end
    frames_ref, finals_ref = [], []
    for b in range(B):
        ns = oracle.OracleSolver((h, w), DT, VISC, K)
        fr = []
        for t in range(T):
            for x, y, r, i in rows_as_lists(sched, t)[b]:
                ns.add_smoke_source(x, y, r, i)
            fr.append(ns.step())
        frames_ref.append(np.stack(fr))
        finals_ref.append((ns.u, ns.v, ns.p, ns.density))
    z = lambda *s: torch.zeros(s, dtype=torch.float32)
    state = (z(B, h + 1, w), z(B, h, w + 1), z(B, h, w), z(B, h, w))
    with torch.no_grad():
        frames, final = rollout_sched(state, T, DT, VISC, K, xy=sched[0], radius=sched[1],
                                      intensities=torch.from_numpy(sched[2]), weight=c_weight)
    for b in range(B):
        for name, got, want in zip("uvpd", final, finals_ref[b]):
            np.testing.assert_array_equal(got[b].numpy(), want, err_msg=name)
    assert_same(frames.numpy(), np.stack(frames_ref), "frames")
    # the emitters do move: consecutive rows differ
    assert not np.array_equal(sched[0][0], sched[0][1]) and not np.array_equal(sched[2][0], sched[2][1])
