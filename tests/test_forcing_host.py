"""CPU checks of velocity forcing (no GPU): pack_forcing's padding, step-major order, chunk pointers and every ValueError, the new ABI
entries declared, exported and bound, and the torch restatement (forcing_oracle.py: add, then the step) against the C oracle's step
with the same add done between steps, bit for bit."""
import re
import subprocess

import numpy as np
import pytest
import torch

import oracle
from forcing_oracle import rollout as rollout_forced, wind
from helpers import assert_same

DT, VISC = 0.01, 0.001
CPU = torch.device("cpu")


def _pair(T, B, h, w, seed=0):
    rng = np.random.default_rng(seed)
    lead = (T, B) if T else (B,)
    return (rng.standard_normal(lead + (h + 1, w)).astype(np.float32), rng.standard_normal(lead + (h, w + 1)).astype(np.float32))


@pytest.mark.parametrize("kind", ["numpy", "tensor"])
@pytest.mark.parametrize("T", [0, 3])
@pytest.mark.parametrize("hw", [(5, 7), (4, 8), (1, 3)])
def test_pack_forcing_padding_and_order(kind, T, hw):
    from smokephysai_b200.navier_stokes import FieldLayout, pack_forcing
    h, w = hw
    B = 2
    du, dv = _pair(T, B, h, w)
    arg = (du, dv) if kind == "numpy" else (torch.from_numpy(du), torch.from_numpy(dv))
    fu, fv, per_step = pack_forcing(arg, T or 9, B, h, w, CPU)
    L = FieldLayout(h, w, B)
    assert per_step == bool(T)
    assert fu.dtype == fv.dtype == torch.float32 and fu.is_contiguous() and fv.is_contiguous()
    assert tuple(fu.shape) == (T or 1, B, h + 1, L.pitch_u) and tuple(fv.shape) == (T or 1, B, h, L.pitch_v)
    # one simulation is stride_u / stride_v elements: the grid's strides
    assert fu[0, 0].numel() == L.stride_u and fv[0, 0].numel() == L.stride_v
    want_u, want_v = (du, dv) if T else (du[None], dv[None])
    assert fu[..., :w].numpy().tobytes() == want_u.tobytes()
    assert fv[..., :w + 1].numpy().tobytes() == want_v.tobytes()
    assert not fu[..., w:].any() and not fv[..., w + 1:].any()              # zero padding
    # step-major: row t of simulation b starts at element (t * B + b) * stride
    flat_u = fu.reshape(-1)
    for t in range(T or 1):
        for b in range(B):
            k = (t * B + b) * L.stride_u
            assert flat_u[k: k + L.stride_u].view(h + 1, L.pitch_u)[:, :w].numpy().tobytes() == want_u[t, b].tobytes()


def test_pack_forcing_drops_the_batch_dimension_for_one_simulation():
    from smokephysai_b200.navier_stokes import pack_forcing
    du, dv = _pair(0, 1, 6, 5)
    a = pack_forcing((du[0], dv[0]), None, 1, 6, 5, CPU)
    b = pack_forcing((du, dv), None, 1, 6, 5, CPU)
    assert a[2] is False and torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_chunk_pointers():
    """Each chunk of steps t0 .. of a per-step forcing passes the base plus t0 * B * stride of the same upload (as schedules pass
    offsets + t0 * B); a constant forcing passes the base whatever t0."""
    from smokephysai_b200.navier_stokes import FieldLayout, forcing_pointers, pack_forcing
    T, B, h, w = 7, 3, 9, 6
    L = FieldLayout(h, w, B)
    fu, fv, per_step = pack_forcing(_pair(T, B, h, w), T, B, h, w, CPU)
    assert forcing_pointers(None, L) == (None, None, 0)
    for n in (1, 2, 3):
        for t0 in range(0, T, n):
            pu, pv, flag = forcing_pointers((fu, fv, per_step, t0), L)
            assert flag == 1 and pu == fu[t0].data_ptr() and pv == fv[t0].data_ptr()
            assert pu == fu.data_ptr() + 4 * t0 * B * L.stride_u and pv == fv.data_ptr() + 4 * t0 * B * L.stride_v
    cu, cv, cflag = pack_forcing(_pair(0, B, h, w), T, B, h, w, CPU)
    assert forcing_pointers((cu, cv, cflag, 5), L) == (cu.data_ptr(), cv.data_ptr(), 0)


def test_pack_forcing_errors():
    from smokephysai_b200.navier_stokes import pack_forcing
    h, w, B, T = 5, 7, 2, 3
    du, dv = _pair(0, B, h, w)
    su, sv = _pair(T, B, h, w)
    bad = [
        (None, T, B),
        ((du,), T, B),                                                  # one array
        ((du, dv, dv), T, B),                                           # three
        ((du.tolist(), dv), T, B),                                      # a list
        ((du, sv), T, B),                                               # constant du, per-step dv
        ((du[:, :-1], dv), T, B),                                       # u rows != h + 1
        ((du, dv[..., :-1]), T, B),                                     # v cols != w + 1
        ((du.transpose(0, 2, 1), dv), T, B),                            # swapped axes
        ((du[:1], dv[:1]), T, B),                                       # batch 1, simulator batch 2
        ((du[0], dv[0]), T, B),                                         # no batch dimension with batch 2
        ((du.astype(np.float64), dv), T, B),                            # float64
        ((du, dv.astype(np.float16)), T, B),                            # float16
        ((su, sv), T + 1, B),                                           # T != nsteps
        ((su[:, :1], sv[:, :1]), T, B),                                 # per-step batch 1
        ((su, sv), None, B),                                            # per-step where only a constant forcing fits
        ((su[None], sv[None]), T, B),                                   # 5-D
    ]
    for f, n, b in bad:
        with pytest.raises(ValueError):
            pack_forcing(f, n, b, h, w, CPU)
    with pytest.raises(ValueError):                                     # a CUDA tensor of another device than the call's
        pack_forcing((torch.from_numpy(du).to("meta"), torch.from_numpy(dv)), T, B, h, w, CPU)


def test_rollout_forcing_errors():
    from smokephysai_b200 import autodiff
    z = lambda *s: torch.zeros(s)
    for bad, two_d in (((z(9, 8),), True), ((z(9, 8).double(), z(8, 9)), True), ((z(9, 8).numpy(), z(8, 9)), True),
                       ((z(2, 2, 9, 8), z(2, 2, 8, 9)), True), ((z(9, 8), z(8, 9)), False)):
        with pytest.raises(ValueError):
            autodiff._check_forcing(bad, two_d, CPU)
    assert len(autodiff._check_forcing((z(9, 8), z(8, 9)), True, CPU)) == 2


def test_new_entries_are_declared_exported_and_bound():
    from smokephysai_b200 import _lib, build
    so = build.build()
    syms = subprocess.check_output(["nm", "-D", "--defined-only", so]).decode()
    header = open(build.os.path.join(build.HERE, "..", "include", "smoke_b200.h")).read()
    for name, n in (("smk_run_steps_force_ex", 20), ("smk_add_forcing", 6)):
        assert re.search(r" T %s\b" % name, syms), name
        m = re.search(r"SMK_API int %s\(([^;]*)\);" % name, header)
        assert m and len(m.group(1).split(",")) == n, name
        assert len(_lib.SIGNATURES[name]) == n, name
    # the forcing triple sits right after offsets_step_stride; everything else is smk_run_steps_sched_ex's
    sched = list(_lib.SIGNATURES["smk_run_steps_sched_ex"])
    force = list(_lib.SIGNATURES["smk_run_steps_force_ex"])
    assert force[:12] + force[15:] == sched
    assert force[12:15] == [_lib.c_p, _lib.c_p, _lib.c_i32]
    assert int(re.search(r"#define SMK_ABI_VERSION (\d+)", header).group(1)) == 7


@pytest.mark.parametrize("hw", [(24, 24), (17, 29), (1, 40)])
@pytest.mark.parametrize("per_step", [False, True])
def test_restatement_with_forcing_bit_equal_to_c_oracle_loop(hw, per_step):
    h, w = hw
    T, B, K = 5, 2, 20
    du, dv = wind(T, B, h, w, seed=h * w)
    if not per_step:
        du, dv = du[0], dv[0]
    frames_ref, finals_ref = [], []
    for b in range(B):
        ns = oracle.OracleSolver((h, w), DT, VISC, K)
        ns.add_smoke_source(w // 2, h // 2, max(1, min(h, w) // 3), 1.5)
        fr = []
        for t in range(T):
            ns.u += du[t, b] if per_step else du[b]
            ns.v += dv[t, b] if per_step else dv[b]
            fr.append(ns.step())
        frames_ref.append(np.stack(fr))
        finals_ref.append((ns.u.copy(), ns.v.copy(), ns.p.copy(), ns.density.copy()))
    d0 = np.zeros((h, w), np.float32)
    oracle.splat(d0, w // 2, h // 2, max(1, min(h, w) // 3), 1.5)
    z = lambda *s: torch.zeros(s, dtype=torch.float32)
    state = (z(B, h + 1, w), z(B, h, w + 1), z(B, h, w), torch.from_numpy(np.stack([d0] * B)))
    with torch.no_grad():
        frames, final = rollout_forced(state, T, DT, VISC, K, du=torch.from_numpy(du), dv=torch.from_numpy(dv))
    for b in range(B):
        for name, got, want in zip("uvpd", final, finals_ref[b]):
            np.testing.assert_array_equal(got[b].numpy(), want, err_msg=name)
    assert_same(frames.numpy(), np.stack(frames_ref), "frames")
    # the forcing is strong enough to carry a back-trace beyond a cell somewhere
    assert DT * max(np.abs(finals_ref[0][0]).max(), np.abs(finals_ref[0][1]).max()) > 1.0
