"""Solid obstacles on the phase kernels: frames and u, v, p, density bit-equal (numeric ==) to the obstacle oracle
(tests/obstacle_oracle.c) on every tile configuration of the masked Jacobi, with obstacles on the seams of overlapped tiles, on
the ring, over whole rows and whole simulations, per simulation and shared; the combinations with sources, schedules, forcing,
frame dtypes, fmul, a deferred reset and generate_sequences; the invariants; and every rejection before any launch."""
import ctypes as C

import numpy as np
import pytest
import torch

import obstacle_oracle as O
from helpers import emitters_for_sequence
from schedule_oracle import moving_schedule, rows_as_lists

pytestmark = pytest.mark.gpu

DT, VISC = 0.01, 0.001
DEV = "cuda:0"
FIELDS = ("u", "v", "p", "density")


def N(t):
    return t.detach().float().cpu().numpy().copy()


def same(a, b, what):
    np.testing.assert_array_equal(np.asarray(a), np.asarray(b), err_msg=what)


def make(h, w, B, K, **kw):
    from smokephysai_b200 import NavierStokesSimulator
    return NavierStokesSimulator((h, w), DT, VISC, DEV, jacobi_iters=K, batch=B, **kw)


def batched(x, B):
    return x if B > 1 else x[None]


def seeded(ns, B, seed):
    """Emitters splatted once (by the library, so the oracle starts from the same density) and a random velocity."""
    h, w = ns.h, ns.w
    ns.add_sources([[(x * w // 128, y * h // 128, max(1, 8 * min(h, w) // 128), i) for x, y, _, i in emitters_for_sequence(seed + b)]
                    for b in range(B)])
    rng = np.random.default_rng(seed)
    ns.u = torch.from_numpy(rng.standard_normal(tuple(ns.u.shape)).astype(np.float32) * 20)
    ns.v = torch.from_numpy(rng.standard_normal(tuple(ns.v.shape)).astype(np.float32) * 20)
    return [batched(N(getattr(ns, k)), B) for k in FIELDS]


def oracle_run(state, masks, K, T, force=None, fmul=None):
    """state: [B, ...] numpy u, v, p, d; masks [B, h, w]; force (du [T, B, ..], dv) -> frames [B, T, h, w], final fields."""
    u, v, p, d = (np.ascontiguousarray(x.copy()) for x in state)
    B = d.shape[0]
    frames = np.empty((B, T) + d.shape[1:], np.float32)
    for b in range(B):
        ub, vb, pb, db = (np.ascontiguousarray(x[b]) for x in (u, v, p, d))
        for t in range(T):
            if force is not None:
                ub += force[0][t, b]
                vb += force[1][t, b]
            fr, _ = O.step_obst(ub, vb, pb, db, masks[b], DT, VISC, K)
            frames[b, t] = fr if fmul is None else fr + fmul * fr
        u[b], v[b], p[b], d[b] = ub, vb, pb, db
    return frames, (u, v, p, d)


def check_against_oracle(h, w, B, K, T, masks, shared=False, seed=1, fmul=None, **kw):
    ns = make(h, w, B, K, **kw)
    state = seeded(ns, B, seed)
    ns.set_obstacles(masks[0] if shared else masks)
    fr = batched(N(ns.run_steps(T, fmul=fmul)), B)
    got = [batched(N(getattr(ns, k)), B) for k in FIELDS]
    want_fr, want = oracle_run(state, np.broadcast_to(masks, (B, h, w)) if shared else masks, K, T,
                               fmul=None if fmul is None else N(fmul)[:, :w])
    same(fr, want_fr, "frames")
    for k, g, wnt in zip(FIELDS, got, want):
        same(g, wnt, k)
    invariants(ns, np.broadcast_to(masks, (B, h, w)), fr[:, -1], K)
    return ns


def invariants(ns, masks, last_frame, K):
    B = masks.shape[0]
    u, v, p, d = (batched(N(getattr(ns, k)), B) for k in FIELDS)
    for b in range(B):
        S = np.asarray(masks[b])
        cu, cv = O.faces(S)
        for name, f, c in (("u", u[b], cu), ("v", v[b], cv), ("density", d[b], S), ("frame", last_frame[b], S)) + \
                          ((("p", p[b], S),) if K >= 1 else ()):
            assert not f[c].any() and not np.signbit(f[c]).any(), "%s: not +0 on a closed face / solid cell" % name


def box_masks(B, h, w, seed=0):
    rng = np.random.default_rng(seed)
    m = np.zeros((B, h, w), bool)
    for b in range(B):
        r0, c0 = rng.integers(h // 8, h // 2), rng.integers(w // 8, w // 2)
        m[b, r0:r0 + h // 6, c0:c0 + w // 5] = True
        m[b, h // 2 + 2: h // 2 + 4, : w // 3] = True
        m[b] |= rng.random((h, w)) < 0.02
    return m


@pytest.mark.parametrize("B", [1, 40])
def test_full_size_batches_on_the_phase_path(B):
    """128^2 at batch 1 and 40 would run on k_step_cluster / k_step_fused without a mask; with one they run on the phase path."""
    ns = check_against_oracle(128, 128, B, 20, 4, box_masks(B, 128, 128, B))
    assert not ns.step_is_fused(4)


@pytest.mark.parametrize("hw", [(96, 96), (17, 29)])
def test_k100_small_grids(hw):
    h, w = hw
    check_against_oracle(h, w, 2, 100, 3, box_masks(2, h, w, h))


def seam_mask(h, w, T, TH=128):
    """Cells on the columns and rows where tiles of run_cfg meet for T sweeps per launch: advances ox = 128 - 2 HX, oy = TH - 2 T,
    tile kx keeps columns [kx ox + HX, kx ox + 128 - HX), so neighbouring kept ranges meet at HX + k ox (rows: T + k oy)."""
    HX = (T + 3) & ~3
    ox, oy = 128 - 2 * HX, TH - 2 * T
    S = np.zeros((h, w), bool)
    for k in range(w // ox + 1):
        c = HX + k * ox
        for dc in (-2, -1, 0, 1):
            if 1 <= c + dc < w - 1:
                S[3 + 5 * k: 40 + 5 * k: 3, c + dc] = True          # dotted columns across the seam
        if c < w:
            S[200:260, max(0, c - 1):c + 1] = True                  # a wall on it
    for k in range(h // oy + 1):
        r = T + k * oy
        for dr in (-2, -1, 0, 1):
            if 1 <= r + dr < h - 1:
                S[r + dr, 5 + 7 * k: w - 5: 4] = True
        if r < h:
            S[max(0, r - 1):r + 1, 300:360] = True
    S[0, 10:20] = S[-1, 30:50] = S[40:60, 0] = S[70:90, -1] = True   # touching the ring
    return S


def test_1024_multi_launch_seams():
    """1024^2, K = 100, 10 sweeps per launch: ten overlapped-tile launches of k_jacobi_obst<8, 16>; obstacles on the seams."""
    S = seam_mask(1024, 1024, 10)
    check_against_oracle(1024, 1024, 1, 100, 2, S[None], sweeps_per_launch=10)


def test_1024_default_sweeps():
    check_against_oracle(1024, 1024, 1, 100, 2, box_masks(1, 1024, 1024, 3))


def test_many_tiles_branch():
    """Six 1024^2 simulations reach launch_jacobi's many-waves branch (64 x 128 tiles, k_jacobi_obst<8, 8>)."""
    check_against_oracle(1024, 1024, 6, 30, 2, box_masks(6, 1024, 1024, 4))


def test_mask_shapes_per_simulation_and_shared():
    h, w, B = 64, 96, 5
    m = np.zeros((B, h, w), bool)
    m[0, 0, :] = True
    m[0, :, -1] = True                     # along the ring
    m[1, h // 2, :] = True                 # a whole row
    m[2, :, :] = True                      # a whole simulation solid
    m[3] = box_masks(1, h, w, 9)[0]
    m[4, 10:20, 10:20] = True
    m[4, 11:19, 11:19] = False             # an enclosed pocket
    check_against_oracle(h, w, B, 20, 4, m)
    check_against_oracle(h, w, B, 20, 4, m[3:4].repeat(B, 0), shared=True)


def test_all_fluid_mask_equals_no_mask():
    for B, kw in ((40, {}), (1, {}), (3, {"step_kernel": "phases"})):
        a, b = make(128, 128, B, 20, **kw), make(128, 128, B, 20, **kw)
        seeded(a, B, 5)
        seeded(b, B, 5)
        b.set_obstacles(np.zeros((128, 128), bool))
        same(N(b.run_steps(3)), N(a.run_steps(3)), "frames")
        for k in FIELDS:
            same(N(getattr(b, k)), N(getattr(a, k)), k)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_frames(dtype):
    h = w = 128
    m = box_masks(3, h, w, 11)
    ns = make(h, w, 3, 20)
    seeded(ns, 3, 6)
    ns.set_obstacles(m)
    ref = make(h, w, 3, 20)
    seeded(ref, 3, 6)
    ref.set_obstacles(m)
    half = ns.run_steps(4, frame_dtype=dtype)
    full = ref.run_steps(4)
    assert half.dtype == dtype
    assert torch.equal(half.view(torch.int16), full.to(dtype).view(torch.int16))     # +0 on solids, bit for bit
    for k in FIELDS:
        same(N(getattr(ns, k)), N(getattr(ref, k)), k)


def test_fractal_multiplier():
    from smokephysai_b200.fractal_generator import FractalGenerator
    fmul = FractalGenerator(DEV).multiplier((128, 128), 0.05)
    check_against_oracle(128, 128, 3, 20, 3, box_masks(3, 128, 128, 12), fmul=fmul)


def host_loop(h, w, B, K, T, masks, heads):
    """The phase path with the mask, the head of each step done by hand: heads(ns, t)."""
    ns = make(h, w, B, K, step_kernel="phases")
    seeded(ns, B, 21)
    ns.set_obstacles(masks)
    frames = []
    for t in range(T):
        heads(ns, t)
        frames.append(N(ns.step()))
    return np.stack(frames, axis=-3), [N(getattr(ns, k)) for k in FIELDS]


def test_continuous_sources_and_schedule_inside_an_obstacle():
    h = w = 128
    B, T = 3, 5
    m = box_masks(B, h, w, 13)
    csrc = [[(x, y, 8, i) for x, y, _, i in emitters_for_sequence(300 + b)] for b in range(B)]
    want_fr, want = host_loop(h, w, B, 20, T, m, lambda ns, t: ns.add_sources(csrc))
    ns = make(h, w, B, 20)
    seeded(ns, B, 21)
    ns.set_obstacles(m)
    ns.set_continuous_sources(csrc)
    same(N(ns.run_steps(T)), want_fr, "frames (continuous)")
    for k, wnt in zip(FIELDS, want):
        same(N(getattr(ns, k)), wnt, k)
    sched = moving_schedule(T, B, h, w, seed=4)
    r0, c0 = np.argwhere(m[0])[0]
    sched[0][:, 0, 0] = (c0, r0)                     # emitter 0 of simulation 0 sits inside an obstacle
    want_fr, want = host_loop(h, w, B, 20, T, m, lambda ns, t: ns.add_sources(rows_as_lists(sched, t)))
    ns = make(h, w, B, 20)
    seeded(ns, B, 21)
    ns.set_obstacles(m)
    fr = N(ns.run_steps(T, schedule=sched))
    same(fr, want_fr, "frames (schedule)")
    for k, wnt in zip(FIELDS, want):
        same(N(getattr(ns, k)), wnt, k)
    invariants(ns, m, fr[:, -1], 20)


def test_forcing_into_a_wall():
    h = w = 96
    B, T = 2, 4
    m = np.zeros((B, h, w), bool)
    m[:, 20:76, 60:64] = True                        # a wall across the wind
    du = np.zeros((T, B, h + 1, w), np.float32)
    dv = np.zeros((T, B, h, w + 1), np.float32)
    du[:, :, 10:86, 20:70] = 150.0                   # blowing in +x, into the wall
    ns = make(h, w, B, 20)
    state = seeded(ns, B, 7)
    ns.set_obstacles(m)
    fr = N(ns.run_steps(T, forcing=(du, dv)))
    want_fr, want = oracle_run(state, m, 20, T, force=(du, dv))
    same(fr, want_fr, "frames")
    for k, wnt in zip(FIELDS, want):
        same(N(getattr(ns, k)), wnt, k)


def test_reset_and_one_shot_splat():
    """A pending reset with one splat is not consumed on the phase path: it is materialized and the call made again."""
    h = w = 128
    m = box_masks(20, h, w, 14)
    init = [[(x, y, 8, i) for x, y, _, i in emitters_for_sequence(b)] for b in range(20)]
    a = make(h, w, 20, 20)
    seeded(a, 20, 3)
    a.set_obstacles(m)
    a.run_steps(2)
    a.setup_grid()
    a.add_sources(init)
    b = make(h, w, 20, 20)
    b.add_sources(init)
    b.set_obstacles(m)
    same(N(a.run_steps(3)), N(b.run_steps(3)), "frames")
    for k in FIELDS:
        same(N(getattr(a, k)), N(getattr(b, k)), k)


@pytest.mark.parametrize("spc", [1, 2, 3])
def test_generate_sequences(spc):
    from smokephysai_b200 import SmokeSimulator
    h = w = 128
    B, T = 4, 7
    m = box_masks(B, h, w, 15)
    em = [[((x, y), i) for x, y, _, i in emitters_for_sequence(b)] for b in range(B)]
    sim = SmokeSimulator((h, w), DT, VISC, DEV, batch=B)
    ref = N(sim.generate_sequences(em, T, obstacles=m))
    assert sim.ns_solver.obstacles is None                       # the simulator's own (none) is restored
    got = sim.generate_sequences(em, T, to_host=True, steps_per_copy=spc, obstacles=m)
    same(N(got), ref, "to_host frames")
    # the same call through the simulator's own mask
    sim.set_obstacles(m)
    same(N(sim.generate_sequences(em, T)), ref, "own mask")
    assert np.array_equal(sim.ns_solver.obstacles, m)
    for b in range(B):
        assert not ref[b][:, m[b]].any()


@pytest.mark.parametrize("K,T", [(1, 0), (7, 3), (40, 10), (100, 0), (100, 24)])
@pytest.mark.parametrize("hw", [(30, 100), (128, 128), (600, 700)])
def test_jacobi_obst_entry(K, T, hw):
    from smokephysai_b200 import _lib
    from smokephysai_b200.navier_stokes import FieldLayout
    h, w = hw
    B = 2
    L = FieldLayout(h, w, B)
    rng = np.random.default_rng(K + h)
    P = rng.standard_normal((B, h, w)).astype(np.float32)
    D = rng.standard_normal((B, h, w)).astype(np.float32)
    S = np.stack([seam_mask(h, w, max(T, 1), 128) if h > 128 else box_masks(1, h, w, K)[0], box_masks(1, h, w, K + 1)[0]])
    pad = lambda a, dt: torch.from_numpy(np.pad(a, ((0, 0), (0, 0), (0, L.pitch_c - w)))).to(DEV, dt).contiguous()
    p, d, s = pad(P, torch.float32), pad(D, torch.float32), pad(S.astype(np.uint8), torch.uint8)
    scratch = torch.zeros_like(p)
    flag = C.c_int32(0)
    g = L.grid_struct()
    _lib.call("smk_jacobi_obst", C.byref(g), d.data_ptr(), p.data_ptr(), scratch.data_ptr(), s.data_ptr(), h * L.pitch_c, K, T,
              C.byref(flag), torch.cuda.current_stream().cuda_stream)
    out = (scratch if flag.value else p)[..., :w].cpu().numpy()
    for b in range(B):
        same(out[b], O.jacobi_obst(P[b], D[b], S[b], K), "simulation %d" % b)


def test_clearing_brings_back_the_fused_launch():
    from smokephysai_b200 import _lib
    ns = make(128, 128, 40, 20)
    seeded(ns, 40, 8)
    ns.set_obstacles(box_masks(1, 128, 128, 16)[0])
    assert not ns.step_is_fused(5)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    ns.run_steps(5, return_frames=False)
    assert _lib.launch_count() - n0 > 5
    ns.set_obstacles(None)
    assert ns.obstacles is None and ns.step_is_fused(5)
    n0 = _lib.launch_count()
    ns.run_steps(5, return_frames=False)
    assert _lib.launch_count() - n0 == 1


def test_residual_norms_use_the_mask():
    """After a masked step, jacobi_residual_norms is the change one more masked sweep (the oracle's) would make."""
    ns = make(96, 96, 1, 400, step_kernel="phases")
    seeded(ns, 1, 9)
    m = box_masks(1, 96, 96, 17)[0]
    ns.set_obstacles(m)
    ns.step()
    masked = ns.jacobi_residual_norms()[0, 0].item()
    p = N(ns.p)
    div = ns._field("div")
    want = O.jacobi_obst(p, N(div), m, 1) - p
    assert masked == pytest.approx(float(np.abs(want).max()), rel=1e-6, abs=1e-12)


def test_rejections_before_any_launch():
    from smokephysai_b200 import _lib
    h = w = 64
    ns = make(h, w, 2, 20)
    m = np.zeros((h, w), bool)
    m[5, 7] = True
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for bad in (m.astype(np.float32), m[:-1], np.stack([m] * 3), m.astype(np.int8) * 3, m.tolist()):
        with pytest.raises(ValueError):
            ns.set_obstacles(bad)
    assert ns.obstacles is None
    with pytest.raises(ValueError):
        make(h, w, 2, 20, step_kernel="fused").set_obstacles(m)
    ns.set_obstacles(m)
    ns.step_kernel = "fused"
    for call in (lambda: ns.step(), lambda: ns.run_steps(3)):
        with pytest.raises(ValueError):
            call()
    ns.step_kernel = "auto"
    assert _lib.launch_count() == n0
    # the C ABI: a misaligned mask, a bad stride, SMK_STEP_FUSED with a mask
    buf = ns._solid[1]
    done = C.c_int32(0)
    L = ns._layout
    prm = ns._params()
    for solid, stride, kernel in ((buf.data_ptr() + 1, 0, 0), (buf.data_ptr(), 7, 0), (buf.data_ptr(), L.h * L.pitch_c + 4, 0),
                                  (None, L.h * L.pitch_c, 0), (buf.data_ptr(), 0, 2)):
        prm.step_kernel = kernel
        rc = ns._lib.smk_run_steps_obst_ex(C.byref(ns._grid), C.byref(ns._state), C.byref(prm), 2, None, 0, 0, None, 0, None, None, 0,
                                           None, None, 0, solid, stride, 0, None, None, C.byref(done),
                                           torch.cuda.current_stream().cuda_stream)
        assert rc != 0
    assert _lib.launch_count() == n0
