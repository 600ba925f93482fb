"""Deferred reset: setup_grid() on an existing state records the reset, a splat right after it is recorded too, and the next
k_step_fused launch builds that state on chip.  Every case runs the same sequence twice -- deferred, and with the eager
reset (memset + k_splat, then the run) -- and compares frames and fields bit for bit, also after phase-kernel steps that
read the copies the fused launch does not write."""
import numpy as np
import pytest
import torch

from helpers import assert_same, emitters_for_sequence, smk_env

pytestmark = pytest.mark.gpu

FIELDS = ("u", "v", "p", "density")


def N(t):
    return t.detach().float().cpu().numpy()


def make(h, w, B, K, device="cuda:0", **kw):
    from smokephysai_b200 import NavierStokesSimulator
    return NavierStokesSimulator((h, w), 0.01, 0.001, device, jacobi_iters=K, batch=B, **kw)


def eager(ns):
    """Force the eager reset: the pending reset is never offered to a step call, so the next launch applies it with memset +
    k_splat."""
    ns._offer_reset = lambda: None
    return ns


def emitters(B, h, w, seed):
    return [[(x % w, y % h, r, i) for x, y, r, i in emitters_for_sequence(seed + s, h, w)] for s in range(B)]


def dirty(ns, B, h, w):
    """Leave every copy of the state non-zero, so a reset has something to clear."""
    ns.add_sources(emitters(B, h, w, 9000))
    ns.run_steps(3, return_frames=False)
    ns.step_kernel, kernel = "phases", ns.step_kernel
    ns.step()
    ns.step_kernel = kernel


def snapshot(ns):
    out = {k: N(getattr(ns, k)).copy() for k in FIELDS}
    out["boundary"] = N(ns.boundary).copy()
    return out


def run_pair(h, w, B, K, T, splats, read_between=False, frame_dtype=torch.float32, env=None, **kw):
    results = []
    for deferred in (True, False):
        with smk_env(**(env or {})):
            ns = make(h, w, B, K, **kw)
            if not deferred:
                eager(ns)
            dirty(ns, B, h, w)
            ns.setup_grid()
            for k in range(splats):
                src, off, _ = ns.upload_sources(emitters(B, h, w, 100 * k))
                ns.splat_uploaded(src, off)
            between = N(ns.density).copy() if read_between else None
            fr = N(ns.run_steps(T, frame_dtype=frame_dtype))
            after = snapshot(ns)
            ns.step_kernel = "phases"           # reads the copies the fused launch left alone
            ns.run_steps(2, return_frames=False)
            phases = snapshot(ns)
            results.append((fr, after, phases, between))
    (f0, a0, p0, b0), (f1, a1, p1, b1) = results
    assert_same(f0, f1, "frames")
    for k in a0:
        assert_same(a0[k], a1[k], k + " after the run")
        assert_same(p0[k], p1[k], k + " after phase steps")
    if read_between:
        assert_same(b0, b1, "density read between the reset and the run")


def test_c2_size_time_sliced_one_launch():
    """256 simulations of 128 x 128 at K = 40, 20 steps: the time-sliced schedule; the reset and the splat cost no launch."""
    from smokephysai_b200 import _lib
    run_pair(128, 128, 256, 40, 20, 1)
    ns = make(128, 128, 256, 40)
    src, off, _ = ns.upload_sources(emitters(256, 128, 128, 0))
    ns.run_steps(2, return_frames=False)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    ns.setup_grid()
    ns.splat_uploaded(src, off)
    ns.run_steps(20, return_frames=False)
    assert _lib.launch_count() - n0 == 1


@pytest.mark.parametrize("splats", [0, 2, 3])
def test_several_or_no_splats(splats):
    run_pair(128, 128, 160, 20, 6, splats)


def test_field_read_between_reset_and_run():
    run_pair(128, 128, 160, 20, 5, 1, read_between=True)


def test_one_cta_per_simulation_and_cluster_batches():
    run_pair(128, 128, 150, 20, 5, 1, env={"SMK_FUSED_SLICE": "0"})
    run_pair(128, 128, 8, 20, 5, 1)             # k_step_cluster: the reset is applied eagerly


def test_generic_instantiation_and_odd_k():
    run_pair(96, 100, 40, 7, 5, 1, step_kernel="fused")
    run_pair(128, 128, 160, 7, 4, 2)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_half_frames(dtype):
    run_pair(128, 128, 160, 20, 4, 1, frame_dtype=dtype)


def test_single_step_consumes_the_reset():
    results = []
    for deferred in (True, False):
        ns = make(128, 128, 64, 20, step_kernel="fused")
        if not deferred:
            eager(ns)
        dirty(ns, 64, 128, 128)
        ns.setup_grid()
        ns.add_sources(emitters(64, 128, 128, 5))
        fr = N(ns.step())
        results.append((fr, snapshot(ns)))
    assert_same(results[0][0], results[1][0], "frame")
    for k in results[0][1]:
        assert_same(results[0][1][k], results[1][1][k], k)


def test_cpu_mirror_edited_between_splat_and_run():
    results = []
    for deferred in (True, False):
        ns = make(128, 128, 160, 20, device="cpu")
        if not deferred:
            eager(ns)
        dirty(ns, 160, 128, 128)
        ns.setup_grid()
        ns.add_sources(emitters(160, 128, 128, 7))
        d = ns.density
        d[:, 40:60, 40:60] += 0.25
        fr = N(ns.run_steps(4))
        results.append((fr, snapshot(ns)))
    assert_same(results[0][0], results[1][0], "frames")
    for k in results[0][1]:
        assert_same(results[0][1][k], results[1][1][k], k)


def test_generate_sequences():
    from smokephysai_b200 import SmokeSimulator
    B, T = 160, 5
    lists = [[((x % 128, y % 128), i) for x, y, _, i in emitters_for_sequence(s, 128, 128)] for s in range(B)]
    out = {}
    for deferred in (True, False):
        sim = SmokeSimulator((128, 128), 0.01, 0.001, "cuda:0", jacobi_iters=20, batch=B)
        if not deferred:
            eager(sim.ns_solver)
        for dtype in (torch.float32, torch.bfloat16):
            for _ in range(2):              # the second call resets a state the first one left behind
                fr = sim.generate_sequences(lists, T, to_host=False, frame_dtype=dtype)
            out[deferred, dtype] = N(fr).copy()
    for dtype in (torch.float32, torch.bfloat16):
        assert_same(out[True, dtype], out[False, dtype], str(dtype))


def test_autodiff_rollout_after_reset():
    from smokephysai_b200 import autodiff
    res = []
    for deferred in (True, False):
        ns = make(128, 128, 16, 20)
        if not deferred:
            eager(ns)
        dirty(ns, 16, 128, 128)
        ns.setup_grid()
        ns.add_sources(emitters(16, 128, 128, 3))
        state = tuple(getattr(ns, k).clone().requires_grad_(True) for k in ("u", "v", "p", "density"))
        frames, *_ = autodiff.rollout(state, 3, dt=0.01, viscosity=0.001, jacobi_iters=20)
        frames.square().sum().backward()
        res.append([N(frames)] + [N(t.grad) for t in state])
    for a, b in zip(*res):
        assert_same(a, b, "rollout")
    assert np.any(res[0][0])
