"""Half-precision frame output (SMK_FRAME_F16 / _BF16) of every frame-writing kernel, against fp32 twins.

Two simulators start from the same seeded state (emitter-like density, velocities large enough that back-traces leave
the advection tiles); one writes fp32 frames, the other fp16 or bf16.  The half frames must be bit-equal to torch's
conversion of the fp32 frames -- on the cells and on every padding column the fp32 path writes (both buffers start
as NaN, so a position one path writes and the other skips shows) -- and the final u, v, p, density of the twins must
be bit-equal: the frame format never touches the solver.
"""
import ctypes as C
import zlib

import numpy as np
import pytest
import torch

from helpers import smk_env

pytestmark = pytest.mark.gpu

from smokephysai_b200 import NavierStokesSimulator, SmokeSimulator, _lib  # noqa: E402

FIELDS = ("u", "v", "p", "density")
HALF = [torch.float16, torch.bfloat16]


def make(h, w, B=1, K=12, dt=0.02, nu=0.004, **kw):
    return NavierStokesSimulator((h, w), dt, nu, "cuda", jacobi_iters=K, batch=B, **kw)


def seeded_state(h, w, B, seed, vel=300.0, density_scale=None):
    rng = np.random.default_rng(seed)
    st = {
        "u": ((rng.random((B, h + 1, w)) - 0.5) * vel).astype(np.float32),
        "v": ((rng.random((B, h, w + 1)) - 0.5) * vel).astype(np.float32),
        "p": rng.standard_normal((B, h, w)).astype(np.float32),
        "density": rng.random((B, h, w)).astype(np.float32),
    }
    if density_scale is not None:
        st["density"] = (st["density"] * density_scale(rng, (B, h, w))).astype(np.float32)
    return st


def load(ns, st):
    for k in FIELDS:
        t = torch.from_numpy(st[k]).cuda()
        setattr(ns, k, t if ns.batch > 1 else t[0])


def bits(t):
    t = t.contiguous()
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def assert_state_equal(a, b, what):
    for k in FIELDS:
        assert torch.equal(bits(getattr(a, k)), bits(getattr(b, k))), "%s: %s differs between the fp32 and the half twin" % (what, k)


def assert_frames_cast(half, f32, dtype, what):
    """half == f32.to(dtype) bit for bit (torch's CPU conversion), NaN sentinels included."""
    half, want = half.cpu(), f32.cpu().to(dtype)
    assert half.dtype == dtype and half.shape == want.shape, "%s: %s %s vs %s" % (what, half.dtype, tuple(half.shape), tuple(want.shape))
    nh, nw = torch.isnan(half), torch.isnan(want)
    assert torch.equal(nh, nw), "%s: %d positions written by one path only" % (what, int((nh ^ nw).sum()))
    hb, wb = bits(half)[~nh], bits(want)[~nh]
    if not torch.equal(hb, wb):
        k = int(torch.nonzero(hb != wb)[0])
        raise AssertionError("%s: %d elements differ, first %r vs %r (fp32 %r)" % (
            what, int((hb != wb).sum()), half[~nh][k].item(), want[~nh][k].item(), f32.cpu()[~nh][k].item()))


def twins(h, w, B, n, dtype, with_fmul, seed, env=None, vel=300.0, density_scale=None, **kw):
    """Run n steps of the fp32 twin and the `dtype` twin into NaN-filled [B, n, h, pitch_c] buffers; check frames, state and
    launch counts; return (fp32 frames, half frames)."""
    env = env or {}
    with smk_env(**env):
        sims = {dt: make(h, w, B, **kw) for dt in (torch.float32, dtype)}
        st = seeded_state(h, w, B, seed, vel, density_scale)
        pc = sims[torch.float32]._layout.pitch_c
        g = torch.Generator().manual_seed(seed)
        fmul = (torch.rand(h, pc, generator=g) * 0.05).cuda() if with_fmul else None
        out, launched = {}, {}
        for dt, ns in sims.items():
            load(ns, st)
            out[dt] = torch.full((B, n, h, pc), float("nan"), dtype=dt, device="cuda")
            n0 = _lib.launch_count()
            ns.run_steps(n, fmul=fmul, out=out[dt])
            launched[dt] = _lib.launch_count() - n0
        torch.cuda.synchronize()
    what = "%dx%d x%d, %d steps, %s, fmul %s, %s" % (h, w, B, n, dtype, with_fmul, env)
    assert launched[dtype] == launched[torch.float32], "%s: %d launches against %d for fp32" % (what, launched[dtype], launched[torch.float32])
    assert not torch.isnan(out[torch.float32][..., :w]).any(), what + ": fp32 frames incomplete"
    assert_frames_cast(out[dtype], out[torch.float32], dtype, what)
    assert_state_equal(sims[torch.float32], sims[dtype], what)
    return out[torch.float32], out[dtype]


# ---- every frame writer --------------------------------------------------------------------------------------------
CASES = {
    # k_advect (the phase path's direct advection): small batch, and a ragged width that is not a multiple of 4
    "k_advect_64x64x3": dict(h=64, w=64, B=3, n=3, step_kernel="phases"),
    "k_advect_61x83": dict(h=61, w=83, B=2, n=3, step_kernel="phases"),
    # k_advect_tiled forced, interior tiles staged by TMA and with cp.async everywhere; ragged grid with interior and edge tiles
    "k_advect_tiled_tma": dict(h=133, w=389, B=2, n=2, step_kernel="phases", env={"SMK_ADVECT_TILED": 1}),
    "k_advect_tiled_cp_async": dict(h=133, w=389, B=2, n=2, step_kernel="phases", env={"SMK_ADVECT_TILED": 1, "SMK_ADVECT_TMA": 0}),
    # k_step_fused: one CTA per simulation at 128 x 128, the generic size, and the time-sliced schedule
    "k_step_fused_128x128x12": dict(h=128, w=128, B=12, n=4, step_kernel="fused", env={"SMK_FUSED_CLUSTER": 0, "SMK_FUSED_SLICE": 0}),
    "k_step_fused_60x128": dict(h=60, w=128, B=3, n=4, step_kernel="fused", env={"SMK_FUSED_CLUSTER": 0, "SMK_FUSED_SLICE": 0}),
    "k_step_fused_sliced": dict(h=128, w=128, B=5, n=7, step_kernel="fused", env={"SMK_FUSED_CLUSTER": 0, "SMK_FUSED_SLICE": 3}),
    # k_step_cluster: a simulation on a cluster of 2 / 4 CTAs
    "k_step_cluster_2": dict(h=128, w=128, B=3, n=3, step_kernel="fused", env={"SMK_FUSED_CLUSTER": 2, "SMK_FUSED_SLICE": 0}),
    "k_step_cluster_4": dict(h=128, w=128, B=3, n=3, step_kernel="fused", env={"SMK_FUSED_CLUSTER": 4, "SMK_FUSED_SLICE": 0}),
}


@pytest.mark.parametrize("with_fmul", [False, True])
@pytest.mark.parametrize("dtype", HALF, ids=["f16", "bf16"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_half_frames_of_every_writer_equal_the_fp32_frames_cast(case, dtype, with_fmul):
    kw = dict(CASES[case])
    env = kw.pop("env", None)
    twins(kw.pop("h"), kw.pop("w"), kw.pop("B"), kw.pop("n"), dtype, with_fmul, seed=zlib.crc32(case.encode()) & 0xffff, env=env, **kw)


@pytest.mark.parametrize("with_fmul", [False, True])
@pytest.mark.parametrize("dtype", HALF, ids=["f16", "bf16"])
def test_half_frames_default_dispatch_at_full_size(dtype, with_fmul):
    """2560^2 (6.6 M cells) with no SMK_* override: the library's own choice for big grids (tiled advection with the gradient
    subtract fused into the u advection, TMA staging)."""
    with smk_env(**{k: None for k in ("SMK_ADVECT_TILED", "SMK_ADVECT_TMA", "SMK_PROJECT_FUSED", "SMK_FUSED_CLUSTER", "SMK_FUSED_SLICE")}):
        twins(2560, 2560, 1, 2, dtype, with_fmul, seed=2560, K=20)


# ---- range: subnormals and overflow ---------------------------------------------------------------------------------
def block_magnitudes(rng, shape):
    """Per 16 x 16 block a magnitude from 1e-44 to 1e6 (evenly spaced exponents, shuffled): the interior of a block is out
    of reach of its neighbours for a few small-dt steps, so tiny blocks stay tiny."""
    B, h, w = shape
    e = rng.permutation(np.linspace(-44.0, 6.0, B * (h // 16) * (w // 16))).reshape(B, h // 16, w // 16)
    return np.repeat(np.repeat(10.0 ** e, 16, axis=1), 16, axis=2)


@pytest.mark.parametrize("dtype", HALF, ids=["f16", "bf16"])
@pytest.mark.parametrize("kind", ["phases", "fused"])
def test_half_frames_round_like_torch_across_the_range(dtype, kind):
    """Density blocks from 1e-44 to 1e6 (dt = 1e-3 keeps the buoyant velocities at a fraction of a cell per step): the fp32
    frames hold fp32 subnormals, fp16 subnormals and values above 65504 (fp16 overflow); the half frames must still equal
    torch's conversion -- inf, subnormals, rounding."""
    h = w = 64 if kind == "phases" else 128
    env = {"SMK_FUSED_CLUSTER": 0, "SMK_FUSED_SLICE": 0}
    f32, _ = twins(h, w, 2, 2, dtype, False, seed=77, env=env, vel=1.0, density_scale=block_magnitudes, step_kernel=kind, dt=1e-3)
    a = f32[..., :w].abs().cpu()
    assert ((a > 0) & (a < 1.1754944e-38)).any(), "no fp32 subnormal in the frames"
    assert ((a > 6e-8) & (a < 6.1035156e-05)).any(), "no fp16 subnormal in the frames"
    assert (a > 65504).any(), "no value above the fp16 range in the frames"


# ---- the Python surface ---------------------------------------------------------------------------------------------
def pair(h=64, w=64, B=2, **kw):
    st = seeded_state(h, w, B, 4321)
    a, b = make(h, w, B, **kw), make(h, w, B, **kw)
    load(a, st)
    load(b, st)
    return a, b


@pytest.mark.parametrize("dtype", HALF, ids=["f16", "bf16"])
@pytest.mark.parametrize("kernel", ["phases", "fused"])
def test_api_step_step_into_run_steps(dtype, kernel):
    a, b = pair(step_kernel=kernel)
    L = a._layout
    fmul = torch.rand(L.h, L.pitch_c, device="cuda") * 0.05
    # step(): dtype, shape, value
    f32, fh = a.step(fmul=fmul), b.step(fmul=fmul, frame_dtype=dtype)
    assert fh.dtype == dtype and tuple(fh.shape) == (2, 64, 64)
    assert_frames_cast(fh, f32, dtype, "step()")
    # step_into(): a caller-owned half buffer
    buf32 = torch.full((2, L.h, L.pitch_c), float("nan"), device="cuda")
    bufh = torch.full((2, L.h, L.pitch_c), float("nan"), dtype=dtype, device="cuda")
    a.step_into(buf32, fmul)
    b.step_into(bufh, fmul)
    assert_frames_cast(bufh, buf32, dtype, "step_into()")
    # run_steps(): allocated, and into out= (whose dtype is the frame dtype)
    f32, fh = a.run_steps(3), b.run_steps(3, frame_dtype=dtype)
    assert fh.dtype == dtype and tuple(fh.shape) == (2, 3, 64, 64)
    assert_frames_cast(fh, f32, dtype, "run_steps()")
    o32 = torch.full((2, 2, L.h, L.pitch_c), float("nan"), device="cuda")
    oh = torch.full((2, 2, L.h, L.pitch_c), float("nan"), dtype=dtype, device="cuda")
    r32, rh = a.run_steps(2, out=o32), b.run_steps(2, out=oh, frame_dtype=dtype)
    assert rh.dtype == dtype
    assert_frames_cast(oh, o32, dtype, "run_steps(out=)")
    # run_steps_time_major()
    t32 = torch.full((3, 2, L.h, L.pitch_c), float("nan"), device="cuda")
    th = torch.full((3, 2, L.h, L.pitch_c), float("nan"), dtype=dtype, device="cuda")
    a.run_steps_time_major(3, t32, fmul=fmul)
    b.run_steps_time_major(3, th, fmul=fmul)
    assert_frames_cast(th, t32, dtype, "run_steps_time_major()")
    torch.cuda.synchronize()
    assert_state_equal(a, b, "API sequence")


def test_api_cpu_output_device_with_half_frames():
    st = seeded_state(48, 52, 1, 99)
    a = NavierStokesSimulator((48, 52), 0.02, 0.004, "cpu", jacobi_iters=8)
    b = NavierStokesSimulator((48, 52), 0.02, 0.004, "cuda", jacobi_iters=8)
    load(a, st)
    load(b, st)
    fa = a.step(frame_dtype=torch.bfloat16)
    fb = b.step()
    assert fa.device.type == "cpu" and fa.dtype == torch.bfloat16 and tuple(fa.shape) == (48, 52)
    assert_frames_cast(fa, fb, torch.bfloat16, "device='cpu' step()")
    ra = a.run_steps(2, frame_dtype=torch.float16)
    rb = b.run_steps(2)
    assert ra.device.type == "cpu" and ra.dtype == torch.float16
    assert_frames_cast(ra, rb, torch.float16, "device='cpu' run_steps()")


def emitters(B, seed=5):
    rng = np.random.default_rng(seed)
    return [[((int(rng.integers(20, 108)), int(rng.integers(20, 108))), float(rng.uniform(0.5, 2.0)))
             for _ in range(int(rng.integers(1, 4)))] for _ in range(B)]


@pytest.mark.parametrize("kernel", ["phases", "fused"])
def test_api_generate_sequences(kernel):
    B, T = 4, 5
    ems = emitters(B)
    sim = SmokeSimulator((128, 128), device="cuda", batch=B, jacobi_iters=40, step_kernel=kernel)
    ref = sim.generate_sequences(ems, T).clone()
    for dtype in HALF:
        d = sim.generate_sequences(ems, T, frame_dtype=dtype)
        assert d.is_cuda and d.dtype == dtype and tuple(d.shape) == (B, T, 128, 128)
        assert_frames_cast(d, ref, dtype, "generate_sequences(to_host=False, %s)" % dtype)
    # to_host: alternating fp32 / fp16 / bf16 / fp32 calls on one simulator; each dtype keeps its own pinned buffer
    h32 = sim.generate_sequences(ems, T, to_host=True)
    assert h32.is_pinned() and h32.dtype == torch.float32 and tuple(h32.shape) == (B, T, 128, 128)
    assert torch.equal(bits(h32), bits(ref.cpu())), "to_host fp32 vs device fp32"
    first = h32.clone()
    for dtype in HALF:
        hh = sim.generate_sequences(ems, T, to_host=True, frame_dtype=dtype)
        assert hh.is_pinned() and hh.dtype == dtype and tuple(hh.shape) == (B, T, 128, 128)
        assert_frames_cast(hh, first, dtype, "generate_sequences(to_host=True, %s)" % dtype)
        assert torch.equal(bits(h32), bits(first)), "a %s call overwrote the fp32 call's host frames" % dtype
    again = sim.generate_sequences(ems, T, to_host=True, steps_per_copy=2)
    assert torch.equal(bits(again), bits(first)), "fp32 after fp16 / bf16 calls differs from the first fp32 call"


@pytest.mark.parametrize("kernel", ["phases", "fused"])
def test_half_frames_take_no_extra_launch(kernel):
    """The conversion is inside the frame-writing kernels: the half call launches exactly what the fp32 call launches."""
    a, b = pair(128, 128, 2, step_kernel=kernel)
    counts = []
    for ns, dt in ((a, torch.float32), (b, torch.float16)):
        n0 = _lib.launch_count()
        ns.run_steps(3, frame_dtype=dt)
        n1 = _lib.launch_count()
        ns.step(frame_dtype=dt)
        counts.append((n1 - n0, _lib.launch_count() - n1))
    assert counts[0] == counts[1] and counts[0][0] >= 1


# ---- rejections -----------------------------------------------------------------------------------------------------
def test_unsupported_frame_dtypes_are_refused():
    ns = make(32, 32)
    L = ns._layout
    for bad in (torch.float64, torch.int8):
        with pytest.raises(ValueError, match="bfloat16"):
            ns.step(frame_dtype=bad)
        with pytest.raises(ValueError, match="bfloat16"):
            ns.run_steps(2, frame_dtype=bad)
        with pytest.raises(ValueError, match="bfloat16"):
            ns.step_into(torch.zeros(1, L.h, L.pitch_c, dtype=bad, device="cuda"))
        with pytest.raises(ValueError, match="bfloat16"):
            ns.run_steps_time_major(2, torch.zeros(2, 1, L.h, L.pitch_c, dtype=bad, device="cuda"))
    with pytest.raises(ValueError, match="disagrees"):
        ns.run_steps(2, out=torch.zeros(1, 2, L.h, L.pitch_c, dtype=torch.float16, device="cuda"), frame_dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="disagrees"):
        ns.run_steps(2, out=torch.zeros(1, 2, L.h, L.pitch_c, device="cuda"), frame_dtype=torch.float16)
    sim = SmokeSimulator((32, 32), device="cuda")
    with pytest.raises(ValueError, match="bfloat16"):
        sim.generate_sequences([[((16, 16), 1.0)]], 3, to_host=True, frame_dtype=torch.float64)


def test_abi_rejects_bad_frame_format_and_misaligned_half_frames():
    ns = make(32, 32, step_kernel="phases")
    L, lib = ns._layout, _lib.load()
    buf = torch.zeros(1, 2, L.h, L.pitch_c + 8, dtype=torch.float16, device="cuda")
    prm = ns._params()
    s = _lib.stream_on(ns._cuda)
    step_stride, batch_stride = L.h * L.pitch_c, 2 * L.h * L.pitch_c

    def run(ptr, fmt):
        return lib.smk_run_steps_ex(C.byref(ns._grid), C.byref(ns._state), C.byref(prm), 2, ptr, step_stride, batch_stride,
                                    None, fmt, s)
    n0 = _lib.launch_count()
    assert run(buf.data_ptr(), 3) == -1 and b"frame_format" in lib.smk_last_error_string()
    assert run(buf.data_ptr(), -1) == -1
    assert run(buf.data_ptr() + 2, _lib.FRAME_FORMATS[torch.float16]) == -1 and b"aligned" in lib.smk_last_error_string()
    assert run(buf.data_ptr() + 4, _lib.FRAME_FORMATS[torch.bfloat16]) == -1
    assert lib.smk_step_ex(C.byref(ns._grid), C.byref(ns._state), C.byref(prm), buf.data_ptr() + 2, step_stride, None, 1, s) == -1
    assert lib.smk_step_ex(C.byref(ns._grid), C.byref(ns._state), C.byref(prm), buf.data_ptr(), step_stride, None, 7, s) == -1
    assert _lib.launch_count() == n0, "a rejected call launched kernels"
    # 8-byte alignment is enough for a half frame (4 elements): accepted
    assert run(buf.data_ptr() + 8, _lib.FRAME_FORMATS[torch.float16]) == 0
    torch.cuda.synchronize()
    assert _lib.launch_count() > n0
