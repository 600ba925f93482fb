"""CPU checks of the gradient oracle (oracle/torch_step.py), no GPU: its fp32 forward is bit-equal to the C oracle, so torch
autograd through it is the gradient of the reference's arithmetic; and, where the unmodified reference is installed in
baseline/_ref, its gradients equal autograd through the reference's own NavierStokesSimulator."""
import importlib.util
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import torch_step as ts
from conftest import ROOT
from helpers import assert_same, nerr

DT, VISC = 0.01, 0.001


def random_state(B, h, w, seed, vel=150.0):
    """Velocities of a few cells per step (dt = 0.01): back-traces cross cells and hit the clamps."""
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    return [f(B, h + 1, w) * np.float32(vel), f(B, h, w + 1) * np.float32(vel), f(B, h, w) * np.float32(0.1),
            rng.random((B, h, w)).astype(np.float32)]


def rest_state(B, h, w):
    """At rest, with emitters splatted by the C oracle (the splat's expf is held to ulps, not bits)."""
    d = np.zeros((B, h, w), np.float32)
    for b in range(B):
        oracle.splat(d[b], w // 2 + b, h // 3, 6, 1.5)
        oracle.splat(d[b], w // 4, h // 2, 5, 0.7 + b)
    return [np.zeros((B, h + 1, w), np.float32), np.zeros((B, h, w + 1), np.float32), np.zeros((B, h, w), np.float32), d]


@pytest.mark.parametrize("K", [1, 20])
@pytest.mark.parametrize("kind", ["random", "rest"])
def test_restatement_forward_bit_equal_to_c_oracle(K, kind):
    B, h, w, T = 2, 37, 53, 4
    state = random_state(B, h, w, 11 + K) if kind == "random" else rest_state(B, h, w)
    ref = [a.copy() for a in state]
    frames_ref = oracle.run_batch(*ref, DT, VISC, K, T)
    with torch.no_grad():
        frames, final = ts.rollout(tuple(torch.from_numpy(a) for a in state), T, DT, VISC, K)
    assert_same(frames.numpy(), frames_ref, "frames")
    for name, got, want in zip("uvpd", final, ref):
        assert_same(got.numpy(), want, name)


def test_restatement_forward_with_fractal_bit_equal_to_c_oracle():
    B, n, T = 2, 40, 3
    state = random_state(B, n, n, 5, vel=80.0)
    fmul = (np.random.default_rng(3).random((n, n)) * 0.05).astype(np.float32)
    ref = [a.copy() for a in state]
    frames_ref = oracle.run_batch(*ref, DT, VISC, 20, T, fmul=fmul)
    with torch.no_grad():
        frames, _ = ts.rollout(tuple(torch.from_numpy(a) for a in state), T, DT, VISC, 20, fmul=torch.from_numpy(fmul))
    assert_same(frames.numpy(), frames_ref, "fractal frames")


def _reference_navier_stokes():
    path = os.path.join(ROOT, "baseline", "_ref", "src", "physics", "navier_stokes.py")
    if not os.path.exists(path):
        pytest.skip("the unmodified reference is not installed in baseline/_ref")
    spec = importlib.util.spec_from_file_location("reference_navier_stokes", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_restatement_gradients_equal_reference_autograd():
    ref_mod = _reference_navier_stokes()
    h, w, T, K = 12, 12, 2, 20
    state = [torch.from_numpy(a[0]) for a in random_state(1, h, w, 21, vel=120.0)]
    rng = np.random.default_rng(8)
    wf = torch.from_numpy(rng.standard_normal((T, h, w)).astype(np.float32))
    wd = torch.from_numpy(rng.standard_normal((h, w)).astype(np.float32))

    def grads(run):
        leaves = [a.clone().requires_grad_(True) for a in state]
        frames, d = run(leaves)
        ((frames * wf).sum() + (d * wd).sum()).backward()
        return [a.grad.numpy() for a in leaves]

    def reference(leaves):
        ns = ref_mod.NavierStokesSimulator((h, w), DT, VISC, "cpu")
        ns.u, ns.v, ns.p, ns.density = (a.clone() for a in leaves)
        frames = torch.stack([ns.step() for _ in range(T)])
        return frames, ns.density

    def restated(leaves):
        frames, (_, _, _, d) = ts.rollout(tuple(leaves), T, DT, VISC, K)
        return frames, d

    for name, a, b in zip("uvpd", grads(restated), grads(reference)):
        assert nerr(a, b) < 1e-6, (name, nerr(a, b))
