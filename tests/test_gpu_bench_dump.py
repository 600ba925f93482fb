"""bench.py --dump-outputs on the GPU: the files hold exactly what the last timed bench step left, bit for bit.  c2 resets
its state every bench step; c4 carries it from step to step, so only the state after the last timed step matches there."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from conftest import ROOT

pytestmark = pytest.mark.gpu

WARMUP, STEPS = 3, 2


def run_bench(workload, out):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", workload, "--steps", str(STEPS),
           "--warmup", str(WARMUP), "--no-cpu-baseline", "--dump-outputs", str(out)]
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]


def assert_dumped(out, workload, arrays):
    assert sorted(os.listdir(out)) == sorted("%s_%s.npy" % (workload, n) for n in arrays)
    for name, t in arrays.items():
        got = np.load(os.path.join(out, "%s_%s.npy" % (workload, name)))
        assert got.dtype == np.float32
        assert np.array_equal(got, bench.dump_sample(t)), name


def test_c2_dump_is_the_last_timed_step(tmp_path):
    run_bench("c2", tmp_path)
    from smokephysai_b200 import SmokeSimulator
    wl = bench.WORKLOADS["c2"]
    h, w, B, T = wl["h"], wl["w"], wl["batch"], wl["tsteps"]
    sim = SmokeSimulator((h, w), 0.01, 0.001, "cuda:0", jacobi_iters=wl["K"], batch=B)
    ns = sim.ns_solver
    frames = torch.empty(B, T, h, ns._layout.pitch_c, dtype=torch.float32, device="cuda:0")
    src, off, _ = ns.upload_sources([bench.emitters_for_sequence(s, h, w) for s in range(B)])
    ns.setup_grid()
    ns.splat_uploaded(src, off)
    ns.run_steps(T, fmul=sim.fractal_gen.multiplier((h, w), 0.05), out=frames)
    torch.cuda.synchronize()
    assert_dumped(tmp_path, "c2", {"frames": frames[..., :w], "u": ns.u, "v": ns.v, "p": ns.p, "density": ns.density})


def test_c4_dump_is_the_last_timed_step(tmp_path):
    run_bench("c4", tmp_path)
    from smokephysai_b200.slab import SlabNavierStokes
    wl = bench.WORKLOADS["c4"]
    h, w = wl["h"], wl["w"]
    slab = SlabNavierStokes((h, w), 0.01, 0.001, torch.device("cuda", 0), rank=0, world=1, jacobi_iters=wl["K"], sweeps_per_launch=10)
    slab.add_sources(bench.emitters_for_sequence(0, h, w))
    slab.step()                                       # bench.run_slab's eager first step
    for _ in range(WARMUP + STEPS):                   # warm-up and timed bench steps
        slab.run_steps(wl["tsteps"])
    torch.cuda.synchronize()
    assert_dumped(tmp_path, "c4", {name: slab.owned(k) for k, name in (("u", "u"), ("v", "v"), ("p", "p"), ("d", "density"))})
