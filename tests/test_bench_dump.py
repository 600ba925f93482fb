"""bench.py --dump-outputs and --steps, host side: what the dump writes of an output array is bounded, fp32, named by
workload and rank, and the same rows in every process; --steps reaches every workload of the line."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

import bench
from conftest import ROOT


def test_small_array_is_dumped_whole():
    t = torch.arange(24.0).reshape(2, 3, 4)
    assert np.array_equal(bench.dump_sample(t), t.numpy())


def pitched_rows(rows, pitch, cols):
    """A pitched buffer cropped to its logical columns, as the frames and state views are; every row holds its own index."""
    return torch.arange(rows, dtype=torch.float32)[:, None].expand(rows, pitch).reshape(100, rows // 100, pitch)[..., :cols]


def test_large_array_is_a_fixed_sample_of_its_rows():
    t = pitched_rows(100 * 100, 132, 129)
    a = bench.dump_sample(t)
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_MAX_VALUES // 129, 129)
    assert (a == a[:, :1]).all()                     # whole rows
    assert (np.diff(a[:, 0]) > 0).all()              # distinct rows, in order
    # another process picks the same rows
    code = ("import sys; sys.path.insert(0, %r); import bench, torch; from test_bench_dump import pitched_rows; "
            "print(bench.dump_sample(pitched_rows(100 * 100, 132, 129))[:, 0].astype(int).tolist())"
            % os.path.join(ROOT, "tests"))
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, check=True,
                         env=dict(os.environ, PYTHONPATH=ROOT))
    assert json.loads(out.stdout) == a[:, 0].astype(int).tolist()


@pytest.mark.parametrize("world", [1, 4])
def test_dump_outputs_names_dtype_and_budget(tmp_path, world):
    arrays = {"frames": pitched_rows(100 * 100, 132, 129), "density": torch.ones(3, 5, dtype=torch.float64)}
    written = {}
    for rank in range(world):
        ctx = types.SimpleNamespace(world=world, rank=rank, args=types.SimpleNamespace(dump_outputs=str(tmp_path / "d")))
        bench.dump_outputs(ctx, "c2", arrays)
    for name in sorted(os.listdir(tmp_path / "d")):
        written[name] = np.load(tmp_path / "d" / name)
    want = ["c2_%s.npy" % n for n in ("density", "frames")] if world == 1 else \
        sorted("c2_rank%d_%s.npy" % (r, n) for r in range(world) for n in ("density", "frames"))
    assert sorted(written) == want
    assert all(a.dtype == np.float32 for a in written.values())
    assert sum(a.size for n, a in written.items() if "frames" in n) <= bench.DUMP_MAX_VALUES   # the budget holds over all ranks
    assert all(np.array_equal(a, np.ones((3, 5))) for n, a in written.items() if "density" in n)


@pytest.mark.parametrize("world,want", [(1, ["c2", "c3", "c4"]), (2, ["c2", "c2s", "c4"])])
def test_steps_reach_every_workload(monkeypatch, capsys, world, want):
    seen = []

    class Ctx:
        def __init__(self, args):
            self.args, self.world, self.rank = args, world, 0
            self.dist = types.SimpleNamespace(destroy_process_group=lambda: None)

    def run(ctx, key, steps, warmup):
        seen.append((key, steps, warmup))
        return {"value": 0.0}
    monkeypatch.setattr(bench, "Ctx", Ctx)
    monkeypatch.setattr(bench, "run_batched", run)
    monkeypatch.setattr(bench, "run_slab", run)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "37", "--warmup", "4", "--no-cpu-baseline"])
    assert bench.main() == 0
    assert seen == [(k, 37, 4) for k in want]
    json.loads(capsys.readouterr().out)
