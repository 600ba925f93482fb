"""CPU-only checks of the half-precision frame output: the SMK_FRAME_* codes of the header agree with the ctypes map, the
Python side rejects dtypes it cannot write, and the library's frame-writing kernels hold the fp32 -> f16 / bf16 packing
conversions (so the rounding happens in their epilogue, not in a separate cast)."""
import os
import re
import shutil
import subprocess

import pytest
import torch

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "smoke_b200.h")


@pytest.fixture(scope="module")
def so_path():
    from smokephysai_b200 import build
    return build.build()


def test_frame_format_codes_match_the_header():
    from smokephysai_b200 import _lib
    src = open(HEADER).read()
    m = re.search(r"enum\s*\{\s*(SMK_FRAME_F32[^}]*)\}", src)
    assert m, "SMK_FRAME_* enum missing from the header"
    codes = {k: int(v) for k, v in re.findall(r"(SMK_FRAME_\w+)\s*=\s*(\d+)", m.group(1))}
    assert codes == {"SMK_FRAME_F32": 0, "SMK_FRAME_F16": 1, "SMK_FRAME_BF16": 2}
    assert _lib.FRAME_FORMATS == {torch.float32: codes["SMK_FRAME_F32"], torch.float16: codes["SMK_FRAME_F16"],
                                  torch.bfloat16: codes["SMK_FRAME_BF16"]}
    for dt, code in _lib.FRAME_FORMATS.items():
        assert _lib.frame_format(dt) == code
    for bad in (torch.float64, torch.int8, torch.float8_e4m3fn, torch.int16):
        with pytest.raises(ValueError, match="float16"):
            _lib.frame_format(bad)


def test_abi_version_unchanged_and_ex_entries_exported(so_path):
    from smokephysai_b200 import _lib
    lib = _lib.load()
    assert lib.smk_version() == 7
    syms = subprocess.check_output(["nm", "-D", "--defined-only", so_path]).decode()
    assert re.search(r" T smk_step_ex$", syms, flags=re.M) and re.search(r" T smk_run_steps_ex$", syms, flags=re.M)


def _sass_functions(so_path):
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([tool, "-sass", so_path], capture_output=True, text=True, check=True).stdout
    out = {}
    for part in re.split(r"\n\s*Function : ", sass)[1:]:
        name, body = part.split("\n", 1)
        out[name.strip()] = body
    return out


@pytest.mark.parametrize("kernel", ["k_step_fusedILb0", "k_step_fusedILb1", "k_step_clusterILi2", "k_step_clusterILi4",
                                    "k_advectILb0", "k_advect_tiledILb0ELi0"])
def test_frame_writers_convert_in_their_epilogue(so_path, kernel):
    """Every kernel that writes a frame carries both packing conversions: F2FP.F16.F32.PACK_AB (cvt.rn.f16x2.f32) and
    F2FP.BF16.F32.PACK_AB (cvt.rn.bf16x2.f32)."""
    funcs = {n: b for n, b in _sass_functions(so_path).items() if kernel in n}
    assert funcs, "no SASS function matches %s" % kernel
    for name, body in funcs.items():
        assert "F2FP.F16.F32.PACK_AB" in body, "%s: no fp32 -> f16 conversion" % name
        assert "F2FP.BF16.F32.PACK_AB" in body, "%s: no fp32 -> bf16 conversion" % name
