"""Codegen canaries for the two exhaustive scan kernels since the stage-1 prefilter (csrc/kernels_bi_scan.cuh):
bi_scan_sqrt_kernel — the square-root filter alone, which runs pruned passes and smaller tours — keeps the properties
tests/test_codegen.py watches on bi_scan_kernel, and the prefilter kernel keeps its square roots off the column loop."""
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT

LIB = os.path.join(ROOT, "tsp_optimization_b200", "lib")
SHAPES = ["ILi64ELi8ELb0ELb1ELb0ELb1", "ILi64ELi8ELb0ELb0ELb0ELb1", "ILi64ELi8ELb1ELb1ELb0ELb1", "ILi64ELi8ELb0ELb1ELb0ELb0",
          "ILi128ELi8ELb0ELb1ELb0ELb0", "ILi128ELi16ELb0ELb1ELb0ELb0"]


def _obj_of(shape: str) -> str:
    if shape.startswith("ILi128E"):
        return os.path.join(LIB, "kernels_bi_128.o")
    if shape.startswith("ILi256E"):
        return os.path.join(LIB, "kernels_bi_256.o")
    return os.path.join(LIB, "kernels_bi_s64.o" if shape.endswith("ELb1") else "kernels_bi_p64.o")


def _sass(kernel: str, shape: str) -> str:
    obj = _obj_of(shape)
    if not shutil.which("cuobjdump") or not os.path.exists(obj):
        pytest.skip("cuobjdump or the built object is not available")
    mangled = f"_ZN4tspb{len(kernel)}{kernel}{shape}EEEvNS_6BiArgsE"
    r = subprocess.run(["cuobjdump", "-sass", "-fun", mangled, obj], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "Function" in r.stdout, r.stderr[-500:]
    return r.stdout


@pytest.mark.parametrize("shape", SHAPES)
def test_sqrt_scan_hot_loop_stays_in_the_uniform_datapath(shape):
    """bi_scan_sqrt_kernel<T, R, ATT, EXACT32, PRUNED=false, SHUF>: LDS.128 [UR + imm] column reads, packed FP32x2, one
    MUFU.SQRT per distance, the TMA bulk copy and (shuffle variant) SHFL.DOWN"""
    sass = _sass("bi_scan_sqrt_kernel", shape)
    assert len(re.findall(r"LDS\.128 R\d+, \[UR", sass)) >= 4
    assert "FFMA2" in sass and "FADD2" in sass and "UBLKCP" in sass
    assert sass.count("MUFU.SQRT") >= 8 * int(re.match(r"ILi\d+ELi(\d+)E", shape).group(1))
    if shape.endswith("ELb1"):
        assert "SHFL.DOWN" in sass


@pytest.mark.parametrize("shape", [s for s in SHAPES if s.startswith("ILi64")])
def test_prefilter_scan_has_no_square_root_per_distance(shape):
    """bi_scan_kernel (prefilter): the column loop computes squared distances only; the few MUFU.SQRT left belong to the
    inline stage-2 re-check of a hit (two per loop copy), against tens in every copy of the square-root kernel's loop"""
    assert _sass("bi_scan_kernel", shape).count("MUFU.SQRT") <= 8
