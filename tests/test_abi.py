"""CPU tests of the C-ABI boundary: the shared libraries load, export every symbol the headers declare, the
`instance` mirror matches the compiled reference's layout, and the product fails loudly without a GPU."""
import ctypes as C
import os
import re

import pytest

from conftest import HAVE_GPU, ROOT
from tsp_optimization_b200 import engine as eng


def _declared(header):
    txt = open(os.path.join(ROOT, "include", header)).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(tspb200_[a-z0-9_]+|calc_dist|alg_2opt_tabu|alg_2opt|reverse_path|greedy|HEU_Greedy_iter|HEU_extramileage)\s*\(", txt)))


def test_libtspb200_exports_every_declared_symbol():
    L = eng.load_library()
    names = [n for n in _declared("tspb200.h")]
    assert set(names) == set(eng.ABI_SYMBOLS)
    for nm in names:
        assert hasattr(L, nm), nm


def test_dropin_exports_reference_symbols():
    L = C.CDLL(eng.DROPIN_PATH)
    for nm in _declared("tspb200_dropin.h"):
        assert hasattr(L, nm), nm
    for nm in ("calc_dist", "alg_2opt", "alg_2opt_tabu", "reverse_path", "greedy", "HEU_Greedy_iter", "HEU_extramileage"):
        assert hasattr(L, nm) and nm in _declared("tspb200_dropin.h")


def test_instance_mirror_matches_reference_layout(reference_outputs, reflib_if_built):
    L = C.CDLL(eng.DROPIN_PATH)
    buf = (C.c_longlong * 32)()
    k = L.tspb200_dropin_layout(buf, 32)
    mine = [int(buf[t]) for t in range(k)]
    assert mine == reference_outputs["layout"]
    if reflib_if_built:
        ref = reflib_if_built.layout()
        assert mine == [ref[key] for key in reflib_if_built.LAYOUT_KEYS]
    assert mine[0] == 152 and mine[4] == 80 and mine[8] == 120 and mine[9] == 128  # SURVEY.md §8(b)


def test_dropin_reverse_path_matches_reference_semantics(oracle):
    """reverse_path works on host arrays (no GPU involved): compare with the oracle's restatement."""
    import numpy as np
    from test_gpu_parity import RefInstance
    n = 12
    succ = np.roll(np.arange(n, dtype=np.int32), -1)
    inst = RefInstance(np.zeros((n, 2)), 0, succ)
    prev = np.roll(np.arange(n, dtype=np.int32), 1).copy()
    L = C.CDLL(eng.DROPIN_PATH)
    L.reverse_path.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    # apply the 2-opt move (a=2, b=7): succ[a]=b; succ[a1]=b1; reverse_path(b, a1)
    a, b = 2, 7
    a1, b1 = int(succ[a]), int(succ[b])
    s2, p2 = succ.copy(), prev.copy()
    for arr in (None,):
        inst.set_succ_entry(a, b)
        inst.set_succ_entry(a1, b1)
    s2[a] = b
    s2[a1] = b1
    L.reverse_path(C.byref(inst.c), b, a1, prev.ctypes.data)
    oracle.L.orc_reverse_path(n, s2, b, a1, p2)
    assert (inst.succ() == s2).all() and (prev == p2).all()


@pytest.mark.skipif(HAVE_GPU, reason="only meaningful without a GPU")
def test_product_fails_loudly_without_gpu():
    with pytest.raises(eng.TspB200Error) as ei:
        eng.Engine(0)
    assert "no CPU fallback" in str(ei.value)


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "tsp_optimization_b200")):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dirpath, fn)).read()
                assert "tsp_oracle" not in txt and "from oracle" not in txt and "import oracle" not in txt, fn


def test_c_example_compiles_against_the_public_header(tmp_path):
    """examples/two_opt_greedy.c: plain C against include/tspb200.h + libtspb200.so (no CUDA headers on the caller's side).
    Without a GPU it must stop with the library's own error message, not run on the CPU."""
    import subprocess
    exe = str(tmp_path / "two_opt_greedy")
    lib = os.path.dirname(eng.LIB_PATH)
    r = subprocess.run(["gcc", "-O2", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "two_opt_greedy.c"), "-L" + lib, "-ltspb200", "-Wl,-rpath," + lib, "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    tsp = tmp_path / "sq.tsp"
    tsp.write_text("NAME : sq\nTYPE : TSP\nDIMENSION : 5\nEDGE_WEIGHT_TYPE : EUC_2D\nNODE_COORD_SECTION\n"
                   "1 0 0\n2 10 0\n3 0 10\n4 10 10\n5 5 5\nEOF\n")
    r = subprocess.run([exe, str(tsp)], capture_output=True, text=True)
    if HAVE_GPU:
        assert r.returncode == 0 and "2-opt (first improvement)" in r.stdout, r.stdout + r.stderr
    else:
        assert r.returncode == 1 and "no CPU fallback" in r.stderr


def test_vns_session_example_compiles_and_runs(tmp_path):
    """examples/vns_resident.c: the reference's HEU_VNS loop on the resident-session entry points, plain C.  On a GPU it must
    finish with the restored incumbent equal to the best cost it saw; without one it stops with the library's error."""
    import subprocess
    exe = str(tmp_path / "vns_resident")
    lib = os.path.dirname(eng.LIB_PATH)
    r = subprocess.run(["gcc", "-O2", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "vns_resident.c"), "-L" + lib, "-ltspb200", "-Wl,-rpath," + lib, "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe, "1500", "12", "123"], capture_output=True, text=True)
    if HAVE_GPU:
        assert r.returncode == 0 and "best tour after 12 kicks" in r.stdout, r.stdout + r.stderr
    else:
        assert r.returncode == 1 and "no CPU fallback" in r.stderr
