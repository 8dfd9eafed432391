"""The stage-1 prefilter in its dot-product form (csrc/kernels_bi_scan.cuh, pf_dot_const; DESIGN.md §3) on the inputs its
rounding margins depend on: coordinates far from the origin that the engine translates exactly, and coordinates it cannot
translate.  Move logs, tours and costs with the prefilter on must equal those with it off and the oracle's.  Plus a codegen
canary on the column loop the headline pass runs."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import GOLD_DIR, ROOT
from test_gpu_prefilter import _check
from tsp_optimization_b200 import engine as eng
from tsp_optimization_b200.instances import uniform_instance

BI = eng.BI


def _offset_instance(n, seed):
    """integer coordinates in 2^23 - 10^4 + [0, 10^4]: FP32-exact, translated by about 2^23 - 5000"""
    rng = np.random.default_rng(seed)
    return 2.0 ** 23 - 1e4 + np.floor(rng.random((n, 2)) * 1e4)


def _untranslatable_instance(n, seed):
    """FP32-exact non-integer coordinates in [0, 1000) plus one point near 0: no exact integer translation exists"""
    rng = np.random.default_rng(seed)
    xy = (rng.random((n, 2)) * 1e3).astype(np.float32).astype(np.float64)
    xy[0] = [np.float32(1e-3), np.float32(2e-3)]
    return xy


@pytest.mark.gpu
@pytest.mark.parametrize("make", [_offset_instance, _untranslatable_instance])
def test_dot_prefilter_on_off_oracle(engine, oracle, make):
    xy = make(2500, 7)
    succ, _ = oracle.nn_tour(xy, 0, 0)
    _check(engine, oracle, xy, 0, succ, max_passes=60)


@pytest.mark.gpu
@pytest.mark.parametrize("make", [_offset_instance, _untranslatable_instance])
def test_dot_prefilter_auto_at_scale(engine, make):
    """n = 45 000: the automatic rule runs the prefilter kernel (stage-1 hits are counted); the same moves, tour and cost
    as with the square-root kernel alone"""
    xy = make(45000, 8)
    engine.set_instance(xy, 0)
    engine.set_option("prune", 0)
    out, hits = {}, {}
    try:
        succ0, _ = engine.nn_tour(0)
        for pf in (-1, 0):
            engine.set_option("prefilter", pf)
            s, obj, st, log = engine.two_opt(BI, succ0, 0.0, max_iters=25, log_cap=1000)
            out[pf] = (s.tolist(), obj, st.moves, log.tolist())
            hits[pf] = engine.info("pf_hits")  # counted since the call's tour upload
    finally:
        engine.set_option("prefilter", -1)
        engine.set_option("prune", -1)
    assert hits[-1] > 0 and hits[0] == 0
    assert out[-1] == out[0] and out[0][2] == 25


@pytest.mark.gpu
def test_dot_prefilter_uni100000_first_moves(engine):
    """the headline instance from its committed NN tour: the first 12 moves of the committed move log; exact-path calls
    at the square-root kernel's rate, stage-1 hits reported"""
    mv = np.load(os.path.join(GOLD_DIR, "uni100000_bi_moves.npz"))["moves"]
    succ = np.load(os.path.join(GOLD_DIR, "nn_uni100000.npz"))["succ"]
    engine.set_instance(uniform_instance(100000), 0)
    engine.set_option("prune", 0)
    cold, hits = {}, {}
    try:
        for pf in (0, 1):
            engine.set_option("prefilter", pf)
            engine.tour_upload(succ, log_cap=64)
            c0, h0 = engine.info("cold_calls"), engine.info("pf_hits")
            st = engine.bi_run(12)
            log = engine.tour_log(64)
            assert st.moves == 12 and log[:, :3].astype(np.int64).tolist() == mv[:12].astype(np.int64).tolist(), pf
            cold[pf], hits[pf] = engine.info("cold_calls") - c0, engine.info("pf_hits") - h0
    finally:
        engine.set_option("prefilter", -1)
        engine.set_option("prune", -1)
    print(f"uni100000, 12 passes: pf_hits {hits[1]}, cold_calls {cold[1]} (square-root kernel: {cold[0]})")
    assert hits[0] == 0 and hits[1] >= cold[1] > 0
    assert abs(cold[1] - cold[0]) <= 0.1 * cold[0] + 100


@pytest.mark.parametrize("att,exact32", [(0, 1), (1, 1), (0, 0), (1, 0)])
def test_dot_prefilter_column_loop_codegen(att, exact32):
    """bi_scan_kernel<64, 8, ATT, EXACT32, PRUNED=0, SHUF=1> (the row-shuffle kernels the prefilter runs for FP32-exact
    coordinates, the headline pass among them, and for coordinates FP32 cannot hold): no spills (ptxas), and the column loop
    is the packed FMA chain — 4 FFMA2 per row pair, 16 per column step, 64 per 4-column block — with no local-memory traffic"""
    obj = os.path.join(ROOT, "tsp_optimization_b200", "lib", "kernels_bi_s64.o")
    if not shutil.which("cuobjdump") or not os.path.exists(obj):
        pytest.skip("cuobjdump or the built object is not available")
    fn = f"_ZN4tspb14bi_scan_kernelILi64ELi8ELb{att}ELb{exact32}ELb0ELb1EEEvNS_6BiArgsE"
    r = subprocess.run(["cuobjdump", "-sass", "-fun", fn, obj], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "Function" in r.stdout, r.stderr[-500:]
    ops = [(int(a, 16), t) for a, t in re.findall(r"/\*([0-9a-f]{4,})\*/\s+([^;]*);", r.stdout)]
    log = os.path.join(os.path.dirname(obj), "kernels_bi_s64.ptxas.log")  # written next to the object by the build
    if os.path.exists(log):
        m = re.search(re.escape(fn) + r"'.*?(\d+) bytes spill stores, (\d+) bytes spill loads", open(log).read(), re.S)
        assert m and m.group(1) == "0" and m.group(2) == "0"
    # the column loops: backward branches whose body holds the FMA chain; count up to the warp ballot
    at = {a: i for i, (a, _) in enumerate(ops)}
    loops = 0
    for i, (a, t) in enumerate(ops):
        m = re.search(r"\bBRA\S*\s+(?:\S+,\s*)?0x([0-9a-f]+)\s*$", t)
        if not m or int(m.group(1), 16) >= a or int(m.group(1), 16) not in at:
            continue
        body = []
        for _, u in ops[at[int(m.group(1), 16)]:i + 1]:
            body.append(u)
            if "VOTE.ANY" in u and "VOTEU" not in u:
                break
        ffma2 = sum(1 for u in body if re.search(r"\bFFMA2\b", u))
        if ffma2 >= 16 * 4 and len(body) < 200:
            loops += 1
            assert not any(re.search(r"\b(FADD2|FMUL2|MUFU|STL|LDL)\b", u) for u in body)
    assert loops >= 2  # the regular and the diagonal tile


@pytest.mark.gpu
def test_dot_prefilter_offset_is_translated(engine):
    """the offset instance filters as well as the same instance moved to the origin: its translation was applied (without
    it the margins, ~ 2^-19 of |P|^2 ~ 2^28, would let nearly every block through to stage 2)"""
    base = _offset_instance(45000, 9) - (2.0 ** 23 - 1e4)
    hits = {}
    engine.set_option("prune", 0)
    engine.set_option("prefilter", 1)
    try:
        for name, xy in (("origin", base), ("offset", base + (2.0 ** 23 - 1e4))):
            engine.set_instance(xy, 0)
            succ0, _ = engine.nn_tour(0)
            engine.two_opt(BI, succ0, 0.0, max_iters=10, log_cap=0)
            hits[name] = engine.info("pf_hits")
    finally:
        engine.set_option("prefilter", -1)
        engine.set_option("prune", -1)
    assert 0 < hits["offset"] <= 1.1 * hits["origin"] + 100, hits
