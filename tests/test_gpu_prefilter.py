"""The scan kernel's stage-1 prefilter (option "prefilter", csrc/kernels_bi_scan.cuh, DESIGN.md §3): squared distances
against per-row and per-column bounds in front of the square-root filter.  It may only add work, never change a move:
move logs, tours, costs and counters with the prefilter on must equal those with it off and the oracle's.  Exhaustive scans
only: pruned passes always run the square-root kernel (tests/test_gpu_parity.py covers them against the oracle)."""
import os

import numpy as np
import pytest

from conftest import GOLD_DIR
from tsp_optimization_b200 import engine as eng
from tsp_optimization_b200.instances import order_to_succ, uniform_instance

pytestmark = pytest.mark.gpu
BI = eng.BI


def _runs(engine, succ0, max_passes):
    out = {}
    engine.set_option("prune", 0)
    for pf in (1, 0):
        engine.set_option("prefilter", pf)
        s, obj, st, log = engine.two_opt(BI, succ0, 0.0, max_iters=max_passes, log_cap=100000)
        out[pf] = (s, obj, st.moves, st.passes, log)
    engine.set_option("prefilter", -1)
    engine.set_option("prune", -1)
    return out


def _check(engine, oracle, xy, wt, succ0, max_passes=-1):
    engine.set_instance(xy, wt)
    assert engine.info("fp32_ok") == 1
    os_, oobj, ost, olog = oracle.two_opt_bi(xy, wt, succ0, max_passes=max_passes, log_cap=100000)
    for key, (s, obj, moves, passes, log) in _runs(engine, succ0, max_passes).items():
        assert log.tolist() == olog.tolist(), key
        assert (s == os_).all() and obj == oobj, key
        assert moves == ost.moves and passes == ost.passes, key


def test_prefilter_on_off_oracle_tsplib(engine, oracle, instances):
    """every TSPLIB fixture of a metric the FP32 path serves (EUC_2D, CEIL_2D, ATT), to the local optimum"""
    done = 0
    for nm, (xy, wt) in sorted(instances.items()):
        if wt not in (0, 3, 5):
            continue
        succ, _ = oracle.nn_tour(xy, wt, 0)
        _check(engine, oracle, xy, wt, succ)
        done += 1
    assert done >= 20


@pytest.mark.parametrize("nm", ["fl3795", "pla7397"])
def test_prefilter_on_off_oracle_large(engine, oracle, nm):
    """decimal coordinates FP32 cannot hold (fl3795) and CEIL_2D around 10^6 (pla7397)"""
    z = np.load(os.path.join(GOLD_DIR, "large.npz"))
    xy, wt = z[nm + "__xy"], int(z[nm + "__wt"])
    succ, _ = oracle.nn_tour(xy, wt, 0)
    _check(engine, oracle, xy, wt, succ, max_passes=40)


def _hard_cases():
    rng = np.random.default_rng(2024)
    cases = [("non_fp32_coords", rng.random((1800, 2)) * 1000.0 + 0.1, 0),
             ("duplicates", np.repeat(np.floor(rng.random((450, 2)) * 5000.0), 4, axis=0), 0),
             ("integer_ties", np.floor(rng.random((2000, 2)) * 40.0), 0),
             ("ceil_ties", np.floor(rng.random((1500, 2)) * 60.0), 3),
             ("att_decimal", rng.random((1500, 2)) * 3000.0, 5),
             ("big_box", np.floor(rng.random((1500, 2)) * 2.5e6), 0)]
    return cases


@pytest.mark.parametrize("case", range(len(_hard_cases())))
def test_prefilter_on_off_oracle_hard_inputs(engine, oracle, case):
    nm, xy, wt = _hard_cases()[case]
    rng = np.random.default_rng(case)
    succ, _ = oracle.nn_tour(xy, wt, 0)
    _check(engine, oracle, xy, wt, succ, max_passes=60)
    _check(engine, oracle, xy, wt, order_to_succ(rng.permutation(len(xy)).astype(np.int32)), max_passes=8)


@pytest.mark.parametrize("T,R,TJ,shuffle", [(64, 8, 256, 1), (64, 8, 88, 0), (64, 4, 64, 1), (64, 2, 32, 0), (128, 8, 128, 0),
                                            (128, 16, 64, 0), (256, 4, 36, 0), (256, 16, 64, 0)])
def test_prefilter_on_off_oracle_tile_shapes(engine, oracle, T, R, TJ, shuffle):
    xy = uniform_instance(2300)
    engine.set_option("block_threads", T)
    engine.set_option("rows_per_thread", R)
    engine.set_option("tile_cols", TJ)
    engine.set_option("row_shuffle", shuffle)
    try:
        succ, _ = oracle.nn_tour(xy, 0, 0)
        _check(engine, oracle, xy, 0, succ, max_passes=30)
        assert (engine.info("block_threads"), engine.info("rows_per_thread"), engine.info("tile_cols")) == (T, R, TJ)
    finally:
        engine.set_option("block_threads", 0)
        engine.set_option("rows_per_thread", 0)
        engine.set_option("tile_cols", 0)
        engine.set_option("row_shuffle", -1)


def test_prefilter_uni100000_first_moves_and_counters(engine):
    """the headline instance from its committed NN tour: the first 12 moves of the committed move log with the prefilter on
    and off; the exact path sees the same number of blocks either way, and stage-1 hits are counted"""
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
    assert hits[0] == 0 and hits[1] >= cold[1] > 0
    assert abs(cold[1] - cold[0]) <= 0.1 * cold[0] + 100
