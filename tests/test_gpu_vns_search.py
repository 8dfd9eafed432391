"""One VNS search on the resident tour (tspb200_vns_search): every iteration of a call (kick, first-improvement 2-opt, keep or
go back to the incumbent) is driven from the device.  Replayed on the CPU as in test_gpu_vns_chains.py (oracle.vns_kick,
oracle.two_opt_fi, strict '<': reference HEU_VNS, src/vns.c:125-177) and compared bit for bit: trace, best cost, the final
resident tour and the move and sweep counts.  Larger tours are compared with population_vns (one chain) and with the
single-tour session loop (vns_kick + fi_run + tour_save / tour_restore)."""
import numpy as np
import pytest

from test_gpu_vns_chains import _fi_optima, _kicks, _metric_cases, _replay
from tsp_optimization_b200 import engine as eng
from tsp_optimization_b200.instances import is_tour, order_to_succ, uniform_instance

pytestmark = pytest.mark.gpu


def _run_and_check(engine, oracle, xy, wt, start, kicks):
    engine.tour_upload(start)
    best, trace, st = engine.vns_search(kicks)
    ob, osucc, otr, om, op = _replay(oracle, xy, wt, start, kicks)
    assert trace.tolist() == otr
    assert best == ob
    final, cost = engine.tour_download()
    assert (final == osucc).all() and cost == ob
    assert st.moves == om and st.passes == op
    assert st.launches > 1 and st.gpu_ms > 0 and st.evals > 0
    return best, trace, st


def test_vns_search_euc2d_uni400(engine, oracle):
    n = 400
    xy = uniform_instance(n)
    engine.set_instance(xy, 0)
    start = _fi_optima(oracle, xy, 0, [3])[0]
    kicks = _kicks(n, [100], 14)[0]
    kicks[2] = (0, n // 2, n - 1)  # the last tour index as the largest: f wraps to tour index 0
    kicks[5] = (n // 3, 0, n - 5)  # idx1 = 0, given out of order
    c0 = oracle.succ_cost(xy, 0, start)
    _, trace, st = _run_and_check(engine, oracle, xy, 0, start, kicks)
    assert st.path == 0
    inc, acc, rej = c0, 0, 0
    for c in trace:
        acc, rej = acc + (c < inc), rej + (c >= inc)
        inc = min(inc, c)
    assert acc >= 1 and rej >= 1, (acc, rej)


@pytest.mark.parametrize("case", range(6))
def test_vns_search_metrics_and_paths(engine, oracle, instances, case):
    name, xy, wt, how = _metric_cases(instances)[case]
    n = len(xy)
    engine.set_instance(xy, wt)
    if how == "matrix":
        engine.dist_matrix_build()
    if how == "path1":
        engine.set_option("force_path", 1)
    try:
        if how == "fp32_unsafe":
            assert engine.info("fp32_ok") == 0
        start = _fi_optima(oracle, xy, wt, [n // 2])[0]
        _, _, st = _run_and_check(engine, oracle, xy, wt, start, _kicks(n, [21 + case], 8)[0])
        if how == "matrix":
            assert st.path == 2
        if how == "path1":
            assert st.path == 1
    finally:
        engine.set_option("force_path", -1)
        if how == "matrix":
            engine.dist_matrix_free()


def test_vns_search_lattice_tie_is_rejected(engine, oracle):
    """16 x 16 lattice: an iteration that ends at exactly the incumbent's cost is rejected (strict '<', vns.c:167)"""
    xy = np.stack(np.meshgrid(np.arange(16), np.arange(16)), -1).reshape(-1, 2).astype(np.float64) * 100
    n = len(xy)
    engine.set_instance(xy, 0)
    start = _fi_optima(oracle, xy, 0, [0])[0]
    c0 = oracle.succ_cost(xy, 0, start)
    _, trace, _ = _run_and_check(engine, oracle, xy, 0, start, _kicks(n, [1], 12)[0])
    assert trace[0] == c0  # seed 1: the first kick comes back to a tie


def test_vns_search_random_start(engine, oracle):
    """a start that is no local optimum: the first iteration's kick is applied to it as it is"""
    n = 500
    xy = uniform_instance(n, seed=41)
    engine.set_instance(xy, 0)
    start = order_to_succ(np.random.default_rng(2).permutation(n).astype(np.int32))
    _run_and_check(engine, oracle, xy, 0, start, _kicks(n, [8], 6)[0])


@pytest.mark.parametrize("n,kicks", [(5, [(0, 2, 4), (4, 2, 0), (2, 0, 4)]),
                                     (6, [(0, 2, 4), (1, 3, 5), (5, 0, 2), (0, 3, 5)]),
                                     (7, [(0, 2, 4), (2, 4, 6), (6, 1, 3), (0, 3, 6), (1, 4, 6)])])
def test_vns_search_tiny_tours(engine, oracle, n, kicks):
    """hand-picked triples: vns_kick_indices can loop forever on such tours (n = 5: i1 = 1, i2 = 3 leave no i3)"""
    xy = uniform_instance(n, seed=n)
    engine.set_instance(xy, 0)
    start = order_to_succ(np.random.default_rng(n).permutation(n).astype(np.int32))
    _run_and_check(engine, oracle, xy, 0, start, np.array(kicks, dtype=np.int32))


def _population_vns(engine, start, kicks):
    engine.population_upload(start[None], as_order=False)
    best, trace, _ = engine.population_vns(kicks[None])
    return best[0], trace[0], engine.population_download(1, as_order=False)[0]


@pytest.mark.parametrize("n,iters", [(2000, 6), (7919, 3)])
def test_vns_search_equals_population_vns(engine, n, iters):
    xy = uniform_instance(n, seed=n)
    engine.set_instance(xy, 0)
    nn, _ = engine.nn_tour(0)
    start, _, _, _ = engine.two_opt(eng.FI, nn)
    kicks = _kicks(n, [n + 3], iters)[0]
    pbest, ptrace, pfinal = _population_vns(engine, start, kicks)
    engine.tour_upload(start)
    best, trace, st = engine.vns_search(kicks)
    assert trace.tolist() == ptrace.tolist() and best == pbest
    assert (engine.tour_download()[0] == pfinal).all()
    assert st.path == 0


def _session_loop(engine, start, kicks):
    engine.tour_upload(start)
    inc = engine.tour_cost()
    engine.tour_save(0)
    costs = []
    for i1, i2, i3 in kicks:
        c = engine.vns_kick(i1, i2, i3) + engine.fi_run(-1).obj_delta
        costs.append(c)
        if c < inc:
            inc = c
            engine.tour_save(0)
        else:
            engine.tour_restore(0)
    final, cost = engine.tour_download()
    return inc, costs, final


@pytest.mark.parametrize("n,iters", [(10000, 4), (19997, 3)])
def test_vns_search_equals_session_beyond_one_block(engine, n, iters):
    """tours the one-block chain kernel cannot hold"""
    xy = uniform_instance(n, seed=n + 1)
    engine.set_instance(xy, 0)
    nn, _ = engine.nn_tour(0)
    start, _, _, _ = engine.two_opt(eng.FI, nn)
    kicks = _kicks(n, [n], iters)[0]
    inc, costs, sfinal = _session_loop(engine, start, kicks)
    engine.tour_upload(start)
    best, trace, st = engine.vns_search(kicks)
    assert trace.tolist() == costs and best == inc
    assert (engine.tour_download()[0] == sfinal).all()
    assert st.moves > 0 and st.passes >= iters


def test_vns_search_options_pdl_and_late_selection(engine):
    n = 2000
    xy = uniform_instance(n, seed=n)
    engine.set_instance(xy, 0)
    nn, _ = engine.nn_tour(0)
    start, _, _, _ = engine.two_opt(eng.FI, nn)
    kicks = _kicks(n, [n + 3], 6)[0]
    ref = _population_vns(engine, start, kicks)
    try:
        for pdl in (0, 1):
            for late in (0, 1):
                engine.set_option("pdl", pdl)
                engine.set_option("fi_late", late)
                engine.tour_upload(start)
                best, trace, _ = engine.vns_search(kicks)
                assert best == ref[0] and trace.tolist() == ref[1].tolist(), (pdl, late)
                assert (engine.tour_download()[0] == ref[2]).all(), (pdl, late)
    finally:
        engine.set_option("pdl", 1)
        engine.set_option("fi_late", 1)


def test_vns_search_continuation_and_interplay(engine, oracle):
    n = 300
    xy = uniform_instance(n, seed=9)
    engine.set_instance(xy, 0)
    start = _fi_optima(oracle, xy, 0, [4])[0]
    other = _fi_optima(oracle, xy, 0, [150])[0]
    kicks = _kicks(n, [61], 12)[0]
    engine.tour_upload(start)
    b12, t12, _ = engine.vns_search(kicks)
    f12, _ = engine.tour_download()
    # a tour saved in slot 0 survives a call
    engine.tour_upload(other)
    engine.tour_save(0)
    engine.tour_upload(start)
    b5, t5, _ = engine.vns_search(kicks[:5])
    b7, t7, _ = engine.vns_search(kicks[5:])
    assert b7 == b12 and np.concatenate([t5, t7]).tolist() == t12.tolist()
    assert (engine.tour_download()[0] == f12).all()
    # iters = 0: the current cost, nothing changes
    b0, t0, st0 = engine.vns_search(np.zeros((0, 3), dtype=np.int32))
    assert b0 == b12 == engine.tour_cost() and len(t0) == 0 and st0.moves == 0 and st0.passes == 0
    assert (engine.tour_download()[0] == f12).all()
    # the incumbent is an FI optimum: a first-improvement run finds nothing in one sweep
    st = engine.fi_run(-1)
    assert st.moves == 0 and st.passes == 1
    engine.tour_restore(0)
    assert (engine.tour_download()[0] == other).all()
    # best improvement after a call sees the incumbent
    engine.tour_upload(start)
    engine.vns_search(kicks[:3])
    inc, _ = engine.tour_download()
    engine.bi_run()
    osucc, ocost, _, _ = oracle.two_opt_bi(xy, 0, inc)
    got, cost = engine.tour_download()
    assert (got == osucc).all() and cost == ocost


def test_vns_search_errors(engine):
    n = 200
    xy = uniform_instance(n, seed=3)
    engine.set_instance(uniform_instance(n + 1, seed=3), 0)
    engine.set_instance(xy, 0)  # a new instance: no tour
    with pytest.raises(eng.TspB200Error) as ei:
        engine.vns_search(_kicks(n, [0], 2)[0])
    assert ei.value.code == 3
    tour = order_to_succ(np.random.default_rng(0).permutation(n).astype(np.int32))
    engine.tour_upload(tour)
    good = _kicks(n, [4], 3)[0]
    for bad in [(0, 1, 50), (10, 60, 61), (5, 5, 90), (7, 7, 7), (-1, 40, 90), (3, 40, n), (0, 2, n + 5)]:
        k = good.copy()
        k[1] = bad
        with pytest.raises(eng.TspB200Error) as ei:
            engine.vns_search(k)
        assert ei.value.code == 2 and "iteration 1" in str(ei.value), bad
        assert (engine.tour_download()[0] == tour).all(), bad
    rc = engine.L.tspb200_vns_search(engine.h, None, 2, None, None, None)  # kicks = NULL with iters > 0
    assert rc == 2
    assert is_tour(engine.tour_download()[0])
