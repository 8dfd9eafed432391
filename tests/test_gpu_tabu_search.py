"""One tabu search on the resident tour (tspb200_tabu_search): the masked passes are grid-wide (FP32-filter scan with the tabu
test in its exact path, or the exact scan), each preceded by the pass's exact lazy expiry, and the kick is drawn on the
device.  Replayed on the CPU as in test_gpu_tabu_chains.py (GlibcRandom, oracle.two_opt_bi with the list, oracle.tabu_kick)
and compared bit for bit: trace, draws, best cost, best and current tours, the list and the next iteration number.  Larger
tours are compared with population_tabu (one chain) and with the single-tour session loop."""
import numpy as np
import pytest

from test_gpu_tabu_chains import _Chain, _metric_cases, _nn_tours, _step_tenures
from tsp_optimization_b200 import BI
from tsp_optimization_b200 import engine as eng
from tsp_optimization_b200.instances import GlibcRandom, is_tour, uniform_instance

pytestmark = pytest.mark.gpu


def _check(engine, chain, best, trace, draws):
    assert trace.tolist() == chain.trace
    assert draws.tolist() == chain.draws
    assert best == chain.best
    cur, _ = engine.tour_download()
    tl, it, bst = engine.tabu_search_fetch()
    assert (cur == chain.succ).all() and (bst == chain.best_succ).all()
    assert it == chain.it
    assert (tl == chain.tl).all(), int((tl != chain.tl).sum())


def _run_and_check(engine, oracle, xy, wt, start, seed, tenures):
    engine.tour_upload(start)
    engine.tabu_search_begin(seed)
    best, trace, draws, st = engine.tabu_search(tenures)
    ch = _Chain(oracle, xy, wt, start, seed)
    ch.run(tenures)
    _check(engine, ch, best, trace, draws)
    assert st.moves == ch.moves and st.passes == ch.passes
    n = len(xy)
    assert st.evals == st.passes * (n * (n - 3) // 2) and st.launches > 1
    return st, ch


def test_tabu_search_euc2d_uni400_step_tenure(engine, oracle):
    n = 400
    xy = uniform_instance(n)
    engine.set_instance(xy, 0)
    start = _nn_tours(oracle, xy, 0, [5])[0]
    st, ch = _run_and_check(engine, oracle, xy, 0, start, 200, _step_tenures(1, 15)[0])
    assert st.path == 0 and st.gpu_ms > 0 and st.moves > 0
    assert max(ch.draws) > 1  # some kicks met a tabu or adjacent pair first
    engine.tabu_search_end()


@pytest.mark.parametrize("case", range(5))
def test_tabu_search_metrics_and_paths(engine, oracle, instances, case):
    name, xy, wt, how = _metric_cases(instances)[case]
    n = len(xy)
    engine.set_instance(xy, wt)
    if how == "matrix":
        engine.dist_matrix_build()
    try:
        if how == "fp32_unsafe":
            assert engine.info("fp32_ok") == 0
        start = _nn_tours(oracle, xy, wt, [n // 2])[0]
        st, _ = _run_and_check(engine, oracle, xy, wt, start, 31 + case, _step_tenures(1, 8)[0])
        assert st.path == {"att532": 0, "ceil": 0, "gr229_matrix": 2, "man": 1, "fp32_unsafe": 1}[name]
        engine.tabu_search_end()
    finally:
        if how == "matrix":
            engine.dist_matrix_free()


@pytest.mark.parametrize("tenure", [-1, 0, 3, 50, 100000])
def test_tabu_search_tenure_sweep(engine, oracle, tenure):
    """tenure -1 (check_tenure never blocks nor expires), 0, 3, 50, and one >= iters (nothing expires)"""
    n, iters = 300, 20
    xy = uniform_instance(n, seed=17)
    engine.set_instance(xy, 0)
    start = _nn_tours(oracle, xy, 0, [2])[0]
    _run_and_check(engine, oracle, xy, 0, start, 6, np.full(iters, tenure, dtype=np.int32))
    engine.tabu_search_end()


def test_tabu_search_table_overflow(engine, oracle):
    """more than 256 live stamps: the table overflows and the expiry walks the whole list until the survivors fit again.
    Search 1 stays overflowed (tenure >= iters); search 2 overflows unmasked (tenure -1), then the masked passes at tenure 3
    expire the old entries and the table fits again."""
    xy = uniform_instance(800, seed=23)
    engine.set_instance(xy, 0)
    starts = _nn_tours(oracle, xy, 0, [3, 70])
    _, ch = _run_and_check(engine, oracle, xy, 0, starts[0], 9, np.full(190, 100000, dtype=np.int32))
    assert (ch.tl != 0).sum() > 256
    _, ch = _run_and_check(engine, oracle, xy, 0, starts[1], 10, np.array([-1] * 180 + [3] * 10, dtype=np.int32))
    assert (ch.tl != 0).sum() < 16
    engine.tabu_search_end()


@pytest.mark.parametrize("n,iters", [(2000, 6), (7919, 3)])
def test_tabu_search_equals_population_tabu(engine, n, iters):
    xy = uniform_instance(n, seed=n)
    engine.set_instance(xy, 0)
    nn, _ = engine.nn_tour_batch(np.array([0], dtype=np.int32))
    start = nn[0]
    ten = _step_tenures(1, iters)
    engine.population_upload(np.stack([start, start]), as_order=False)
    engine.population_tabu_begin([77])
    pbest, ptrace, pdraws, _ = engine.population_tabu(ten)
    cur_p, best_p = engine.population_download(2, as_order=False)
    ptl, pit = engine.population_tabu_list(0)
    engine.population_tabu_end()
    engine.tour_upload(start)
    engine.tabu_search_begin(77)
    best, trace, draws, st = engine.tabu_search(ten[0])
    assert st.path == 0
    cur, _ = engine.tour_download()
    tl, it, bst = engine.tabu_search_fetch()
    assert trace.tolist() == ptrace[0].tolist() and draws.tolist() == pdraws[0].tolist() and best == pbest[0]
    assert (cur == cur_p).all() and (bst == best_p).all() and it == pit and (tl == ptl).all()
    engine.tabu_search_end()


def _session_loop(engine, start, seed, tenures):
    """the single-tour session: tabu_run, tour_save of a better tour, one-candidate tabu_kick calls"""
    n = len(start)
    engine.tour_upload(start)
    inc = engine.tour_cost()
    engine.tour_save(1)
    engine.tabu_begin()
    g = GlibcRandom(seed)
    costs, nd = [], []
    for t, tenure in enumerate(tenures):
        it, tenure = t + 1, int(tenure)
        c = engine.tabu_run(it, tenure).cost
        costs.append(c)
        if c < inc:
            inc = c
            engine.tour_save(1)
        d = 0
        while True:
            d += 1
            if engine.tabu_kick([[g.rand_choice(0, n), g.rand_choice(0, n)]], it, tenure) == 0:
                break
        nd.append(d)
    cur, _ = engine.tour_download()
    tl = engine.tabu_end(want_list=True)
    engine.tour_restore(1)
    bst, bc = engine.tour_download()
    return inc, costs, nd, cur, bst, tl


@pytest.mark.parametrize("n,iters", [(10000, 5), (19997, 3)])
def test_tabu_search_equals_session_beyond_one_block(engine, n, iters):
    """tours the one-block chain kernel cannot hold; the start is a 2-opt local optimum, so each iteration is a few passes"""
    xy = uniform_instance(n, seed=n + 1)
    engine.set_instance(xy, 0)
    nn, _ = engine.nn_tour(0)
    start, _, _, _ = engine.two_opt(BI, nn)
    ten = np.array([3, 15, 0, 3, 3][:iters], dtype=np.int32)
    inc, costs, nd, cur_s, bst_s, tl_s = _session_loop(engine, start, 123, ten)
    engine.tour_upload(start)
    engine.tabu_search_begin(123)
    best, trace, draws, st = engine.tabu_search(ten)
    assert st.path == 0 and st.passes >= iters
    cur, _ = engine.tour_download()
    tl, it, bst = engine.tabu_search_fetch()
    assert trace.tolist() == costs and draws.tolist() == nd and best == inc
    assert (cur == cur_s).all() and (bst == bst_s).all() and it == iters + 1 and (tl == tl_s).all()
    engine.tabu_search_end()


def test_tabu_search_continuation_zero_iterations_and_replaced_tour(engine, oracle):
    n = 300
    xy = uniform_instance(n, seed=9)
    engine.set_instance(xy, 0)
    starts = _nn_tours(oracle, xy, 0, [0, 7])
    ten = _step_tenures(1, 12)[0]
    engine.tour_upload(starts[0])
    engine.tabu_search_begin(50)
    b12, t12, d12, _ = engine.tabu_search(ten)
    c12, _ = engine.tour_download()
    l12 = engine.tabu_search_fetch()
    # K1 = 5, then K2 = 7
    engine.tour_upload(starts[0])
    engine.tabu_search_begin(50)
    _, t5, d5, _ = engine.tabu_search(ten[:5])
    b7, t7, d7, _ = engine.tabu_search(ten[5:])
    assert b7 == b12 and np.concatenate([t5, t7]).tolist() == t12.tolist() and np.concatenate([d5, d7]).tolist() == d12.tolist()
    assert (engine.tour_download()[0] == c12).all()
    l = engine.tabu_search_fetch()
    assert l[1] == l12[1] == 13 and (l[0] == l12[0]).all() and (l[2] == l12[2]).all()
    # iters = 0: nothing changes
    b0, t0, d0, st0 = engine.tabu_search(np.zeros(0, dtype=np.int32))
    assert b0 == b12 and len(t0) == 0 and st0.moves == 0 and st0.passes == 0
    assert (engine.tour_download()[0] == c12).all() and engine.tabu_search_fetch()[1] == 13
    # a 2-opt run after the search sees the resident tour as usual
    assert engine.bi_run().passes >= 1
    # the tour replaced between calls: the search continues from the new tour with its list, stream and best tour
    ch = _Chain(oracle, xy, 0, starts[0], 50)
    ch.run(ten)
    ch.succ = starts[1].copy()
    ch.trace, ch.draws = [], []
    ch.run(ten[:4])
    engine.tour_upload(starts[1])
    best, trace, draws, _ = engine.tabu_search(ten[:4])
    _check(engine, ch, best, trace, draws)
    engine.tabu_search_end()


def test_tabu_search_errors(engine, oracle):
    n = 120
    xy = uniform_instance(n, seed=3)
    engine.set_instance(xy, 0)
    ring = np.roll(np.arange(n, dtype=np.int32), -1)
    engine.tour_upload(ring)
    # no begin
    with pytest.raises(eng.TspB200Error) as ei:
        engine.tabu_search(np.full(3, 3, dtype=np.int32))
    assert ei.value.code == 3
    with pytest.raises(eng.TspB200Error) as ei:
        engine.tabu_search_fetch()
    assert ei.value.code == 3
    # max_draws: a seed whose first pair has a == b stops the search at iteration 0
    def first_pair_equal(s):
        g = GlibcRandom(s)
        return g.rand_choice(0, n) == g.rand_choice(0, n)

    bad = next(s for s in range(1, 100000) if first_pair_equal(s))
    engine.tabu_search_begin(bad)
    with pytest.raises(eng.TspB200Error) as ei:
        engine.tabu_search(np.full(2, 3, dtype=np.int32), max_draws=1)
    assert ei.value.code == 6 and "iteration 0" in str(ei.value), str(ei.value)
    with pytest.raises(eng.TspB200Error) as ei:
        engine.tabu_search(np.full(2, 3, dtype=np.int32), max_draws=0)
    assert ei.value.code == 2
    # a new instance ends the search
    engine.set_instance(uniform_instance(n, seed=4), 0)
    engine.tour_upload(ring)
    with pytest.raises(eng.TspB200Error) as ei:
        engine.tabu_search(np.full(2, 3, dtype=np.int32))
    assert ei.value.code == 3
    engine.tabu_search_begin(1)
    engine.tabu_search_end()
    with pytest.raises(eng.TspB200Error) as ei:
        engine.tabu_search_end()
    assert ei.value.code == 3
    # n > 46340: the reference's int list index
    big = 46341
    engine.set_instance(uniform_instance(big, seed=5), 0)
    engine.tour_upload(np.roll(np.arange(big, dtype=np.int32), -1))
    with pytest.raises(eng.TspB200Error) as ei:
        engine.tabu_search_begin(1)
    assert ei.value.code == 5
    assert is_tour(engine.tour_download()[0])
