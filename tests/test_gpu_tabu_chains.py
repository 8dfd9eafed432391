"""Independent tabu chains on the resident population (tspb200_population_tabu): masked best improvement, best-tour copy and
the random kick run on the device for every chain and iteration in one launch, each chain drawing from its own glibc
random() stream.  Every replayed chain is run on the CPU with GlibcRandom(seed_b) (instances.py, pinned to libc in
tests/test_host_logic.py), oracle.two_opt_bi with the list, iter and tenure (alg_2opt_tabu, reference
src/tabusearch.c:107-178) and oracle.tabu_kick one drawn candidate at a time (:262-309), and compared bit for bit: trace,
draws, best costs, current and best tours, the list and the next iteration number."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from tsp_optimization_b200 import engine as eng
from tsp_optimization_b200.instances import GlibcRandom, is_tour, order_to_succ, uniform_instance

pytestmark = pytest.mark.gpu


def _step_tenures(chains, iters):
    """the session test's schedule: 3, switching between 3 and 15 every 6 iterations"""
    row = [3 if (t // 6) % 2 == 0 else 15 for t in range(iters)]
    return np.tile(np.array(row, dtype=np.int32), (chains, 1))


class _Chain:
    """one chain replayed on the CPU"""

    def __init__(self, oracle, xy, wt, succ, seed):
        self.oracle, self.xy, self.wt = oracle, xy, wt
        self.n = len(xy)
        self.g = GlibcRandom(int(seed))
        self.succ = np.array(succ, dtype=np.int32)
        self.best_succ = self.succ.copy()
        self.best = oracle.succ_cost(xy, wt, self.succ)
        self.tl = np.zeros(self.n * (self.n - 1) // 2, dtype=np.int32)
        self.it = 1
        self.trace, self.draws = [], []
        self.moves = self.passes = 0

    def run(self, tenures, max_draws=None):
        """-> None, or the index of the iteration whose kick needed more than max_draws pairs"""
        for t, ten in enumerate(tenures):
            ten = int(ten)
            self.succ, c, st, _ = self.oracle.two_opt_bi(self.xy, self.wt, self.succ, skip_edge=self.tl, iter_=self.it, tenure=ten)
            self.trace.append(c)
            self.moves += st.moves
            self.passes += st.passes
            if c < self.best:
                self.best, self.best_succ = c, self.succ.copy()
            d = 0
            while True:
                if max_draws is not None and d == max_draws:
                    return t
                a, b = self.g.rand_choice(0, self.n), self.g.rand_choice(0, self.n)
                d += 1
                acc, self.succ, self.tl = self.oracle.tabu_kick(self.succ, self.tl, [[a, b]], self.it, ten)
                if acc == 0:
                    break
            self.draws.append(d)
            self.it += 1
        return None


def _check(engine, chain, b, slot, best_slot, best, trace, draws):
    assert trace[b].tolist() == chain.trace, b
    assert draws[b].tolist() == chain.draws, b
    assert best[b] == chain.best, b
    cur, bst = engine.population_download(slots=[slot, best_slot], as_order=False)
    assert (cur == chain.succ).all() and (bst == chain.best_succ).all(), b
    tl, it = engine.population_tabu_list(b)
    assert it == chain.it, b
    assert (tl == chain.tl).all(), (b, int((tl != chain.tl).sum()))


def _run_and_check(engine, oracle, xy, wt, starts, seeds, tenures, sample=None):
    """population = starts + as many spare tours (the best slots); chain b: slot b, best slot count + b"""
    k = len(starts)
    pop = np.concatenate([starts, starts])
    engine.population_upload(pop, as_order=False)
    engine.population_tabu_begin(seeds)
    best, trace, draws, st = engine.population_tabu(tenures)
    assert st.launches == 1 and trace.shape == tenures.shape and draws.shape == tenures.shape
    idx = range(k) if sample is None else sample
    chains = {}
    for b in idx:
        ch = _Chain(oracle, xy, wt, starts[b], seeds[b])
        ch.run(tenures[b])
        _check(engine, ch, b, b, k + b, best, trace, draws)
        chains[b] = ch
    if sample is None:
        assert st.moves == sum(c.moves for c in chains.values()) and st.passes == sum(c.passes for c in chains.values())
    return best, trace, draws, st, chains


def _nn_tours(oracle, xy, wt, starts):
    return np.stack([oracle.nn_tour(xy, wt, int(s))[0] for s in starts])


def test_tabu_chains_euc2d_uni400_step_tenure(engine, oracle):
    n, k, iters = 400, 24, 15
    xy = uniform_instance(n)
    engine.set_instance(xy, 0)
    starts = _nn_tours(oracle, xy, 0, range(0, 5 * k, 5))
    seeds = np.arange(200, 200 + k)
    best, trace, draws, st, _ = _run_and_check(engine, oracle, xy, 0, starts, seeds, _step_tenures(k, iters))
    assert st.gpu_ms > 0 and st.evals > 0 and st.moves > 0
    assert (draws >= 1).all() and (draws > 1).any()  # some kicks met a tabu or adjacent pair first
    engine.population_tabu_end()


def _metric_cases(instances):
    rng = np.random.default_rng(7)
    return [
        ("att532", *instances["att532"], None),
        ("ceil", rng.integers(0, 4000, size=(300, 2)).astype(np.float64), 3, None),
        ("gr229_matrix", *instances["gr229"], "matrix"),
        ("man", rng.integers(0, 5000, size=(250, 2)).astype(np.float64), 2, None),
        ("fp32_unsafe", rng.integers(0, 3_500_000, size=(250, 2)).astype(np.float64), 3, "fp32_unsafe"),
    ]


@pytest.mark.parametrize("case", range(5))
def test_tabu_chains_metrics_and_paths(engine, oracle, instances, case):
    name, xy, wt, how = _metric_cases(instances)[case]
    n = len(xy)
    engine.set_instance(xy, wt)
    if how == "matrix":
        engine.dist_matrix_build()
    try:
        if how == "fp32_unsafe":
            assert engine.info("fp32_ok") == 0
        starts = _nn_tours(oracle, xy, wt, [0, n // 2, n - 1])
        _, _, _, st, _ = _run_and_check(engine, oracle, xy, wt, starts, [31, 32, 33], _step_tenures(3, 8))
        if how == "matrix":
            assert st.path == 2
    finally:
        if how == "matrix":
            engine.dist_matrix_free()


def test_tabu_chains_tenure_sweep_in_one_launch(engine, oracle):
    """tenure -1 (check_tenure never blocks nor expires), 0, 3 and 50, one per chain, in one launch"""
    n, iters = 300, 20
    xy = uniform_instance(n, seed=17)
    engine.set_instance(xy, 0)
    starts = _nn_tours(oracle, xy, 0, [1, 2, 3, 4])
    ten = np.array([[-1], [0], [3], [50]], dtype=np.int32).repeat(iters, axis=1)
    _, _, _, _, chains = _run_and_check(engine, oracle, xy, 0, starts, [5, 6, 7, 8], ten)
    assert (chains[0].tl != 0).sum() > (chains[2].tl != 0).sum()  # nothing expires at tenure -1


def test_tabu_chains_long_tenure_and_table_overflow(engine, oracle):
    """tenure >= iters: nothing expires, the table of possibly non-zero entries only grows; with more than 256 live
    entries it overflows and the chain falls back to rebuilding it from the whole list (every node marked)"""
    n = 200
    xy = uniform_instance(n, seed=23)
    engine.set_instance(xy, 0)
    starts = _nn_tours(oracle, xy, 0, [0, 50])
    ten = np.array([[40] * 40, [100000] * 40], dtype=np.int32)
    _run_and_check(engine, oracle, xy, 0, starts, [1, 2], ten)
    # more than 256 stamps on distinct edges; a larger n so that the kicks still find pairs whose edges are not tabu.  Chain 1
    # runs unmasked (tenure -1: its table overflows without being rebuilt), then masked at tenure 3: the first masked pass
    # marks every node and expires the old entries, and the table fits again
    xy = uniform_instance(800, seed=23)
    engine.set_instance(xy, 0)
    starts = _nn_tours(oracle, xy, 0, [3, 70])
    ten = np.array([[100000] * 190, [-1] * 180 + [3] * 10], dtype=np.int32)
    _, _, _, _, chains = _run_and_check(engine, oracle, xy, 0, starts, [9, 10], ten)
    assert (chains[0].tl != 0).sum() > 256 and (chains[1].tl != 0).sum() < 16


def test_tabu_chains_equal_the_single_tour_session(engine, oracle):
    """two chains through population_tabu == the same chains through tabu_begin, tabu_run, one-candidate tabu_kick calls
    and tour_save, lists included"""
    n, iters = 350, 14
    xy = uniform_instance(n, seed=41)
    engine.set_instance(xy, 0)
    starts = _nn_tours(oracle, xy, 0, [10, 20])
    seeds = [71, 72]
    ten = _step_tenures(2, iters)
    engine.population_upload(np.concatenate([starts, starts]), as_order=False)
    engine.population_tabu_begin(seeds)
    best, trace, draws, _ = engine.population_tabu(ten)
    finals = engine.population_download(4, as_order=False)
    lists = [engine.population_tabu_list(b)[0] for b in range(2)]
    for b in range(2):
        engine.tour_upload(starts[b])
        inc = engine.tour_cost()
        engine.tour_save(1)
        engine.tabu_begin()
        g = GlibcRandom(seeds[b])
        costs, nd = [], []
        for t in range(iters):
            it, tenure = t + 1, int(ten[b, t])
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
        assert trace[b].tolist() == costs and draws[b].tolist() == nd, b
        assert best[b] == inc == bc, b
        assert (finals[b] == cur).all() and (finals[2 + b] == bst).all(), b
        assert (lists[b] == tl).all(), b


def test_tabu_chains_continuation_slots_and_zero_iterations(engine, oracle):
    n, k = 300, 6
    xy = uniform_instance(n, seed=9)
    engine.set_instance(xy, 0)
    starts = _nn_tours(oracle, xy, 0, range(k))
    seeds = np.arange(50, 50 + k)
    ten = _step_tenures(k, 12)
    ten[1] = 0
    pop = np.concatenate([starts, starts])
    # K1 + K2 in one call
    engine.population_upload(pop, as_order=False)
    engine.population_tabu_begin(seeds)
    b12, t12, d12, _ = engine.population_tabu(ten)
    f12 = engine.population_download(2 * k, as_order=False)
    l12 = [engine.population_tabu_list(b) for b in range(k)]
    # K1 = 5, then K2 = 7
    engine.population_upload(pop, as_order=False)
    engine.population_tabu_begin(seeds)
    b5, t5, d5, _ = engine.population_tabu(ten[:, :5])
    b7, t7, d7, _ = engine.population_tabu(ten[:, 5:])
    assert (b7 == b12).all() and (np.concatenate([t5, t7], 1) == t12).all() and (np.concatenate([d5, d7], 1) == d12).all()
    assert (engine.population_download(2 * k, as_order=False) == f12).all()
    for b in range(k):
        tl, it = engine.population_tabu_list(b)
        assert it == l12[b][1] == 13 and (tl == l12[b][0]).all(), b
    # iters = 0: the best costs, nothing changes
    b0, t0, d0, st0 = engine.population_tabu(np.zeros((k, 0), dtype=np.int32))
    assert (b0 == b12).all() and t0.shape == (k, 0) and st0.moves == 0
    assert (b0 == engine.population_costs(slots=np.arange(k, 2 * k))).all()
    assert (engine.population_download(2 * k, as_order=False) == f12).all()
    assert all(engine.population_tabu_list(b)[1] == 13 for b in range(k))
    engine.population_tabu_end()
    # non-contiguous slots and best slots: only those move
    pop10 = np.concatenate([starts, starts[:4]])
    engine.population_upload(pop10, as_order=False)
    sl, bs = np.array([7, 2, 4], dtype=np.int32), np.array([0, 9, 5], dtype=np.int32)
    sel_seeds = seeds[[1, 3, 5]]
    engine.population_tabu_begin(sel_seeds, slots=sl, best_slots=bs)
    tsel = ten[[1, 3, 5]]
    best, trace, draws, _ = engine.population_tabu(tsel)
    for q in range(3):
        ch = _Chain(oracle, xy, 0, pop10[sl[q]], sel_seeds[q])
        ch.run(tsel[q])
        _check(engine, ch, q, int(sl[q]), int(bs[q]), best, trace, draws)
    after = engine.population_download(10, as_order=False)
    for s in set(range(10)) - set(sl.tolist()) - set(bs.tolist()):
        assert (after[s] == pop10[s]).all(), s
    # a slot overwritten between calls: the chain continues from that tour
    engine.population_upload(starts[:1], slots=[7], as_order=False)
    ch = _Chain(oracle, xy, 0, pop10[7], sel_seeds[0])
    ch.run(tsel[0])
    ch.succ = starts[0].copy()
    ch.trace, ch.draws = [], []
    ch.run(tsel[0, :3])
    best, trace, draws, _ = engine.population_tabu(tsel[:, :3])
    _check(engine, ch, 0, 7, 0, best, trace, draws)
    engine.population_tabu_end()


def test_tabu_chains_n2000_many_chains(engine, oracle):
    n, k, iters = 2000, 128, 3
    xy = uniform_instance(n)
    engine.set_instance(xy, 0)
    nn, _ = engine.nn_tour_batch(np.arange(k, dtype=np.int32))
    seeds = np.arange(1000, 1000 + k)
    _, _, _, st, _ = _run_and_check(engine, oracle, xy, 0, nn, seeds, _step_tenures(k, iters), sample=[0, 45, 127])
    assert st.moves > 0 and all(is_tour(s) for s in engine.population_download(2 * k, as_order=False))
    engine.population_tabu_end()


def test_tabu_chains_errors(engine, oracle):
    n = 120
    xy = uniform_instance(n, seed=3)
    engine.set_instance(xy, 0)
    rng = np.random.default_rng(0)
    tours = np.stack([order_to_succ(rng.permutation(n).astype(np.int32)) for _ in range(8)])
    engine.population_upload(tours, as_order=False)

    def untouched():
        return (engine.population_download(8, as_order=False) == tours).all()

    # no chain set
    engine.population_tabu_begin([1, 2])  # copies slots 0, 1 to the best slots 2, 3
    engine.population_tabu_end()
    engine.population_upload(tours, as_order=False)
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_tabu(np.full((2, 3), 3, dtype=np.int32))
    assert ei.value.code == 3 and untouched()
    # overlapping slots
    for sl, bs in [([0, 1], [1, 2]), ([0, 0], [2, 3]), ([0, 1], [2, 8])]:
        with pytest.raises(eng.TspB200Error) as ei:
            engine.population_tabu_begin([1, 2], slots=sl, best_slots=bs)
        assert ei.value.code == 2 and untouched(), (sl, bs)
    # a failed begin ends the previous chain set: the library no longer holds 3 chains when the caller has arrays for 2
    engine.population_tabu_begin([1, 2, 3])
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_tabu_begin([1, 2], slots=[0, 1], best_slots=[1, 2])
    assert ei.value.code == 2
    ref = engine.population_download(8, as_order=False)
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_tabu(np.full((2, 3), 3, dtype=np.int32))
    assert ei.value.code == 3
    ten2 = np.full((2, 3), 3, dtype=np.int32)
    best2, trace2, draws2 = np.empty(2), np.empty((2, 3)), np.empty((2, 3), dtype=np.int32)
    rc = engine.L.tspb200_population_tabu(engine.h, ten2.ctypes.data, 3, 16, best2.ctypes.data, trace2.ctypes.data,
                                          draws2.ctypes.data, None)
    assert rc == 3 and (engine.population_download(8, as_order=False) == ref).all()
    # a short tenure array, max_draws < 1: the population stays as begin left it
    engine.population_tabu_begin([1, 2, 3])
    ref = engine.population_download(8, as_order=False)
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_tabu(np.full((2, 3), 3, dtype=np.int32))
    assert ei.value.code == 2 and (engine.population_download(8, as_order=False) == ref).all()
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_tabu(np.full((3, 3), 3, dtype=np.int32), max_draws=0)
    assert ei.value.code == 2 and (engine.population_download(8, as_order=False) == ref).all()
    assert all(engine.population_tabu_list(b)[1] == 1 for b in range(3))  # no iteration ran
    # a re-created population
    engine.population_upload(tours, as_order=False)
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_tabu(np.full((3, 3), 3, dtype=np.int32))
    assert ei.value.code == 3 and untouched()
    # a slot that is not one cycle
    broken = tours[1].copy()
    broken[[3, 4]] = broken[[4, 3]]
    assert not is_tour(broken)
    engine.population_upload(broken[None], slots=[1], as_order=False)
    engine.population_tabu_begin([1, 2, 3])
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_tabu(np.full((3, 2), 3, dtype=np.int32))
    assert ei.value.code == 6 and "chain 1" in str(ei.value)
    engine.population_upload(tours, as_order=False)
    # max_draws = 1: a seed whose first pair has a == b stops its chain at iteration 0; the other chains' seeds have kicks
    # that pass at their first pair, so they finish and match the oracle
    def first_pair_equal(s):
        g = GlibcRandom(s)
        return g.rand_choice(0, n) == g.rand_choice(0, n)

    bad = next(s for s in range(1, 100000) if first_pair_equal(s))
    good, s = [], 1
    for b in (0, 1, 3):
        while s == bad or _Chain(oracle, xy, 0, tours[b], s).run([3, 3], max_draws=1) is not None:
            s += 1
        good.append(s)
        s += 1
    seeds = [good[0], good[1], bad, good[2]]
    engine.population_tabu_begin(seeds)
    ten = np.full((4, 2), 3, dtype=np.int32)
    best, trace, draws = np.empty(4), np.empty((4, 2)), np.empty((4, 2), dtype=np.int32)
    rc = engine.L.tspb200_population_tabu(engine.h, ten.ctypes.data, 2, 1, best.ctypes.data, trace.ctypes.data,
                                          draws.ctypes.data, None)
    msg = engine.L.tspb200_last_error(engine.h).decode()
    assert rc == 6 and "chain 2, iteration 0" in msg, msg
    for b in (0, 1, 3):
        ch = _Chain(oracle, xy, 0, tours[b], seeds[b])
        ch.run(ten[b])
        _check(engine, ch, b, b, 4 + b, best, trace, draws)
    engine.population_tabu_end()
    # the memory check: 6000 chains' lists at n = 4000 need 192 GB
    big = 4000
    engine.set_instance(uniform_instance(big), 0)
    ring = np.roll(np.arange(big, dtype=np.int32), -1)
    engine.population_upload(np.tile(ring, (12000, 1)), as_order=False)
    import torch
    torch.cuda.mem_get_info(0)  # the first call creates torch's context
    free0 = torch.cuda.mem_get_info(0)[0]
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_tabu_begin(np.arange(6000))
    assert ei.value.code == 5 and "191952000000 bytes" in str(ei.value), str(ei.value)
    assert torch.cuda.mem_get_info(0)[0] >= free0 - (64 << 20)  # no list was allocated
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_tabu(np.zeros((6000, 1), dtype=np.int32))
    assert ei.value.code == 3


def test_tabu_chains_two_ranks_one_device():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29553", os.path.join(ROOT, "tools", "tabu_chains.py"), "--size", "500", "--chains", "32",
           "--iters", "8", "--session-chains", "2"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and '"shards_equal_single_gpu": true' in r.stdout and '"session_equals_chains": true' in r.stdout, \
        r.stdout[-2000:] + r.stderr[-2000:]
