"""Independent VNS chains on the resident population (tspb200_population_vns): kick, first-improvement 2-opt and keep /
restore run on the device for every chain and iteration in one launch.  Every chain is replayed on the CPU with the oracle
(oracle.vns_kick, oracle.two_opt_fi on the kicked tour and cost, strict '<' keep / restore: reference HEU_VNS,
src/vns.c:125-177), with the kicks drawn from GlibcRandom(seed_b) per chain (instances.vns_kick_indices)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from tsp_optimization_b200 import engine as eng
from tsp_optimization_b200.instances import GlibcRandom, is_tour, order_to_succ, uniform_instance, vns_kick_indices

FI = eng.FI
pytestmark = pytest.mark.gpu


def _kicks(n, seeds, iters):
    out = np.empty((len(seeds), iters, 3), dtype=np.int32)
    for b, s in enumerate(seeds):
        g = GlibcRandom(int(s))
        for t in range(iters):
            out[b, t] = vns_kick_indices(g, n)
    return out


def _fi_optima(oracle, xy, wt, starts):
    """FI local optima of the NN tours from `starts` (oracle), as successor arrays"""
    out = []
    for s in starts:
        succ, c = oracle.nn_tour(xy, wt, int(s))
        out.append(oracle.two_opt_fi(xy, wt, succ, c)[0])
    return np.stack(out)


def _replay(oracle, xy, wt, succ, kicks):
    """one chain on the CPU -> (incumbent cost, incumbent tour, trace, moves, sweeps)"""
    best_succ = np.asarray(succ, dtype=np.int32)
    best = oracle.succ_cost(xy, wt, best_succ)
    trace, moves, passes = [], 0, 0
    for i1, i2, i3 in kicks:
        ks, kc = oracle.vns_kick(xy, wt, best_succ, i1, i2, i3)
        s, c, st, _ = oracle.two_opt_fi(xy, wt, ks, kc)
        trace.append(c)
        moves += st.moves
        passes += st.passes
        if c < best:
            best, best_succ = c, s
    return best, best_succ, trace, moves, passes


def _check_chains(engine, oracle, xy, wt, starts_succ, kicks, sample=None):
    """uploads the start tours, runs population_vns, compares the sampled chains (all by default) with the oracle"""
    engine.population_upload(starts_succ, as_order=False)
    best, trace, st = engine.population_vns(kicks)
    final = engine.population_download(len(starts_succ), as_order=False)
    assert st.launches == 1
    idx = range(len(starts_succ)) if sample is None else sample
    tot_moves = tot_passes = 0
    for b in idx:
        ob, osucc, otr, om, op = _replay(oracle, xy, wt, starts_succ[b], kicks[b])
        assert trace[b].tolist() == otr, b
        assert best[b] == ob, b
        assert (final[b] == osucc).all(), b
        tot_moves += om
        tot_passes += op
    if sample is None:
        assert st.moves == tot_moves and st.passes == tot_passes
    return best, trace, st, final


def _accepted_rejected(engine_start_costs, trace):
    acc = rej = 0
    for b in range(len(trace)):
        inc = engine_start_costs[b]
        for c in trace[b]:
            if c < inc:
                acc, inc = acc + 1, c
            else:
                rej += 1
    return acc, rej


def test_vns_chains_euc2d_uni400(engine, oracle):
    n, chains, iters = 400, 24, 12
    xy = uniform_instance(n)
    engine.set_instance(xy, 0)
    starts = _fi_optima(oracle, xy, 0, range(0, 3 * chains, 3))
    kicks = _kicks(n, range(100, 100 + chains), iters)
    kicks[0, 2] = (0, n // 2, n - 1)  # the last tour index as the largest: f wraps to tour index 0
    kicks[1, 0] = (n // 3, 0, n - 5)  # idx1 = 0, given out of order
    c0 = [oracle.succ_cost(xy, 0, s) for s in starts]
    best, trace, st, final = _check_chains(engine, oracle, xy, 0, starts, kicks)
    acc, rej = _accepted_rejected(c0, trace)
    assert acc >= 1 and rej >= 1, (acc, rej)
    assert all(is_tour(s) for s in final)
    assert st.evals > 0 and st.gpu_ms > 0


def _metric_cases(instances):
    rng = np.random.default_rng(5)
    return [
        ("att532", *instances["att532"], None),
        ("dsj1000", *instances["dsj1000"], None),
        ("gr666_matrix", *instances["gr666"], "matrix"),
        ("gr666_path1", *instances["gr666"], "path1"),
        ("man", rng.integers(0, 5000, size=(350, 2)).astype(np.float64), 2, None),
        ("fp32_unsafe", rng.integers(0, 3_500_000, size=(300, 2)).astype(np.float64), 3, "fp32_unsafe"),
    ]


@pytest.mark.parametrize("case", range(6))
def test_vns_chains_metrics_and_paths(engine, oracle, instances, case):
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
        starts = _fi_optima(oracle, xy, wt, [0, n // 2, n - 1])
        kicks = _kicks(n, [11, 12, 13], 6)
        _, _, st, _ = _check_chains(engine, oracle, xy, wt, starts, kicks)
        if how == "matrix":
            assert st.path == 2
        if how == "path1":
            assert st.path == 1
    finally:
        engine.set_option("force_path", -1)
        if how == "matrix":
            engine.dist_matrix_free()


def test_vns_chains_lattice_tie_is_rejected(engine, oracle):
    """a 16 x 16 lattice: equal-cost local optima are everywhere; an iteration that ends exactly at the incumbent's cost
    is not an improvement (strict '<', vns.c:167) and the chain goes back to the incumbent's tour"""
    xy = np.stack(np.meshgrid(np.arange(16), np.arange(16)), -1).reshape(-1, 2).astype(np.float64) * 100
    n = len(xy)
    engine.set_instance(xy, 0)
    starts = _fi_optima(oracle, xy, 0, [0, 37, 101, 200])
    kicks = _kicks(n, [1, 2, 3, 4], 6)
    c0 = [oracle.succ_cost(xy, 0, s) for s in starts]
    best, trace, _, final = _check_chains(engine, oracle, xy, 0, starts, kicks)
    assert trace[0][0] == c0[0] == best[0]  # seed 1: the first kick of chain 0 comes back to a tie, rejected
    ties = 0
    for b in range(len(starts)):
        inc = c0[b]
        for c in trace[b]:
            ties += c == inc
            inc = min(inc, c)
    assert ties >= 1


def test_vns_chains_equal_the_single_tour_session(engine, oracle):
    """one chain through population_vns == the same kicks through vns_kick + fi_run + tour_save / tour_restore"""
    n, iters = 500, 15
    xy = uniform_instance(n, seed=31)
    engine.set_instance(xy, 0)
    start = _fi_optima(oracle, xy, 0, [7])
    kicks = _kicks(n, [77], iters)
    engine.population_upload(start, as_order=False)
    best, trace, _ = engine.population_vns(kicks)
    chain_final = engine.population_download(1, as_order=False)[0]
    engine.set_option("single_block", 0)
    try:
        engine.tour_upload(start[0])
        inc = engine.tour_cost()
        engine.tour_save(0)
        costs = []
        for i1, i2, i3 in kicks[0]:
            c = engine.vns_kick(i1, i2, i3)
            c += engine.fi_run(-1).obj_delta
            costs.append(c)
            if c < inc:
                inc = c
                engine.tour_save(0)
            else:
                engine.tour_restore(0)
        sess_final, sess_cost = engine.tour_download()
    finally:
        engine.set_option("single_block", -1)
    assert trace[0].tolist() == costs
    assert best[0] == inc == sess_cost
    assert (chain_final == sess_final).all()


def test_vns_chains_continuation_isolation_and_zero_iterations(engine, oracle):
    n, pop = 300, 10
    xy = uniform_instance(n, seed=9)
    engine.set_instance(xy, 0)
    starts = _fi_optima(oracle, xy, 0, range(pop))
    kicks = _kicks(n, range(50, 50 + pop), 12)
    # iters = 12 in one call
    engine.population_upload(starts, as_order=False)
    b12, t12, s12 = engine.population_vns(kicks)
    f12 = engine.population_download(pop, as_order=False)
    # iters = 5, then the next 7
    engine.population_upload(starts, as_order=False)
    b5, t5, _ = engine.population_vns(kicks[:, :5])
    b7, t7, _ = engine.population_vns(kicks[:, 5:])
    f57 = engine.population_download(pop, as_order=False)
    assert (b7 == b12).all() and (np.concatenate([t5, t7], axis=1) == t12).all() and (f57 == f12).all()
    assert (b5 >= b12).all()
    # iters = 0: current costs, nothing changes
    b0, t0, st0 = engine.population_vns(np.zeros((pop, 0, 3), dtype=np.int32))
    assert (b0 == b12).all() and t0.shape == (pop, 0) and st0.moves == 0
    assert (b0 == engine.population_costs(pop)).all()
    assert (engine.population_download(pop, as_order=False) == f12).all()
    # with slots: only the listed individuals move
    engine.population_upload(starts, as_order=False)
    sel = np.array([7, 2, 4], dtype=np.int32)
    bs, ts, _ = engine.population_vns(kicks[sel], slots=sel, want_trace=False)
    assert ts is None and (bs == b12[sel]).all()
    after = engine.population_download(pop, as_order=False)
    for k in range(pop):
        assert (after[k] == (f12[k] if k in sel else starts[k])).all(), k


def test_vns_chains_n2000_many_chains(engine, oracle):
    n, chains, iters = 2000, 256, 4
    xy = uniform_instance(n)
    engine.set_instance(xy, 0)
    nn, costs = engine.nn_tour_batch(np.arange(chains, dtype=np.int32))
    engine.population_upload(nn, as_order=False)
    engine.population_two_opt(FI, count=chains, obj=costs)
    starts = engine.population_download(chains, as_order=False)
    kicks = _kicks(n, range(1000, 1000 + chains), iters)
    _, _, st, final = _check_chains(engine, oracle, xy, 0, starts, kicks, sample=[0, 1, 37, 100, 128, 201, 254, 255])
    assert all(is_tour(s) for s in final)
    assert st.moves > 0


def test_vns_chains_errors(engine):
    n = 200
    xy = uniform_instance(n, seed=3)
    engine.set_instance(xy, 0)
    rng = np.random.default_rng(0)
    tours = np.stack([order_to_succ(rng.permutation(n).astype(np.int32)) for _ in range(4)])
    engine.population_upload(tours, as_order=False)
    good = _kicks(n, range(4), 3)
    for bad in [(0, 1, 50), (10, 60, 61), (5, 5, 90), (7, 7, 7), (-1, 40, 90), (3, 40, n), (0, 2, n + 5)]:
        k = good.copy()
        k[2, 1] = bad
        with pytest.raises(eng.TspB200Error) as ei:
            engine.population_vns(k)
        assert ei.value.code == 2 and "chain 2, iteration 1" in str(ei.value), bad
        assert (engine.population_download(4, as_order=False) == tours).all(), bad
    with pytest.raises(eng.TspB200Error):
        engine.population_vns(good[:1], slots=[4])
    # a slot that is not one cycle
    broken = tours[1].copy()
    broken[[3, 4]] = broken[[4, 3]]
    if not is_tour(broken):
        engine.population_upload(broken[None], slots=[1], as_order=False)
        with pytest.raises(eng.TspB200Error) as ei:
            engine.population_vns(good[:2])
        assert ei.value.code == 6
    # no population for this instance
    engine.set_instance(uniform_instance(n + 1, seed=3), 0)
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_vns(_kicks(n + 1, [0], 1))
    assert ei.value.code == 3
    # beyond one block's shared memory (28 bytes per node)
    big = 9000
    engine.set_instance(uniform_instance(big), 0)
    engine.population_upload(np.roll(np.arange(big, dtype=np.int32), -1)[None], as_order=False)
    with pytest.raises(eng.TspB200Error) as ei:
        engine.population_vns(_kicks(big, [0], 1))
    assert ei.value.code == 5


def test_vns_chains_sharded_equal_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(ROOT, "tools", "vns_chains.py"), "--size", "600", "--chains", "64",
           "--iters", "8", "--session-chains", "1"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and '"shards_equal_single_gpu": true' in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
