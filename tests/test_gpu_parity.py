"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through the C ABI
(libtspb200.so / libtspb200_dropin.so) and is compared bit-for-bit with the oracle (oracle/tsp_oracle.c,
itself pinned to the compiled reference) and with the committed golden fixtures."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from tsp_optimization_b200 import engine as eng
from tsp_optimization_b200.instances import is_tour, order_to_succ, random_tours, uniform_instance

FI, BI = eng.FI, eng.BI


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# ---- ctypes mirror of the reference `instance` (include/tspb200_dropin.h) ---------------------------------
class _Method(C.Structure):
    _fields_ = [("id", C.c_int), ("edge_type", C.c_int), ("name", C.c_char_p), ("use_cplex", C.c_int)]


class _Params(C.Structure):
    _fields_ = [("file_path", C.c_char_p), ("num_threads", C.c_int), ("time_limit", C.c_int), ("method", _Method),
                ("verbose", C.c_int), ("integer_cost", C.c_int), ("seed", C.c_int), ("perf_prof", C.c_int),
                ("callback_2opt", C.c_int)]


class _Solution(C.Structure):
    _fields_ = [("obj_best", C.c_double), ("edges", C.c_void_p), ("time_to_solve", C.c_double), ("xbest", C.c_void_p)]


class _Instance(C.Structure):
    _fields_ = [("params", _Params), ("name", C.c_char_p), ("comment", C.c_char_p), ("nodes", C.c_void_p),
                ("num_nodes", C.c_int), ("weight_type", C.c_int), ("num_columns", C.c_long), ("ind", C.c_void_p),
                ("thread_seeds", C.c_void_p), ("solution", _Solution)]


class RefInstance:
    """A reference-layout instance living in numpy buffers (what the reference's parser + TSP_heuc build)."""

    def __init__(self, xy, wt, succ, obj=0.0):
        assert C.sizeof(_Instance) == 152
        self.xy = np.ascontiguousarray(xy, dtype=np.float64)
        n = len(self.xy)
        self.edges = np.empty((n, 2), dtype=np.int32)
        self.edges[:, 0] = np.arange(n)
        self.edges[:, 1] = succ
        c = _Instance()
        c.params.integer_cost = 1
        c.params.perf_prof = 1
        c.params.time_limit = 0
        c.nodes = self.xy.ctypes.data
        c.num_nodes = n
        c.weight_type = wt
        c.num_columns = n * (n - 1) // 2
        c.solution.obj_best = obj
        c.solution.edges = self.edges.ctypes.data
        self.c = c

    def succ(self):
        return self.edges[:, 1].copy()

    def set_succ_entry(self, k, v):
        self.edges[k, 1] = v


pytestmark = pytest.mark.gpu

EUC = ["berlin52", "eil51", "pr299", "a280", "lin318", "rd400", "pcb442", "pr439", "d493", "u574", "rat575", "p654",
       "d657", "u724", "rat783", "pr1002", "vm1084"]


# ---- distance matrix ------------------------------------------------------------------------------------------
def test_matrix_bit_exact_all_golden_instances(engine, instances, goldens, oracle):
    """every (i,j) of every fixture instance == calc_dist (EUC_2D, CEIL_2D, ATT, GEO incl. the GEO diagonal 1)."""
    for nm, (xy, wt) in sorted(instances.items()):
        engine.set_instance(xy, wt)
        m = engine.dist_matrix()
        g = goldens["instances"][nm]
        if sha(m) != g["matrix_sha256"]:
            ref = oracle.dist_matrix(xy, wt)
            bad = np.argwhere(m != ref)
            pytest.fail(f"{nm}: {len(bad)} entries differ, first {bad[:5].tolist()} got {m[tuple(bad[0])]} want {ref[tuple(bad[0])]}")
        assert int(m.sum(dtype=np.int64)) == g["matrix_sum"]
    engine.dist_matrix_free()


@pytest.mark.parametrize("wt", [0, 3, 5, 1, 2, 99])
def test_matrix_random_coordinates(engine, oracle, wt):
    rng = np.random.default_rng(100 + wt)
    for n, hi, frac in [(257, 50, False), (1031, 10000, False), (700, 3000, True), (515, 1_400_000, False)]:
        xy = rng.integers(0, hi, size=(n, 2)).astype(np.float64)
        if frac:
            xy += rng.integers(0, 1000, size=(n, 2)) / 1000.0  # not FP32-representable -> FP64 path
        engine.set_instance(xy, wt)
        m = engine.dist_matrix()
        ref = oracle.dist_matrix(xy, wt)
        assert (m == ref).all(), (wt, n, hi, np.argwhere(m != ref)[:3].tolist())
    engine.dist_matrix_free()


def test_matrix_adversarial_half_boundaries(engine, oracle):
    """distances engineered to sit on / next to the .5 (EUC) and integer (CEIL, ATT) rounding boundaries."""
    pts = [(0.0, 0.0)]
    for k in range(1, 400):
        pts.append((float(k), float(k + 1)))      # s = 2k^2+2k+1 : sqrt close to k*sqrt2 + .7
        pts.append((0.0, float(k) + 0.5))          # exact .5
        pts.append((3.0 * k, 4.0 * k))             # exact integers 5k
    for k in range(1, 300):
        s = k * k + k                              # sqrt(s) = k + .5 - 1/(8k): nearest approach from below
        pts.append((float(s), 0.0))
    xy = np.array(pts, dtype=np.float64)
    xy2 = np.sqrt(np.abs(xy)) if False else xy
    for wt in (0, 3, 5):
        engine.set_instance(xy2, wt)
        m = engine.dist_matrix()
        ref = oracle.dist_matrix(xy2, wt)
        assert (m == ref).all(), (wt, np.argwhere(m != ref)[:3].tolist())
    engine.dist_matrix_free()


@pytest.mark.parametrize("wt", [0, 3, 5])
def test_matrix_full_compare_n4096(engine, oracle, wt):
    """16.7 M entries per metric against the oracle, entry by entry: exercises the deferred exact re-evaluation of
    rows flagged by the FP32 guard band (integer coordinates -> exact FP64 compare; quarter-integer coordinates ->
    reference operation order in FP64) and both the full-block and the tail-row code paths (4100 % 32 != 0)."""
    rng = np.random.default_rng(4096 + wt)
    for n, scale in [(4096, 1.0), (4100, 0.25)]:
        xy = rng.integers(0, 40000, size=(n, 2)).astype(np.float64) * scale
        engine.set_instance(xy, wt)
        assert engine.info("exact32") == 1 and engine.info("int_coords") == (1 if scale == 1.0 else 0)
        m = engine.dist_matrix()
        ref = oracle.dist_matrix(xy, wt)
        assert (m == ref).all(), (wt, n, np.argwhere(m != ref)[:3].tolist())
    engine.dist_matrix_free()


def test_matrix_large_checksum_property(engine, oracle):
    """n = 6000 (144 MB matrix): symmetry, zero diagonal, and 64 sampled rows == oracle."""
    xy = uniform_instance(6000)
    engine.set_instance(xy, 0)
    m = engine.dist_matrix()
    assert (m == m.T).all() and (np.diag(m) == 0).all()
    rows = np.random.default_rng(1).integers(0, 6000, size=64)
    for i in rows:
        out = np.empty(6000, dtype=np.int32)
        oracle.L.orc_dist_row(np.ascontiguousarray(xy), 6000, 0, int(i), out)
        assert (m[i] == out).all()
    engine.dist_matrix_free()


# ---- 2-opt, single tour --------------------------------------------------------------------------------------
def _check_bi(engine, oracle, xy, wt, succ0, max_passes=-1, force_path=-1):
    """grid kernels (single_block 0) AND, when the run goes to the local optimum and the tour fits, the one-block kernel
    (single_block 1): both must reproduce the oracle's move log, tour, cost and counters."""
    engine.set_option("force_path", force_path)
    engine.set_instance(xy, wt)
    if force_path == 2 or (force_path == -1 and wt in (1, 2, 4)):
        engine.dist_matrix_build()
    os_, oobj, ost, olog = oracle.two_opt_bi(xy, wt, succ0, max_passes=max_passes, log_cap=100000)
    st = None
    # (route, prune): grid kernels exhaustive, grid kernels with exact tile pruning (must select the very same moves), one-block
    combos = [(0, 0), (0, 1)] + ([(1, 0)] if (max_passes < 0 and len(xy) <= 2000) else [])
    for route, prune in combos:
        engine.set_option("single_block", route)
        engine.set_option("prune", prune)
        s, obj, st_r, log = engine.two_opt(BI, succ0, 0.0, max_iters=max_passes, log_cap=100000)
        assert log.tolist() == olog.tolist(), (route, prune)
        assert (s == os_).all() and obj == oobj, (route, prune)
        assert st_r.moves == ost.moves and st_r.passes == ost.passes, (route, prune)
        if prune and st_r.tiles_total:
            assert st_r.evals <= ost.evals and 0 <= st_r.tiles_scanned <= st_r.tiles_total
        else:
            assert st_r.evals == ost.evals, (route, prune)
        assert st_r.launches == 1 or route == 0
        st = st or st_r
    engine.set_option("single_block", -1)
    engine.set_option("prune", -1)
    engine.set_option("force_path", -1)
    return st


def _check_fi(engine, oracle, xy, wt, succ0, obj0, force_path=-1):
    engine.set_option("force_path", force_path)
    engine.set_instance(xy, wt)
    if force_path == 2 or (force_path == -1 and wt in (1, 2, 4)):
        engine.dist_matrix_build()
    os_, oobj, ost, olog = oracle.two_opt_fi(xy, wt, succ0, obj0, log_cap=100000)
    st = None
    for route in ((0, 1) if len(xy) <= 5000 else (0,)):
        engine.set_option("single_block", route)
        s, obj, st_r, log = engine.two_opt(FI, succ0, obj0, log_cap=100000)
        assert log.tolist() == olog.tolist(), route
        assert (s == os_).all() and obj == oobj, route
        assert st_r.moves == ost.moves and st_r.passes == ost.passes, route
        st = st or st_r
    engine.set_option("single_block", -1)
    engine.set_option("force_path", -1)
    return st


def test_berlin52_known_answers(engine, oracle, instances, goldens):
    xy, wt = instances["berlin52"]
    succ, cost = oracle.nn_tour(xy, wt, 0)
    engine.set_instance(xy, wt)
    s, obj, st, log = engine.two_opt(BI, succ, 0.0, log_cap=100)
    assert obj == 7842 and st.moves == 11 and st.evals == 15288
    assert log.tolist() == goldens["instances"]["berlin52"]["bi_log"]
    s, obj, st, log = engine.two_opt(FI, succ, cost, log_cap=100)
    assert obj == 8083 and st.moves == 20 and st.passes == 5
    assert log.tolist() == goldens["instances"]["berlin52"]["fi_log"]


@pytest.mark.parametrize("nm", ["berlin52", "pr299", "att532", "dsj1000", "pr1002", "att48", "eil51"])
def test_bi_grid_kernel_move_log_parity(engine, oracle, instances, nm):
    xy, wt = instances[nm]
    succ, _ = oracle.nn_tour(xy, wt, 0)
    st = _check_bi(engine, oracle, xy, wt, succ)
    assert st.path == 0 and st.status == 0


@pytest.mark.parametrize("nm", ["gr666", "ulysses22", "burma14", "gr96"])
def test_bi_geo_matrix_and_exact_paths(engine, oracle, instances, nm):
    xy, wt = instances[nm]
    succ, _ = oracle.nn_tour(xy, wt, 0)
    assert _check_bi(engine, oracle, xy, wt, succ).path == 2            # matrix lookup
    assert _check_bi(engine, oracle, xy, wt, succ, force_path=1).path == 1  # FP64 on the fly


def test_bi_golden_costs_all_instances(engine, instances, goldens, oracle):
    for nm, (xy, wt) in sorted(instances.items()):
        g = goldens["instances"][nm]
        if "bi_cost" not in g:
            continue
        succ, _ = oracle.nn_tour(xy, wt, 0)
        engine.set_instance(xy, wt)
        if wt == 4:
            engine.dist_matrix_build()
        s, obj, st, _ = engine.two_opt(BI, succ, 0.0)
        assert obj == g["bi_cost"] and sha(s) == g["bi_sha256"] and st.moves == g["bi_moves"], nm


@pytest.mark.parametrize("nm", ["berlin52", "pr299", "att532", "gr666", "dsj1000", "ulysses16"])
def test_fi_grid_kernel_move_log_parity(engine, oracle, instances, nm):
    xy, wt = instances[nm]
    succ, cost = oracle.nn_tour(xy, wt, 0)
    _check_fi(engine, oracle, xy, wt, succ, cost)


def test_fi_reference_csv_goldens(engine, instances, goldens, oracle):
    """the reference's published 2OPT_GREEDY column (results/constructive_heuristics_2opt_new.csv), 18 instances."""
    for nm, row in sorted(goldens["reference_csv"].items()):
        xy, wt = instances[nm]
        g = goldens["instances"][nm]
        succ, cost = oracle.nn_tour(xy, wt, 0)
        assert cost == row["GREEDY"]
        engine.set_instance(xy, wt)
        if wt == 4:
            engine.dist_matrix_build()
        s, obj, st, _ = engine.two_opt(FI, succ, cost)
        assert obj == row["2OPT_GREEDY"], nm
        assert sha(s) == g["fi_sha256"] and st.moves == g["fi_moves"] and st.passes == g["fi_sweeps"], nm


@pytest.mark.parametrize("T,R,TJ,fuse", [(256, 2, 32, -1), (256, 2, 64, 0), (256, 4, 64, 1), (256, 8, 128, -1), (256, 8, 256, 0),
                                         (256, 4, 36, 1), (256, 16, 64, -1), (128, 16, 64, -1), (128, 16, 256, 1), (128, 8, 128, 1), (128, 4, 64, 0), (64, 8, 64, 1),
                                         (64, 8, 128, 0), (64, 4, 32, -1), (64, 2, 64, 1)])
def test_bi_tile_shapes(engine, oracle, T, R, TJ, fuse):
    """every supported (block threads, rows per thread) shape, with the move applied by a separate launch (fuse 0) and by
    the scan kernel's last block (fuse 1)."""
    xy = uniform_instance(1500)
    succ, _ = oracle.nn_tour(xy, 0, 0)
    engine.set_option("block_threads", T)
    engine.set_option("rows_per_thread", R)
    engine.set_option("tile_cols", TJ)
    engine.set_option("fuse_apply", fuse)
    try:
        _check_bi(engine, oracle, xy, 0, succ, max_passes=25)
        assert (engine.info("block_threads"), engine.info("rows_per_thread"), engine.info("tile_cols")) == (T, R, TJ)
    finally:
        engine.set_option("block_threads", 0)
        engine.set_option("rows_per_thread", 0)
        engine.set_option("tile_cols", 0)
        engine.set_option("fuse_apply", -1)


@pytest.mark.parametrize("T,R,TJ", [(64, 8, 256), (64, 8, 88), (64, 4, 64), (64, 2, 32)])
@pytest.mark.parametrize("shuffle", [0, 1])
def test_bi_row_shuffle_variant_equals_plain_variant(engine, oracle, T, R, TJ, shuffle):
    """bi_scan_kernel<..., SHUF>: a warp owns 32 R - 1 rows and takes the distance below a lane's rows from the next lane
    (csrc/kernels_bi_scan.cuh); the plain variant computes it.  Same move log, exhaustive and pruned, from an NN start and from a
    random start (wrap-around reversals), tile rows 32 R - 1 per warp vs 32 R."""
    xy = uniform_instance(2300)
    engine.set_option("block_threads", T)
    engine.set_option("rows_per_thread", R)
    engine.set_option("tile_cols", TJ)
    engine.set_option("row_shuffle", shuffle)
    try:
        succ, _ = oracle.nn_tour(xy, 0, 0)
        _check_bi(engine, oracle, xy, 0, succ, max_passes=30)
        assert engine.info("row_shuffle") == shuffle and engine.info("tile_rows") == ((T // 32) * (32 * R - 1) if shuffle else T * R)
        rnd = order_to_succ(np.random.default_rng(17).permutation(len(xy)))
        _check_bi(engine, oracle, xy, 0, rnd, max_passes=12)
    finally:
        engine.set_option("block_threads", 0)
        engine.set_option("rows_per_thread", 0)
        engine.set_option("tile_cols", 0)
        engine.set_option("row_shuffle", -1)


def test_bi_random_start_and_wraparound_reversals(engine, oracle):
    """random permutations: most moves have pos[a] > pos[b] for some step, i.e. the reversed forward path wraps."""
    rng = np.random.default_rng(5)
    for n, wt in [(333, 0), (400, 3), (257, 5), (64, 0), (5, 0), (4, 0), (7, 0)]:
        xy = rng.integers(0, 2000, size=(n, 2)).astype(np.float64)
        succ = order_to_succ(rng.permutation(n).astype(np.int32))
        _check_bi(engine, oracle, xy, wt, succ)
        _check_fi(engine, oracle, xy, wt, succ, oracle.succ_cost(xy, wt, succ))


def test_duplicate_points_and_ties(engine, oracle):
    """many equal deltas: the (delta, i, j) tie-break must pick the reference's lowest (i, j)."""
    rng = np.random.default_rng(9)
    xy = rng.integers(0, 12, size=(300, 2)).astype(np.float64)  # heavy duplicates, tiny integer distances
    succ = order_to_succ(rng.permutation(300).astype(np.int32))
    _check_bi(engine, oracle, xy, 0, succ)
    _check_fi(engine, oracle, xy, 0, succ, oracle.succ_cost(xy, 0, succ))
    grid = np.array([(x, y) for x in range(20) for y in range(20)], dtype=np.float64) * 10
    succ = order_to_succ(rng.permutation(400).astype(np.int32))
    _check_bi(engine, oracle, grid, 0, succ)
    _check_fi(engine, oracle, grid, 3, succ, oracle.succ_cost(grid, 3, succ))


def test_non_fp32_coordinates_use_fp64_exact_check(engine, oracle):
    rng = np.random.default_rng(21)
    xy = rng.integers(0, 300000, size=(500, 2)) + rng.integers(0, 1000, size=(500, 2)) / 1000.0
    succ, cost = oracle.nn_tour(xy, 0, 0)
    engine.set_instance(xy, 0)
    assert engine.info("exact32") == 0 and engine.info("fp32_ok") == 1
    _check_bi(engine, oracle, xy, 0, succ)
    _check_fi(engine, oracle, xy, 0, succ, cost)


def test_uni4000_bi_first_passes_and_fi_full(engine, oracle):
    xy = uniform_instance(4000)
    succ, cost = oracle.nn_tour(xy, 0, 0)
    assert cost == 565693  # SURVEY.md §8(c)
    _check_bi(engine, oracle, xy, 0, succ, max_passes=40)
    st = _check_fi(engine, oracle, xy, 0, succ, cost)
    assert st.moves == 1156 and st.passes == 9


def test_uni10000_bi_passes_match_oracle(engine, oracle):
    """BASELINE config 3 at full size: the first 3 passes move-for-move, then properties to the local optimum."""
    xy = uniform_instance(10000)
    succ, cost = oracle.nn_tour(xy, 0, 0)
    _check_bi(engine, oracle, xy, 0, succ, max_passes=3)
    engine.set_instance(xy, 0)
    s, obj, st, log = engine.two_opt(BI, succ, 0.0, log_cap=4000)
    assert st.status == 0 and is_tour(s)
    assert obj == oracle.succ_cost(xy, 0, s) == cost + log[:, 2].sum()
    assert (log[:, 2] < 0).all() and (log[:, 0] < log[:, 1]).all()
    # idempotence: a 2-opt local optimum has no improving move left -> exactly one more scan, no move
    s2, obj2, st2, _ = engine.two_opt(BI, s, 0.0)
    assert (s2 == s).all() and st2.moves == 0 and st2.passes == 1
    # and the oracle agrees that nothing improves (one full CPU scan)
    _, _, key = oracle.bi_scan_rows_mt(xy, 0, s, 0, 10000, 8)
    assert key[0] == 0


# ---- batched 2-opt -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [FI, BI])
def test_batch_kernel_parity(engine, oracle, instances, mode):
    for nm, batch in [("berlin52", 40), ("pr299", 12), ("att48", 20), ("ulysses22", 10)]:
        xy, wt = instances[nm]
        n = len(xy)
        tours = random_tours(n, batch, seed=n)
        tours[0], _ = oracle.nn_tour(xy, wt, 0)
        engine.set_instance(xy, wt)
        obj0 = np.array([oracle.succ_cost(xy, wt, t) for t in tours])
        out, obj, st = engine.two_opt_batch(mode, tours, obj0)
        for b in range(batch):
            if mode == BI:
                es, eo, est, _ = oracle.two_opt_bi(xy, wt, tours[b])
            else:
                es, eo, est, _ = oracle.two_opt_fi(xy, wt, tours[b], obj0[b])
            assert (out[b] == es).all() and obj[b] == eo, (nm, b)


def test_batch_ga_population_uni1000(engine, oracle):
    """BASELINE config 5 shape: random population on uni1000, FI repair == reference alg_2opt per tour."""
    xy = uniform_instance(1000)
    tours = random_tours(1000, 64, seed=1000)
    engine.set_instance(xy, 0)
    obj0 = engine.tour_costs(tours, as_order=False)
    for b in range(4):
        assert obj0[b] == oracle.succ_cost(xy, 0, tours[b])
    out, obj, st = engine.two_opt_batch(FI, tours, obj0)
    for b in (0, 17, 63):
        es, eo, _, _ = oracle.two_opt_fi(xy, 0, tours[b], obj0[b])
        assert (out[b] == es).all() and obj[b] == eo
    for b in range(64):
        assert is_tour(out[b]) and obj[b] == oracle.succ_cost(xy, 0, out[b])


# ---- NN + costs ----------------------------------------------------------------------------------------------
def test_nn_tour_parity(engine, oracle, instances, goldens):
    for nm in ["berlin52", "att532", "gr666", "dsj1000", "pr1002"]:
        xy, wt = instances[nm]
        engine.set_instance(xy, wt)
        s, c = engine.nn_tour(0)
        g = goldens["instances"][nm]
        assert c == g["nn_cost"] and sha(s) == g["nn_sha256"], nm
    xy = uniform_instance(5000)
    engine.set_instance(xy, 0)
    for start in (0, 4999, 1234):
        s, c = engine.nn_tour(start)
        es, ec = oracle.nn_tour(xy, 0, start)
        assert (s == es).all() and c == ec


def test_tour_costs_order_and_succ(engine, oracle, instances):
    xy, wt = instances["att532"]
    n = len(xy)
    rng = np.random.default_rng(2)
    orders = np.stack([rng.permutation(n).astype(np.int32) for _ in range(9)])
    engine.set_instance(xy, wt)
    got = engine.tour_costs(orders, as_order=True)
    for b in range(9):
        assert got[b] == oracle.order_cost(xy, wt, orders[b])
    succs = np.stack([order_to_succ(o) for o in orders])
    assert (engine.tour_costs(succs, as_order=False) == got).all()


# ---- the reference-named drop-in symbols ------------------------------------------------------------------------
def test_dropin_symbols_on_reference_instance(oracle, instances):
    L = C.CDLL(eng.DROPIN_PATH)
    L.calc_dist.restype = C.c_double
    L.calc_dist.argtypes = [C.c_int, C.c_int, C.c_void_p]
    L.alg_2opt.argtypes = [C.c_void_p]
    L.alg_2opt_tabu.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    for nm in ["pr299", "att532", "gr666"]:
        xy, wt = instances[nm]
        n = len(xy)
        succ, cost = oracle.nn_tour(xy, wt, 0)
        inst = RefInstance(xy, wt, succ, cost)
        for (i, j) in [(0, 0), (0, 1), (5, 17), (n - 1, 3)]:
            assert L.calc_dist(i, j, C.byref(inst.c)) == oracle.dist(xy, wt, i, j)
        assert L.alg_2opt(C.byref(inst.c)) == 0
        es, eo, _, _ = oracle.two_opt_fi(xy, wt, succ, cost)
        assert (inst.succ() == es).all() and inst.c.solution.obj_best == eo
        inst2 = RefInstance(xy, wt, succ, 123.0)
        prev = np.full(n, -1, dtype=np.int32)
        assert L.alg_2opt_tabu(C.byref(inst2.c), None, prev.ctypes.data, 1, 1) == 0
        bs, bo, _, _, bprev = oracle.two_opt_bi(xy, wt, succ, want_prev=True)
        assert (inst2.succ() == bs).all() and inst2.c.solution.obj_best == bo and (prev == bprev).all()
    L.tspb200_dropin_reset()


def test_errors_are_loud(engine):
    engine.set_instance(uniform_instance(50), 0)
    bad = np.arange(50, dtype=np.int32)  # self loops: not a cycle
    with pytest.raises(eng.TspB200Error):
        engine.tour_upload(bad)
    with pytest.raises(eng.TspB200Error):
        engine.set_option("rows_per_thread", 3)


def test_upload_ranks_the_successor_array_on_the_device(engine, oracle):
    """tour upload: visiting order from the successor array by pointer jumping on the device (csrc/kernels_misc.cu
    launch_succ_to_order, default for n >= 2048) == the host walk: same state, same 2-opt run; and the same loud rejection of
    everything that is not one Hamiltonian cycle."""
    rng = np.random.default_rng(3)
    for n in (5, 64, 1000, 2049, 5000):
        xy = np.floor(rng.random((n, 2)) * 3000.0)
        engine.set_instance(xy, 0)
        succ = order_to_succ(rng.permutation(n).astype(np.int32))
        res = {}
        for mode in (0, 1):
            engine.set_option("upload_rank", mode)
            engine.tour_upload(succ, log_cap=16)
            s0, c0 = engine.tour_download()
            engine.bi_run(5)
            res[mode] = (s0, c0, engine.tour_log(16).tolist(), engine.tour_download())
        assert (res[0][0] == succ).all() and (res[1][0] == succ).all() and res[0][1] == res[1][1] == oracle.succ_cost(xy, 0, succ), n
        assert res[0][2] == res[1][2] and (res[0][3][0] == res[1][3][0]).all() and res[0][3][1] == res[1][3][1], n
    n = 3000
    engine.set_instance(np.floor(rng.random((n, 2)) * 3000.0), 0)
    good = order_to_succ(rng.permutation(n).astype(np.int32))
    two_cycles = good.copy()                      # cut the cycle in two: swap the successors of two nodes
    a, b = 17, int(good[good[good[17]]])
    two_cycles[a], two_cycles[b] = good[b], good[a]
    out_of_range = good.copy(); out_of_range[5] = n
    negative = good.copy(); negative[7] = -1
    not_a_permutation = good.copy(); not_a_permutation[9] = good[11]
    self_loops = np.arange(n, dtype=np.int32)
    try:
        for mode in (0, 1):
            engine.set_option("upload_rank", mode)
            for bad in (two_cycles, out_of_range, negative, not_a_permutation, self_loops):
                with pytest.raises(eng.TspB200Error):
                    engine.tour_upload(bad)
                with pytest.raises(eng.TspB200Error):
                    engine.bi_run(1)          # nothing resident after a rejected upload
            engine.tour_upload(good)
            assert (engine.tour_download()[0] == good).all()
    finally:
        engine.set_option("upload_rank", -1)


# ---- tabu-masked best improvement (reference src/tabusearch.c:83-92,137-149) ---------------------------------
@pytest.mark.parametrize("n,wt,density,iter_,tenure", [(60, 0, 0.2, 30, 12), (200, 0, 0.05, 100, 20), (299, 5, 0.3, 50, 49),
                                                       (150, 4, 0.1, 40, 5), (120, 3, 0.5, 10, -1), (500, 0, 0.02, 1000, 50)])
def test_tabu_masked_bi_equals_oracle(engine, oracle, n, wt, density, iter_, tenure):
    """same move log, tour, cost AND the same lazily-expired tabu list as the oracle (itself pinned to the compiled
    reference by tests/test_oracle.py::test_tabu_mask_restatement)."""
    rng = np.random.default_rng(n + iter_)
    xy = rng.integers(0, 1000, size=(n, 2)).astype(np.float64)
    if wt == 4:
        xy = xy / 10.0 - 50.0  # GEO: degrees.minutes
    succ = order_to_succ(rng.permutation(n).astype(np.int32))
    ncols = n * (n - 1) // 2
    mask = np.where(rng.random(ncols) < density, rng.integers(1, iter_ + 1, size=ncols), 0).astype(np.int32)
    m_ref = mask.copy()
    es, eobj, est, elog = oracle.two_opt_bi(xy, wt, succ, skip_edge=m_ref, iter_=iter_, tenure=tenure, log_cap=100000)
    engine.set_instance(xy, wt)
    for use_matrix in (False, True):
        if use_matrix:
            engine.dist_matrix_build()
        s, obj, st, log, m_out = engine.two_opt_tabu(succ, mask, iter_, tenure, log_cap=100000)
        assert log.tolist() == elog.tolist()
        assert (s == es).all() and obj == eobj and st.moves == est.moves and st.passes == est.passes
        assert (m_out == m_ref).all(), int((m_out != m_ref).sum())
    engine.dist_matrix_free()


def _two_exchange(succ, a, b):
    """The tabu kick (reference src/tabusearch.c:293-295): succ[a]=b; succ[a1]=b1; reverse_path(b, a1)."""
    succ = succ.copy()
    a1, b1 = int(succ[a]), int(succ[b])
    path = [a1]
    while path[-1] != b:
        path.append(int(succ[path[-1]]))
    succ[a] = b
    for k in range(len(path) - 1, 0, -1):
        succ[path[k]] = path[k - 1]
    succ[a1] = b1
    return succ


def test_tabu_search_iterations_replayed(engine, oracle):
    """A deterministic replay of the reference's tabu() loop (src/tabusearch.c:228-311): masked 2-opt, random
    non-adjacent kick, the two removed edges enter the list with the iteration stamp, the tenure steps between two
    values (so expired entries can become tabu again unless the lazy expiry zeroed them).  The device path must track
    the oracle for 40 iterations: tours, costs and the list itself."""
    rng = np.random.default_rng(5)
    n = 180
    xy = rng.integers(0, 2000, size=(n, 2)).astype(np.float64)
    engine.set_instance(xy, 0)
    succ_o, _ = oracle.nn_tour(xy, 0, 0)
    succ_g = succ_o.copy()
    ncols = n * (n - 1) // 2
    tl_o = np.zeros(ncols, dtype=np.int32)
    tl_g = np.zeros(ncols, dtype=np.int32)

    def pos(i, j):
        if i > j:
            i, j = j, i
        return i * n + j - ((i + 1) * (i + 2)) // 2

    tenure = 4
    for it in range(1, 41):
        succ_o, obj_o, _, _ = oracle.two_opt_bi(xy, 0, succ_o, skip_edge=tl_o, iter_=it, tenure=tenure)
        succ_g, obj_g, _, _, tl_g = engine.two_opt_tabu(succ_g, tl_g, it, tenure)
        assert (succ_o == succ_g).all() and obj_o == obj_g and (tl_o == tl_g).all(), it
        while True:
            a, b = int(rng.integers(0, n)), int(rng.integers(0, n))
            a1, b1 = int(succ_o[a]), int(succ_o[b])
            if a != b and a1 != b and b1 != a:
                break
        succ_o = _two_exchange(succ_o, a, b)
        succ_g = succ_o.copy()
        for tl in (tl_o, tl_g):
            tl[pos(a, a1)] = it
            tl[pos(b, b1)] = it
        if it % 10 == 0:
            tenure = 18 if tenure == 4 else 4


# ---- batched nearest neighbour (reference HEU_Greedy_iter, src/heuristics.c:168-205) -------------------------------
@pytest.mark.parametrize("nm", ["berlin52", "pr299", "att532", "gr666", "dsj1000", "ulysses22"])
def test_nn_batch_every_start_equals_oracle(engine, oracle, instances, nm):
    xy, wt = instances[nm]
    n = len(xy)
    engine.set_instance(xy, wt)
    starts = np.arange(n, dtype=np.int32) if n <= 300 else np.random.default_rng(1).choice(n, size=64, replace=False).astype(np.int32)
    for use_matrix in (False, True):
        if use_matrix:
            engine.dist_matrix_build()
        succ, costs = engine.nn_tour_batch(starts)
        for b, s0 in enumerate(starts):
            osucc, ocost = oracle.nn_tour(xy, wt, int(s0))
            assert (succ[b] == osucc).all() and costs[b] == ocost, (nm, int(s0))
    engine.dist_matrix_free()


def test_greedy_iter_equals_reference_driver(engine, reference_outputs, reflib_if_built, instances):
    """best-of-n-starts == the reference's own HEU_Greedy_iter (first strictly better start wins)."""
    for nm in ("berlin52", "pr299", "rd400"):
        xy, wt = instances[nm]
        engine.set_instance(xy, wt)
        best, succ, cost = engine.greedy_iter()
        r = reference_outputs["greedy_iter"][nm]
        assert cost == r["cost"] and sha(succ) == r["sha256"], nm
        if reflib_if_built:
            st, rsucc, robj = reflib_if_built.run_method("HEU_Greedy_iter", xy, wt)
            assert st == 0 and cost == robj and (succ == rsucc).all(), nm


def test_nn_batch_duplicate_points_and_ties(engine, oracle):
    rng = np.random.default_rng(9)
    xy = rng.integers(0, 12, size=(200, 2)).astype(np.float64)  # many equal distances and coincident nodes
    engine.set_instance(xy, 0)
    starts = np.arange(200, dtype=np.int32)
    succ, costs = engine.nn_tour_batch(starts)
    for b in range(0, 200, 7):
        osucc, ocost = oracle.nn_tour(xy, 0, b)
        assert (succ[b] == osucc).all() and costs[b] == ocost


# ---- edge cases: tiny tours, caps, limits ------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6, 7, 9, 33, 64, 65, 129])
def test_tiny_instances_all_paths(engine, oracle, n):
    """n < 4 has no non-adjacent pair at all (one empty pass / sweep); n = 4, 5 have 2 and 5.  Every entry point must agree
    with the oracle: matrix, NN, BI (grid, exact, matrix and batched kernels), FI (grid and batched), tour costs."""
    rng = np.random.default_rng(n)
    xy = rng.integers(0, 50, size=(n, 2)).astype(np.float64)
    engine.set_instance(xy, 0)
    assert (engine.dist_matrix() == oracle.dist_matrix(xy, 0)).all()
    engine.dist_matrix_free()
    succ0 = order_to_succ(rng.permutation(n).astype(np.int32))
    cost0 = oracle.succ_cost(xy, 0, succ0)
    assert engine.tour_costs(succ0[None, :], as_order=False)[0] == cost0
    nn, nnc = engine.nn_tour(0)
    onn, onnc = oracle.nn_tour(xy, 0, 0)
    assert (nn == onn).all() and nnc == onnc
    es, eobj, est, elog = oracle.two_opt_bi(xy, 0, succ0, log_cap=1000)
    for fp in (-1, 1, 2):
        engine.set_option("force_path", fp)
        if fp == 2:
            engine.dist_matrix_build()
        s, obj, st, log = engine.two_opt(BI, succ0, 0.0, log_cap=1000)
        assert log.tolist() == elog.tolist() and (s == es).all() and obj == eobj and st.passes == est.passes, (n, fp)
    engine.set_option("force_path", -1)
    engine.dist_matrix_free()
    fs, fobj, fst, flog = oracle.two_opt_fi(xy, 0, succ0, cost0, log_cap=1000)
    s, obj, st, log = engine.two_opt(FI, succ0, cost0, log_cap=1000)
    assert log.tolist() == flog.tolist() and (s == fs).all() and obj == fobj and st.passes == fst.passes
    sb, ob, _ = engine.two_opt_batch(BI, np.stack([succ0, succ0]), np.array([0.0, 0.0]))
    assert (sb[0] == es).all() and (sb[1] == es).all() and ob[0] == eobj
    sb, ob, _ = engine.two_opt_batch(FI, np.stack([succ0]), np.array([cost0]))
    assert (sb[0] == fs).all() and ob[0] == fobj


def test_pass_and_move_caps_resume_where_they_stopped(engine, oracle):
    """max_passes / max_moves stop early with status STOPPED_BY_CAP; repeated capped calls on the resident tour walk through
    exactly the oracle's move sequence."""
    xy = uniform_instance(700)
    succ0, c0 = oracle.nn_tour(xy, 0, 0)
    engine.set_instance(xy, 0)
    _, _, est, elog = oracle.two_opt_bi(xy, 0, succ0, log_cap=100000)
    engine.tour_upload(succ0, log_cap=100000)
    total = 0
    while True:
        st = engine.bi_run(7)
        total += st.passes
        if st.status == eng.LOCAL_OPTIMUM:
            break
        assert st.status == eng.STOPPED_BY_CAP and st.passes == 7
    assert total == est.passes and engine.tour_log(100000).tolist() == elog.tolist()
    _, _, fst, flog = oracle.two_opt_fi(xy, 0, succ0, c0, log_cap=100000)
    engine.tour_upload(succ0, log_cap=100000)
    while True:
        st = engine.fi_run(5)
        if st.status == eng.LOCAL_OPTIMUM:
            break
        assert st.status == eng.STOPPED_BY_CAP and st.moves == 5
    assert engine.tour_log(100000).tolist() == flog.tolist()


def test_time_limit_returns_reference_status(engine):
    """a 1 ms budget on a 20 000-node tour: status TIME_LIMIT_EXCEEDED (reference include/heuristics.h:7), tour still valid."""
    xy = uniform_instance(20000)
    engine.set_instance(xy, 0)
    succ0, _ = engine.nn_tour(0)
    engine.set_option("time_limit_ms", 1)
    try:
        s, obj, st, _ = engine.two_opt(BI, succ0, 0.0)
        assert st.status == eng.TIME_LIMIT_EXCEEDED and is_tour(s)
        assert obj == engine.tour_costs(s[None, :], as_order=False)[0]
    finally:
        engine.set_option("time_limit_ms", 0)


def test_large_coordinates_take_the_exact_path(engine, oracle):
    """pla85900-like coordinates (~1.4e6, beyond the FP32 filter's validity window dmax < 4e6 only just): parity on BI."""
    rng = np.random.default_rng(77)
    xy = rng.integers(0, 3_500_000, size=(400, 2)).astype(np.float64)
    succ0, _ = oracle.nn_tour(xy, 3, 0)
    _check_bi(engine, oracle, xy, 3, succ0)
    assert engine.info("fp32_ok") == 0


def test_nn_uni100000_equals_committed_fixture(engine):
    """the headline instance's start tour: GPU nearest neighbour (10^10 exact distances, 0.4 s) == the oracle's tour
    committed as tests/golden/nn_uni100000.npz (2 min of CPU, tests/golden/make_nn_uni100000.py)."""
    import os
    from conftest import GOLD_DIR
    z = np.load(os.path.join(GOLD_DIR, "nn_uni100000.npz"))
    engine.set_instance(uniform_instance(100000), 0)
    succ, cost = engine.nn_tour(0)
    assert (succ == z["succ"]).all() and cost == float(z["cost"])


def _nn_grid_cases():
    rng = np.random.default_rng(77)
    cases = []
    cases.append(("uniform_int_ties", np.floor(rng.random((3000, 2)) * 60.0), 0))            # small integer box: masses of equal distances
    cases.append(("duplicates", np.repeat(np.floor(rng.random((500, 2)) * 1000.0), 4, axis=0), 0))
    cl = np.concatenate([rng.normal(c, 30.0, (600, 2)) for c in ((0, 0), (5000, 200), (-3000, 9000), (100000, 100000))])
    cases.append(("clusters_far_apart", np.round(cl, 3), 0))                                 # long jumps: rings run out, whole-block scan
    cases.append(("collinear", np.stack([np.floor(rng.random(2000) * 1e5), np.zeros(2000)], axis=1), 0))
    cases.append(("ceil_decimal", np.round(rng.random((2500, 2)) * 5000.0, 2), 3))
    cases.append(("att", np.floor(rng.random((2500, 2)) * 8000.0), 5))
    cases.append(("negative_half_integers", np.floor(rng.random((2000, 2)) * 4000.0) / 2.0 - 1000.0, 0))
    cases.append(("tall_box", np.stack([np.floor(rng.random(1500) * 30.0), np.floor(rng.random(1500) * 1e6)], axis=1), 0))
    return cases


@pytest.mark.parametrize("case", _nn_grid_cases(), ids=lambda c: c[0])
def test_nn_bucket_grid_walk_equals_oracle(engine, oracle, case):
    """reference src/heuristics.c:18-78 greedy on the bucket grid (csrc/kernels_nn.cu): the tour of the oracle's full scan, node
    for node, whatever the ties / empty neighbourhoods, and the same tour as the grid-wide kernel it replaces."""
    nm, xy, wt = case
    engine.set_instance(xy, wt)
    try:
        for start in (0, len(xy) - 1, len(xy) // 3):
            engine.set_option("nn_grid", 1)
            s, c = engine.nn_tour(start)
            es, ec = oracle.nn_tour(xy, wt, start)
            assert (s == es).all() and c == ec, (nm, start)
        engine.set_option("nn_grid", 0)
        s0, c0 = engine.nn_tour(0)
        es, ec = oracle.nn_tour(xy, wt, 0)
        assert (s0 == es).all() and c0 == ec, nm
    finally:
        engine.set_option("nn_grid", -1)


def test_nn_bucket_grid_small_and_degenerate(engine, oracle):
    """forced onto the bucket grid: tiny instances, all points equal, two points"""
    for n in (2, 3, 5, 17, 64, 255):
        xy = np.floor(np.random.default_rng(n).random((n, 2)) * 50.0)
        engine.set_instance(xy, 0)
        engine.set_option("nn_grid", 1)
        try:
            s, c = engine.nn_tour(n - 1)
        finally:
            engine.set_option("nn_grid", -1)
        es, ec = oracle.nn_tour(xy, 0, n - 1)
        assert (s == es).all() and c == ec, n
    xy = np.full((300, 2), 7.0)
    engine.set_instance(xy, 0)
    s, c = engine.nn_tour(5)
    es, ec = oracle.nn_tour(xy, 0, 5)
    assert (s == es).all() and c == ec


# ---- extra mileage (reference HEU_extramileage, src/heuristics.c:208-314) and the remaining published CSV columns ------
@pytest.mark.parametrize("nm", ["berlin52", "pr299", "att532", "gr666", "dsj1000", "ulysses22", "eil51"])
def test_extra_mileage_equals_reference_driver(engine, reference_outputs, reflib_if_built, instances, nm):
    xy, wt = instances[nm]
    engine.set_instance(xy, wt)
    if wt == 4:
        engine.dist_matrix_build()
    succ, cost = engine.extra_mileage()
    r = reference_outputs["extra_mileage"][nm]
    assert cost == r["cost"] and sha(succ) == r["sha256"], nm
    if reflib_if_built:
        st, rsucc, robj = reflib_if_built.run_method("HEU_extramileage", xy, wt)
        assert st == 0 and cost == robj and (succ == rsucc).all(), nm
    engine.dist_matrix_free()


def test_extra_mileage_ties_and_duplicates(engine, oracle):
    rng = np.random.default_rng(21)
    for n in (2, 3, 4, 9, 40, 150, 400):
        xy = rng.integers(0, 9, size=(n, 2)).astype(np.float64)  # few distinct points: ties everywhere, zero distances
        for wt in (0, 3, 5):
            engine.set_instance(xy, wt)
            succ, cost = engine.extra_mileage()
            osucc, ocost = oracle.extra_mileage(xy, wt)
            assert cost == ocost and (succ == osucc).all(), (n, wt)


def test_constructive_kernels_equal_oracle_on_fixtures(engine, oracle, instances):
    for nm in ("pr299", "att532", "gr666", "rd400", "ulysses16"):
        xy, wt = instances[nm]
        engine.set_instance(xy, wt)
        if wt == 4:
            engine.dist_matrix_build()
        s, c = engine.extra_mileage()
        os_, oc = oracle.extra_mileage(xy, wt)
        assert c == oc and (s == os_).all(), nm
        b, s, c = engine.greedy_iter()
        ob, os_, oc = oracle.greedy_iter(xy, wt)
        assert (b, c) == (ob, oc) and (s == os_).all(), nm
        engine.dist_matrix_free()


def test_reference_csv_all_deterministic_columns(engine, instances, goldens):
    """GREEDY_ITER, EXTR_MILE (results/constructive_heuristics_new.csv) and 2OPT_GREEDY_ITER, 2OPT_EXTR_MIL
    (results/constructive_heuristics_2opt_new.csv), 18 instances: construction on the GPU, then alg_2opt on the GPU, must
    land on the reference's published objective values."""
    for nm, row in sorted(goldens["reference_csv"].items()):
        xy, wt = instances[nm]
        engine.set_instance(xy, wt)
        if wt == 4:
            engine.dist_matrix_build()
        _, s_gi, c_gi = engine.greedy_iter()
        assert c_gi == row["GREEDY_ITER"], nm
        _, o_gi, _, _ = engine.two_opt(FI, s_gi, c_gi)
        assert o_gi == row["2OPT_GREEDY_ITER"], nm
        s_em, c_em = engine.extra_mileage()
        assert c_em == row["EXTR_MILE"], nm
        _, o_em, _, _ = engine.two_opt(FI, s_em, c_em)
        assert o_em == row["2OPT_EXTR_MIL"], nm
        engine.dist_matrix_free()


def test_synthetic_full_runs_reach_the_reference_known_answers(engine):
    """SURVEY.md §8(c) known answers, produced by the compiled reference during the survey (NN start from node 0):
    uni2000 BI 339437 / 315 moves, FI 345191 / 630 moves / 6 sweeps; uni4000 BI 476692 / 604 moves, FI 491876 / 1156 / 9;
    uni10000 FI 781189.  Full runs to the local optimum through both single-tour routes where they apply."""
    for n, nn, bi, fi, fi_full in ((2000, 406727, (339437, 315), (345191, 630, 6), True), (4000, 565693, (476692, 604), (491876, 1156, 9), True),
                                   (10000, None, None, (781189, None, None), False)):
        xy = uniform_instance(n)
        engine.set_instance(xy, 0)
        succ, cost = engine.nn_tour(0)
        if nn is not None:
            assert cost == nn
        if bi is not None:
            for prune in (0, 1):  # exhaustive scan / exact tile pruning: same moves, same local optimum
                engine.set_option("prune", prune)
                s, obj, st, _ = engine.two_opt(BI, succ, 0.0)
                assert (obj, st.moves) == bi and st.passes == bi[1] + 1, (n, prune)
                full = (bi[1] + 1) * (n * (n - 3) // 2)
                assert st.evals == full if not prune else st.evals <= full, (n, prune)
            engine.set_option("prune", -1)
        for route in ((0, 1) if n <= 4096 else (0,)):
            engine.set_option("single_block", route)
            s, obj, st, _ = engine.two_opt(FI, succ, cost)
            assert obj == fi[0], (n, route)
            if fi_full:
                assert (st.moves, st.passes) == fi[1:], (n, route)
        engine.set_option("single_block", -1)


def test_fi_late_selection_equals_published_move_path(engine, oracle):
    """first improvement on one GPU: the apply launch that reads the search's winner itself (option fi_late = 1, the default;
    csrc/kernels_bi.cu apply_move_kernel) against the search kernel's last-block tail (fi_late = 0) and the oracle — move logs,
    tours, costs — in one go, in single moves (every run ends with a parked position entry to flush and starts with fresh
    hit words) and interleaved with best-improvement passes, which read the position table first improvement only writes."""
    xy = uniform_instance(1800)
    succ0, c0 = oracle.nn_tour(xy, 0, 0)
    engine.set_instance(xy, 0)
    engine.set_option("single_block", 0)
    try:
        fs, fobj, fst, flog = oracle.two_opt_fi(xy, 0, succ0, c0, log_cap=100000)
        for late in (1, 0):
            engine.set_option("fi_late", late)
            s, obj, st, log = engine.two_opt(FI, succ0, c0, log_cap=100000)
            assert log.tolist() == flog.tolist() and (s == fs).all() and obj == fobj and st.moves == fst.moves, late
        engine.set_option("fi_late", 1)
        # one move per run, 40 runs: the log must be the oracle's first 40 moves and the tour what they lead to
        engine.tour_upload(succ0, log_cap=64)
        for _ in range(40):
            st = engine.fi_run(1)
            assert st.moves == 1
        es, eobj, est, elog = oracle.two_opt_fi(xy, 0, succ0, c0, max_moves=40, log_cap=64)
        s, cost = engine.tour_download()
        assert engine.tour_log(64).tolist() == elog.tolist() and (s == es).all() and cost == eobj
        # fi_run(k) -> bi_run(m) -> fi_run(-1), each checked against the oracle started from the previous stage's tour
        engine.tour_upload(succ0)
        engine.fi_run(25)
        s1, c1 = engine.tour_download()
        e1, o1, _, _ = oracle.two_opt_fi(xy, 0, succ0, c0, max_moves=25)
        assert (s1 == e1).all() and c1 == o1
        engine.bi_run(9)
        s2, c2 = engine.tour_download()
        e2, o2, _, _ = oracle.two_opt_bi(xy, 0, e1, max_passes=9)
        assert (s2 == e2).all() and c2 == o2
        engine.fi_run(-1)
        s3, c3 = engine.tour_download()
        e3, o3, _, _ = oracle.two_opt_fi(xy, 0, e2, float(o2))
        assert (s3 == e3).all() and c3 == o3
    finally:
        engine.set_option("fi_late", 1)
        engine.set_option("single_block", -1)


def test_capped_runs_can_be_continued_in_either_mode(engine, oracle):
    """include/tspb200.h: repeated calls on the resident tour continue where the previous one stopped.  fi_run(k) then
    fi_run(-1) is the oracle's full first-improvement run; bi_run(k) then fi_run(-1) is the oracle's first-improvement
    run started from the tour k best-improvement passes lead to (node-space tables rebuilt, fresh sweep)."""
    xy = uniform_instance(900)
    succ0, c0 = oracle.nn_tour(xy, 0, 0)
    engine.set_instance(xy, 0)
    engine.set_option("single_block", 0)
    try:
        fs, fobj, fst, flog = oracle.two_opt_fi(xy, 0, succ0, c0, log_cap=100000)
        engine.tour_upload(succ0, log_cap=100000)
        st = engine.fi_run(7)
        assert st.status == eng.STOPPED_BY_CAP and st.moves == 7
        st = engine.fi_run(-1)
        assert st.status == eng.LOCAL_OPTIMUM and st.moves == fst.moves - 7
        s, cost = engine.tour_download()
        assert engine.tour_log(100000).tolist() == flog.tolist() and (s == fs).all() and cost == fobj
        # a finished run stays finished: one more call of either mode does nothing
        assert engine.fi_run(-1).moves == 0 and engine.bi_run(-1).moves == 0

        bs, bobj, bst, blog = oracle.two_opt_bi(xy, 0, succ0, max_passes=9, log_cap=100000)
        es, eobj, est, elog = oracle.two_opt_fi(xy, 0, bs, bobj, log_cap=100000)
        engine.tour_upload(succ0, log_cap=100000)
        st = engine.bi_run(9)
        assert st.status == eng.STOPPED_BY_CAP and st.moves == 9
        st = engine.fi_run(-1)
        assert st.status == eng.LOCAL_OPTIMUM and st.moves == est.moves
        s, cost = engine.tour_download()
        assert engine.tour_log(100000).tolist() == blog.tolist() + elog.tolist()
        assert (s == es).all() and cost == eobj
        # and the other way round: a capped first-improvement run followed by best improvement to the end
        ps, pobj, pst, plog = oracle.two_opt_fi(xy, 0, succ0, c0, max_moves=11, log_cap=100000)
        qs, qobj, qst, qlog = oracle.two_opt_bi(xy, 0, ps, log_cap=100000)
        engine.tour_upload(succ0, log_cap=100000)
        assert engine.fi_run(11).moves == 11
        st = engine.bi_run(-1)
        assert st.status == eng.LOCAL_OPTIMUM and st.moves == qst.moves
        s, cost = engine.tour_download()
        assert engine.tour_log(100000).tolist() == plog.tolist() + qlog.tolist() and (s == qs).all() and cost == qobj
    finally:
        engine.set_option("single_block", -1)


def test_edge_lengths_up_to_2_pow_24_and_loud_rejection_beyond(engine, oracle):
    """coordinates ~1e7: distances up to 1.4e7 still fit the FP32 edge-length words exactly (exact path, FP64 distances);
    coordinates ~1e8 do not — the 2-opt entry points must refuse instead of silently rounding."""
    rng = np.random.default_rng(123)
    xy = rng.integers(0, 10_000_000, size=(300, 2)).astype(np.float64)
    succ0 = order_to_succ(rng.permutation(300).astype(np.int32))
    _check_bi(engine, oracle, xy, 0, succ0)
    assert engine.info("fp32_ok") == 0 and engine.info("dist_bound") < (1 << 24)
    _check_fi(engine, oracle, xy, 0, succ0, oracle.succ_cost(xy, 0, succ0))
    big = rng.integers(0, 100_000_000, size=(300, 2)).astype(np.float64)
    engine.set_instance(big, 0)
    assert (engine.dist_matrix() == oracle.dist_matrix(big, 0)).all()  # distances themselves are fine
    engine.dist_matrix_free()
    for call in (lambda: engine.two_opt(BI, succ0, 0.0), lambda: engine.two_opt(FI, succ0, 0.0),
                 lambda: engine.two_opt_batch(BI, succ0[None, :])):
        with pytest.raises(eng.TspB200Error) as ei:
            call()
        assert ei.value.code == 5  # TSPB200_E_UNSUPPORTED


def test_pruned_scan_skips_tiles_but_not_moves(engine, oracle):
    """exact tile pruning on a spatially coherent tour: most tiles are provably dead, the move log is unchanged."""
    xy = uniform_instance(6000)
    succ0, _ = oracle.nn_tour(xy, 0, 0)
    engine.set_instance(xy, 0)
    logs = {}
    for prune in (0, 1):
        engine.set_option("prune", prune)
        s, obj, st, log = engine.two_opt(BI, succ0, 0.0, max_iters=120, log_cap=200)
        logs[prune] = (log.tolist(), s.tolist(), obj, st)
    engine.set_option("prune", -1)
    assert logs[0][:3] == logs[1][:3]
    st = logs[1][3]
    assert st.tiles_total > 0 and st.tiles_scanned < 0.7 * st.tiles_total
    es, eobj, est, elog = oracle.two_opt_bi(xy, 0, succ0, max_passes=120, log_cap=200)
    assert logs[1][0] == elog.tolist() and logs[1][2] == eobj


def test_batch_bi_position_space_kernel_equals_node_space_kernel_and_oracle(engine, oracle):
    """the position-space block kernel (csrc/kernels_batch.cu two_opt_batch_bi_kernel) against the node-space one and the
    oracle: random tours (wrap-around reversals), every FP32-path metric, sizes around the warp-tile boundaries."""
    rng = np.random.default_rng(31)
    for n, wt, batch in [(1000, 0, 6), (257, 3, 5), (256, 5, 5), (129, 0, 4), (128, 0, 4), (61, 5, 6), (33, 0, 3), (9, 0, 3), (5, 0, 2),
                         (4, 0, 2), (3, 0, 1), (700, 0, 3)]:
        xy = rng.integers(0, 3000, size=(n, 2)).astype(np.float64)
        if n == 700:
            xy = xy + rng.integers(0, 1000, size=(n, 2)) / 1000.0  # not FP32-exact: FP64 exact check from the node table
        tours = random_tours(n, batch, 1000 + n)
        engine.set_instance(xy, wt)
        res = {}
        for kern in (0, 1):
            engine.set_option("batch_kernel", kern)
            res[kern] = engine.two_opt_batch(BI, tours)
        engine.set_option("batch_kernel", 0)
        assert (res[0][0] == res[1][0]).all() and (res[0][1] == res[1][1]).all(), (n, wt)
        assert (res[0][2].moves, res[0][2].passes, res[0][2].evals) == (res[1][2].moves, res[1][2].passes, res[1][2].evals)
        for b in range(min(batch, 2)):
            es, eobj, est, _ = oracle.two_opt_bi(xy, wt, tours[b])
            assert (res[0][0][b] == es).all() and res[0][1][b] == eobj, (n, wt, b)


def test_batches_of_tours_too_large_for_one_block_run_on_the_grid_path(engine, oracle):
    """n = 12 000 exceeds the shared-memory tour of both block kernels: the batch entry point must still deliver (each tour goes
    through the grid kernels), with the same result as the single-tour call."""
    xy = uniform_instance(12000)
    engine.set_instance(xy, 0)
    s0, c0 = engine.nn_tour(0)
    s1, c1 = engine.nn_tour(5)
    tours = np.stack([s0, s1])
    sb, ob, st = engine.two_opt_batch(FI, tours, np.array([c0, c1]))
    for b, (s, c) in enumerate(((s0, c0), (s1, c1))):
        es, eo, _, _ = engine.two_opt(FI, s, c)
        assert (sb[b] == es).all() and ob[b] == eo
    assert is_tour(sb[0]) and ob[0] == oracle.succ_cost(xy, 0, sb[0])


def test_geo_matrix_reports_no_entry_on_a_rounding_boundary(engine, instances, oracle):
    """GEO depends on library cos / acos (CUDA vs glibc): the matrix kernel counts entries whose value handed to nint() lies
    within 1e-9 (1e-6 below 10 km) of a rounding boundary; none of the reference's GEO instances has one, so equality with
    the CPU is not luck."""
    seen = 0
    for nm, (xy, wt) in sorted(instances.items()):
        if wt != 4:
            continue
        engine.set_instance(xy, wt)
        m = engine.dist_matrix()
        assert (m == oracle.dist_matrix(xy, wt)).all(), nm
        assert engine.info("geo_near_boundary") == 0, nm
        engine.dist_matrix_free()
        seen += 1
    assert seen >= 5


def test_rows_on_demand_and_limits_the_reference_does_not_have(engine, oracle):
    """dist_row without a resident matrix; extra mileage with its state in global memory (forced at a size the oracle can
    check); batched nearest neighbour beyond the shared-memory limit falls back to the grid kernel per start."""
    xy = uniform_instance(1200)
    engine.set_instance(xy, 0)
    full = oracle.dist_matrix(xy, 0)
    for i in (0, 7, 1199):
        assert (engine.dist_row(i) == full[i]).all()
    es, ec = oracle.extra_mileage(xy, 0)
    for forced in (0, 1):
        engine.set_option("em_global", forced)
        s, c = engine.extra_mileage()
        assert (s == es).all() and c == ec, forced
    engine.set_option("em_global", 0)
    big = uniform_instance(23000)
    engine.set_instance(big, 0)
    succ, costs = engine.nn_tour_batch(np.array([0, 11], dtype=np.int32))
    for b, start in enumerate((0, 11)):
        s1, c1 = engine.nn_tour(start)
        assert (succ[b] == s1).all() and costs[b] == c1 and is_tour(succ[b])


def test_dropin_calc_dist_beyond_the_host_mirror_and_after_in_place_edits(oracle):
    """scalar calc_dist on an instance too large for the n x n host mirror (rows fetched from the device on demand, no abort),
    and on an instance whose nodes[] the caller rewrote IN PLACE between two calls (same pointer, same n): the sampled
    hash must notice and the stale matrix must not be served."""
    L = C.CDLL(eng.DROPIN_PATH)
    L.calc_dist.restype = C.c_double
    L.calc_dist.argtypes = [C.c_int, C.c_int, C.c_void_p]
    n = 17000
    xy = uniform_instance(n)
    succ = order_to_succ(np.arange(n, dtype=np.int32))
    inst = RefInstance(xy, 0, succ, 0.0)
    rng = np.random.default_rng(3)
    for i, j in rng.integers(0, n, size=(200, 2)):
        assert L.calc_dist(int(i), int(j), C.byref(inst.c)) == oracle.dist(xy, 0, int(i), int(j))
    small = uniform_instance(400)
    inst2 = RefInstance(small, 0, order_to_succ(np.arange(400, dtype=np.int32)), 0.0)
    assert L.calc_dist(3, 9, C.byref(inst2.c)) == oracle.dist(small, 0, 3, 9)
    moved = small[::-1].copy()
    inst2.xy[...] = moved  # rewrite the coordinates in place: same nodes pointer, same n
    for i, j in ((3, 9), (0, 399), (17, 250)):
        assert L.calc_dist(i, j, C.byref(inst2.c)) == oracle.dist(moved, 0, i, j)
    L.tspb200_dropin_reset()


def test_dropin_keeps_several_instances_resident(oracle):
    """a caller that alternates between instances (csrc/dropin.cpp: up to four resident contexts, least recently used first to
    go): every call is answered for the right instance, coming back to an instance does not evict the others, a fifth one
    replaces the least recently used, and alg_2opt on an instance still sees that instance's coordinates."""
    L = C.CDLL(eng.DROPIN_PATH)
    L.calc_dist.restype = C.c_double
    L.calc_dist.argtypes = [C.c_int, C.c_int, C.c_void_p]
    L.alg_2opt.argtypes = [C.c_void_p]
    L.tspb200_dropin_reset()
    rng = np.random.default_rng(11)
    insts = []
    for k, (n, wt) in enumerate(((300, 0), (300, 0), (450, 3), (200, 5), (350, 0))):
        xy = np.floor(rng.random((n, 2)) * 5000.0) + k
        succ, cost = oracle.nn_tour(xy, wt, 0)
        insts.append((xy, wt, RefInstance(xy, wt, succ, cost), succ, cost))
    for rounds in range(3):
        for k in (0, 1, 2, 3, 0, 2, 1, 3):
            xy, wt, ri, _, _ = insts[k]
            i, j = int(rng.integers(0, len(xy))), int(rng.integers(0, len(xy)))
            assert L.calc_dist(i, j, C.byref(ri.c)) == oracle.dist(xy, wt, i, j), (rounds, k)
        assert L.tspb200_dropin_resident() == 4
    xy, wt, ri, succ, cost = insts[4]                      # a fifth problem: replaces the least recently used (instance 0)
    assert L.alg_2opt(C.byref(ri.c)) == 0
    es, eobj, _, _ = oracle.two_opt_fi(xy, wt, succ, cost)
    assert (ri.succ() == es).all() and ri.c.solution.obj_best == eobj and L.tspb200_dropin_resident() == 4
    for k in (3, 1, 2, 0):                                 # instance 0 comes back (evicting another one): still the right answers
        xy, wt, ri, succ, cost = insts[k]
        assert L.calc_dist(1, 7, C.byref(ri.c)) == oracle.dist(xy, wt, 1, 7)
    xy, wt, ri, succ, cost = insts[2]
    assert L.alg_2opt(C.byref(ri.c)) == 0
    es, eobj, _, _ = oracle.two_opt_fi(xy, wt, succ, cost)
    assert (ri.succ() == es).all() and ri.c.solution.obj_best == eobj
    L.tspb200_dropin_reset()
    assert L.tspb200_dropin_resident() == 0

