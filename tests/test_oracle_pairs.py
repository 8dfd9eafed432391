"""oracle.bi_pairs_le (oracle/tsp_oracle.c orc_bi_pairs_le): every legal pair of one best-improvement scan whose exact
delta is at or below a threshold.  tests/test_gpu_filter_probe.py holds the device's FP32 filters against this set, so it
is checked here against the oracle's own scan, a plain numpy restatement and, where it is built, the compiled reference."""
import numpy as np
import pytest

from tsp_optimization_b200.instances import order_to_succ, uniform_instance

EUC_2D, CEIL_2D, ATT = 0, 3, 5


def _np_dist(xy, a, b, wt):
    """reference src/distutil.c calc_euc2d / calc_pseudo_euc / calc_ceil2d, one IEEE double operation at a time"""
    ex = xy[a, 0] - xy[b, 0]
    ey = xy[a, 1] - xy[b, 1]
    s = ex * ex + ey * ey
    if wt == ATT:
        r = np.sqrt(s / 10.0)
        t = np.trunc(r + 0.5)
        return np.where(t < r, t + 1.0, t)
    r = np.sqrt(s)
    return np.ceil(r) if wt == CEIL_2D else np.trunc(r + 0.5)


def _np_pairs_le(xy, wt, succ, H):
    n = len(xy)
    a, b = np.triu_indices(n, 1)
    a1, b1 = succ[a], succ[b]
    legal = (b != a1) & (b1 != a)
    a, b, a1, b1 = a[legal], b[legal], a1[legal], b1[legal]
    delta = _np_dist(xy, a, b, wt) + _np_dist(xy, a1, b1, wt) - _np_dist(xy, a, a1, wt) - _np_dist(xy, b, b1, wt)
    keep = delta <= H
    return np.stack([a[keep], b[keep], delta[keep].astype(np.int64)], axis=1)


def _cases():
    rng = np.random.default_rng(11)
    return [("uniform", uniform_instance(300), EUC_2D),
            ("lattice_ties", np.floor(rng.random((260, 2)) * 12.0), EUC_2D),
            ("decimal", rng.random((240, 2)) * 1000.0 + 0.3, EUC_2D),
            ("ceil", np.floor(rng.random((250, 2)) * 400.0), CEIL_2D),
            ("ceil_axis_lattice", np.stack(np.meshgrid(np.arange(16.0), np.arange(15.0)), -1).reshape(-1, 2) * 7.0, CEIL_2D),
            ("att", np.floor(rng.random((270, 2)) * 5000.0), ATT),
            ("att_decimal", rng.random((220, 2)) * 3000.0, ATT),
            ("duplicates", np.repeat(np.floor(rng.random((70, 2)) * 300.0), 3, axis=0), EUC_2D)]


def _tours(oracle, xy, wt, seed):
    succ, _ = oracle.nn_tour(xy, wt, 0)
    rnd = order_to_succ(np.random.default_rng(seed).permutation(len(xy)).astype(np.int32))
    return [("nn", succ), ("random", rnd)]


@pytest.mark.parametrize("case", range(len(_cases())))
def test_pairs_le_equal_numpy_restatement(oracle, case):
    nm, xy, wt = _cases()[case]
    for tour, succ in _tours(oracle, xy, wt, case):
        _, _, (m, _, _) = oracle.bi_scan_rows_mt(xy, wt, succ, 0, len(xy), 4)
        for H in sorted({m, -1, 0, m // 2}):
            got = oracle.bi_pairs_le(xy, wt, succ, H, threads=3)
            want = _np_pairs_le(xy, wt, np.asarray(succ), H)
            assert got.tolist() == want.tolist(), (nm, tour, H)
        if m < 0:
            assert (got[:, 2] <= 0).all() and len(got) > 0


@pytest.mark.parametrize("case", range(len(_cases())))
def test_pairs_le_minimum_is_the_scan_key(oracle, reflib_if_built, case):
    """the smallest delta of the set at H = -1, with its lowest (i, j), is the scan's (delta, i, j); at H = m the set holds
    the ties of the minimum only"""
    nm, xy, wt = _cases()[case]
    for tour, succ in _tours(oracle, xy, wt, 100 + case):
        ev, _, key = oracle.bi_scan_rows_mt(xy, wt, succ, 0, len(xy), 4)
        if reflib_if_built is not None:
            assert reflib_if_built.bi_scan_rows_mt(xy, wt, succ, 0, len(xy), 4)[2] == key, (nm, tour)
        m = key[0]
        if m >= 0:
            assert len(oracle.bi_pairs_le(xy, wt, succ, -1)) == 0
            continue
        pairs = oracle.bi_pairs_le(xy, wt, succ, -1)
        lo = pairs[pairs[:, 2] == pairs[:, 2].min()]
        assert (lo[0, 2], lo[0, 0], lo[0, 1]) == key, (nm, tour)
        ties = oracle.bi_pairs_le(xy, wt, succ, m)
        assert ties.tolist() == lo.tolist(), (nm, tour)
        # every legal pair at H = +inf: the scan's evaluation count
        assert len(oracle.bi_pairs_le(xy, wt, succ, 1 << 40)) == ev


def test_pairs_le_thread_count_does_not_matter(oracle):
    xy = uniform_instance(1500)
    succ, _ = oracle.nn_tour(xy, EUC_2D, 0)
    one = oracle.bi_pairs_le(xy, EUC_2D, succ, -1, threads=1)
    assert len(one) > 100
    assert oracle.bi_pairs_le(xy, EUC_2D, succ, -1, threads=7).tolist() == one.tolist()
