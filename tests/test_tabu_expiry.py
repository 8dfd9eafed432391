"""The exact lazy-expiry rule of the resident tabu search (kernels_tabu_search.cu, DESIGN.md §4.9), restated in numpy and
checked against the oracle: the entries one masked best-improvement pass (oracle.two_opt_bi with the list, max_passes=1,
i.e. one scan of alg_2opt_tabu, reference src/tabusearch.c:126-156) zeroes are exactly the expired non-zero entries that
T1-T4 say some non-adjacent pair reaches.  No GPU needed."""
import numpy as np
import pytest

from tsp_optimization_b200.instances import order_to_succ, uniform_instance


def _idx(x, y, n):
    """reference src/utility.c:17-30 x_udir_pos"""
    if x > y:
        x, y = y, x
    return x * n + y - (x + 1) * (x + 2) // 2


def expire_model(succ, tl, it, tenure):
    """-> the list after the lazy expiry of one masked pass over tour `succ`, by rules T1-T4"""
    n = len(succ)
    out = tl.copy()
    if it < 0 or tenure < 0:
        return out
    pred = np.empty(n, dtype=np.int64)
    pred[succ] = np.arange(n)

    def in_u(x, y):
        v = int(tl[_idx(x, y, n)])
        return v != 0 and it - v <= tenure

    def reached(x, y):
        if succ[x] != y and succ[y] != x:  # T1
            return True
        t, u = (x, y) if succ[x] == y else (y, x)
        for b in range(t + 1, n):  # T2
            if b != u and succ[b] != t and not in_u(t, b):
                return True
        for a in range(t):  # T3
            if a != u and succ[a] != t and not in_u(a, t) and not in_u(a, int(succ[a])):
                return True
        for a, b1 in ((x, y), (y, x)):  # T4
            b, a1 = int(pred[b1]), int(succ[a])
            if a < b and b != a1 and not in_u(a, b) and not in_u(a, a1) and not in_u(b, b1):
                return True
        return False

    for x in range(n):
        for y in range(x + 1, n):
            v = int(tl[_idx(x, y, n)])
            if v != 0 and it - v > tenure and reached(x, y):
                out[_idx(x, y, n)] = 0
    return out


def _case(rng, n, it, tenure, density):
    """a random tour and a list with stamps on tour edges and off them, on both sides of the tenure"""
    succ = order_to_succ(rng.permutation(n).astype(np.int32))
    tl = np.zeros(n * (n - 1) // 2, dtype=np.int32)
    lo = max(1, it - max(tenure, 0) - 4)
    for x in range(n):  # tour edges
        if rng.random() < density:
            tl[_idx(x, int(succ[x]), n)] = rng.integers(lo, it + 1)
    if density >= 1.0:  # saturated: every entry blocks except a few expired tour edges, which no pair can then reach
        tl[:] = it
        for x in rng.choice(n, 2, replace=False):
            tl[_idx(int(x), int(succ[x]), n)] = lo
        return succ, tl
    k = max(1, int(density * n))
    for _ in range(k):  # anywhere
        x, y = rng.choice(n, 2, replace=False)
        tl[_idx(int(x), int(y), n)] = rng.integers(lo, it + 1)
    return succ, tl


@pytest.mark.parametrize("tenure", [-1, 0, 3])
def test_expiry_model_equals_one_oracle_pass(oracle, tenure):
    rng = np.random.default_rng(100 + tenure)
    cases = 0
    zeroed = kept = 0
    for n in list(range(5, 20)) + [24, 31, 40, 60]:
        xy = uniform_instance(n, seed=n)
        for density in (0.15, 0.5, 0.9, 1.0):
            it = int(rng.integers(4, 12))
            succ, tl = _case(rng, n, it, tenure, density)
            want = expire_model(succ, tl, it, tenure)
            got = tl.copy()
            oracle.two_opt_bi(xy, 0, succ, max_passes=1, skip_edge=got, iter_=it, tenure=tenure)
            assert (got == want).all(), (n, density, np.nonzero(got != want))
            cases += 1
            expired = (tl != 0) & (it - tl > tenure) if tenure >= 0 else np.zeros_like(tl, dtype=bool)
            zeroed += int((expired & (want == 0)).sum())
            kept += int((expired & (want != 0)).sum())
    assert cases == 76
    if tenure >= 0:
        assert zeroed > 0 and kept > 0  # both outcomes occur: some expired entries are not reached by any pair
