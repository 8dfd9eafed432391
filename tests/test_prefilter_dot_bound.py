"""CPU model (numpy, FP32 rounding emulated) of the scan kernel's stage-1 prefilter in its dot-product form
(csrc/kernels_bi_scan.cuh, pf_dot_const; DESIGN.md §3): the translation chosen at set_instance, the row and column constants
A_p and B_q, the four-FMA chain and the final sum.  Every pair whose exact delta is <= the threshold, and every pair the
square-root FP32 filter passes, must pass it — including pairs placed exactly on the boundary d1 + d2 = a + b — and padding
must never pass nor produce a NaN.  One case shows that the rounding margins are needed."""
import numpy as np

from test_prefilter_bound import _window, exact_dist, fma32, pf_bound, sqrt_filter, stage1

f32 = np.float32
DOT_REL = np.ldexp(1.0, -19)
DOT_ABS = np.ldexp(1.0, -100)


def center(x, y):
    """engine.cu, tspb200_set_instance: the bounding box's center rounded to an integer, if it moves every FP32
    coordinate exactly; else no translation"""
    cx, cy = np.rint(0.5 * (x.min() + x.max())), np.rint(0.5 * (y.min() + y.max()))
    if max(abs(cx), abs(cy)) >= 2.0 ** 24:
        return 0.0, 0.0
    tx = x.astype(f32).astype(np.float64) - cx
    ty = y.astype(f32).astype(np.float64) - cy
    if (tx.astype(f32) == tx).all() and (ty.astype(f32) == ty).all():
        return float(cx), float(cy)
    return 0.0, 0.0


@np.errstate(invalid="ignore", over="ignore")
def dot_const(nrm, pf, margin=True):
    t = (nrm - pf).astype(f32)
    if not margin:
        return t
    low = (fma32(f32(-DOT_REL), (nrm + np.abs(pf)).astype(f32), t) - f32(DOT_ABS)).astype(f32)
    return np.where(pf == -np.inf, t, low)


def norm2(X, Y, i):
    return (fma32(Y[i], Y[i], (X[i] * X[i]).astype(f32)) + fma32(Y[i + 1], Y[i + 1], (X[i + 1] * X[i + 1]).astype(f32))).astype(f32)


@np.errstate(over="ignore")
def stage1_dot(x, y, ds, p, q, thr, E, att, c, margin=True):
    """min over rows of A_p + w_p . v_q, plus B_q, <= 0 — in FP32, as bi_scan_kernel computes it"""
    h = (f32(0.5) * (f32(thr) + f32(E))).astype(f32)
    X = (x.astype(f32) - f32(c[0])).astype(f32)
    Y = (y.astype(f32) - f32(c[1])).astype(f32)
    A = dot_const(norm2(X, Y, p), pf_bound(ds[p], h, att), margin)
    B = dot_const(norm2(X, Y, q), pf_bound(ds[q], h, att), margin)
    m2 = f32(-2.0)
    with np.errstate(invalid="raise"):
        acc = fma32(m2 * X[p], X[q], A)
        acc = fma32(m2 * Y[p], Y[q], acc)
        acc = fma32(m2 * X[p + 1], X[q + 1], acc)
        acc = fma32(m2 * Y[p + 1], Y[q + 1], acc)
        return (acc + B).astype(f32) <= 0


def _check_tour(xy, wt, order, expect_center=None, filters=True):
    n = len(order)
    x, y = xy[order, 0], xy[order, 1]
    x, y = np.append(x, x[0]), np.append(y, y[0])
    c = center(xy[:, 0], xy[:, 1])
    if expect_center is not None:
        assert c == expect_center
    idx = np.arange(n)
    ds = exact_dist(x, y, idx, idx + 1, wt)
    ds = np.append(ds, ds[0])
    W, E = _window(x, y, wt)
    p, q = np.triu_indices(n, 2)
    keep = ~((p == 0) & (q == n - 1))
    p, q = p[keep], q[keep]
    delta = exact_dist(x, y, p, q, wt) + exact_dist(x, y, p + 1, q + 1, wt) - ds[p] - ds[q]
    att = wt == 5
    for t in sorted({float(delta.min()), float(np.quantile(delta, 1e-3)), float(np.quantile(delta, 1e-2)), 0.0}):
        thr = f32(t + W)
        pass1 = stage1_dot(x, y, ds, p, q, thr, E, att, c)
        assert pass1[delta <= t].all(), t
        assert pass1[sqrt_filter(x, y, ds, p, q, thr, att)].all(), t
        if filters and t == float(delta.min()):  # and it filters about as well as the squared-distance form
            assert pass1.mean() <= stage1(x, y, ds, x, y, ds, p, q, thr, E, att).mean() + 1e-3
    return c


def _nn_order(xy):
    n = len(xy)
    left, cur, order = set(range(1, n)), 0, [0]
    while left:
        rest = np.fromiter(left, int)
        cur = int(rest[np.argmin(np.hypot(*(xy[rest] - xy[cur]).T))])
        left.remove(cur)
        order.append(cur)
    return np.array(order)


def test_dot_stage1_random_instances():
    rng = np.random.default_rng(21)
    for n, scale, wt, integer in [(400, 1e4, 0, True), (400, 1e4, 3, True), (400, 3e3, 5, True), (300, 2.5e6, 0, True),
                                  (300, 1e3, 0, False), (300, 1.0, 0, False)]:
        xy = rng.random((n, 2)) * scale
        if integer:
            xy = np.floor(xy)
        c = _check_tour(xy, wt, rng.permutation(n))
        if integer:
            assert c != (0.0, 0.0)
        _check_tour(xy, wt, _nn_order(xy))


def test_dot_stage1_duplicates_and_ties():
    rng = np.random.default_rng(22)
    xy = np.repeat(np.floor(rng.random((80, 2)) * 50), 4, axis=0)  # duplicate points: s = 0, ds = 0
    _check_tour(xy, 0, rng.permutation(len(xy)))
    _check_tour(np.floor(rng.random((300, 2)) * 20), 3, rng.permutation(300))


def test_dot_stage1_large_common_offset():
    """integer coordinates in 2^23 - 10^4 + [0, 10^4]: the translation is exact and brings them near the origin"""
    rng = np.random.default_rng(23)
    xy = 2.0 ** 23 - 1e4 + np.floor(rng.random((300, 2)) * 1e4)
    c = _check_tour(xy, 0, _nn_order(xy))
    assert c != (0.0, 0.0) and abs(c[0] - (2.0 ** 23 - 5e3)) < 1e2
    _check_tour(xy, 5, rng.permutation(300))


def test_dot_stage1_without_translation():
    """non-integer coordinates the translation would round: no translation (c = 0), still sound"""
    rng = np.random.default_rng(24)
    xy = (rng.random((300, 2)) * 1e3).astype(f32).astype(np.float64)
    xy[0] = [1e-3, 2e-3]
    _check_tour(xy, 0, _nn_order(xy), expect_center=(0.0, 0.0))
    # not FP32-exact, far from the origin: sound, but the margins (~ 2^-19 of |P|^2) let far more pairs through
    xy = 1e5 + rng.random((300, 2)) * 1e3
    xy[0] = [1e-3, 1e5]
    _check_tour(xy, 0, _nn_order(xy), expect_center=(0.0, 0.0), filters=False)


def _boundary_pairs(rng, count, spread, same_second=False):
    """d1 + d2 = a + b exactly (Pythagorean distances, integer ds), points anywhere in [-spread, spread]^2"""
    triples = [(3, 4, 5), (5, 12, 13), (8, 15, 17), (7, 24, 25), (20, 21, 29), (9, 40, 41), (12, 35, 37)]
    for _ in range(count):
        (a1, b1, c1), (a2, b2, c2) = triples[rng.integers(len(triples))], triples[rng.integers(len(triples))]
        k1, k2 = int(rng.integers(1, 40)), (0 if same_second else int(rng.integers(1, 40)))
        d1, d2 = c1 * k1, c2 * k2
        o1, o2 = rng.integers(-spread, spread, 2), rng.integers(-spread, spread, 2)
        x = np.array([o1[0], o2[0], o1[0] + a1 * k1, o2[0] + a2 * k2], dtype=np.float64)  # rows p, p+1; columns q, q+1
        y = np.array([o1[1], o2[1], o1[1] + b1 * k1, o2[1] + b2 * k2], dtype=np.float64)
        E = f32(4.0 * (np.hypot(4 * spread, 4 * spread) * 2.0 ** -20))
        L = d1 + d2
        if same_second:  # a = b: the squares' step (a + b)^2 <= 2a^2 + 2b^2 and d1^2 + d2^2 <= (d1 + d2)^2 are both tight
            dsp = dsq = float(L // 2)
        else:
            dsp = float(rng.integers(0, L + 1))
            dsq = float(rng.integers(-L // 4, L - dsp + 1))
        thr = f32(L - dsp - dsq - float(E))  # puts a + b exactly at d1 + d2
        yield x, y, np.array([dsp, 0.0, dsq, 0.0]), thr, E


def test_dot_stage1_on_its_boundary():
    rng = np.random.default_rng(25)
    for spread in (100, 5000, 2 ** 22):
        for x, y, ds, thr, E in _boundary_pairs(rng, 1500, spread):
            assert stage1_dot(x, y, ds, 0, 2, thr, E, False, (0.0, 0.0)), (x, y, ds)
        for x, y, ds, thr, E in _boundary_pairs(rng, 1500, spread, same_second=True):
            assert stage1_dot(x, y, ds, 0, 2, thr, E, False, (0.0, 0.0)), (x, y, ds)


def test_dot_stage1_needs_its_margins():
    """the same tight boundary pairs far from the origin: without the margins of pf_dot_const the FMA chain's rounding
    rejects some of them (so the boundary test above can fail)"""
    rng = np.random.default_rng(26)
    rejected = sum(not stage1_dot(x, y, ds, 0, 2, thr, E, False, (0.0, 0.0), margin=False)
                   for x, y, ds, thr, E in _boundary_pairs(rng, 1500, 5000, same_second=True))
    assert rejected > 0


@np.errstate(over="ignore")
def test_dot_stage1_padding_never_passes():
    """padding rows / columns (ds = -BIG, coordinates 0 or a real point's): A = B = +inf, never a hit, never a NaN"""
    big = 1e30
    x = np.array([0.0, 0.0, 37.0, 0.0, 12.0, 40.0])
    y = np.array([0.0, 0.0, -5.0, 0.0, 9.0, 3.0])
    ds = np.array([-big, -big, -big, -big, 3.0, 5.0])
    for p, q in [(0, 2), (4, 2), (0, 4), (2, 4)]:
        for c in [(0.0, 0.0), (5000.0, 5000.0)]:
            assert not stage1_dot(x, y, ds, p, q, f32(1e4), f32(0.0), False, c)
    h = f32(10.0)
    assert dot_const(f32(25.0), pf_bound(-f32(big), h, False)) == np.inf
    assert dot_const(f32(25.0), pf_bound(-f32(big), h, True)) == np.inf
