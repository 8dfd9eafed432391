"""CPU model (numpy, FP32 rounding emulated) of the scan kernel's stage-1 prefilter (csrc/kernels_bi_scan.cuh, pf_bound;
DESIGN.md §3): every pair whose exact delta is <= the threshold, and every pair the square-root FP32 filter passes, must pass
the squared-distance test — including pairs placed exactly on its boundary D1 + D2 = a + b."""
import numpy as np

f32 = np.float32
PF_REL = np.ldexp(1.0, -16)
PF_ABS = np.ldexp(1.0, -100)


def fma32(a, b, c):
    """fmaf: the product of two floats is exact in double; one rounding of the sum to float (double rounding is far
    below the bound's slack)"""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(f32)


def pf_bound(ds, h, att):
    a = (f32(ds) + f32(h)).astype(f32)
    t = (a * f32(20.0 if att else 2.0)).astype(f32)
    v = fma32(f32(PF_REL), a, np.abs(a))
    return fma32(t, v, f32(PF_ABS))


def sq32(ax, ay, bx, by):
    dx = (f32(ax) - f32(bx)).astype(f32)
    dy = (f32(ay) - f32(by)).astype(f32)
    return fma32(dy, dy, (dx * dx).astype(f32))


def stage1(xr, yr, dsr, xc, yc, dsc, p, q, thr, E, att):
    """(s(p,q) + cp_p) + s(p+1,q+1) <= C_q in FP32, as the kernel computes it"""
    h = (f32(0.5) * (f32(thr) + f32(E))).astype(f32)
    cp = -pf_bound(dsr[p], h, att)
    s1 = sq32(xr[p], yr[p], xc[q], yc[q])
    s2 = sq32(xr[p + 1], yr[p + 1], xc[q + 1], yc[q + 1])
    lhs = ((s1 + cp).astype(f32) + s2).astype(f32)
    return lhs <= pf_bound(dsc[q], h, att)


def sqrt_filter(x, y, ds, p, q, thr, att):
    """bi_cold_warp's FP32 filter: (D1 - ds_p) + D2 <= thr + ds_q"""
    def d32(i, j):
        s = sq32(x[i], y[i], x[j], y[j])
        if att:
            s = (s * f32(0.1)).astype(f32)
        return np.sqrt(s).astype(f32)
    qv = ((d32(p, q) - f32(ds[p])).astype(f32) + d32(p + 1, q + 1)).astype(f32)
    return qv <= (f32(thr) + f32(ds[q])).astype(f32)


def exact_dist(x, y, i, j, wt):
    r = np.hypot(x[i] - x[j], y[i] - y[j]) if wt != 5 else np.sqrt(((x[i] - x[j]) ** 2 + (y[i] - y[j]) ** 2) / 10.0)
    if wt == 0:
        return np.floor(r + 0.5)
    if wt == 3:
        return np.ceil(r)
    t = np.floor(r + 0.5)
    return np.where(t < r, t + 1, t)


def _window(x, y, wt):
    dmax = float(np.hypot(np.ptp(x), np.ptp(y)))
    dc = max(float(np.max(np.abs(x.astype(f32).astype(np.float64) - x))), float(np.max(np.abs(y.astype(f32).astype(np.float64) - y))))
    eps = dmax * 2.0 ** -20 + 4.0 * dc
    return (0.125 if wt in (3, 5) else 1.0) + 4.0 * eps, 4.0 * eps


def _check_tour(xy, wt, order):
    """position space as the kernel sees it: rows and columns are the tour's points; all non-adjacent pairs"""
    n = len(order)
    x, y = xy[order, 0], xy[order, 1]
    x, y = np.append(x, x[0]), np.append(y, y[0])
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
        pass1 = stage1(x, y, ds, x, y, ds, p, q, thr, E, att)
        assert pass1[delta <= t].all(), t
        assert pass1[sqrt_filter(x, y, ds, p, q, thr, att)].all(), t
        if t == float(delta.min()):
            assert pass1.mean() < 0.5  # and it does filter


def test_stage1_random_instances():
    rng = np.random.default_rng(11)
    for n, scale, wt, integer in [(400, 1e4, 0, True), (400, 1e4, 3, True), (400, 3e3, 5, True), (300, 1e3, 0, False),
                                  (300, 2.5e6, 0, True), (300, 1.0, 0, False)]:
        xy = rng.random((n, 2)) * scale
        if integer:
            xy = np.floor(xy)
        _check_tour(xy, wt, rng.permutation(n))
        # a good tour: greedy nearest neighbour from node 0 (long closing edges, many small deltas)
        left, cur, order = set(range(1, n)), 0, [0]
        while left:
            rest = np.fromiter(left, int)
            cur = int(rest[np.argmin(np.hypot(*(xy[rest] - xy[cur]).T))])
            left.remove(cur)
            order.append(cur)
        _check_tour(xy, wt, np.array(order))


def test_stage1_duplicates_and_ties():
    rng = np.random.default_rng(12)
    xy = np.repeat(np.floor(rng.random((80, 2)) * 50), 4, axis=0)  # duplicate points: s = 0, ds = 0
    _check_tour(xy, 0, rng.permutation(len(xy)))
    _check_tour(np.floor(rng.random((300, 2)) * 20), 3, rng.permutation(300))


def test_stage1_on_its_boundary():
    """d1 + d2 = a + b exactly (Pythagorean distances, integer ds): balanced and very unbalanced splits, b < 0 < a + b"""
    rng = np.random.default_rng(13)
    triples = [(3, 4, 5), (5, 12, 13), (8, 15, 17), (7, 24, 25), (20, 21, 29), (9, 40, 41), (12, 35, 37)]
    for _ in range(4000):
        (a1, b1, c1), (a2, b2, c2) = triples[rng.integers(len(triples))], triples[rng.integers(len(triples))]
        k1, k2 = int(rng.integers(1, 4000)), int(rng.integers(1, 4000))
        d1, d2 = c1 * k1, c2 * k2
        x = np.array([0.0, 1e5, a1 * k1, 1e5 + a2 * k2])  # rows p, p+1; columns q, q+1
        y = np.array([0.0, 0.0, b1 * k1, b2 * k2])
        E = f32(4.0 * (np.hypot(2e5, 2e5) * 2.0 ** -20))
        L = d1 + d2
        dsp = float(rng.integers(0, L + 1))
        dsq = float(rng.integers(-L // 4, L - dsp + 1))  # then thr = L - dsp - dsq - E puts a + b exactly at d1 + d2
        thr = f32(L - dsp - dsq - float(E))
        xr, yr, xc, yc = x[[0, 1]], y[[0, 1]], x[[2, 3]], y[[2, 3]]
        assert stage1(xr, yr, np.array([dsp, 0.0]), xc, yc, np.array([dsq, 0.0]), 0, 0, thr, E, False), (d1, d2, dsp, dsq)


@np.errstate(over="ignore")
def test_stage1_padding_never_passes():
    big = f32(1e30)
    h = f32(10.0)
    assert np.isinf(pf_bound(-big, h, False)) and pf_bound(-big, h, False) < 0  # padding column: C = -inf
    cp = -pf_bound(-big, h, True)                                                 # padding row: cp = +inf
    lhs = (f32(5.0) + cp).astype(f32) + f32(7.0)
    assert np.isinf(lhs) and not (lhs <= pf_bound(f32(1e6), h, False))
