"""The FP32 filters of the best-improvement scan, pair by pair, against an FP64 enumeration (DESIGN.md §3).

FP32 is only a filter: every pair whose exact delta is at or below the threshold must reach the FP64 judge.  The probe build
(TSPB_FILTER_PROBE=1, csrc/tsp_state.cuh) pins the threshold of one pass at H + W — nothing lowers it, so which pairs pass
depends on (tour, H, kernel shape) alone — and its cold paths record every pair of each R x 4 block they are handed whose
exact delta is <= H, with the FP32 value qv = (D1 - ds_p) + D2 the filter compared and its verdict.  For every case:

1. no miss: the records are exactly oracle.bi_pairs_le(H), each pair once, each with passed = 1.  A missing pair was
   rejected by the hot loop, the prefilter's stage 1 or stage 2, or tile pruning; passed = 0 by the cold path's re-test;
2. the pin held: every record's threshold is float32(H) + W, bit for bit;
3. error model: |qv - Q64| <= 1.75 eps_fp32, Q64 = the same quantity in FP64 from the FP32 coordinates the device reads,
   eps_fp32 = dmax 2^-20 (the coordinate-rounding term of eps does not enter: Q64 uses the rounded coordinates);
4. determinism: a second probe pass records the same set.

Kernels: the square-root kernel and the prefilter kernel at every tile shape of tests/test_gpu_prefilter.py, pruned
passes, the one-block position-space kernel of two_opt_batch, and the headline kernel at n = 100 000."""
import os
import subprocess
import time

import numpy as np
import pytest

from conftest import GOLD_DIR, ROOT
from test_oracle_pairs import _np_dist
from tsp_optimization_b200 import engine as eng
from tsp_optimization_b200.instances import order_to_succ, succ_to_order_fast, uniform_instance

pytestmark = pytest.mark.gpu
BI = eng.BI
EUC_2D, CEIL_2D, ATT = 0, 3, 5
CSRC = os.path.join(ROOT, "tsp_optimization_b200", "csrc")
PROBE_LIB = os.path.join(ROOT, "tsp_optimization_b200", "lib", "probe", "libtspb200.so")
#: largest |qv - Q64| / (dmax 2^-23) seen, per metric (printed at the end of the module)
WORST = {}


@pytest.fixture(scope="module")
def probe():
    """the probe build of the engine (make's dependency tracking: rebuilt only when a source changed)"""
    t0 = time.time()
    r = subprocess.run(["make", "-C", CSRC, f"-j{os.cpu_count() or 4}", "OUT=../lib/probe", "EXTRA=-DTSPB_FILTER_PROBE=1",
                        "../lib/probe/libtspb200.so"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    print(f"\nprobe build: {time.time() - t0:.1f} s")
    e = eng.Engine(0, lib_path=PROBE_LIB)
    yield e
    e.close()
    for wt, v in sorted(WORST.items()):
        print(f"max |qv - Q64| / (dmax 2^-23), metric {wt}: {v:.3f}")


def _set(e, **opts):
    for k, v in opts.items():
        e.set_option(k, v)


def _records(e, cap):
    count = e.info("probe_count")
    assert 0 <= count <= cap, f"probe buffer overflow: {count} records, room for {cap}"
    buf = np.zeros((max(cap, 1), 8), dtype=np.int32)
    e._ck(e.L.tspb200_debug_fetch(e.h, b"probe", buf.ctypes.data, buf.nbytes))
    return buf[:count]


def _probe_pass(e, succ, H, cap, batch):
    """one pass with the threshold pinned at H; the records, sorted by (i, j)"""
    _set(e, probe_cap=cap, probe=H)
    try:
        if batch:
            _, _, st = e.two_opt_batch(BI, np.asarray(succ)[None, :])
        else:
            e.tour_upload(succ)
            st = e.bi_run(1)
    finally:
        e.set_option("probe", 0)
    assert st.moves == 0  # the cold paths return no key: the pass ends with "no move"
    rec = _records(e, cap)
    return rec[np.argsort(rec[:, 0].astype(np.int64) * len(succ) + rec[:, 1], kind="stable")]


class Case:
    """an instance with its oracle enumerations, shared by every kernel that probes it"""

    def __init__(self, oracle, xy, wt, succ):
        self.xy, self.wt, self.succ = np.asarray(xy, np.float64), wt, np.asarray(succ, np.int32)
        n = len(xy)
        self.pos = np.empty(n, np.int64)
        self.pos[succ_to_order_fast(self.succ)] = np.arange(n)
        lo, hi = self.xy.min(0), self.xy.max(0)
        self.dmax = float(np.hypot(*(hi - lo)))
        full = oracle.bi_pairs_le(self.xy, wt, self.succ, -1)
        self.m = int(full[:, 2].min()) if len(full) else 0
        self.full = full
        self.x32 = self.xy.astype(np.float32).astype(np.float64)

    def thresholds(self):
        if self.m >= 0:
            return []
        mid = int(np.quantile(self.full[:, 2], 0.25, method="lower"))  # a large set between the two ends
        return sorted({self.m, min(-1, max(self.m, mid)), -1})

    def want(self, H):
        return self.full[self.full[:, 2] <= H]

    def check(self, e, H, batch=False):
        want = self.want(H)
        cap = len(want) + 64
        rec = _probe_pass(e, self.succ, H, cap, batch)
        got = rec[:, :3].astype(np.int64)
        miss = len(want) - len(got)
        assert np.array_equal(got, want), (f"H={H}: {len(got)} records, {len(want)} pairs <= H in FP64 "
                                           f"({miss} fewer), first differences: {_diff(got, want)}")
        assert (rec[:, 5] == 1).all(), f"H={H}: the cold path's FP32 re-test rejected {(rec[:, 5] != 1).sum()} pairs"
        W = np.array([e.info("window_bits")], np.uint32).view(np.float32)[0]
        thr = rec[:, 4].view(np.float32)
        assert (thr == np.float32(np.float32(H) + W)).all(), f"H={H}: the threshold moved"
        if len(rec):
            self._error_model(rec)
        again = _probe_pass(e, self.succ, H, cap, batch)
        assert np.array_equal(again, rec), f"H={H}: a second probe pass recorded a different set"
        return len(rec)

    def _error_model(self, rec):
        i, j = rec[:, 0].astype(np.int64), rec[:, 1].astype(np.int64)
        p = np.where(self.pos[i] < self.pos[j], i, j)  # the row: the pair's node that comes first in the tour
        q = np.where(p == i, j, i)
        ds_p = _np_dist(self.xy, p, self.succ[p], self.wt)

        def d64(a, b):
            s = (self.x32[a, 0] - self.x32[b, 0]) ** 2 + (self.x32[a, 1] - self.x32[b, 1]) ** 2
            return np.sqrt(s / 10.0 if self.wt == ATT else s)

        q64 = d64(p, q) - ds_p + d64(self.succ[p], self.succ[q])
        err = np.abs(rec[:, 3].view(np.float32).astype(np.float64) - q64)
        worst = float(err.max()) / (self.dmax * 2.0 ** -23)
        WORST[self.wt] = max(WORST.get(self.wt, 0.0), worst)
        assert err.max() <= 1.75 * self.dmax * 2.0 ** -20, f"|qv - Q64| = {err.max()} = {worst:.2f} dmax 2^-23"


def _diff(got, want):
    g, w = {tuple(r) for r in got.tolist()}, {tuple(r) for r in want.tolist()}
    return {"missing": sorted(w - g)[:5], "extra": sorted(g - w)[:5], "duplicates": len(got) - len(g)}


def _tours(oracle, xy, wt, seed):
    """an NN tour, a random permutation and the permutation after three oracle best-improvement passes"""
    nn, _ = oracle.nn_tour(xy, wt, 0)
    rnd = order_to_succ(np.random.default_rng(seed).permutation(len(xy)).astype(np.int32))
    moved, _, _, _ = oracle.two_opt_bi(xy, wt, rnd, max_passes=3)
    return {"nn": nn, "random": rnd, "random+3": moved}


# ---- kernels and shapes ------------------------------------------------------------------------------------------------
SHAPES = [(64, 8, 256, 1), (64, 8, 88, 0), (64, 4, 64, 1), (64, 2, 32, 0), (128, 8, 128, 0), (128, 16, 64, 0), (256, 4, 36, 0),
          (256, 16, 64, 0)]


@pytest.fixture(scope="module")
def shape_cases(oracle):
    xy = uniform_instance(1700)
    return {nm: Case(oracle, xy, EUC_2D, s) for nm, s in _tours(oracle, xy, EUC_2D, 5).items()}


@pytest.mark.parametrize("pf", [0, 1])
@pytest.mark.parametrize("T,R,TJ,shuffle", SHAPES)
def test_probe_tile_shapes(probe, oracle, shape_cases, T, R, TJ, shuffle, pf):
    """the square-root kernel (pf = 0) and the prefilter kernel (pf = 1) at every tile shape"""
    probe.set_instance(shape_cases["nn"].xy, EUC_2D)
    _set(probe, block_threads=T, rows_per_thread=R, tile_cols=TJ, row_shuffle=shuffle, prune=0, prefilter=pf)
    try:
        for nm, c in shape_cases.items():
            for H in c.thresholds():
                c.check(probe, H)
        assert (probe.info("block_threads"), probe.info("rows_per_thread"), probe.info("tile_cols")) == (T, R, TJ)
    finally:
        _set(probe, block_threads=0, rows_per_thread=0, tile_cols=0, row_shuffle=-1, prune=-1, prefilter=-1)


# ---- where the margins are thin -----------------------------------------------------------------------------------------
def _margin_cases():
    rng = np.random.default_rng(77)
    g = np.stack(np.meshgrid(np.arange(40.0), np.arange(38.0)), -1).reshape(-1, 2)
    return [
        # EUC_2D in a box just under the FP32 path's limit (dmax < 4e6): eps = dmax 2^-20 ~ 3.7
        ("big_box_int", np.floor(rng.random((1600, 2)) * 2.76e6), EUC_2D),
        ("big_box_decimal", rng.random((1500, 2)) * 2.76e6, EUC_2D),       # exact32 = 0: dc > 0
        ("ceil_int", np.floor(rng.random((1500, 2)) * 2.76e6), CEIL_2D),
        ("ceil_lattice", g * 997.0, CEIL_2D),                               # axis-aligned pairs: integer exact distances
        ("att_int", np.floor(rng.random((1500, 2)) * 2.76e6), ATT),
        ("att_lattice", g * 3163.0, ATT),
        ("ties_lattice", np.floor(rng.random((1600, 2)) * 30.0), EUC_2D),  # many tied deltas
        ("duplicates", np.repeat(np.floor(rng.random((400, 2)) * 4.0e5), 4, axis=0), EUC_2D),
        ("offset", 2.0 ** 23 - 1e4 + np.floor(rng.random((1500, 2)) * 1e4), EUC_2D),
        ("untranslatable", np.concatenate([[[np.float32(1e-3), np.float32(2e-3)]],
                                           (rng.random((1499, 2)) * 1e3).astype(np.float32)]).astype(np.float64), EUC_2D),
    ]


MARGIN = _margin_cases()


@pytest.mark.parametrize("case", range(len(MARGIN)), ids=[c[0] for c in MARGIN])
def test_probe_thin_margins(probe, oracle, case):
    """each instance from three tours, with the square-root kernel, the prefilter kernel and pruned passes"""
    nm, xy, wt = MARGIN[case]
    probe.set_instance(xy, wt)
    assert probe.info("fp32_ok") == 1
    recs = 0
    for tour, succ in _tours(oracle, xy, wt, case).items():
        c = Case(oracle, xy, wt, succ)
        for opts in ({"prune": 0, "prefilter": 0}, {"prune": 0, "prefilter": 1}, {"prune": 1}):
            _set(probe, **opts)
            try:
                for H in c.thresholds():
                    recs += c.check(probe, H)
            finally:
                _set(probe, prune=-1, prefilter=-1)
    assert recs > 0


# ---- the one-block position-space kernel ---------------------------------------------------------------------------------
BATCH = [("uniform", uniform_instance(1500), EUC_2D), MARGIN[0], MARGIN[3], MARGIN[5], MARGIN[7]]


@pytest.mark.parametrize("case", range(len(BATCH)), ids=[c[0] for c in BATCH])
def test_probe_batch_kernel(probe, oracle, case):
    nm, xy, wt = BATCH[case]
    probe.set_instance(xy, wt)
    for tour, succ in _tours(oracle, xy, wt, 40 + case).items():
        c = Case(oracle, xy, wt, succ)
        for H in c.thresholds():
            c.check(probe, H, batch=True)


# ---- the headline shape ---------------------------------------------------------------------------------------------------
def test_probe_headline_uni100000(probe, oracle):
    """the headline kernel at its real size: uni100000 from its committed NN tour, prefilter on, H = m and H = -1"""
    xy = uniform_instance(100000)
    succ = np.load(os.path.join(GOLD_DIR, "nn_uni100000.npz"))["succ"]
    t0 = time.time()
    c = Case(oracle, xy, EUC_2D, succ)
    print(f"\nuni100000: {len(c.full)} improving pairs, m = {c.m}, enumerated in {time.time() - t0:.1f} s")
    probe.set_instance(xy, EUC_2D)
    _set(probe, prune=0, prefilter=1)
    try:
        for H in (c.m, -1):
            c.check(probe, H)
        assert probe.info("row_shuffle") == 1 and probe.info("block_threads") == 64
    finally:
        _set(probe, prune=-1, prefilter=-1)
