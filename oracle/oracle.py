"""ctypes bindings for the two CPU checkers under oracle/ — TEST INFRASTRUCTURE ONLY.

* ``Oracle``  — our C restatement (oracle/tsp_oracle.c -> oracle/_build/libtsporacle.so).
* ``RefLib``  — the UNMODIFIED reference compiled from /root/reference/src with a stub cplex.h
  (oracle/Makefile -> oracle/_ref/libtspref.so), driven through the reference's own symbols
  ``calc_dist`` (src/distutil.c:73), ``greedy`` (src/heuristics.c:18), ``alg_2opt``
  (src/heuristics.c:438) and ``alg_2opt_tabu`` (src/tabusearch.c:107).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / ``--impl reference`` leg may import
this module; the product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(_HERE, "_build", "libtsporacle.so")
REF_SO = os.path.join(_HERE, "_ref", "libtspref.so")
#: the same reference objects linked against the product's drop-in symbols (oracle/Makefile, INTEGRATION.md §2)
REF_GPU_SO = os.path.join(_HERE, "_ref", "libtspref_gpu.so")
#: the reference's drivers restated on the drop-in header, linked against libtspb200_dropin.so (oracle/dropin_callers.c)
CALLERS_SO = os.path.join(_HERE, "_build", "libdropin_callers.so")

EUC_2D, MAX_2D, MAN_2D, CEIL_2D, GEO, ATT = 0, 1, 2, 3, 4, 5

_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")


class OrcMove(C.Structure):
    _fields_ = [("i", C.c_int32), ("j", C.c_int32), ("delta", C.c_int64)]


class OrcStats(C.Structure):
    _fields_ = [("evals", C.c_int64), ("moves", C.c_int64), ("passes", C.c_int64),
                ("logged", C.c_int64), ("status", C.c_int32)]


def build(force: bool = False) -> None:
    """Build the checkers (make -C oracle). The reference lib is rebuilt only if /root/reference exists."""
    if force or not os.path.exists(ORACLE_SO) or (os.path.isdir("/root/reference/src") and not os.path.exists(REF_SO)):
        subprocess.run(["make", "-C", _HERE], check=True, stdout=subprocess.DEVNULL)


def _as_xy(xy) -> np.ndarray:
    a = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
    return a


def _log_to_array(log, k: int) -> np.ndarray:
    out = np.zeros((k, 3), dtype=np.int64)
    for t in range(k):
        out[t] = (log[t].i, log[t].j, log[t].delta)
    return out


class Oracle:
    """The C restatement."""

    def __init__(self):
        build()
        L = C.CDLL(ORACLE_SO)
        L.orc_dist.restype = C.c_double
        L.orc_dist.argtypes = [_f64p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_dist_matrix.argtypes = [_f64p, C.c_int, C.c_int, _i32p]
        L.orc_dist_row.argtypes = [_f64p, C.c_int, C.c_int, C.c_int, _i32p]
        L.orc_nn_tour.restype = C.c_double
        L.orc_nn_tour.argtypes = [_f64p, C.c_int, C.c_int, C.c_int, _i32p]
        L.orc_order_cost.restype = C.c_double
        L.orc_order_cost.argtypes = [_f64p, C.c_int, C.c_int, _i32p]
        L.orc_succ_cost.restype = C.c_double
        L.orc_succ_cost.argtypes = [_f64p, C.c_int, C.c_int, _i32p]
        L.orc_reverse_path.argtypes = [C.c_int, _i32p, C.c_int, C.c_int, _i32p]
        L.orc_two_opt_fi.argtypes = [_f64p, C.c_int, C.c_int, _i32p, C.POINTER(C.c_double), C.c_int64,
                                     C.c_void_p, C.c_int64, C.POINTER(OrcStats)]
        L.orc_two_opt_bi.argtypes = [_f64p, C.c_int, C.c_int, _i32p, C.POINTER(C.c_double), C.c_void_p,
                                     C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_int64,
                                     C.POINTER(OrcStats)]
        L.orc_bi_scan_rows_mt.restype = C.c_int64
        L.orc_bi_scan_rows_mt.argtypes = [_f64p, C.c_int, C.c_int, _i32p, C.c_int, C.c_int, C.c_int,
                                          C.POINTER(C.c_double), C.POINTER(C.c_int64),
                                          C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        self.L = L

    def dist(self, xy, wt, i, j, integer=1) -> float:
        return self.L.orc_dist(_as_xy(xy), wt, integer, i, j)

    def dist_matrix(self, xy, wt) -> np.ndarray:
        xy = _as_xy(xy)
        n = len(xy)
        out = np.empty((n, n), dtype=np.int32)
        self.L.orc_dist_matrix(xy, n, wt, out)
        return out

    def nn_tour(self, xy, wt, start=0):
        xy = _as_xy(xy)
        n = len(xy)
        succ = np.empty(n, dtype=np.int32)
        cost = self.L.orc_nn_tour(xy, n, wt, start, succ)
        return succ, cost

    def greedy_iter(self, xy, wt):
        """HEU_Greedy_iter -> (best_start, succ, cost)."""
        xy = _as_xy(xy)
        n = len(xy)
        succ = np.empty(n, dtype=np.int32)
        best = C.c_int32(0)
        self.L.orc_greedy_iter.restype = C.c_double
        self.L.orc_greedy_iter.argtypes = [_f64p, C.c_int, C.c_int, _i32p, C.POINTER(C.c_int32)]
        cost = self.L.orc_greedy_iter(xy, n, wt, succ, C.byref(best))
        return best.value, succ, cost

    def extra_mileage(self, xy, wt):
        """HEU_extramileage -> (succ, cost)."""
        xy = _as_xy(xy)
        n = len(xy)
        succ = np.empty(n, dtype=np.int32)
        self.L.orc_extra_mileage.restype = C.c_double
        self.L.orc_extra_mileage.argtypes = [_f64p, C.c_int, C.c_int, _i32p]
        cost = self.L.orc_extra_mileage(xy, n, wt, succ)
        return succ, cost

    def succ_cost(self, xy, wt, succ) -> float:
        xy = _as_xy(xy)
        return self.L.orc_succ_cost(xy, len(xy), wt, np.ascontiguousarray(succ, dtype=np.int32))

    def order_cost(self, xy, wt, order) -> float:
        xy = _as_xy(xy)
        return self.L.orc_order_cost(xy, len(xy), wt, np.ascontiguousarray(order, dtype=np.int32))

    def two_opt_fi(self, xy, wt, succ, obj, max_moves=-1, log_cap=0):
        xy = _as_xy(xy)
        succ = np.array(succ, dtype=np.int32, copy=True)
        o = C.c_double(obj)
        st = OrcStats()
        log = (OrcMove * max(1, log_cap))()
        self.L.orc_two_opt_fi(xy, len(xy), wt, succ, C.byref(o), max_moves,
                              C.cast(log, C.c_void_p) if log_cap else None, log_cap, C.byref(st))
        return succ, o.value, st, _log_to_array(log, st.logged)

    def two_opt_bi(self, xy, wt, succ, max_passes=-1, log_cap=0, skip_edge=None, iter_=1, tenure=1,
                   want_prev=False):
        xy = _as_xy(xy)
        n = len(xy)
        succ = np.array(succ, dtype=np.int32, copy=True)
        o = C.c_double(0.0)
        st = OrcStats()
        log = (OrcMove * max(1, log_cap))()
        prev = np.empty(n, dtype=np.int32) if want_prev else None
        self.L.orc_two_opt_bi(xy, n, wt, succ, C.byref(o),
                              skip_edge.ctypes.data if skip_edge is not None else None,
                              prev.ctypes.data if prev is not None else None, iter_, tenure, max_passes,
                              C.cast(log, C.c_void_p) if log_cap else None, log_cap, C.byref(st))
        if want_prev:
            return succ, o.value, st, _log_to_array(log, st.logged), prev
        return succ, o.value, st, _log_to_array(log, st.logged)

    def vns_kick(self, xy, wt, succ, idx1, idx2, idx3):
        """reference kick() (src/vns.c:11-100) with the three drawn tour indices -> (succ, cost)."""
        xy = _as_xy(xy)
        succ = np.array(succ, dtype=np.int32, copy=True)
        self.L.orc_vns_kick.restype = C.c_double
        self.L.orc_vns_kick.argtypes = [_f64p, C.c_int, C.c_int, _i32p, C.c_int, C.c_int, C.c_int]
        cost = self.L.orc_vns_kick(xy, len(xy), wt, succ, int(idx1), int(idx2), int(idx3))
        return succ, cost

    def tabu_kick(self, succ, skip, pairs, iter_, tenure):
        """the random kick of tabu() (src/tabusearch.c:262-309) -> (accepted index, succ, skip)."""
        succ = np.array(succ, dtype=np.int32, copy=True)
        skip = np.array(skip, dtype=np.int32, copy=True)
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        self.L.orc_tabu_kick.restype = C.c_int
        self.L.orc_tabu_kick.argtypes = [C.c_int, _i32p, _i32p, _i32p, C.c_int, C.c_int, C.c_int]
        acc = self.L.orc_tabu_kick(len(succ), succ, skip, pairs, len(pairs), int(iter_), int(tenure))
        return acc, succ, skip

    def bi_scan_rows_mt(self, xy, wt, succ, row_begin, row_end, threads):
        xy = _as_xy(xy)
        sec = C.c_double(0)
        bd = C.c_int64(0)
        bi = C.c_int32(0)
        bj = C.c_int32(0)
        ev = self.L.orc_bi_scan_rows_mt(xy, len(xy), wt, np.ascontiguousarray(succ, dtype=np.int32), row_begin,
                                        row_end, threads, C.byref(sec), C.byref(bd), C.byref(bi), C.byref(bj))
        return ev, sec.value, (bd.value, bi.value, bj.value)

    def bi_pairs_le(self, xy, wt, succ, H, threads=None) -> np.ndarray:
        """Every legal pair of one best-improvement scan of `succ` whose exact delta is <= H: an (m, 3) int64 array of
        (i, j, delta), i < j node indices, in (i, j) order."""
        L = self.L
        L.orc_bi_pairs_le.restype = C.c_int64
        L.orc_bi_pairs_le.argtypes = [_f64p, C.c_int, C.c_int, _i32p, C.c_int64, C.c_int, C.POINTER(C.POINTER(OrcMove))]
        L.orc_free.argtypes = [C.c_void_p]
        xy = _as_xy(xy)
        out = C.POINTER(OrcMove)()
        m = L.orc_bi_pairs_le(xy, len(xy), wt, np.ascontiguousarray(succ, dtype=np.int32), int(H),
                              threads or os.cpu_count() or 1, C.byref(out))
        if m < 0:
            raise MemoryError("orc_bi_pairs_le: out of memory")
        try:
            rec = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_int32)), shape=(4 * m,)) if m else np.zeros(0, np.int32)
            rec = rec.reshape(m, 4)
            res = np.empty((m, 3), dtype=np.int64)
            res[:, 0] = rec[:, 0]
            res[:, 1] = rec[:, 1]
            res[:, 2] = rec[:, 2:4].copy().view(np.int64)[:, 0]
        finally:
            L.orc_free(out)
        return res


class _InstanceLib:
    """A library that keeps reference `instance`s through the refshim_* calls and exports the reference's driver symbols."""

    def _bind_instance_calls(self, L):
        L.refshim_new.restype = C.c_void_p
        L.refshim_new.argtypes = [C.c_int, _f64p, C.c_int]
        L.refshim_free.argtypes = [C.c_void_p]
        L.refshim_num_nodes.argtypes = [C.c_void_p]
        L.refshim_obj.restype = C.c_double
        L.refshim_obj.argtypes = [C.c_void_p]
        L.refshim_get_succ.argtypes = [C.c_void_p, _i32p]
        L.refshim_set_succ.argtypes = [C.c_void_p, _i32p]
        L.alg_2opt_tabu.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        self.L = L

    def run_method(self, name: str, xy, wt, time_limit: int = -1):
        """Runs one of the reference's own heuristic drivers (e.g. HEU_2opt_greedy, src/heuristics.c:572) on a fresh
        instance, as solve_problem_HEUC (src/solver.c:114-151) would; returns (status, succ, obj_best)."""
        h = self.new(xy, wt)
        # -1 = unlimited for every driver (HEU_Greedy_iter treats 0 as "0 seconds", src/heuristics.c:181)
        self.L.refshim_set_time_limit.argtypes = [C.c_void_p, C.c_int]
        self.L.refshim_set_time_limit(h, time_limit)
        fn = getattr(self.L, name)
        fn.argtypes = [C.c_void_p]
        fn.restype = C.c_int
        status = fn(h)
        out = status, self.get_succ(h), self.L.refshim_obj(h)
        self.free(h)
        return out

    def new(self, xy, wt):
        xy = _as_xy(xy)
        return self.L.refshim_new(len(xy), xy, wt)

    def free(self, h):
        self.L.refshim_free(h)

    def get_succ(self, h) -> np.ndarray:
        succ = np.empty(self.L.refshim_num_nodes(h), dtype=np.int32)
        self.L.refshim_get_succ(h, succ)
        return succ

    def two_opt_bi(self, xy, wt, succ, skip_edge=None, iter_=1, tenure=1, want_prev=False):
        """alg_2opt_tabu(inst, skip_edge, stored_prev, iter, tenure); returns (succ, obj_best[, prev])."""
        h = self.new(xy, wt)
        n = self.L.refshim_num_nodes(h)
        self.L.refshim_set_succ(h, np.ascontiguousarray(succ, dtype=np.int32))
        prev = np.empty(n, dtype=np.int32) if want_prev else None
        self.L.alg_2opt_tabu(h, skip_edge.ctypes.data if skip_edge is not None else None,
                             prev.ctypes.data if prev is not None else None, iter_, tenure)
        out = (self.get_succ(h), self.L.refshim_obj(h)) + ((prev,) if want_prev else ())
        self.free(h)
        return out


class DropinCallers(_InstanceLib):
    """oracle/dropin_callers.c -> oracle/_build/libdropin_callers.so: the reference drivers HEU_greedy / HEU_2opt_greedy /
    HEU_2opt_greedy_iter / HEU_2opt_extramileage restated on top of libtspb200_dropin.so (needs a GPU at call time).
    Raises FileNotFoundError when it is not built."""

    def __init__(self):
        build()
        if not os.path.exists(CALLERS_SO):  # an oracle built before the product library has no callers library yet
            subprocess.run(["make", "-C", _HERE, "callers"], check=True, stdout=subprocess.DEVNULL)
        if not os.path.exists(CALLERS_SO):
            raise FileNotFoundError(CALLERS_SO)
        self._bind_instance_calls(C.CDLL(CALLERS_SO))


class RefLib(_InstanceLib):
    """The unmodified reference, compiled.  Raises FileNotFoundError when oracle/_ref is absent."""

    LAYOUT_KEYS = ["sizeof_instance", "off_time_limit", "off_integer_cost", "off_perf_prof", "off_nodes",
                   "off_num_nodes", "off_weight_type", "off_num_columns", "off_obj_best", "off_edges",
                   "sizeof_point", "sizeof_edge", "off_verbose", "off_seed"]

    def __init__(self, gpu_link: bool = False):
        """gpu_link=True loads libtspref_gpu.so: the reference's callers run unmodified, but calc_dist / alg_2opt /
        alg_2opt_tabu / reverse_path resolve to the product's CUDA-backed definitions (needs a GPU at call time)."""
        build()
        so = REF_GPU_SO if gpu_link else REF_SO
        if not os.path.exists(so):
            raise FileNotFoundError(so)
        L = C.CDLL(so)
        self._bind_instance_calls(L)
        L.refshim_parse.restype = C.c_void_p
        L.refshim_parse.argtypes = [C.c_char_p]
        L.refshim_weight_type.argtypes = [C.c_void_p]
        L.refshim_set_obj.argtypes = [C.c_void_p, C.c_double]
        L.refshim_get_xy.argtypes = [C.c_void_p, _f64p]
        L.refshim_dist_matrix.argtypes = [C.c_void_p, _i32p]
        L.refshim_layout.argtypes = [C.POINTER(C.c_int64), C.c_int]
        L.refshim_bi_scan_rows_mt.restype = C.c_int64
        L.refshim_bi_scan_rows_mt.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double),
                                              C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        # the reference's own entry points
        L.calc_dist.restype = C.c_double
        L.calc_dist.argtypes = [C.c_int, C.c_int, C.c_void_p]
        L.greedy.argtypes = [C.c_void_p, C.c_int]
        L.alg_2opt.argtypes = [C.c_void_p]
        L.reverse_path.argtypes = [C.c_void_p, C.c_int, C.c_int, _i32p]

    def layout(self) -> dict:
        buf = (C.c_int64 * 32)()
        k = self.L.refshim_layout(buf, 32)
        return {name: int(buf[t]) for t, name in zip(range(k), self.LAYOUT_KEYS)}

    def parse(self, path: str):
        """Reference TSPLIB parser -> (xy, weight_type). weight_type -1 (unset) is returned as is."""
        h = self.L.refshim_parse(path.encode())
        n = self.L.refshim_num_nodes(h)
        xy = np.empty((n, 2), dtype=np.float64)
        self.L.refshim_get_xy(h, xy)
        wt = self.L.refshim_weight_type(h)
        self.L.refshim_free(h)
        return xy, wt

    def dist_matrix(self, xy, wt) -> np.ndarray:
        h = self.new(xy, wt)
        n = len(_as_xy(xy))
        out = np.empty((n, n), dtype=np.int32)
        self.L.refshim_dist_matrix(h, out)
        self.free(h)
        return out

    def nn_tour(self, xy, wt, start=0):
        h = self.new(xy, wt)
        self.L.greedy(h, start)
        succ, cost = self.get_succ(h), self.L.refshim_obj(h)
        self.free(h)
        return succ, cost

    def two_opt_fi(self, xy, wt, succ, obj):
        """alg_2opt on a caller-supplied tour; returns (succ, obj_best)."""
        h = self.new(xy, wt)
        self.L.refshim_set_succ(h, np.ascontiguousarray(succ, dtype=np.int32))
        self.L.refshim_set_obj(h, obj)
        self.L.alg_2opt(h)
        out = self.get_succ(h), self.L.refshim_obj(h)
        self.free(h)
        return out

    def vns_kick_stock(self, xy, wt, succ, seed):
        """The reference's own kick() (src/vns.c:11) after srandom(seed): it draws its three indices from glibc random()."""
        libc = C.CDLL("libc.so.6")
        h = self.new(xy, wt)
        self.L.refshim_set_succ(h, np.ascontiguousarray(succ, dtype=np.int32))
        libc.srandom(C.c_uint(seed))
        self.L.kick.argtypes = [C.c_void_p]
        self.L.kick(h)
        out = self.get_succ(h), self.L.refshim_obj(h)
        self.free(h)
        return out

    def bi_scan_rows_mt(self, xy, wt, succ, row_begin, row_end, threads):
        h = self.new(xy, wt)
        self.L.refshim_set_succ(h, np.ascontiguousarray(succ, dtype=np.int32))
        sec = C.c_double(0)
        bd = C.c_int64(0)
        bi = C.c_int32(0)
        bj = C.c_int32(0)
        ev = self.L.refshim_bi_scan_rows_mt(h, row_begin, row_end, threads, C.byref(sec), C.byref(bd),
                                            C.byref(bi), C.byref(bj))
        self.free(h)
        return ev, sec.value, (bd.value, bi.value, bj.value)


def have_ref() -> bool:
    return os.path.exists(REF_SO) or os.path.isdir("/root/reference/src")
