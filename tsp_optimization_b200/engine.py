"""ctypes binding of libtspb200.so (include/tspb200.h) — the host-side mirror of the reference's hot-path
interface for Python callers (tests, bench, the torch.distributed bootstrap).

The reference is a C program whose 2-opt / distance entry points take an ``instance*``
(reference include/heuristics.h:82 ``alg_2opt``, src/tabusearch.c:107 ``alg_2opt_tabu``,
include/distutil.h:137 ``calc_dist``); ``Engine`` exposes the same operations on numpy arrays:
``xy`` = the instance's ``point[]`` (n x 2 float64), ``succ`` = ``solution.edges[k].j``.

There is no CPU fallback: if the CUDA library is missing, cannot be loaded, or no GPU is present,
construction raises ``TspB200Error``.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtspb200.so")
DROPIN_PATH = os.path.join(_HERE, "lib", "libtspb200_dropin.so")

EUC_2D, MAX_2D, MAN_2D, CEIL_2D, GEO, ATT = 0, 1, 2, 3, 4, 5
FI, BI = 0, 1
LOCAL_OPTIMUM, TIME_LIMIT_EXCEEDED, STOPPED_BY_CAP = 0, 2, 3

#: every symbol include/tspb200.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "tspb200_create", "tspb200_destroy", "tspb200_last_error", "tspb200_set_option", "tspb200_get_info",
    "tspb200_set_instance", "tspb200_dist_matrix_build", "tspb200_dist_matrix_get", "tspb200_dist_matrix",
    "tspb200_dist_matrix_free", "tspb200_dist_row", "tspb200_tour_upload", "tspb200_tour_download", "tspb200_tour_log",
    "tspb200_bi_run", "tspb200_fi_run", "tspb200_two_opt", "tspb200_two_opt_tabu", "tspb200_two_opt_batch", "tspb200_nn_tour", "tspb200_nn_tour_batch", "tspb200_extra_mileage",
    "tspb200_tour_costs", "tspb200_comm_unique_id", "tspb200_comm_init", "tspb200_comm_destroy",
    "tspb200_debug_tile_plan", "tspb200_debug_tile_plan_ex", "tspb200_debug_fetch",
    "tspb200_tour_cost", "tspb200_tour_save", "tspb200_tour_restore", "tspb200_vns_kick",
    "tspb200_tabu_begin", "tspb200_tabu_run", "tspb200_tabu_kick", "tspb200_tabu_end",
    "tspb200_population_upload", "tspb200_population_download", "tspb200_population_costs", "tspb200_population_two_opt",
    "tspb200_population_vns", "tspb200_population_tabu_begin", "tspb200_population_tabu", "tspb200_population_tabu_fetch",
    "tspb200_population_tabu_end", "tspb200_tabu_search_begin", "tspb200_tabu_search", "tspb200_tabu_search_fetch",
    "tspb200_tabu_search_end", "tspb200_vns_search",
]


class TspB200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"tspb200 error {code}: {msg}")
        self.code = code


class _Stats(C.Structure):
    _fields_ = [("passes", C.c_int64), ("moves", C.c_int64), ("evals", C.c_int64), ("launches", C.c_int64),
                ("obj_delta", C.c_int64), ("gpu_ms", C.c_double), ("cost", C.c_double), ("status", C.c_int32),
                ("path", C.c_int32), ("tiles_scanned", C.c_int64), ("tiles_total", C.c_int64)]


class _Move(C.Structure):
    _fields_ = [("i", C.c_int32), ("j", C.c_int32), ("delta", C.c_int64)]


@dataclass
class Stats:
    passes: int
    moves: int
    evals: int
    launches: int
    obj_delta: int
    gpu_ms: float
    cost: float
    status: int
    path: int
    tiles_scanned: int = 0
    tiles_total: int = 0

    @staticmethod
    def of(s: _Stats) -> "Stats":
        return Stats(s.passes, s.moves, s.evals, s.launches, s.obj_delta, s.gpu_ms, s.cost, s.status, s.path,
                     s.tiles_scanned, s.tiles_total)


_libs = {}


def load_library(path: str | None = None) -> C.CDLL:
    """Load libtspb200.so (built in-tree by ``__graft_entry__.build()`` / ``make -C tsp_optimization_b200/csrc``), or another
    build of the same ABI at `path` (e.g. the filter probe build, tests/test_gpu_filter_probe.py).  One handle per path."""
    if path is None:
        path = os.environ.get("TSPB200_LIB", LIB_PATH)  # development: A/B timing of another build of the same ABI
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        raise TspB200Error(-1, f"{path} is missing: build it with `make -C tsp_optimization_b200/csrc` "
                               "(there is no CPU fallback)")
    L = C.CDLL(path)
    vp, i64, i32p = C.c_void_p, C.c_int64, C.POINTER(C.c_int32)
    L.tspb200_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.tspb200_destroy.argtypes = [vp]
    L.tspb200_destroy.restype = None
    L.tspb200_last_error.argtypes = [vp]
    L.tspb200_last_error.restype = C.c_char_p
    L.tspb200_set_option.argtypes = [vp, C.c_char_p, i64]
    L.tspb200_get_info.argtypes = [vp, C.c_char_p]
    L.tspb200_get_info.restype = i64
    L.tspb200_set_instance.argtypes = [vp, C.c_void_p, C.c_int, C.c_int]
    L.tspb200_dist_matrix_build.argtypes = [vp, C.POINTER(C.c_double)]
    L.tspb200_dist_matrix_get.argtypes = [vp, C.c_void_p]
    L.tspb200_dist_matrix.argtypes = [vp, C.c_void_p]
    L.tspb200_dist_matrix_free.argtypes = [vp]
    L.tspb200_tour_upload.argtypes = [vp, C.c_void_p, i64]
    L.tspb200_tour_download.argtypes = [vp, C.c_void_p, C.POINTER(C.c_double)]
    L.tspb200_tour_log.argtypes = [vp, C.c_void_p, i64, C.POINTER(i64)]
    L.tspb200_bi_run.argtypes = [vp, i64, C.POINTER(_Stats)]
    L.tspb200_fi_run.argtypes = [vp, i64, C.POINTER(_Stats)]
    L.tspb200_two_opt.argtypes = [vp, C.c_int, C.c_void_p, C.POINTER(C.c_double), i64, C.POINTER(_Stats),
                                  C.c_void_p, i64, C.POINTER(i64)]
    L.tspb200_two_opt_tabu.argtypes = [vp, C.c_void_p, C.POINTER(C.c_double), C.c_void_p, C.c_int, C.c_int, i64,
                                       C.POINTER(_Stats), C.c_void_p, i64, C.POINTER(i64)]
    L.tspb200_two_opt_batch.argtypes = [vp, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(_Stats)]
    L.tspb200_nn_tour.argtypes = [vp, C.c_int, C.c_void_p, C.POINTER(C.c_double)]
    L.tspb200_nn_tour_batch.argtypes = [vp, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.tspb200_extra_mileage.argtypes = [vp, C.c_void_p, C.POINTER(C.c_double)]
    L.tspb200_tour_costs.argtypes = [vp, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.tspb200_comm_unique_id.argtypes = [C.c_void_p]
    L.tspb200_comm_init.argtypes = [vp, C.c_void_p, C.c_int, C.c_int]
    L.tspb200_comm_destroy.argtypes = [vp]
    L.tspb200_debug_tile_plan.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, i32p, i32p, i32p,
                                          C.c_void_p, C.c_void_p, C.c_int, i32p]
    if hasattr(L, "tspb200_dist_row"):
        L.tspb200_dist_row.argtypes = [vp, C.c_int, C.c_void_p]
    if hasattr(L, "tspb200_tour_cost"):
        L.tspb200_tour_cost.argtypes = [vp, C.POINTER(C.c_double)]
        L.tspb200_tour_save.argtypes = [vp, C.c_int]
        L.tspb200_tour_restore.argtypes = [vp, C.c_int]
        L.tspb200_vns_kick.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
        L.tspb200_tabu_begin.argtypes = [vp]
        L.tspb200_tabu_run.argtypes = [vp, C.c_int, C.c_int, i64, C.POINTER(_Stats)]
        L.tspb200_tabu_kick.argtypes = [vp, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.tspb200_tabu_end.argtypes = [vp, C.c_void_p]
        L.tspb200_population_upload.argtypes = [vp, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.tspb200_population_download.argtypes = [vp, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.tspb200_population_costs.argtypes = [vp, C.c_void_p, C.c_int, C.c_void_p]
        L.tspb200_population_two_opt.argtypes = [vp, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(_Stats)]
    if hasattr(L, "tspb200_population_vns"):
        L.tspb200_population_vns.argtypes = [vp, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                             C.POINTER(_Stats)]
    if hasattr(L, "tspb200_population_tabu"):
        L.tspb200_population_tabu_begin.argtypes = [vp, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.tspb200_population_tabu.argtypes = [vp, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.POINTER(_Stats)]
        L.tspb200_population_tabu_fetch.argtypes = [vp, C.c_int, C.c_void_p, C.POINTER(C.c_int32)]
        L.tspb200_population_tabu_end.argtypes = [vp]
    if hasattr(L, "tspb200_tabu_search"):
        L.tspb200_tabu_search_begin.argtypes = [vp, C.c_uint32]
        L.tspb200_tabu_search.argtypes = [vp, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_void_p, C.c_void_p,
                                          C.POINTER(_Stats)]
        L.tspb200_tabu_search_fetch.argtypes = [vp, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]
        L.tspb200_tabu_search_end.argtypes = [vp]
    if hasattr(L, "tspb200_vns_search"):
        L.tspb200_vns_search.argtypes = [vp, C.c_void_p, C.c_int, C.POINTER(C.c_double), C.c_void_p, C.POINTER(_Stats)]
    if hasattr(L, "tspb200_debug_fetch"):
        L.tspb200_debug_fetch.argtypes = [vp, C.c_char_p, C.c_void_p, i64]
    _libs[path] = L
    return L


def tile_plan(n: int, rows_per_thread: int = 0, tile_cols: int = 0, threads: int = 0, num_sms: int = 148, world: int = 1):
    """Host-only: the BI tile plan -> (T, R, TJ, row_start[ntr+1], row_j0[ntr]); a tile-row is T*R tour positions.
    0 = let the engine choose. Needs no GPU."""
    L = load_library()
    cap = n // 64 + 8
    rs = np.zeros(cap, dtype=np.int32)
    rj = np.zeros(cap, dtype=np.int32)
    t, r, tj, ntr = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
    rc = L.tspb200_debug_tile_plan(n, threads, rows_per_thread, tile_cols, num_sms, world, C.byref(t), C.byref(r),
                                   C.byref(tj), rs.ctypes.data, rj.ctypes.data, cap, C.byref(ntr))
    if rc:
        raise TspB200Error(rc, "tile plan failed")
    return t.value, r.value, tj.value, rs[:ntr.value + 1].copy(), rj[:ntr.value].copy()


def tile_plan_ex(n: int, rows_per_thread: int = 0, tile_cols: int = 0, threads: int = 0, num_sms: int = 148, world: int = 1,
                 row_shuffle: int = 1):
    """Host-only: the plan tspb200_tour_upload makes, row-shuffle variant included -> (T, R, TJ, tile_rows, row_start, row_j0)."""
    L = load_library()
    cap = n // 32 + 8
    rs = np.zeros(cap, dtype=np.int32)
    rj = np.zeros(cap, dtype=np.int32)
    t, r, tj, ti, ntr = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
    L.tspb200_debug_tile_plan_ex.argtypes = [C.c_int] * 7 + [C.POINTER(C.c_int32)] * 4 + [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int32)]
    rc = L.tspb200_debug_tile_plan_ex(n, threads, rows_per_thread, tile_cols, num_sms, world, row_shuffle, C.byref(t), C.byref(r),
                                      C.byref(tj), C.byref(ti), rs.ctypes.data, rj.ctypes.data, cap, C.byref(ntr))
    if rc:
        raise TspB200Error(rc, "tile plan failed")
    return t.value, r.value, tj.value, ti.value, rs[:ntr.value + 1].copy(), rj[:ntr.value].copy()


def key_pack(delta: int, i: int, j: int) -> int:
    """Python mirror of key_pack() in csrc/tsp_device.cuh (the 62-bit key of the per-pass atomicMin and of the
    multi-GPU exchange; n <= 2^17, |delta| < 2^27)."""
    return ((delta + (1 << 27)) << 34) | (i << 17) | j


def key_unpack(p: int):
    return (p >> 34) - (1 << 27), (p >> 17) & 0x1FFFF, p & 0x1FFFF


def _moves_to_array(buf, k: int) -> np.ndarray:
    out = np.zeros((k, 3), dtype=np.int64)
    for t in range(k):
        out[t] = (buf[t].i, buf[t].j, buf[t].delta)
    return out


class Engine:
    """One engine = one CUDA device + stream; holds one instance and one resident tour."""

    def __init__(self, device: int = 0, lib_path: str | None = None):
        self.L = load_library(lib_path)
        self.h = C.c_void_p()
        rc = self.L.tspb200_create(device, C.byref(self.h))
        if rc:
            msg = self.L.tspb200_last_error(self.h).decode() if self.h else "create failed"
            if self.h:
                self.L.tspb200_destroy(self.h)
                self.h = C.c_void_p()
            raise TspB200Error(rc, msg)
        self.n = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.tspb200_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc: int):
        if rc:
            raise TspB200Error(rc, self.L.tspb200_last_error(self.h).decode())

    # -- options / info
    def set_option(self, key: str, value: int):
        self._ck(self.L.tspb200_set_option(self.h, key.encode(), int(value)))

    def info(self, key: str) -> int:
        return int(self.L.tspb200_get_info(self.h, key.encode()))

    def block_times(self) -> np.ndarray:
        """[grid, 2] %globaltimer stamps {start, end} of every block of the last BI pass run with option timing = 2."""
        out = np.zeros((4096, 2), dtype=np.uint64)
        self._ck(self.L.tspb200_debug_fetch(self.h, b"block_times", out.ctypes.data, out.nbytes))
        return out[:self.info("grid_bi")]

    # -- instance
    def set_instance(self, xy, weight_type: int):
        xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
        self._ck(self.L.tspb200_set_instance(self.h, xy.ctypes.data, len(xy), int(weight_type)))
        self.n = len(xy)

    # -- distance matrix (reference calc_dist for all pairs)
    def dist_matrix(self) -> np.ndarray:
        out = np.empty((self.n, self.n), dtype=np.int32)
        self._ck(self.L.tspb200_dist_matrix(self.h, out.ctypes.data))
        return out

    def dist_matrix_build(self) -> float:
        ms = C.c_double(0)
        self._ck(self.L.tspb200_dist_matrix_build(self.h, C.byref(ms)))
        return ms.value

    def dist_matrix_get(self) -> np.ndarray:
        out = np.empty((self.n, self.n), dtype=np.int32)
        self._ck(self.L.tspb200_dist_matrix_get(self.h, out.ctypes.data))
        return out

    def dist_row(self, i: int) -> np.ndarray:
        out = np.empty(self.n, dtype=np.int32)
        self._ck(self.L.tspb200_dist_row(self.h, int(i), out.ctypes.data))
        return out

    def dist_matrix_free(self):
        self._ck(self.L.tspb200_dist_matrix_free(self.h))

    # -- resident tour
    def tour_upload(self, succ, log_cap: int = 0):
        succ = np.ascontiguousarray(succ, dtype=np.int32)
        assert succ.shape == (self.n,)
        self._ck(self.L.tspb200_tour_upload(self.h, succ.ctypes.data, int(log_cap)))

    def tour_download(self):
        succ = np.empty(self.n, dtype=np.int32)
        cost = C.c_double(0)
        self._ck(self.L.tspb200_tour_download(self.h, succ.ctypes.data, C.byref(cost)))
        return succ, cost.value

    def tour_log(self, cap: int) -> np.ndarray:
        buf = (_Move * max(1, cap))()
        cnt = C.c_int64(0)
        self._ck(self.L.tspb200_tour_log(self.h, C.cast(buf, C.c_void_p), cap, C.byref(cnt)))
        return _moves_to_array(buf, min(cap, cnt.value))

    def bi_run(self, max_passes: int = -1) -> Stats:
        st = _Stats()
        self._ck(self.L.tspb200_bi_run(self.h, int(max_passes), C.byref(st)))
        return Stats.of(st)

    def fi_run(self, max_moves: int = -1) -> Stats:
        st = _Stats()
        self._ck(self.L.tspb200_fi_run(self.h, int(max_moves), C.byref(st)))
        return Stats.of(st)

    # -- host-buffer entry points (mirror alg_2opt / alg_2opt_tabu on an instance)
    def two_opt(self, mode: int, succ, obj: float = 0.0, max_iters: int = -1, log_cap: int = 0):
        """Returns (succ, obj, Stats, log[k,3]) — FI == reference alg_2opt, BI == alg_2opt_tabu(NULL list)."""
        succ = np.array(succ, dtype=np.int32, copy=True)
        o = C.c_double(obj)
        st = _Stats()
        buf = (_Move * max(1, log_cap))()
        cnt = C.c_int64(0)
        self._ck(self.L.tspb200_two_opt(self.h, mode, succ.ctypes.data, C.byref(o), int(max_iters), C.byref(st),
                                        C.cast(buf, C.c_void_p) if log_cap else None, log_cap, C.byref(cnt)))
        return succ, o.value, Stats.of(st), _moves_to_array(buf, min(log_cap, cnt.value))

    def two_opt_tabu(self, succ, skip_edge, iter_: int, tenure: int, max_iters: int = -1, log_cap: int = 0):
        """alg_2opt_tabu(inst, skip_edge, NULL, iter, tenure): returns (succ, obj, Stats, log, skip_edge_after)."""
        succ = np.array(succ, dtype=np.int32, copy=True)
        skip = np.array(skip_edge, dtype=np.int32, copy=True)
        assert skip.shape == (self.n * (self.n - 1) // 2,)
        o = C.c_double(0.0)
        st = _Stats()
        buf = (_Move * max(1, log_cap))()
        cnt = C.c_int64(0)
        self._ck(self.L.tspb200_two_opt_tabu(self.h, succ.ctypes.data, C.byref(o), skip.ctypes.data, int(iter_), int(tenure),
                                             int(max_iters), C.byref(st), C.cast(buf, C.c_void_p) if log_cap else None,
                                             log_cap, C.byref(cnt)))
        return succ, o.value, Stats.of(st), _moves_to_array(buf, min(log_cap, cnt.value)), skip

    def two_opt_batch(self, mode: int, succ_batch, obj=None):
        succ_batch = np.array(succ_batch, dtype=np.int32, copy=True)
        b = succ_batch.shape[0]
        assert succ_batch.shape == (b, self.n)
        o = np.zeros(b, dtype=np.float64) if obj is None else np.array(obj, dtype=np.float64, copy=True)
        st = _Stats()
        self._ck(self.L.tspb200_two_opt_batch(self.h, mode, succ_batch.ctypes.data, o.ctypes.data, b, C.byref(st)))
        return succ_batch, o, Stats.of(st)

    def nn_tour(self, start: int = 0):
        succ = np.empty(self.n, dtype=np.int32)
        cost = C.c_double(0)
        self._ck(self.L.tspb200_nn_tour(self.h, start, succ.ctypes.data, C.byref(cost)))
        return succ, cost.value

    def nn_tour_batch(self, starts, want_tours: bool = True):
        """`len(starts)` independent greedy() runs -> (succ[batch, n] or None, costs[batch])."""
        starts = np.ascontiguousarray(starts, dtype=np.int32)
        b = len(starts)
        succ = np.empty((b, self.n), dtype=np.int32) if want_tours else None
        costs = np.empty(b, dtype=np.float64)
        self._ck(self.L.tspb200_nn_tour_batch(self.h, starts.ctypes.data, b, succ.ctypes.data if want_tours else None,
                                              costs.ctypes.data))
        return succ, costs

    def greedy_iter(self):
        """reference HEU_Greedy_iter (src/heuristics.c:168-205): NN from every node, the first strictly better tour wins."""
        _, costs = self.nn_tour_batch(np.arange(self.n, dtype=np.int32), want_tours=False)
        best = int(np.argmin(costs))  # argmin returns the first minimum == reference's strict '<' over increasing starts
        succ, c = self.nn_tour_batch(np.array([best], dtype=np.int32))
        return best, succ[0], float(c[0])

    def extra_mileage(self):
        """reference HEU_extramileage (src/heuristics.c:208-314) -> (succ, cost)."""
        succ = np.empty(self.n, dtype=np.int32)
        cost = C.c_double(0)
        self._ck(self.L.tspb200_extra_mileage(self.h, succ.ctypes.data, C.byref(cost)))
        return succ, cost.value

    def tour_costs(self, tours, as_order: bool) -> np.ndarray:
        tours = np.ascontiguousarray(tours, dtype=np.int32).reshape(-1, self.n)
        out = np.empty(len(tours), dtype=np.float64)
        self._ck(self.L.tspb200_tour_costs(self.h, tours.ctypes.data, len(tours), 1 if as_order else 0, out.ctypes.data))
        return out

    # -- resident sessions (VNS / tabu / GA callers of the path)
    def tour_cost(self) -> float:
        c = C.c_double(0)
        self._ck(self.L.tspb200_tour_cost(self.h, C.byref(c)))
        return c.value

    def tour_save(self, slot: int = 0):
        self._ck(self.L.tspb200_tour_save(self.h, slot))

    def tour_restore(self, slot: int = 0):
        self._ck(self.L.tspb200_tour_restore(self.h, slot))

    def vns_kick(self, idx1: int, idx2: int, idx3: int) -> float:
        """reference kick() (src/vns.c:11-100) on the resident tour -> recomputed cost."""
        c = C.c_double(0)
        self._ck(self.L.tspb200_vns_kick(self.h, int(idx1), int(idx2), int(idx3), C.byref(c)))
        return c.value

    def tabu_begin(self):
        self._ck(self.L.tspb200_tabu_begin(self.h))

    def tabu_run(self, iter_: int, tenure: int, max_passes: int = -1) -> Stats:
        st = _Stats()
        self._ck(self.L.tspb200_tabu_run(self.h, int(iter_), int(tenure), int(max_passes), C.byref(st)))
        return Stats.of(st)

    def tabu_kick(self, pairs, iter_: int, tenure: int) -> int:
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        acc = C.c_int(-1)
        self._ck(self.L.tspb200_tabu_kick(self.h, pairs.ctypes.data, len(pairs), int(iter_), int(tenure), C.byref(acc)))
        return acc.value

    def tabu_end(self, want_list: bool = False):
        out = np.empty(self.n * (self.n - 1) // 2, dtype=np.int32) if want_list else None
        self._ck(self.L.tspb200_tabu_end(self.h, out.ctypes.data if want_list else None))
        return out

    def population_upload(self, tours, slots=None, as_order: bool = True):
        tours = np.ascontiguousarray(tours, dtype=np.int32).reshape(-1, self.n)
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.int32)
        assert sl is None or len(sl) == len(tours)
        self._ck(self.L.tspb200_population_upload(self.h, tours.ctypes.data, None if sl is None else sl.ctypes.data, len(tours),
                                                  1 if as_order else 0))

    def population_download(self, count=None, slots=None, as_order: bool = True) -> np.ndarray:
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.int32)
        k = len(sl) if sl is not None else int(count)
        out = np.empty((k, self.n), dtype=np.int32)
        self._ck(self.L.tspb200_population_download(self.h, out.ctypes.data, None if sl is None else sl.ctypes.data, k,
                                                    1 if as_order else 0))
        return out

    def population_costs(self, count=None, slots=None) -> np.ndarray:
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.int32)
        k = len(sl) if sl is not None else int(count)
        out = np.empty(k, dtype=np.float64)
        self._ck(self.L.tspb200_population_costs(self.h, None if sl is None else sl.ctypes.data, k, out.ctypes.data))
        return out

    def population_two_opt(self, mode: int, count=None, slots=None, obj=None):
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.int32)
        k = len(sl) if sl is not None else int(count)
        o = np.zeros(k, dtype=np.float64) if obj is None else np.array(obj, dtype=np.float64, copy=True)
        st = _Stats()
        self._ck(self.L.tspb200_population_two_opt(self.h, mode, None if sl is None else sl.ctypes.data, k, o.ctypes.data, C.byref(st)))
        return o, Stats.of(st)

    def population_vns(self, kicks, count=None, slots=None, want_trace: bool = True):
        """Independent VNS chains (reference HEU_VNS, src/vns.c:103-183) on the listed slots (the first `count` when slots is
        None): kicks[b, t] = chain b's three tour indices of iteration t, shape (chains, iters, 3) (instances.vns_kick_indices).
        -> (best[chains] incumbent costs, trace[chains, iters] cost after each iteration's 2-opt or None, Stats)."""
        kicks = np.ascontiguousarray(kicks, dtype=np.int32)
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.int32)
        k = len(sl) if sl is not None else (int(count) if count is not None else kicks.shape[0])
        assert kicks.ndim == 3 and kicks.shape[0] == k and kicks.shape[2] == 3, kicks.shape
        iters = kicks.shape[1]
        best = np.empty(k, dtype=np.float64)
        trace = np.empty((k, iters), dtype=np.float64) if want_trace else None
        st = _Stats()
        self._ck(self.L.tspb200_population_vns(self.h, None if sl is None else sl.ctypes.data, k, kicks.ctypes.data, iters,
                                               best.ctypes.data, trace.ctypes.data if want_trace else None, C.byref(st)))
        return best, trace, Stats.of(st)

    def population_tabu_begin(self, seeds, slots=None, best_slots=None):
        """Independent tabu searches (reference tabu(), src/tabusearch.c:188-320) on the resident population, one per seed:
        chain b works on slot slots[b] (default b) and keeps its best tour in best_slots[b] (default count + b); its random
        stream is srandom(seeds[b])."""
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
        k = len(seeds)
        sl = np.arange(k, dtype=np.int32) if slots is None else np.ascontiguousarray(slots, dtype=np.int32)
        bs = np.arange(k, 2 * k, dtype=np.int32) if best_slots is None else np.ascontiguousarray(best_slots, dtype=np.int32)
        if sl.shape != (k,) or bs.shape != (k,):
            raise TspB200Error(2, f"need {k} slots and {k} best slots, got {sl.shape} and {bs.shape}")
        self._tabu_chains = 0  # a begin, even a failed one, ends the previous chain set
        self._ck(self.L.tspb200_population_tabu_begin(self.h, sl.ctypes.data, bs.ctypes.data, k, seeds.ctypes.data))
        self._tabu_chains = k

    def population_tabu(self, tenures, max_draws: int = 1 << 20):
        """`iters` iterations of every chain in one launch; tenures[b, t] = chain b's tenure of iteration t, shape (chains,
        iters).  -> (best[chains], trace[chains, iters] recomputed cost after each masked 2-opt, draws[chains, iters] pairs
        drawn by each kick, Stats)."""
        tenures = np.ascontiguousarray(tenures, dtype=np.int32)
        k = getattr(self, "_tabu_chains", 0)
        if k == 0:
            # no chain set begun through this binding: no array crosses (the library sizes them by its own chain count)
            self._ck(self.L.tspb200_population_tabu(self.h, None, 0, int(max_draws), None, None, None, None))
            raise TspB200Error(3, "no tabu chain set (population_tabu_begin)")
        if tenures.ndim != 2 or tenures.shape[0] != k:
            raise TspB200Error(2, f"tenures must have shape ({k}, iters), got {tenures.shape}")
        iters = tenures.shape[1]
        best = np.empty(k, dtype=np.float64)
        trace = np.empty((k, iters), dtype=np.float64)
        draws = np.empty((k, iters), dtype=np.int32)
        st = _Stats()
        self._ck(self.L.tspb200_population_tabu(self.h, tenures.ctypes.data, iters, int(max_draws), best.ctypes.data,
                                                trace.ctypes.data, draws.ctypes.data, C.byref(st)))
        return best, trace, draws, Stats.of(st)

    def population_tabu_list(self, chain: int):
        """-> (chain's tabu list, n(n-1)/2 int32 in the reference's x_udir_pos layout, its next iteration number)"""
        out = np.empty(self.n * (self.n - 1) // 2, dtype=np.int32)
        it = C.c_int32(0)
        self._ck(self.L.tspb200_population_tabu_fetch(self.h, int(chain), out.ctypes.data, C.byref(it)))
        return out, it.value

    def population_tabu_end(self):
        self._ck(self.L.tspb200_population_tabu_end(self.h))
        self._tabu_chains = 0

    def tabu_search_begin(self, seed: int):
        """One tabu search (reference tabu(), src/tabusearch.c:188-320) on the resident tour: zeroes its list, next
        iteration 1, random stream srandom(seed), best tour = the resident tour."""
        self._ck(self.L.tspb200_tabu_search_begin(self.h, int(seed) & 0xffffffff))

    def tabu_search(self, tenures, max_draws: int = 1 << 20):
        """len(tenures) iterations on the device (tenures[t] = the tenure of iteration t).  -> (best cost, trace[iters]
        recomputed cost after each masked 2-opt, draws[iters] pairs drawn by each kick, Stats)."""
        tenures = np.ascontiguousarray(tenures, dtype=np.int32).reshape(-1)
        iters = len(tenures)
        best = C.c_double(0.0)
        trace = np.empty(iters, dtype=np.float64)
        draws = np.empty(iters, dtype=np.int32)
        st = _Stats()
        self._ck(self.L.tspb200_tabu_search(self.h, tenures.ctypes.data, iters, int(max_draws), C.byref(best), trace.ctypes.data,
                                            draws.ctypes.data, C.byref(st)))
        return best.value, trace, draws, Stats.of(st)

    def tabu_search_fetch(self):
        """-> (tabu list, n(n-1)/2 int32 in the reference's x_udir_pos layout, next iteration number, best tour's successors)"""
        out = np.empty(self.n * (self.n - 1) // 2, dtype=np.int32)
        it = C.c_int32(0)
        best = np.empty(self.n, dtype=np.int32)
        self._ck(self.L.tspb200_tabu_search_fetch(self.h, out.ctypes.data, C.byref(it), best.ctypes.data))
        return out, it.value, best

    def tabu_search_end(self):
        self._ck(self.L.tspb200_tabu_search_end(self.h))

    def vns_search(self, kicks):
        """One VNS search (reference HEU_VNS, src/vns.c:103-183) on the resident tour: kicks[t] = the three tour indices of
        iteration t, shape (iters, 3) (instances.vns_kick_indices).  The resident tour is left as the incumbent.
        -> (incumbent cost, trace[iters] cost after each iteration's 2-opt, Stats)."""
        kicks = np.ascontiguousarray(kicks, dtype=np.int32).reshape(-1, 3)
        iters = len(kicks)
        best = C.c_double(0.0)
        trace = np.empty(iters, dtype=np.float64)
        st = _Stats()
        self._ck(self.L.tspb200_vns_search(self.h, kicks.ctypes.data, iters, C.byref(best), trace.ctypes.data, C.byref(st)))
        return best.value, trace, Stats.of(st)

    # -- multi-GPU
    @staticmethod
    def comm_unique_id() -> bytes:
        L = load_library()
        buf = C.create_string_buffer(128)
        rc = L.tspb200_comm_unique_id(buf)
        if rc:
            raise TspB200Error(rc, "ncclGetUniqueId failed (is libnccl.so.2 loadable?)")
        return buf.raw

    def comm_init(self, uid: bytes, rank: int, world: int):
        assert len(uid) == 128
        self._ck(self.L.tspb200_comm_init(self.h, uid, rank, world))

    def comm_destroy(self):
        self._ck(self.L.tspb200_comm_destroy(self.h))
