#!/usr/bin/env python
"""bench.py — 2-opt move evaluations per second on the BASELINE.json headline workload.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload (config.workload): synthetic uniform EUC_2D instance uni<n> (n = 100000, SURVEY.md §8(c) generator),
nearest-neighbour start tour built on the GPU, best-improvement 2-opt with on-the-fly distances.
One STEP = one best-improvement pass = all n(n-3)/2 move deltas evaluated + argmin + move applied.
  value   = passes * n(n-3)/2 / device time, tour resident in HBM, EXHAUSTIVE scan (exact tile pruning off), every pass
            preceded by an L2 flush and timed by its own CUDA event pair on the engine's stream
  e2e     = the same through the host-buffer C-ABI calls tspb200_set_instance() + tspb200_two_opt(): the tour uploaded
            from pinned host memory (the coordinates are a constant of the job: compared on the host, re-sent only when
            they change), K passes, tour and cost downloaded, wall clock around the calls
  N > 1   : the pair tiles are dealt round-robin over the ranks (strong scaling, same instance); per pass every rank's
            packed argmin key is stored into every peer's slots over NVLink by the scan kernel itself (CUDA IPC peer
            memory; NCCL only bootstraps the handles and is the fallback); max over ranks of the device time.
Self-checks: the tour after the timed passes, after the e2e call and after the full run is compared (sha256) with the tour
obtained by replaying the committed single-GPU move log tests/golden/uni100000_bi_moves.npz on the host, on every rank.
--impl reference times the reference's own CPU code (oracle/_ref: its calc_dist and x_udir_pos driven over rows of one
best-improvement scan exactly like src/tabusearch.c:126-156, all host threads) on the same instance and start tour, and the
stock single-thread alg_2opt_tabu() on uni2000 next to it.
--dump-outputs DIR writes what the timed passes returned to a caller (tour and cost after the last step, pass counters) as
float64 .npy files, so that two builds can be compared output for output on the same seeded inputs.
Nothing is written into the repository tree; the CPU nearest-neighbour tour of an uncommitted size is cached in the
system's temporary directory.
"""
import argparse
import hashlib
import json
import os
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ from the imports below

METRIC = "2opt_move_evals_per_sec"
UNIT = "evals/s"
FP32_INSTR_PER_EVAL = 18  # SURVEY.md §8(d): per-unit figure of the on-the-fly 2-opt roofline
FIXTURE = os.path.join(ROOT, "tests", "golden", "uni100000_bi_moves.npz")
NCU_KEYED = os.path.join(ROOT, "profiles", "ncu_by_tile_shape.json")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=100000)
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tlo", action="store_true", help="skip the time-to-local-optimum runs (uni100000 on N GPUs, uni10000)")
    ap.add_argument("--no-extras", action="store_true", help="skip ga_batch / matrix roofline / per-pass breakdown")
    ap.add_argument("--rows-per-thread", type=int, default=0)
    ap.add_argument("--tile-cols", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed path's outputs of its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def workload_config(n: int) -> dict:
    """Identical in both arms (the driver compares the two lines' config)."""
    return {"workload": f"uni{n} EUC_2D (SURVEY.md §8c generator), nearest-neighbour start, best-improvement 2-opt passes with "
                        f"on-the-fly distances (BASELINE configs[3])",
            "n": n, "pairs_per_step": n * (n - 3) // 2,
            "l2": "GPU arm: 256 MB written before every timed pass on the engine's stream, outside the per-pass event pairs "
                  "(at N > 1 followed by a peer-slot barrier so that no rank's flush time lands in a peer's timed pass); "
                  "CPU arm: not applicable"}


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.int32).tobytes()).hexdigest()


class ClockSampler:
    """SM clock and throttle reasons read IN-PROCESS through NVML (pynvml) every few milliseconds from a thread that is
    started before the warm-up, so that even a 30 ms timed region holds samples; stop(t0, t1) reports the samples taken
    inside [t0, t1] (perf_counter), falling back to the samples of the whole run under load."""

    def __init__(self, gpu_index: int, period_s: float = 0.002):
        self.idx, self.period, self.samples, self._stop = gpu_index, period_s, [], False
        self.err = None
        self.max_mhz = None
        self.t = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.err = f"NVML unavailable: {e}"
            return self
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def _run(self):
        nv, h = self.nv, self.h
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop:
            try:
                self.samples.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(reasons_fn(h))))
            except Exception as e:  # noqa: BLE001
                self.err = str(e)
                return
            time.sleep(self.period)

    def stop(self, t0: float, t1: float) -> dict:
        self._stop = True
        if self.t:
            self.t.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [self.err or "no samples"], "samples": 0, "source": "nvml"}
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        where = "timed region"
        if len(inside) < 3:  # a region shorter than a few sampling periods: the whole run, upper half of the clock range
            top = max(s[1] for s in self.samples)
            inside = [s for s in self.samples if s[1] >= 0.5 * top]
            where = "warm-up + timed region (timed region shorter than 3 sampling periods)"
        bits = 0
        for s in inside:
            bits |= s[2]
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        return {"sm_mhz": float(np.median([s[1] for s in inside])), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(v for k, v in names.items() if bits & k), "samples": len(inside), "source": f"nvml, {where}"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0}, "fallback"


def pinned(arr: np.ndarray) -> np.ndarray:
    import torch
    t = torch.empty(arr.shape, dtype=getattr(torch, str(arr.dtype)), pin_memory=torch.cuda.is_available())
    out = t.numpy()
    out[...] = arr
    out_holder.append(t)
    return out


out_holder = []


# ---- CPU reference (test infrastructure: the only place bench.py touches oracle/) ---------------------------------------
def _ref_lib():
    from oracle.oracle import Oracle, RefLib, REF_SO
    if os.path.exists(REF_SO):
        return RefLib(), "reference"
    return Oracle(), "port"


def cpu_baseline_sample(xy, succ, seconds_budget: float):
    """Rows of ONE best-improvement scan on the host cores, the loop of reference src/tabusearch.c:126-156 line by line
    (adjacency test, the four x_udir_pos calls, the NULL tabu-list test, four calc_dist calls) with the reference's own
    compiled calc_dist / x_udir_pos when oracle/_ref is present (kind "reference"), else the oracle port."""
    n = len(xy)
    threads = os.cpu_count() or 1
    lib, kind = _ref_lib()
    # calibrate on a few rows, then size the sample for the time budget
    ev, sec, _ = lib.bi_scan_rows_mt(xy, 0, succ, 0, min(n - 1, 16 * threads), threads)
    rate = ev / max(sec, 1e-6)
    want = rate * seconds_budget
    total_pairs = n * (n - 3) // 2
    if want >= total_pairs:
        rows = n - 1
    else:  # rows r with r*n - r^2/2 ~= want
        rows = int(n - np.sqrt(max(0.0, float(n) * n - 2.0 * want)))
        rows = max(16 * threads, min(n - 1, rows))
    ev, sec, _ = lib.bi_scan_rows_mt(xy, 0, succ, 0, rows, threads)
    return {"value": ev / sec, "unit": UNIT, "cores": threads, "kind": kind, "value_per_core": ev / sec / threads,
            "sample": f"rows [0,{rows}) of one best-improvement scan of uni{n} from the NN start = {ev} pair evaluations "
                      f"in {sec:.2f} s; {'reference calc_dist + x_udir_pos (oracle/_ref)' if kind == 'reference' else 'oracle port'}, "
                      f"{threads} threads, rows dealt in blocks of 16"}, rows


def stock_one_core(m: int = 2000):
    """The UNMODIFIED alg_2opt_tabu(inst, NULL, NULL, 1, 1) (reference src/tabusearch.c:107) run to completion on uni<m>
    from the nearest-neighbour start, one thread: the stock single-core figure BASELINE.md §3 asks for.  Known answer at
    m = 2000 (SURVEY.md §8c): cost 339437, 315 moves, 631 052 000 evaluations."""
    from oracle.oracle import REF_SO, RefLib
    from tsp_optimization_b200.instances import uniform_instance
    if not os.path.exists(REF_SO):
        return None
    lib = RefLib()
    xy = uniform_instance(m)
    succ, _ = lib.nn_tour(xy, 0, 0)
    t0 = time.perf_counter()
    s, cost = lib.two_opt_bi(xy, 0, succ)
    sec = time.perf_counter() - t0
    # moves = passes - 1; the reference does not count, so replay the count from the cost trajectory of the port
    from oracle.oracle import Oracle
    _, ocost, ost, _ = Oracle().two_opt_bi(xy, 0, succ)
    ok = bool(cost == ocost)
    return {"workload": f"uni{m} NN start -> alg_2opt_tabu(inst, NULL, NULL, 1, 1) to the local optimum, unmodified reference, 1 thread",
            "seconds": sec, "final_cost": cost, "passes": int(ost.passes), "moves": int(ost.moves), "evals": int(ost.evals),
            "value": ost.evals / sec, "unit": UNIT, "cores": 1, "cost_equals_port": ok}


def run_reference(args, rank):
    """--impl reference: the reference CPU implementation on the same workload (rank 0 only)."""
    if rank != 0:
        return
    from tsp_optimization_b200.instances import uniform_instance
    n = args.n
    xy = uniform_instance(n)
    succ = start_tour_cpu_or_cached(xy, n)
    total = max(1, args.steps + args.warmup)
    per_step = max(0.3, min(8.0, 120.0 / total))
    base, rows = cpu_baseline_sample(xy, succ, per_step)
    lib, _ = _ref_lib()
    threads = os.cpu_count() or 1
    for _ in range(args.warmup):
        lib.bi_scan_rows_mt(xy, 0, succ, 0, rows, threads)
    ev_sum, sec_sum = 0, 0.0
    for _ in range(args.steps):
        ev, sec, _ = lib.bi_scan_rows_mt(xy, 0, succ, 0, rows, threads)
        ev_sum += ev
        sec_sum += sec
    val = ev_sum / sec_sum
    base["value"] = val
    base["value_per_core"] = val / threads
    stock = stock_one_core(2000 if n >= 10000 else 600)
    if stock:
        base["stock_1core"] = stock
        base["harness_per_core_over_stock_1core"] = val / threads / stock["value"]
    line = {"metric": METRIC, "value": val, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sec_sum / max(1, args.steps), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(n), "cpu_baseline": base,
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def start_tour_cpu_or_cached(xy, n):
    """NN start tour without a GPU (reference arm).  greedy() is O(n^2) on the CPU (10^10 calc_dist calls at n = 100 000),
    so the committed fixture tests/golden/nn_uni<n>.npz (generated by tests/golden/make_nn_uni100000.py with the oracle; the
    GPU nearest-neighbour kernel is tested against it) is used when it exists, then a cache from an earlier run."""
    from oracle.oracle import Oracle
    fixture = os.path.join(ROOT, "tests", "golden", f"nn_uni{n}.npz")
    if os.path.exists(fixture):
        return np.load(fixture)["succ"].astype(np.int32)
    cache = nn_cache_path(n)
    if os.path.exists(cache):
        return np.load(cache)
    succ, _ = Oracle().nn_tour(xy, 0, 0)
    try:
        np.save(cache, succ)
    except OSError:
        pass
    return succ


def nn_cache_path(n: int) -> str:
    return os.path.join(tempfile.gettempdir(), f"tspb200_bench_nn_uni{n}.npy")


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """DIR/<name>.npy for every array, as float64 (tour indices < 2^53 stay exact)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


class TourFixture:
    """The committed single-GPU move log of the workload (tests/golden/make_uni100000_moves.py): expected tour after P passes
    = the NN start with the first P moves applied on the host."""

    def __init__(self, n: int, succ0):
        self.ok = n == 100000 and os.path.exists(FIXTURE)
        self.succ0 = succ0
        if self.ok:
            z = np.load(FIXTURE)
            self.moves = z["moves"]
            self.final = {"passes": int(z["final_passes"]), "moves": int(z["final_moves"]), "cost": float(z["final_cost"]),
                          "sha256": str(z["final_sha256"])}
            self.ok = sha(succ0) == str(z["nn_sha256"])

    def check_after_passes(self, succ, passes: int) -> dict:
        out = {"tour_sha256": sha(succ), "passes": int(passes)}
        if not self.ok or passes > len(self.moves):
            out["check"] = "no fixture for this workload / pass count"
            return out
        from tsp_optimization_b200.instances import apply_moves
        exp = apply_moves(self.succ0, self.moves[:passes])
        out["expected_sha256"] = sha(exp)
        out["check"] = "ok" if out["expected_sha256"] == out["tour_sha256"] else "MISMATCH"
        return out

    def check_final(self, succ, passes, moves, cost) -> dict:
        out = {"tour_sha256": sha(succ)}
        if not self.ok:
            out["check"] = "no fixture for this workload"
            return out
        f = self.final
        good = out["tour_sha256"] == f["sha256"] and passes == f["passes"] and moves == f["moves"] and cost == f["cost"]
        out["expected_sha256"] = f["sha256"]
        out["check"] = "ok" if good else "MISMATCH"
        return out


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    # stdout carries exactly one JSON line: keep NCCL's "NCCL version ..." banner (NCCL_DEBUG=VERSION in this image) off it
    # (every level from VERSION up prints it, so the variable is dropped rather than raised to WARN)
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        del os.environ["NCCL_DEBUG"]
    import torch
    import torch.distributed as dist

    from tsp_optimization_b200 import BI, FI, Engine
    from tsp_optimization_b200.dist import attach_engine_comm, init_process_group_from_env, shard_batch
    from tsp_optimization_b200.instances import order_to_succ, reference_random_population, uniform_instance

    if world > 1:
        init_process_group_from_env("nccl")
    torch.cuda.set_device(local)
    sampler = ClockSampler(local).start()
    n = args.n
    xy = uniform_instance(n)
    pairs = n * (n - 3) // 2

    def maxr(x: float) -> float:
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ok(flag: bool) -> bool:
        if world == 1:
            return bool(flag)
        t = torch.tensor([1 if flag else 0], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    eng = Engine(local)
    if args.rows_per_thread:
        eng.set_option("rows_per_thread", args.rows_per_thread)
    if args.tile_cols:
        eng.set_option("tile_cols", args.tile_cols)
    eng.set_instance(xy, 0)
    t0 = time.perf_counter()
    succ0, nn_cost = eng.nn_tour(0)  # identical on every rank (deterministic)
    nn_s = time.perf_counter() - t0
    if rank == 0:
        try:
            np.save(nn_cache_path(n), succ0)
        except OSError:
            pass
    fixture = TourFixture(n, succ0)
    if world > 1:
        attach_engine_comm(eng, rank, world)
    eng.set_option("prune", 0)  # throughput = exhaustive scans: every non-adjacent pair of every pass is evaluated
    eng.tour_upload(succ0)

    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # matrix kernel timing only

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- resident-tour timing: W warm-up passes, then exactly K timed passes in ONE engine call --------------------
    # l2_flush_bytes: the engine writes 256 MB (> 126 MB L2) before every pass and times each pass with its own CUDA
    # event pair on its stream; value = K * pairs / sum of the per-pass intervals (max over ranks).  No host round trip
    # between passes, so multi-GPU ranks stay in step through the device-side exchange only.
    eng.bi_run(args.warmup)
    if not args.no_flush:
        eng.set_option("l2_flush_bytes", 256 << 20)
    barrier()
    t_region0 = time.perf_counter()
    st = eng.bi_run(args.steps)
    barrier()
    t_region1 = time.perf_counter()
    wall_s = t_region1 - t_region0
    eng.set_option("l2_flush_bytes", 0)
    gpu_ms, launches, moves, done_passes = maxr(st.gpu_ms), st.launches, st.moves, st.passes
    value = done_passes * pairs / (gpu_ms * 1e-3)
    # the tile shape / grid `value` was measured with (later legs — pruned runs, other sizes — re-plan the tiles)
    shape_value = {k: eng.info(k) for k in ("block_threads", "rows_per_thread", "tile_cols", "grid_bi", "ntiles", "row_shuffle", "tile_rows")}
    tour_after, cost_after = eng.tour_download()
    chk_value = fixture.check_after_passes(tour_after, args.warmup + done_passes)
    clocks = sampler.stop(t_region0, t_region1)

    # ---- e2e: host buffers through the C-ABI, copies inside the timed region -------------------------------
    h_xy = pinned(xy)
    h_succ = pinned(succ0.astype(np.int32))
    e2e_passes = args.steps
    eng.set_instance(h_xy, 0)           # warm-up of the same call sequence
    eng.two_opt(BI, h_succ, 0.0, max_iters=2)
    barrier()
    w0 = time.perf_counter()
    eng.set_instance(h_xy, 0)
    s_out, obj_out, st_e, _ = eng.two_opt(BI, h_succ, 0.0, max_iters=e2e_passes)
    torch.cuda.synchronize()
    e2e_s = maxr(time.perf_counter() - w0)
    e2e_val = st_e.passes * pairs / e2e_s
    chk_e2e = fixture.check_after_passes(s_out, st_e.passes)
    h2d = 4 * n  # the step's input tour; the coordinates are a constant of the job: set_instance compares them on the host and sends nothing
    d2h = 4 * n + 8

    # ---- e2e, strictest reading: EVERY step is its own public call with its own host<->device copies -----------------
    # K calls of tspb200_two_opt(max_iters = 1): each uploads the step's input tour from pinned host memory (4n bytes),
    # runs one pass, downloads the resulting tour and its cost (4n + 8 bytes), which is the next step's input.  The
    # instance (coordinates) stays resident like any constant of the job.
    step_calls = args.steps
    cur = h_succ.copy()
    eng.two_opt(BI, cur, 0.0, max_iters=1)
    barrier()
    w0 = time.perf_counter()
    done_step = 0
    for _ in range(step_calls):
        cur, _, st_s, _ = eng.two_opt(BI, cur, 0.0, max_iters=1)
        done_step += st_s.passes
    torch.cuda.synchronize()
    step_s = maxr(time.perf_counter() - w0)
    e2e_step = {"value": done_step * pairs / step_s, "unit": UNIT, "h2d_bytes_per_step": 4 * n, "d2h_bytes_per_step": 4 * n + 8,
                "steps": step_calls, "seconds": step_s, "call": "tspb200_two_opt(BI, host succ[], max_iters=1) once per step",
                "tour_check": fixture.check_after_passes(cur, done_step)["check"]}

    # ---- where a pass's time goes (device %globaltimer stamps; a separate short run, not part of `value`) -----------
    breakdown = None
    if not args.no_extras:
        eng.set_option("timing", 1)
        eng.tour_upload(succ0)
        eng.bi_run(4)
        eng.tour_upload(succ0)
        barrier()
        stb = eng.bi_run(60)
        cnt = max(1, eng.info("tm_count"))
        breakdown = {k[3:] + "_us": round(eng.info(k) / cnt / 1e3, 2) for k in
                     ("tm_gap", "tm_scan", "tm_spread", "tm_tail", "tm_xwait", "tm_apply_gap", "tm_apply")}
        breakdown.update({"passes": int(stb.passes), "us_per_pass_events": round(1e3 * stb.gpu_ms / max(1, stb.passes), 2),
                          "legend": "per pass, this rank: gap = previous apply's end -> first scan block; scan = first scan block -> "
                                    "last block's ticket; spread = first block done -> last block done (inside scan); tail = ticket -> "
                                    "move published (includes xwait = polling the peers' keys); apply_gap = published -> first "
                                    "apply block; apply = apply kernel.  L2 not flushed in this run."})
        eng.set_option("timing", 0)

    # ---- time to local optimum (BASELINE metric, second half): the same instance and start tour, run to the end ----
    tlo = None
    if not args.no_tlo:
        tlo = {}
        for key, prune in (("exhaustive", 0), ("pruned", 1)):
            eng.set_option("prune", prune)
            eng.set_instance(h_xy, 0)
            barrier()
            w0 = time.perf_counter()
            s_out, obj_out, st_f, _ = eng.two_opt(BI, h_succ, 0.0)
            torch.cuda.synchronize()
            tlo_s = maxr(time.perf_counter() - w0)
            rec = {"time_to_local_optimum_s": tlo_s, "passes": st_f.passes, "moves": st_f.moves, "gpu_ms": st_f.gpu_ms,
                   "start_cost": nn_cost, "final_cost": obj_out, "evals": st_f.evals, "evals_per_s": st_f.evals / tlo_s,
                   "tour_check": fixture.check_final(s_out, st_f.passes, st_f.moves, obj_out)}
            if prune:
                rec.update({"tiles_scanned": st_f.tiles_scanned, "tiles_total": st_f.tiles_total,
                            "tiles_skipped": st_f.tiles_total - st_f.tiles_scanned,
                            "note": "exact tile pruning: tiles whose lower bound exceeds the best exact delta known are not "
                                    "evaluated; same move log, `evals` counts evaluated pairs only (this rank's share)"})
            rec["all_ranks_ok"] = all_ok(rec["tour_check"]["check"] != "MISMATCH")
            if key == "exhaustive":
                tlo.update({"workload": f"uni{n} NN start -> best-improvement 2-opt local optimum on {world} GPU(s), host buffers in and out"})
                tlo.update(rec)
            else:
                tlo["pruned"] = rec
        eng.set_option("prune", 0)
        # first improvement (reference alg_2opt) on the same instance and start tour: on N GPUs the segments of the pair order
        # are dealt over the ranks, the first improving pair is min-exchanged like the best-improvement keys
        barrier()
        w0 = time.perf_counter()
        s_fi, obj_fi, st_fi, _ = eng.two_opt(FI, h_succ, nn_cost)
        torch.cuda.synchronize()
        fi_s = maxr(time.perf_counter() - w0)
        hv = int(sha(s_fi)[:15], 16)
        if world > 1:
            t = torch.tensor([hv, -hv], dtype=torch.int64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            same = bool(t[0].item() == -t[1].item())
        else:
            same = True
        tlo["uni100000_FI" if n == 100000 else f"uni{n}_FI"] = {
            "time_to_local_optimum_s": fi_s, "sweeps": st_fi.passes, "moves": st_fi.moves, "final_cost": obj_fi,
            "us_per_move": 1e6 * fi_s / max(1, st_fi.moves), "tour_sha256": sha(s_fi), "same_tour_on_all_ranks": same}
        if world == 1 and n != 10000:  # BASELINE configs[2]: uni10000, greedy start + 2-opt to the local optimum, 1 B200
            xy2 = uniform_instance(10000)
            eng.set_instance(xy2, 0)
            s2, c2 = eng.nn_tour(0)
            for prune in (0, 1):
                eng.set_option("prune", prune)
                eng.two_opt(BI, s2, 0.0, max_iters=4)  # warm-up of this tile shape
                for mode, nm in ((BI, "BI"), (FI, "FI")):
                    if mode == FI and prune:
                        continue
                    w0 = time.perf_counter()
                    _, o2, st2, _ = eng.two_opt(mode, s2, c2)
                    d2 = time.perf_counter() - w0
                    tlo[f"uni10000_{nm}" + ("_pruned" if prune else "")] = {
                        "time_to_local_optimum_s": d2, "passes": st2.passes, "moves": st2.moves, "final_cost": o2, "evals": st2.evals,
                        "us_per_pass": 1e3 * st2.gpu_ms / max(1, st2.passes) if mode == BI else None}
            eng.set_option("prune", 0)
            eng.set_instance(h_xy, 0)

    # ---- BASELINE configs[4]: GA population 1024 x uni1000, every tour driven to its 2-opt local optimum -----------------
    ga = None
    if not args.no_extras:
        n_ga, pop = 1000, 1024
        xy_ga = uniform_instance(n_ga)
        orders = reference_random_population(n_ga, pop, 123)  # reference genetic.c:349-364, srandom(123)
        succ_ga = np.stack([order_to_succ(o) for o in orders])
        lo, hi = shard_batch(pop, rank, world)
        eng.set_instance(xy_ga, 0)
        ga = {"workload": f"{pop} x uni{n_ga} tours from random_generation() (glibc random(), seed 123), each to its 2-opt local optimum; "
                          f"contiguous shards of {hi - lo} tours per GPU, no data-path collective",
              "population_sha256": sha(orders)}
        mine = np.ascontiguousarray(succ_ga[lo:hi])
        costs0 = eng.tour_costs(mine, as_order=False)
        for mode, nm in ((FI, "FI"), (BI, "BI")):
            eng.two_opt_batch(mode, mine[:8], costs0[:8])  # warm-up
            barrier()
            w0 = time.perf_counter()
            sb, ob, stg = eng.two_opt_batch(mode, mine, costs0)
            torch.cuda.synchronize()
            sec = maxr(time.perf_counter() - w0)
            tot = torch.tensor([float(stg.moves), float(stg.evals), float(ob.sum())], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tot)
            ga[nm] = {"seconds": sec, "tours_per_s": pop / sec, "moves": int(tot[0].item()), "evals": int(tot[1].item()),
                      "evals_per_s": float(tot[1].item()) / sec, "sum_of_final_costs": float(tot[2].item()),
                      "call": "tspb200_two_opt_batch (host buffers in and out, inside the timed region)"}
        eng.set_instance(h_xy, 0)

    if rank != 0:
        eng.close()
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peaks_src = measured_peaks()
    if clocks.get("sm_mhz"):
        sm_mhz, clock_src = clocks["sm_mhz"], f"NVML median over the {clocks['source'].split(', ', 1)[1]}"
    else:
        sm_mhz, clock_src = peaks.get("sm_max_mhz", 1965.0), "no NVML sample: MEASURED_PEAKS.json sm_max_mhz"
    num_sms = eng.info("num_sms")
    per_gpu = value / world
    # Binding unit of bi_scan_kernel: the SFU (MUFU.SQRT, 16 results/clk/SM).  Algorithmic minimum = ONE distance
    # (one sqrt) per evaluated move: every D[p][q] is shared by the two moves that use it (DESIGN.md §4).
    sqrt_peak = num_sms * 16 * sm_mhz * 1e6
    fp32_peak = num_sms * 128 * sm_mhz * 1e6
    T, R, TJ = shape_value["block_threads"], shape_value["rows_per_thread"], shape_value["tile_cols"]
    ncu = {}
    if os.path.exists(NCU_KEYED):
        with open(NCU_KEYED) as f:
            ncu = json.load(f).get(f"{T}x{R}x{TJ}" + ("s" if shape_value["row_shuffle"] else ""), {})
    ipe = ncu.get("thread_instr_per_eval")
    roofline = {"bound": "sfu_sqrt", "achieved": per_gpu / 1e12, "peak": sqrt_peak / 1e12, "unit": "T sqrt/s (= T evals/s)",
                "frac": per_gpu / sqrt_peak, "traffic": ncu.get("dram_bytes_per_launch"), "kernel": "bi_scan_kernel",
                "per_unit": "1 MUFU.SQRT per evaluated move (algorithmic minimum: every distance serves two moves); the kernel issues " +
                            (f"32R/(32R-1) = {32 * R / (32 * R - 1):.4f} (R = {R} rows per thread; the distance below a lane's rows comes "
                             f"from the next lane by shuffle, a warp owns 32R-1 rows)" if shape_value["row_shuffle"]
                             else f"(R+1)/R = {(R + 1) / R:.4f} with R = {R} rows per thread"),
                "peak_source": f"{num_sms} SMs x 16 MUFU/clk x {sm_mhz:.0f} MHz ({clock_src}); MEASURED_PEAKS.json ({peaks_src}) "
                               f"holds HBM and bf16 figures only, neither bounds this kernel",
                "ncu": ncu if ncu else f"no ncu capture committed for tile shape {T}x{R}x{TJ}{'s' if shape_value['row_shuffle'] else ''} (profiles/ncu_by_tile_shape.json)",
                "fp32_issue_view": {"survey_per_unit": FP32_INSTR_PER_EVAL,
                                    "frac_vs_survey_18_instr_model": per_gpu * FP32_INSTR_PER_EVAL / fp32_peak,
                                    "executed_thread_instr_per_eval": ipe,
                                    "frac_issue_slots": per_gpu * ipe / fp32_peak if ipe else None,
                                    "note": "SURVEY.md §8d's 18 lane-instr/eval model evaluates two fresh distances per move with "
                                            "scalar FP32; sharing each distance between its two moves and packed FP32x2 arithmetic "
                                            "bring the executed count far below it, so the 18-instr fraction exceeds 1 and is "
                                            "reported for reference only"}}
    # secondary kernel: distance matrix, HBM-store-bound (4*n*ld bytes written per launch)
    mat = None
    if world == 1 and not args.no_extras:
        nm = 20000  # 1.6 GB of int32 (> L2); the size the ncu --set full capture in profiles/ was taken at
        eng.set_instance(uniform_instance(nm), 0)
        eng.dist_matrix_build()
        ms_list = []
        for _ in range(5):
            if flush is not None:
                flush.zero_()
                torch.cuda.synchronize()
            ms_list.append(eng.dist_matrix_build())
        ld = eng.info("matrix_ld")
        eng.dist_matrix_free()
        ms = float(np.median(ms_list))
        gbs = 4.0 * nm * ld / (ms * 1e-3) / 1e9
        mncu = {}
        if os.path.exists(NCU_KEYED):
            with open(NCU_KEYED) as f:
                mncu = json.load(f).get("dist_matrix_n20000", {})
        mat = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
               "traffic": mncu.get("dram_bytes_per_launch"), "ncu": mncu, "kernel": "dist_matrix_kernel", "n": nm, "ms": ms,
               "per_unit": "4 bytes written per matrix entry (int32), reads O(n)", "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peaks_src})"}
    cfg = workload_config(n)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": gpu_ms / max(1, done_passes), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "engine": {"block_threads": T, "rows_per_thread": R, "tile_cols": TJ, "tile_rows": shape_value["tile_rows"],
                       "row_shuffle": shape_value["row_shuffle"], "grid": shape_value["grid_bi"], "tiles": shape_value["ntiles"],
                       "sharding": ("tiles round-robin over ranks; per pass each rank's 8-byte argmin key is " +
                                    ("stored into every peer's slots over NVLink by the scan kernel (CUDA IPC peer memory)"
                                     if eng.info("exchange_p2p") else "min-allreduced by NCCL")) if world > 1 else "single GPU",
                       "l2_flush": not args.no_flush, "nn_start_s": nn_s, "tile_pruning": "off for value / e2e (exhaustive scans)"},
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d / e2e_passes, "d2h_bytes_per_step": d2h / e2e_passes,
                    "passes": st_e.passes, "seconds": e2e_s,
                    "call": "tspb200_set_instance (unchanged coordinates: compared on the host, not re-sent) + "
                            "tspb200_two_opt(BI, host succ[], max_iters=steps)",
                    "tour_check": chk_e2e, "one_call_per_step": e2e_step},
            "gpu_launches": int(launches), "moves_applied": int(moves), "wall_s": wall_s,
            "tour_check": chk_value, "clocks": clocks, "roofline": roofline}
    if breakdown:
        line["pass_breakdown"] = breakdown
    if mat:
        line["roofline_matrix"] = mat
    if tlo:
        line["time_to_local_optimum"] = tlo
    if ga:
        line["ga_batch"] = ga
    if not args.no_cpu_baseline and world == 1:
        base, _ = cpu_baseline_sample(xy, succ0, 12.0)
        stock = stock_one_core(2000 if n >= 10000 else 600)
        if stock:
            base["stock_1core"] = stock
            base["harness_per_core_over_stock_1core"] = base["value_per_core"] / stock["value"]
        line["cpu_baseline"] = base
    bad = [k for k, c in (("value", chk_value), ("e2e", chk_e2e)) if c.get("check") == "MISMATCH"]
    if tlo and tlo.get("tour_check", {}).get("check") == "MISMATCH":
        bad.append("time_to_local_optimum")
    if tlo and tlo.get("pruned", {}).get("tour_check", {}).get("check") == "MISMATCH":
        bad.append("time_to_local_optimum.pruned")
    line["self_check"] = "ok" if not bad else "MISMATCH in " + ", ".join(bad)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"tour_succ": tour_after, "tour_cost": [cost_after],
                                         "pass_stats": [done_passes, moves, st.evals, st.obj_delta]})
    print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    if bad:
        sys.exit(3)


if __name__ == "__main__":
    main()
