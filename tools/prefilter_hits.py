"""Stage-1 prefilter statistics of the exhaustive best-improvement pass (csrc/kernels_bi_scan.cuh, DESIGN.md §3 / §4.1).

From the committed NN tour of uni100000 (tests/golden/nn_uni100000.npz) it runs K passes with the prefilter off and on and
prints, per pass, the device time, the stage-1 hits (warp ballot blocks that passed the squared-distance test) and the
exact-path calls, then the FP32-pipe fraction of the prefilter kernel.  bench.py's `roofline` block divides by the SFU peak of
the square-root kernel, so for the prefilter kernel it reads above 1; this script gives the number against the unit that
binds it now.

FP32_LANE_OPS_PER_COL: FP32-pipe lane operations per thread and column step in the column loop of
bi_scan_kernel<64, 8, false, true, false, true>, counted from `cuobjdump -sass` between the loop head and the warp ballot,
which covers 4 column steps: per step FFMA2 16 x 2 and FADD 1 = 33 — the four-FMA chain A_p + w_p . v_q of 4 packed row pairs
and the column constant B_q added to the row minimum.  FMNMX3 / FMNMX, LDS and the loop-carried register moves run on other
pipes.  A thread evaluates 8 moves per column step, and a warp 32 x 8 - 1 of the rows it scans.  The fraction assumes the
packed FP32x2 instructions occupy the pipe for two lane-ops each (not measured: no ncu).

With --sizes n1,n2,... it times instead exhaustive passes from an NN tour of uniform_instance(n) with the prefilter forced
off and on (alternating, `passes` each, L2 flushed before every pass): the data behind BI_PREFILTER_MIN_N in csrc/engine.cu.
--world W times one rank's share of W ranks on one GPU (option "debug_shard", rank 0's tiles).  --fractional adds a
fraction to every coordinate, so that they are not FP32-exact and the kernels for such coordinates (EXACT32 = 0) run.

usage: python tools/prefilter_hits.py [passes] [--sizes n1,n2,... [--world W] [--fractional]]
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from tsp_optimization_b200 import Engine
from tsp_optimization_b200.instances import uniform_instance

FP32_LANE_OPS_PER_COL = 33
EVALS_PER_COL = 8 * 255 / 256
LANES_PER_SM = 128  # FP32 lanes per SM and clock


def by_size(passes, sizes, world, fractional):
    eng = Engine(0)
    eng.set_option("prune", 0)
    eng.set_option("l2_flush_bytes", 256 << 20)
    for n in sizes:
        xy = uniform_instance(n)
        if fractional:  # decimal coordinates FP32 cannot hold: the kernels for non-FP32-exact coordinates run
            xy = xy + np.random.default_rng(n).random(xy.shape) * 0.999 + 0.1
        eng.set_instance(xy, 0)
        assert eng.info("exact32") == (0 if fractional else 1)
        succ, _ = eng.nn_tour(0)
        eng.set_option("debug_shard", (world << 8) if world > 1 else 0)
        us = {0: [], 1: []}
        for rep in range(4):
            for pf in (0, 1):
                eng.set_option("prefilter", pf)
                eng.tour_upload(succ)
                st = eng.bi_run(passes)
                us[pf].append(st.gpu_ms * 1e3 / st.passes)
        print(json.dumps({"n": n, "world": world, "fractional": fractional, "passes": passes, "us_per_pass_off": us[0], "us_per_pass_on": us[1],
                          "speedup_median": float(np.median(us[0]) / np.median(us[1]))}), flush=True)
    eng.close()


def main():
    passes = int(sys.argv[1]) if len(sys.argv) > 1 and not sys.argv[1].startswith("--") else 20
    if "--sizes" in sys.argv:
        world = int(sys.argv[sys.argv.index("--world") + 1]) if "--world" in sys.argv else 1
        return by_size(passes, [int(v) for v in sys.argv[sys.argv.index("--sizes") + 1].split(",")], world,
                       "--fractional" in sys.argv)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    succ = np.load(os.path.join(root, "tests", "golden", "nn_uni100000.npz"))["succ"]
    n = len(succ)
    eng = Engine(0)
    eng.set_instance(uniform_instance(n), 0)
    eng.set_option("prune", 0)
    eng.set_option("l2_flush_bytes", 256 << 20)
    pairs = n * (n - 3) // 2
    out = {}
    for pf in (0, 1):
        eng.set_option("prefilter", pf)
        eng.tour_upload(succ)
        rows = []
        for _ in range(passes):
            c0, h0 = eng.info("cold_calls"), eng.info("pf_hits")
            st = eng.bi_run(1)
            rows.append({"us": st.gpu_ms * 1e3, "pf_hits": eng.info("pf_hits") - h0, "cold_calls": eng.info("cold_calls") - c0})
        us = np.array([r["us"] for r in rows[1:]])
        out[pf] = {"prefilter": pf, "passes": passes, "us_median": float(np.median(us)),
                   "evals_per_s": pairs / (float(np.median(us)) * 1e-6),
                   "pf_hits_per_pass": [r["pf_hits"] for r in rows], "cold_calls_per_pass": [r["cold_calls"] for r in rows],
                   "pf_hit_fraction_of_ballots": float(np.mean([r["pf_hits"] for r in rows])) / (pairs / (32 * EVALS_PER_COL * 4))}
        print(json.dumps(out[pf]), flush=True)
    sms = eng.info("num_sms")
    eng.close()
    import subprocess
    clk = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits"], capture_output=True,
                         text=True).stdout.split()
    f_hz = float(clk[0]) * 1e6 if clk else 1.965e9
    ops = out[1]["evals_per_s"] * FP32_LANE_OPS_PER_COL / EVALS_PER_COL
    print(json.dumps({"fp32_pipe_fraction": ops / (sms * LANES_PER_SM * f_hz), "sm_clock_max_hz": f_hz, "num_sms": sms,
                      "speedup_prefilter": out[1]["evals_per_s"] / out[0]["evals_per_s"]}))


if __name__ == "__main__":
    main()
