"""One tabu search (reference tabu(), src/tabusearch.c:188-320) on the resident tour, tspb200_tabu_search: iterations/s on
uni<n> for each `--sizes` entry, from the FI local optimum of the NN tour from node 0, seeded with srandom(--seed) and run
with the step tenure schedule of tests/test_gpu_sessions.py (3, then 15, switching every 6 iterations).  For the same seed
and tenures it also times the single-tour session loop (tabu_begin, tabu_run + one-candidate tabu_kick calls, tour_save)
and asserts the same trace and draws; at the sizes in `--chain-sizes`, population_tabu with one chain on the first `--chain-iters` iterations (asserted equal too).
Per pass (all four launches of a pass: expiry, scan, apply, step) it compares a masked search (tenure 50) with the same
search unmasked (tenure -1), both `--pass-iters` iterations long, and shows an unmasked exhaustive bi_run pass of the same
scan shape (64 x 8, row shuffle, no pruning, no prefilter) from the NN tour (a denser pass: many improving moves); `--profile` adds the kernel times of one search from torch.profiler.  The GPU name,
power limit and SM clock are read in the same process.  One JSON line per size."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from tsp_optimization_b200 import FI, Engine  # noqa: E402
from tsp_optimization_b200.instances import GlibcRandom, uniform_instance  # noqa: E402
from vns_chains import gpu_info  # noqa: E402


def step_tenures(iters):
    return np.array([3 if (t // 6) % 2 == 0 else 15 for t in range(iters)], dtype=np.int32)


def timed_search(eng, start, seed, tenures):
    eng.tour_upload(start)
    eng.tabu_search_begin(seed)
    t0 = time.perf_counter()
    best, trace, draws, st = eng.tabu_search(tenures)
    sec = time.perf_counter() - t0
    eng.tabu_search_end()
    return best, trace, draws, st, sec


def session_loop(eng, start, seed, tenures):
    n = len(start)
    eng.tour_upload(start)
    inc = eng.tour_cost()
    eng.tour_save(1)
    eng.tabu_begin()
    g = GlibcRandom(seed)
    costs, nd = [], []
    t0 = time.perf_counter()
    for t, tenure in enumerate(tenures):
        it, tenure = t + 1, int(tenure)
        c = eng.tabu_run(it, tenure).cost
        costs.append(c)
        if c < inc:
            inc = c
            eng.tour_save(1)
        d = 0
        while True:
            d += 1
            if eng.tabu_kick([[g.rand_choice(0, n), g.rand_choice(0, n)]], it, tenure) == 0:
                break
        nd.append(d)
    sec = time.perf_counter() - t0
    eng.tabu_end()
    return costs, nd, sec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="5000,10000,20000")
    ap.add_argument("--iters", default="1000,400,200", help="search iterations per size")
    ap.add_argument("--session-iters", default="20,10,5", help="session-loop iterations per size (the search's first ones)")
    ap.add_argument("--chain-sizes", default="5000")
    ap.add_argument("--chain-iters", type=int, default=10, help="population_tabu iterations (the search's first ones)")
    ap.add_argument("--pass-iters", type=int, default=100, help="iterations of the masked / unmasked per-pass comparison")
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "r7_tabu_search_w1.jsonl"))
    args = ap.parse_args()
    sizes = [int(x) for x in args.sizes.split(",")]
    iters = [int(x) for x in args.iters.split(",")]
    siters = [int(x) for x in args.session_iters.split(",")]
    chain_sizes = {int(x) for x in args.chain_sizes.split(",") if x}
    eng = Engine(0)
    info = gpu_info(0)
    lines = []
    for n, k, ks in zip(sizes, iters, siters):
        xy = uniform_instance(n)
        eng.set_instance(xy, 0)
        nn, cost = eng.nn_tour(0)
        start, _, _, _ = eng.two_opt(FI, nn, cost)
        ten = step_tenures(k)
        timed_search(eng, start, args.seed + 1, ten[:2])  # warm-up: modules, scratch buffers
        best, trace, draws, st, sec = timed_search(eng, start, args.seed, ten)
        rec = {"workload": f"one tabu search on uni{n} from the FI optimum of the NN tour from node 0, step tenure 3/15 every 6 "
                           f"iterations, seed {args.seed}",
               "n": n, "iters": k, "seconds": sec, "iters_per_s": k / sec, "gpu_ms": st.gpu_ms, "passes": st.passes,
               "moves": st.moves, "launches": st.launches, "ms_per_pass": st.gpu_ms / max(st.passes, 1), "best_cost": best,
               "draws": int(draws.sum())}
        costs, nd, ssec = session_loop(eng, start, args.seed, ten[:ks])
        assert costs == trace[:ks].tolist() and nd == draws[:ks].tolist(), (n, costs, trace[:ks].tolist(), nd, draws[:ks].tolist())
        rec.update({"session_iters": ks, "session_seconds": ssec, "session_iters_per_s": ks / ssec, "session_equals_search": True})
        if n in chain_sizes:
            eng.population_upload(np.stack([start, start]), as_order=False)
            eng.population_tabu_begin([args.seed])
            t0 = time.perf_counter()
            kc = min(args.chain_iters, k)
            pbest, ptrace, pdraws, _ = eng.population_tabu(ten[None, :kc])
            csec = time.perf_counter() - t0
            eng.population_tabu_end()
            cbest, ctrace, cdraws, _, _ = timed_search(eng, start, args.seed, ten[:kc])
            assert ptrace[0].tolist() == ctrace.tolist() == trace[:kc].tolist() and pdraws[0].tolist() == cdraws.tolist()
            assert pbest[0] == cbest
            rec.update({"chain_iters": kc, "chain_seconds": csec, "chain_iters_per_s": kc / csec, "chain_equals_search": True})
        # per pass: masked (tenure 50) vs unmasked (tenure -1) search passes, and the unmasked exhaustive bi_run pass
        pk = args.pass_iters
        for name, tv in (("masked", 50), ("unmasked", -1)):
            _, _, _, pst, _ = timed_search(eng, start, args.seed, np.full(pk, tv, dtype=np.int32))
            rec[f"search_{name}_ms_per_pass"] = pst.gpu_ms / max(pst.passes, 1)
            rec[f"search_{name}_passes"] = pst.passes
        for key, v in (("prune", 0), ("prefilter", 0), ("block_threads", 64), ("rows_per_thread", 8)):
            eng.set_option(key, v)
        eng.tour_upload(nn)
        eng.bi_run(2)
        bst = eng.bi_run(100)
        rec["bi_run_exhaustive_ms_per_pass"] = bst.gpu_ms / max(bst.passes, 1)
        for key, v in (("prune", -1), ("prefilter", -1), ("block_threads", 0), ("rows_per_thread", 0)):
            eng.set_option(key, v)
        if args.profile:
            from torch.profiler import ProfilerActivity, profile
            try:
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    _, _, _, pst, _ = timed_search(eng, start, args.seed, ten[:min(k, 6)])
                    torch.cuda.synchronize()
                ker = {}
                for e in prof.key_averages():
                    t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                    if t and e.count:
                        ker[e.key[:80]] = {"count": e.count, "us_total": round(t, 1)}
                rec["profile_passes"] = pst.passes
                rec["profile_kernels"] = ker
            except Exception as ex:  # the measurement above stands without it
                rec["profile_error"] = repr(ex)[:300]
        rec.update(info)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    eng.close()


if __name__ == "__main__":
    main()
