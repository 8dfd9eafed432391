"""One VNS search (reference HEU_VNS, src/vns.c:103-183) on the resident tour, tspb200_vns_search: iterations/s on uni<n> for
each `--sizes` entry, from the FI local optimum of the NN tour from node 0, with the kicks drawn by
instances.vns_kick_indices(GlibcRandom(--seed), n).  The iteration count of the timed call is sized from a calibration call so
that the window is at least `--window` seconds.  Reported per size: iterations/s, FI moves and sweeps per iteration, host
launches (and per FI move).  On the first `--session-iters` kicks it times the single-tour session loop (vns_kick + fi_run +
tour_save / tour_restore, tools/vns_chains.py) and asserts its costs equal the search's trace; where the tour fits one block
(n <= `--chain-max-n`), population_vns with one chain on the first `--chain-iters` kicks (asserted equal too).  `--caps`
times the search at fixed batch sizes (option "batch") at the sizes in `--cap-sizes`.  `--profile` instead takes the kernel
times of one search from torch.profiler (search, apply, step: the no-op steps and the working ones apart, and the gaps), in
a run of its own.  The GPU name, power limit and SM clock are read in the same process.  One JSON line per size."""
import argparse
import json
import math
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from tsp_optimization_b200 import FI, Engine  # noqa: E402
from tsp_optimization_b200.instances import GlibcRandom, uniform_instance, vns_kick_indices  # noqa: E402
from vns_chains import gpu_info, session_loop  # noqa: E402


def draw(n, seed, iters):
    g = GlibcRandom(seed)
    return np.array([vns_kick_indices(g, n) for _ in range(iters)], dtype=np.int32).reshape(-1, 3)


def timed_search(eng, start, kicks):
    eng.tour_upload(start)
    t0 = time.perf_counter()
    best, trace, st = eng.vns_search(kicks)
    return best, trace, st, time.perf_counter() - t0


def profile_search(eng, start, kicks):
    from torch.profiler import ProfilerActivity, profile
    eng.tour_upload(start)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, _, st = eng.vns_search(kicks)
        torch.cuda.synchronize()
    groups = {"search": "fi_search_kernel", "apply": "apply_move_kernel", "step": "vns_step_kernel"}
    dur = {k: [] for k in groups}
    other = 0.0
    spans = []
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        t0, t1 = e.time_range.start, e.time_range.end
        spans.append((t0, t1))
        for k, name in groups.items():
            if name in e.name:
                dur[k].append(t1 - t0)
                break
        else:
            other += t1 - t0
    out = {"profile_iters": len(kicks), "profile_moves": st.moves, "profile_passes": st.passes}
    for k, v in dur.items():
        out[f"profile_{k}_count"] = len(v)
        out[f"profile_{k}_us"] = round(sum(v), 1)
    # the working steps (the call-start one and one per iteration) are the longest; the others return at once
    steps = sorted(dur["step"])
    work = len(kicks) + 1
    noop, busy = steps[:-work], steps[-work:]
    out["profile_step_noop_us_mean"] = round(sum(noop) / max(len(noop), 1), 2)
    out["profile_step_working_us_mean"] = round(sum(busy) / max(len(busy), 1), 2)
    out["profile_other_kernels_us"] = round(other, 1)
    # with PDL a search is resident (in griddepcontrol.wait) while the apply before it runs, so kernel times overlap: the
    # gaps are the span minus the union of the kernel intervals
    spans.sort()
    busy, end = 0.0, None
    for t0, t1 in spans:
        if end is None or t0 > end:
            busy, end = busy + (t1 - t0), t1
        elif t1 > end:
            busy, end = busy + (t1 - end), t1
    out["profile_span_us"] = round(max(t1 for _, t1 in spans) - spans[0][0], 1) if spans else 0.0
    out["profile_gaps_us"] = round(out["profile_span_us"] - busy, 1)
    out["profile_span_us_per_fi_move"] = round(out["profile_span_us"] / max(st.moves, 1), 2)
    out["profile_launches_per_fi_move"] = round(st.launches / max(st.moves, 1), 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,5000,10000,20000,100000")
    ap.add_argument("--window", type=float, default=0.3, help="least seconds of the timed call")
    ap.add_argument("--max-iters", type=int, default=20000)
    ap.add_argument("--session-iters", default="40,20,10,6,3", help="session-loop iterations per size (the search's first ones)")
    ap.add_argument("--chain-max-n", type=int, default=8296)
    ap.add_argument("--chain-iters", type=int, default=10)
    ap.add_argument("--caps", default="", help="fixed batch sizes to time, e.g. 16,64,256")
    ap.add_argument("--cap-sizes", default="1000,20000")
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--profile-iters", type=int, default=5)
    ap.add_argument("--out", default=None, help="default profiles/r8_vns_search_w1.jsonl (with --profile: "
                                                 "profiles/r8_vns_search_profile_w1.jsonl)")
    args = ap.parse_args()
    if args.out is None:
        args.out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                "r8_vns_search_profile_w1.jsonl" if args.profile else "r8_vns_search_w1.jsonl")
    sizes = [int(x) for x in args.sizes.split(",")]
    siters = [int(x) for x in args.session_iters.split(",")]
    caps = [int(x) for x in args.caps.split(",") if x]
    cap_sizes = {int(x) for x in args.cap_sizes.split(",") if x}
    eng = Engine(0)
    info = gpu_info(0)
    lines = []
    for n, ks in zip(sizes, siters):
        xy = uniform_instance(n)
        eng.set_instance(xy, 0)
        nn, cost = eng.nn_tour(0)
        start, _, _, _ = eng.two_opt(FI, nn, cost)
        rec = {"workload": f"one VNS search on uni{n} from the FI optimum of the NN tour from node 0, kicks from "
                           f"vns_kick_indices(GlibcRandom({args.seed}))", "n": n}
        if args.profile:
            timed_search(eng, start, draw(n, args.seed + 1, 2))  # warm-up: modules, scratch buffers
            rec.update(profile_search(eng, start, draw(n, args.seed, args.profile_iters)))
        else:
            # calibration (also the warm-up), then a call sized for the window
            k0 = 4 if n >= 50000 else 40
            _, _, _, sec0 = timed_search(eng, start, draw(n, args.seed + 1, k0))
            k = int(min(args.max_iters, max(k0, math.ceil(args.window * k0 / sec0))))
            kicks = draw(n, args.seed, max(k, ks, args.chain_iters))
            best, trace, st, sec = timed_search(eng, start, kicks[:k])
            rec.update({"iters": k, "seconds": sec, "iters_per_s": k / sec, "gpu_ms": st.gpu_ms, "moves": st.moves,
                        "sweeps": st.passes, "moves_per_iter": st.moves / k, "sweeps_per_iter": st.passes / k,
                        "launches": st.launches, "launches_per_fi_move": st.launches / max(st.moves, 1), "best_cost": best})
            session_loop(eng, start, kicks[:2])  # warm-up
            costs, ssec = session_loop(eng, start, kicks[:ks])
            ptrace = trace if ks <= k else timed_search(eng, start, kicks[:ks])[1]
            assert costs == ptrace[:ks].tolist(), (n, costs, ptrace[:ks].tolist())
            rec.update({"session_iters": ks, "session_seconds": ssec, "session_iters_per_s": ks / ssec,
                        "session_equals_search": True})
            if n <= args.chain_max_n:
                kc = args.chain_iters
                eng.population_upload(start[None], as_order=False)
                eng.population_vns(kicks[None, :1])  # warm-up
                eng.population_upload(start[None], as_order=False)
                t0 = time.perf_counter()
                pbest, ptr, _ = eng.population_vns(kicks[None, :kc])
                csec = time.perf_counter() - t0
                cbest, ctrace, _, _ = timed_search(eng, start, kicks[:kc])
                assert ptr[0].tolist() == ctrace.tolist() and pbest[0] == cbest
                rec.update({"chain_iters": kc, "chain_seconds": csec, "chain_iters_per_s": kc / csec, "chain_equals_search": True})
            if n in cap_sizes:
                for c in caps:
                    eng.set_option("batch", c)
                    _, ctr, _, csec = timed_search(eng, start, kicks[:k])
                    assert ctr.tolist() == trace.tolist()
                    rec[f"batch{c}_iters_per_s"] = k / csec
                eng.set_option("batch", 0)
        rec.update(info)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    eng.close()


if __name__ == "__main__":
    main()
