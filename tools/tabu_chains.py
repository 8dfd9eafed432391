"""Independent tabu searches (reference tabu(), src/tabusearch.c:188-320) across GPUs: `--chains` chains on uni<n>, chain b
started from the FI local optimum of the NN tour from node b mod n, seeded with srandom(seed + b) (so a shard does not depend
on the world size) and run `--iters` iterations with the step tenure schedule of tests/test_gpu_sessions.py (3, then 15,
switching every 6 iterations).  Run under torchrun: every rank runs its contiguous share of the chains
(tsp_optimization_b200.dist.shard_batch) with one tspb200_population_tabu call on its own engine; at the end
torch.distributed (gloo) finds the best chain (minimum best cost, lowest chain index) and broadcasts its best tour.  Rank r
runs on device r mod (devices present), so the sharded path can be checked with several ranks on one GPU.  Rank 0 then
reruns all chains on its own GPU and compares every shard (SHA-256 of tours, best tours, trace and draws), and times the
single-tour session loop (tabu_begin, tabu_run + one-candidate tabu_kick calls, tour_save) on the first `--session-chains`
chains.  One JSON line; at world = 1 the chain rate is the single-GPU measurement."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from tsp_optimization_b200 import Engine  # noqa: E402
from tsp_optimization_b200.dist import init_process_group_from_env, shard_batch  # noqa: E402
from tsp_optimization_b200.instances import GlibcRandom, uniform_instance  # noqa: E402
from vns_chains import digest, gpu_info, start_tours  # noqa: E402


def step_tenures(chains, iters):
    row = [3 if (t // 6) % 2 == 0 else 15 for t in range(iters)]
    return np.tile(np.array(row, dtype=np.int32), (chains, 1))


def run_chains(eng, n, lo, hi, seed, tenures):
    """chains lo..hi-1 on a fresh population: current tours in slots 0.., best tours after them"""
    starts = start_tours(eng, n, lo, hi)
    eng.population_upload(np.concatenate([starts, starts]), as_order=False)
    eng.population_tabu_begin(np.arange(lo, hi) + seed)
    t0 = time.perf_counter()
    best, trace, draws, st = eng.population_tabu(tenures)
    dt = time.perf_counter() - t0
    tours = eng.population_download(2 * (hi - lo), as_order=False)
    eng.population_tabu_end()
    return best, trace, draws, st, tours, dt


def session_loop(eng, n, start, seed, tenures):
    """the same chain through the single-tour session -> (costs, draws, seconds)"""
    eng.tour_upload(start)
    inc = eng.tour_cost()
    eng.tour_save(1)
    eng.tabu_begin()
    g = GlibcRandom(seed)
    costs, draws = [], []
    t0 = time.perf_counter()
    for t, tenure in enumerate(tenures):
        it = t + 1
        c = eng.tabu_run(it, int(tenure)).cost
        costs.append(c)
        if c < inc:
            inc = c
            eng.tour_save(1)
        d = 0
        while True:
            d += 1
            if eng.tabu_kick([[g.rand_choice(0, n), g.rand_choice(0, n)]], it, int(tenure)) == 0:
                break
        draws.append(d)
    eng.tour_cost()  # ends in a stream synchronisation
    dt = time.perf_counter() - t0
    eng.tabu_end()
    return costs, draws, dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1000)
    ap.add_argument("--chains", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--session-chains", type=int, default=4)
    a = ap.parse_args()
    rank, world, local = init_process_group_from_env("gloo")
    ndev = torch.cuda.device_count()
    local %= ndev
    torch.cuda.set_device(local)
    n, B, K = a.size, a.chains, a.iters
    ten = step_tenures(B, K)
    eng = Engine(local)
    eng.set_instance(uniform_instance(n), 0)
    lo, hi = shard_batch(B, rank, world)
    mine = hi - lo
    if mine > 0:
        run_chains(eng, n, lo, lo + 1, a.seed, ten[:1, :1])  # warm-up (module load)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if mine > 0:
        best, trace, draws, st, tours, dt = run_chains(eng, n, lo, hi, a.seed, ten[lo:hi])
    else:
        best, trace, draws, tours, dt = np.zeros(0), np.zeros((0, K)), np.zeros((0, K), np.int32), np.zeros((0, n), np.int32), 0.0
    # best chain over all ranks: minimum best cost, lowest chain index
    k = int(np.argmin(best)) if mine else 0
    cand = torch.tensor([float(best[k]) if mine else float("inf"), float(lo + k)], dtype=torch.float64)
    tot = torch.tensor([dt, float(st.moves) if mine else 0.0, float(st.evals) if mine else 0.0], dtype=torch.float64)
    if world > 1:
        allc = [torch.zeros_like(cand) for _ in range(world)]
        dist.all_gather(allc, cand)
        allc = torch.stack(allc).numpy()
        tmax = tot.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        tot[0] = tmax[0]
    else:
        allc = cand.numpy()[None]
    owner = int(min(range(world), key=lambda r: (allc[r][0], allc[r][1])))
    best_chain, best_cost = int(allc[owner][1]), float(allc[owner][0])
    tour = torch.tensor(tours[mine + k] if rank == owner else np.zeros(n, dtype=np.int32), dtype=torch.int32)
    if world > 1:
        dist.broadcast(tour, src=owner)
    best_tour = tour.numpy()
    shard = (lo, hi, digest(tours, np.concatenate([trace, draws.astype(np.float64)], 1)))
    hashes = [None] * world
    if world > 1:
        dist.all_gather_object(hashes, shard)
    else:
        hashes = [shard]
    if rank == 0:
        best1, trace1, draws1, _, tours1, dt1 = run_chains(eng, n, 0, B, a.seed, ten)
        ok = True
        for x, y, h in hashes:
            part = np.concatenate([tours1[x:y], tours1[B + x:B + y]])
            ok = ok and digest(part, np.concatenate([trace1[x:y], draws1[x:y].astype(np.float64)], 1)) == h
        ok = ok and best_chain == int(np.argmin(best1)) and best_cost == float(best1.min()) and (best_tour == tours1[B + best_chain]).all()
        S = min(a.session_chains, B)
        starts0 = start_tours(eng, n, 0, S) if S else None
        sess_s, sess_equal = 0.0, True
        for b in range(S):
            costs, nd, s = session_loop(eng, n, starts0[b], a.seed + b, ten[b])
            sess_s += s
            sess_equal = sess_equal and costs == trace1[b].tolist() and nd == draws1[b].tolist()
        out = {"workload": f"tabu chains: {B} chains x {K} iterations on uni{n}, each from the FI optimum of an NN tour, "
                           "step tenure 3/15 every 6 iterations",
               "n": n, "chains": B, "iters": K, "n_ranks": world, "devices": min(world, ndev), "seconds": float(tot[0]),
               "chain_iters_per_s": B * K / float(tot[0]), "moves": int(tot[1]), "evals": int(tot[2]),
               "list_bytes": 4 * B * (n * (n - 1) // 2), "best_chain": best_chain, "best_cost": best_cost,
               "shards_equal_single_gpu": bool(ok), "rank0_all_chains_seconds": dt1}
        if S:
            out.update({"session_chains": S, "session_seconds": sess_s, "session_chain_iters_per_s": S * K / sess_s,
                        "session_equals_chains": bool(sess_equal)})
        out.update(gpu_info(local))
        print(json.dumps(out), flush=True)
        if not ok or not sess_equal:
            sys.exit(1)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
