"""Independent VNS chains (reference HEU_VNS, src/vns.c:103-183) across GPUs: `--chains` chains on uni<n>, each started from
the FI local optimum of the NN tour from node b mod n and kicked `--iters` times with indices drawn from GlibcRandom(seed + b)
(instances.vns_kick_indices).  Run under torchrun: every rank runs its contiguous share of the chains
(tsp_optimization_b200.dist.shard_batch) with one tspb200_population_vns call on its own engine, with no collective on the
data path; at the end torch.distributed finds the best chain (minimum cost, lowest chain index) and broadcasts its tour.
The end-of-run exchange is a few hundred bytes plus one tour, over gloo on CPU tensors; rank r runs on
device r mod (devices present), so the sharded path can also be checked with several ranks on one GPU (`devices` in the
output says how many GPUs the ranks really had).  Rank 0 then reruns all chains on its own GPU and compares every shard
(SHA-256 of final tours + trace), and times the single-tour session loop (vns_kick + fi_run + tour_save / tour_restore)
on the first `--session-chains` chains.  One JSON line; at world = 1 the chain rate is the single-GPU measurement."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from tsp_optimization_b200 import FI, Engine  # noqa: E402
from tsp_optimization_b200.dist import init_process_group_from_env, shard_batch  # noqa: E402
from tsp_optimization_b200.instances import GlibcRandom, uniform_instance, vns_kick_indices  # noqa: E402


def draw_kicks(n, chains, iters, seed):
    out = np.empty((chains, iters, 3), dtype=np.int32)
    for b in range(chains):
        g = GlibcRandom(seed + b)
        for t in range(iters):
            out[b, t] = vns_kick_indices(g, n)
    return out


def start_tours(eng, n, lo, hi):
    """FI local optima of the NN tours from nodes lo..hi-1 (mod n), left as the resident population"""
    nn, costs = eng.nn_tour_batch(np.arange(lo, hi, dtype=np.int32) % n)
    eng.population_upload(nn, as_order=False)
    eng.population_two_opt(FI, count=hi - lo, obj=costs)
    return eng.population_download(hi - lo, as_order=False)


def digest(tours, trace):
    return hashlib.sha256(np.ascontiguousarray(tours).tobytes() + np.ascontiguousarray(trace).tobytes()).hexdigest()


def gpu_info(local):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--id={local}", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power, sm, sm_max = [x.strip() for x in r.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock": sm, "sm_clock_max": sm_max}
    except Exception:
        return {"gpu": torch.cuda.get_device_name(local)}


def session_loop(eng, start, kicks):
    """the same chain through the single-tour session: kick, alg_2opt, keep or restore -> (costs, seconds)"""
    eng.tour_upload(start)
    inc = eng.tour_cost()
    eng.tour_save(0)
    costs = []
    t0 = time.perf_counter()
    for i1, i2, i3 in kicks:
        c = eng.vns_kick(i1, i2, i3) + eng.fi_run(-1).obj_delta
        costs.append(c)
        if c < inc:
            inc = c
            eng.tour_save(0)
        else:
            eng.tour_restore(0)
    eng.tour_cost()  # ends in a stream synchronisation
    return costs, time.perf_counter() - t0


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
    xy = uniform_instance(n)
    kicks = draw_kicks(n, B, K, a.seed)
    eng = Engine(local)
    eng.set_instance(xy, 0)
    lo, hi = shard_batch(B, rank, world)
    mine = hi - lo
    if mine > 0:
        starts = start_tours(eng, n, lo, hi)
        eng.population_vns(kicks[lo:lo + 1, :1], count=1)  # warm-up (module load); the population is uploaded again below
        eng.population_upload(starts, as_order=False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    if mine > 0:
        best, trace, st = eng.population_vns(kicks[lo:hi], count=mine)
        final = eng.population_download(mine, as_order=False)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if mine == 0:
        best, trace, final = np.zeros(0), np.zeros((0, K)), np.zeros((0, n), dtype=np.int32)
    # best chain over all ranks: minimum cost, lowest chain index
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
    tour = torch.tensor(final[k] if rank == owner else np.zeros(n, dtype=np.int32), dtype=torch.int32)
    if world > 1:
        dist.broadcast(tour, src=owner)
    best_tour = tour.numpy()
    shard = (lo, hi, digest(final, trace))
    hashes = [None] * world
    if world > 1:
        dist.all_gather_object(hashes, shard)
    else:
        hashes = [shard]
    if rank == 0:
        eng.population_upload(start_tours(eng, n, 0, B), as_order=False)
        t1 = time.perf_counter()
        best1, trace1, _ = eng.population_vns(kicks, count=B)
        final1 = eng.population_download(B, as_order=False)
        dt1 = time.perf_counter() - t1
        ok = all(digest(final1[x:y], trace1[x:y]) == h for x, y, h in hashes)
        ok = ok and best_chain == int(np.argmin(best1)) and best_cost == float(best1.min()) and (best_tour == final1[best_chain]).all()
        starts0 = start_tours(eng, n, 0, a.session_chains) if a.session_chains else None
        sess_s, sess_equal = 0.0, True
        for b in range(a.session_chains):
            costs, s = session_loop(eng, starts0[b], kicks[b])
            sess_s += s
            sess_equal = sess_equal and costs == trace1[b].tolist()
        out = {"workload": f"VNS chains: {B} chains x {K} iterations on uni{n}, each from the FI optimum of an NN tour",
               "n": n, "chains": B, "iters": K, "n_ranks": world, "devices": min(world, ndev), "seconds": float(tot[0]),
               "chain_iters_per_s": B * K / float(tot[0]), "moves": int(tot[1]), "evals": int(tot[2]),
               "best_chain": best_chain, "best_cost": best_cost, "shards_equal_single_gpu": bool(ok),
               "rank0_all_chains_seconds": dt1}
        if a.session_chains:
            out.update({"session_chains": a.session_chains, "session_seconds": sess_s,
                        "session_chain_iters_per_s": a.session_chains * K / sess_s, "session_equals_chains": bool(sess_equal)})
        out.update(gpu_info(local))
        print(json.dumps(out), flush=True)
        if not ok or not sess_equal:
            sys.exit(1)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
