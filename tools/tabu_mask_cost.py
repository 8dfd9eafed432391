"""What the tabu mask costs per pair: the masked best-improvement pass of tspb200_population_tabu against unmasked passes on
the same tours.  `--chains` chains on uni<n> first run `--warm` tabu iterations (step tenure 3/15, tools/tabu_chains.py) so
that their lists hold live entries.  Then, `--reps` times and alternating, the same random tours (instances.random_tours) go
through one tabu iteration at tenure 15 (masked passes), one at tenure -1 (the same kernel's unmasked pass: check_tenure
never blocks there), and tspb200_population_two_opt in mode BI with option batch_kernel = 1 (two_opt_batch_kernel).  From
random tours the best-improvement search runs hundreds of passes, so the kick, the table refresh and the tour loads of a
tabu iteration are a small share of its time.  Every pass counts n(n-3)/2 pairs; the rate is pairs per second of device
time (the engine's events).  One JSON line."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from tabu_chains import step_tenures  # noqa: E402
from vns_chains import gpu_info, start_tours  # noqa: E402

from tsp_optimization_b200 import BI, Engine  # noqa: E402
from tsp_optimization_b200.instances import random_tours, uniform_instance  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1000)
    ap.add_argument("--chains", type=int, default=1024)
    ap.add_argument("--warm", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    n, B = a.size, a.chains
    eng = Engine(0)
    eng.set_instance(uniform_instance(n), 0)
    starts = start_tours(eng, n, 0, B)
    eng.population_upload(np.concatenate([starts, starts, starts]), as_order=False)
    eng.population_tabu_begin(np.arange(B) + 1)
    eng.population_tabu(step_tenures(B, a.warm))
    rnd = random_tours(n, B, seed=5)
    cur, spare = np.arange(B, dtype=np.int32), np.arange(2 * B, 3 * B, dtype=np.int32)
    rows = {"masked": [], "unmasked_same_kernel": [], "two_opt_batch_kernel": []}
    eng.set_option("batch_kernel", 1)
    for _ in range(a.reps):
        for name, tenure in (("masked", 15), ("unmasked_same_kernel", -1)):
            eng.population_upload(rnd, slots=cur, as_order=False)  # the chains continue from these tours
            _, _, _, st = eng.population_tabu(np.full((B, 1), tenure, dtype=np.int32))
            rows[name].append(st)
        eng.population_upload(rnd, slots=spare, as_order=False)
        _, st = eng.population_two_opt(BI, slots=spare)
        rows["two_opt_batch_kernel"].append(st)
    eng.set_option("batch_kernel", 0)
    eng.population_tabu_end()
    out = {"workload": f"{B} random tours of uni{n} to the best-improvement local optimum; tabu lists after {a.warm} iterations",
           "n": n, "chains": B}
    for name, sts in rows.items():
        out[name] = {"pairs_per_s": [s.evals / (s.gpu_ms * 1e-3) for s in sts], "passes": [s.passes for s in sts],
                     "gpu_ms": [s.gpu_ms for s in sts]}
    med = {k: float(np.median(v["pairs_per_s"])) for k, v in out.items() if isinstance(v, dict)}
    out["masked_over_unmasked_same_kernel"] = med["masked"] / med["unmasked_same_kernel"]
    out["masked_over_two_opt_batch_kernel"] = med["masked"] / med["two_opt_batch_kernel"]
    out.update(gpu_info(0))
    print(json.dumps(out), flush=True)
    eng.close()


if __name__ == "__main__":
    main()
