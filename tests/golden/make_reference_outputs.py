"""Generates tests/golden/reference_outputs.json: the results of the reference's own functions on the inputs of the tests that
compare the oracle restatement, the GPU engine and the drop-in with them (alg_2opt, alg_2opt_tabu with and without a tabu
list and its exported prev[], HEU_Greedy_iter, HEU_extramileage, the HEU_greedy / HEU_2opt_* drivers, kick(), the
`instance` layout).  With the stored values those tests run without a deno750/TSP_Optimization checkout; where the
reference is built (oracle/_ref, `make -C oracle REF=<checkout>`) they still compare with it as well.

Every value is computed with each available source and all must agree before anything is written:
  * the compiled reference, oracle/_ref/libtspref.so (RefLib) — the source of record when it is built;
  * the oracle restatement (oracle/tsp_oracle.c) and the drop-in's mirror of the reference `instance`, always;
  * the reference-derived values goldens.json already holds (NN / FI / BI tours, the published CSV costs) and SURVEY.md §8(b).
Without the compiled reference the script stops unless --restatement is given; the file then records, in "source", that
its values beyond goldens.json / SURVEY.md come from the restatement.  Tours are stored as sha256 of the int32 successor
array, like goldens.json.

    python tests/golden/make_reference_outputs.py [--restatement] [--out FILE]   (after __graft_entry__.build(); no GPU)
"""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.oracle import Oracle, RefLib, have_ref  # noqa: E402
from tsp_optimization_b200.engine import DROPIN_PATH  # noqa: E402
from tsp_optimization_b200.instances import GlibcRandom, order_to_succ, uniform_instance  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
COMPILED_REF_INSTANCES = ["berlin52", "att48", "ulysses22", "pr299", "gr96"]
GREEDY_ITER = ["berlin52", "pr299", "rd400", "att532", "ulysses22", "gr96", "eil51"]
EXTRA_MILEAGE = ["berlin52", "pr299", "att532", "gr666", "dsj1000", "ulysses22", "eil51", "gr96"]
#: (driver, instance) pairs tests/test_gpu_dropin_link.py runs through the drop-in
DRIVERS = [("HEU_2opt_extramileage", "lin318"), ("HEU_2opt_extramileage", "att532"), ("HEU_2opt_greedy_iter", "berlin52"),
           ("HEU_greedy", "gr666"), ("HEU_extramileage", "pr299"), ("HEU_2opt_greedy_iter", "gr431"),
           ("HEU_Greedy_iter", "dsj1000"), ("HEU_extramileage", "gr666"), ("HEU_2opt_extramileage", "dsj1000")]
#: the published CSV column of each driver (goldens.json reference_csv)
CSV_COLUMN = {"HEU_greedy": "GREEDY", "HEU_Greedy_iter": "GREEDY_ITER", "HEU_extramileage": "EXTR_MILE",
              "HEU_2opt_greedy_iter": "2OPT_GREEDY_ITER", "HEU_2opt_extramileage": "2OPT_EXTR_MIL"}


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.int32).tobytes()).hexdigest()


def random_tour_cases():
    """the inputs of test_oracle_equals_reference_on_random_tours_and_coords, in its order"""
    rng = np.random.default_rng(7)
    for wt, n in [(0, 120), (3, 90), (5, 100), (4, 60)]:
        if wt == 4:
            xy = np.round(rng.uniform(-80, 80, size=(n, 2)), 2)
        else:
            xy = rng.integers(0, 3000, size=(n, 2)).astype(np.float64)
            xy[::7] += 0.5  # non-integer but FP32-exact
        yield wt, xy, order_to_succ(rng.permutation(n).astype(np.int32))


def tabu_mask_case():
    """the input of test_tabu_mask_restatement"""
    rng = np.random.default_rng(11)
    n = 60
    xy = rng.integers(0, 1000, size=(n, 2)).astype(np.float64)
    succ = order_to_succ(rng.permutation(n).astype(np.int32))
    ncols = n * (n - 1) // 2
    mask = np.where(rng.random(ncols) < 0.2, rng.integers(1, 30, size=ncols), 0).astype(np.int32)
    return xy, succ, mask


def tiny_extra_mileage_cases():
    """the tie-heavy inputs of test_constructive_restatements_equal_reference_and_csv"""
    rng = np.random.default_rng(4)
    for n in (2, 3, 5, 30):
        yield n, rng.integers(0, 7, size=(n, 2)).astype(np.float64)


def vns_kick_indices(seed: int, n: int):
    """the three indices the reference kick() (src/vns.c:11) draws from glibc random() after srandom(seed)"""
    g = GlibcRandom(seed)
    i1 = g.rand_choice(0, n)
    i2 = i3 = i1
    while i2 == i1 or abs(i1 - i2) <= 1:
        i2 = g.rand_choice(0, n)
    while i3 == i1 or i3 == i2 or abs(i1 - i3) <= 1 or abs(i2 - i3) <= 1:
        i3 = g.rand_choice(0, n)
    return i1, i2, i3


def masked_bi_case(xy):
    """the tabu list of test_reference_masked_bi_through_dropin (berlin52)"""
    n = len(xy)
    rng = np.random.default_rng(3)
    ncols = n * (n - 1) // 2
    return np.where(rng.random(ncols) < 0.15, rng.integers(1, 40, size=ncols), 0).astype(np.int32)


class Restatement:
    """the oracle restatement: src/heuristics.c:160 HEU_greedy = greedy(inst, 0); :572-605 HEU_2opt_<ctor> = the constructive
    heuristic, then alg_2opt from its tour and cost"""
    name = "oracle restatement (oracle/tsp_oracle.c) and the drop-in's `instance` mirror"

    def __init__(self):
        self.o = Oracle()

    def layout(self):
        L = C.CDLL(DROPIN_PATH)
        buf = (C.c_longlong * 32)()
        return [int(buf[t]) for t in range(L.tspb200_dropin_layout(buf, 32))]

    def two_opt_fi(self, xy, wt, succ, cost):
        return self.o.two_opt_fi(xy, wt, succ, cost)[:2]

    def two_opt_bi(self, xy, wt, succ, skip_edge=None, iter_=1, tenure=1, want_prev=False):
        r = self.o.two_opt_bi(xy, wt, succ, skip_edge=skip_edge, iter_=iter_, tenure=tenure, want_prev=want_prev)
        return r[:2] + ((r[4],) if want_prev else ())

    def driver(self, method, xy, wt):
        ctor = method.replace("HEU_2opt_", "HEU_")
        if ctor == "HEU_greedy":
            s, c = self.o.nn_tour(xy, wt, 0)
        elif ctor.lower() == "heu_greedy_iter":
            _, s, c = self.o.greedy_iter(xy, wt)
        else:
            s, c = self.o.extra_mileage(xy, wt)
        if method.startswith("HEU_2opt_"):
            s, c = self.two_opt_fi(xy, wt, s, c)
        return s, c

    def vns_kick(self, xy, succ, seed):
        return self.o.vns_kick(xy, 0, succ, *vns_kick_indices(seed, len(xy)))


class Reference:
    """the compiled, unmodified reference"""
    name = "compiled reference (oracle/_ref/libtspref.so)"

    def __init__(self):
        self.r = RefLib()

    def layout(self):
        d = self.r.layout()
        return [d[k] for k in RefLib.LAYOUT_KEYS]

    def two_opt_fi(self, xy, wt, succ, cost):
        return self.r.two_opt_fi(xy, wt, succ, cost)

    def two_opt_bi(self, xy, wt, succ, skip_edge=None, iter_=1, tenure=1, want_prev=False):
        return self.r.two_opt_bi(xy, wt, succ, skip_edge=skip_edge, iter_=iter_, tenure=tenure, want_prev=want_prev)

    def driver(self, method, xy, wt):
        st, s, c = self.r.run_method(method, xy, wt)
        assert st == 0, (method, st)
        return s, c

    def vns_kick(self, xy, succ, seed):
        return self.r.vns_kick_stock(xy, 0, succ, seed)


def agree(results):
    """results of the same call from every source -> the first one's, after checking that all are bit-identical"""
    first = results[0]
    for r in results[1:]:
        assert len(r) == len(first) and all(np.array_equal(a, b) for a, b in zip(first, r)), "sources disagree"
    return first


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--restatement", action="store_true", help="record from the restatement when the reference is not built")
    ap.add_argument("--out", default=os.path.join(GOLD, "reference_outputs.json"))
    args = ap.parse_args()
    srcs = [Reference()] if have_ref() else []
    if not srcs and not args.restatement:
        sys.exit("oracle/_ref is not built (make -C oracle REF=<reference checkout>); --restatement records from the oracle")
    srcs.append(Restatement())
    orc = srcs[-1].o
    gold = json.load(open(os.path.join(GOLD, "goldens.json")))
    z = np.load(os.path.join(GOLD, "instances.npz"))
    inst = lambda nm: (z[nm + "__xy"], int(z[nm + "__wt"]))  # noqa: E731
    out = {}

    layout = agree([[s.layout()] for s in srcs])[0]
    # SURVEY.md §8(b), offsetof probes of the reference build: sizeof(instance), time_limit, integer_cost, perf_prof, nodes,
    # num_nodes, weight_type, num_columns, solution.obj_best, solution.edges
    assert layout[:10] == [152, 12, 44, 52, 80, 88, 92, 96, 120, 128], layout
    out["layout"] = layout

    out["bi_prev_sha256"] = {}
    for nm in COMPILED_REF_INSTANCES:
        xy, wt = inst(nm)
        g = gold["instances"][nm]
        succ, cost = orc.nn_tour(xy, wt, 0)
        assert sha(succ) == g["nn_sha256"] and cost == g["nn_cost"], nm
        bs, bc, prev = agree([s.two_opt_bi(xy, wt, succ, want_prev=True) for s in srcs])
        assert sha(bs) == g["bi_sha256"] and bc == g["bi_cost"], nm
        out["bi_prev_sha256"][nm] = sha(prev)

    out["random_tours"] = []
    for wt, xy, succ in random_tour_cases():
        c = orc.succ_cost(xy, wt, succ)
        fs, fc = agree([s.two_opt_fi(xy, wt, succ, c) for s in srcs])
        bs, bc = agree([s.two_opt_bi(xy, wt, succ) for s in srcs])
        out["random_tours"].append({"wt": wt, "n": len(xy), "fi_sha256": sha(fs), "fi_cost": fc, "bi_sha256": sha(bs), "bi_cost": bc})

    def masked(xy, wt, succ, mask, iter_, tenure):
        res = []
        for s in srcs:
            m = mask.copy()  # alg_2opt_tabu updates the list in place
            res.append(s.two_opt_bi(xy, wt, succ, skip_edge=m, iter_=iter_, tenure=tenure) + (m,))
        bs, bc, m = agree(res)
        return {"iter": iter_, "tenure": tenure, "bi_sha256": sha(bs), "bi_cost": bc, "mask_after_sha256": sha(m)}

    xy, succ, mask = tabu_mask_case()
    out["tabu_mask"] = masked(xy, 0, succ, mask, 30, 12)

    out["greedy_iter"], out["extra_mileage"], out["drivers"] = {}, {}, {}
    for nm in GREEDY_ITER:
        xy, wt = inst(nm)
        s, c = agree([src.driver("HEU_Greedy_iter", xy, wt) for src in srcs])
        if nm in gold["reference_csv"]:
            assert c == gold["reference_csv"][nm]["GREEDY_ITER"], nm
        out["greedy_iter"][nm] = {"sha256": sha(s), "cost": c}
    for nm in EXTRA_MILEAGE:
        xy, wt = inst(nm)
        s, c = agree([src.driver("HEU_extramileage", xy, wt) for src in srcs])
        if nm in gold["reference_csv"]:
            assert c == gold["reference_csv"][nm]["EXTR_MILE"], nm
        out["extra_mileage"][nm] = {"sha256": sha(s), "cost": c}
    for n, xy in tiny_extra_mileage_cases():
        s, c = agree([src.driver("HEU_extramileage", xy, 0) for src in srcs])
        out["extra_mileage"][f"ties{n}"] = {"sha256": sha(s), "cost": c}
    for method, nm in DRIVERS:
        xy, wt = inst(nm)
        s, c = agree([src.driver(method, xy, wt) for src in srcs])
        csv = gold["reference_csv"].get(nm, {}).get(CSV_COLUMN[method])
        assert csv is None or c == csv, (method, nm, c, csv)
        if method == "HEU_greedy":
            assert sha(s) == gold["instances"][nm]["nn_sha256"], nm
        out["drivers"][f"{method}:{nm}"] = {"sha256": sha(s), "cost": c}

    xy, wt = inst("berlin52")
    succ, _ = orc.nn_tour(xy, wt, 0)
    out["masked_bi_berlin52"] = masked(xy, wt, succ, masked_bi_case(xy), 40, 9)

    n = 300
    xy = uniform_instance(n)
    succ, _ = orc.nn_tour(xy, 0, 0)
    out["vns_kick"] = {"n": n, "seeds": {}}
    for seed in range(1, 40):
        if max(vns_kick_indices(seed, n)) == n - 1:  # there the reference reads one element past its tour array
            continue
        s, c = agree([src.vns_kick(xy, succ, seed) for src in srcs])
        out["vns_kick"]["seeds"][str(seed)] = {"sha256": sha(s), "cost": c}

    out["source"] = (f"tests/golden/make_reference_outputs.py; values from: {' = '.join(s.name for s in srcs)}; checked against the "
                     "reference-derived goldens.json (NN, FI and BI tours, published GREEDY / GREEDY_ITER / EXTR_MILE / 2OPT_* costs) "
                     "and SURVEY.md §8(b)")
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote", args.out, {k: len(v) if hasattr(v, "__len__") else v for k, v in out.items()})


if __name__ == "__main__":
    main()
