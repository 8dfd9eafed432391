"""CPU tests: the oracle restatement (oracle/tsp_oracle.c) against (a) the committed golden fixtures that
were generated from the unmodified reference, (b) the reference's own published CSV goldens, and (c) the
stored results of the reference's functions on further inputs (tests/golden/reference_outputs.json, provenance in its
"source"), and the compiled reference itself when oracle/_ref is built."""
import hashlib

import numpy as np
import pytest

from tsp_optimization_b200.instances import is_tour, order_to_succ, uniform_instance


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


SMALL = ["berlin52", "att48", "burma14", "ulysses16", "ulysses22", "eil51", "gr96", "pr299", "a280", "gr202", "gr229"]


def test_golden_set_covers_all_metrics(goldens):
    wts = {g["wt"] for g in goldens["instances"].values()}
    assert {0, 3, 4, 5} <= wts  # EUC_2D, CEIL_2D, GEO, ATT


def test_matrix_matches_golden(oracle, instances, goldens):
    for nm, (xy, wt) in instances.items():
        g = goldens["instances"][nm]
        m = oracle.dist_matrix(xy, wt)
        assert int(m.sum(dtype=np.int64)) == g["matrix_sum"], nm
        assert sha(m) == g["matrix_sha256"], nm


def test_geo_diagonal_is_one(oracle, instances):
    xy, wt = instances["gr666"]
    assert wt == 4
    assert oracle.dist(xy, wt, 0, 0) == 1.0  # reference distutil.c:69 "+ 1.0" then nint


def test_man_max_follow_the_reference_bug(oracle):
    xy = np.array([[0.0, 0.0], [3.0, 40.0]])
    assert oracle.dist(xy, 2, 0, 1) == 3.0  # MAN_2D: dy = fabs(p2.y - p2.y) == 0
    assert oracle.dist(xy, 1, 0, 1) == 3.0  # MAX_2D
    assert oracle.dist(xy, 99, 0, 1) == 40.0  # unknown weight type -> EUC_2D: nint(40.11)


def test_nn_fi_bi_match_golden(oracle, instances, goldens):
    for nm, (xy, wt) in instances.items():
        g = goldens["instances"][nm]
        succ, cost = oracle.nn_tour(xy, wt, 0)
        assert cost == g["nn_cost"] and sha(succ) == g["nn_sha256"], nm
        if g["n"] > 700:
            continue
        fs, fc, fst, _ = oracle.two_opt_fi(xy, wt, succ, cost)
        assert fc == g["fi_cost"] and sha(fs) == g["fi_sha256"], nm
        assert (fst.moves, fst.passes, fst.evals) == (g["fi_moves"], g["fi_sweeps"], g["fi_evals"]), nm
        if nm in SMALL and "bi_cost" in g:
            bs, bc, bst, _ = oracle.two_opt_bi(xy, wt, succ)
            assert bc == g["bi_cost"] and sha(bs) == g["bi_sha256"], nm
            assert (bst.moves, bst.evals) == (g["bi_moves"], g["bi_evals"]), nm


def test_reference_csv_goldens(oracle, instances, goldens):
    """results/constructive_heuristics_new.csv GREEDY and ..._2opt_new.csv 2OPT_GREEDY (18 instances)."""
    csvg = goldens["reference_csv"]
    assert len(csvg) == 18
    for nm in ["lin318", "rd400", "pcb442", "att532", "ali535", "gr431", "u574"]:
        xy, wt = instances[nm]
        succ, cost = oracle.nn_tour(xy, wt, 0)
        assert cost == csvg[nm]["GREEDY"], nm
        _, fc, _, _ = oracle.two_opt_fi(xy, wt, succ, cost)
        assert fc == csvg[nm]["2OPT_GREEDY"], nm


def test_berlin52_move_logs(oracle, instances, goldens):
    xy, wt = instances["berlin52"]
    succ, cost = oracle.nn_tour(xy, wt, 0)
    assert cost == 8980
    bs, bc, bst, blog = oracle.two_opt_bi(xy, wt, succ, log_cap=100)
    assert bc == 7842 and bst.moves == 11 and bst.evals == 15288
    assert blog.tolist() == goldens["instances"]["berlin52"]["bi_log"]
    assert blog[:3].tolist() == [[10, 50, -257], [28, 45, -267], [0, 20, -231]]  # SURVEY.md §8(c)
    fs, fc, fst, flog = oracle.two_opt_fi(xy, wt, succ, cost, log_cap=100)
    assert fc == 8083 and fst.moves == 20 and fst.passes == 5 and fst.evals == 6380
    assert flog.tolist() == goldens["instances"]["berlin52"]["fi_log"]
    assert is_tour(bs) and is_tour(fs)


def test_oracle_equals_compiled_reference(oracle, instances, goldens, reference_outputs, reflib_if_built):
    """the reference's matrix, NN, FI and BI results (goldens.json) and the prev[] alg_2opt_tabu exports (tabusearch.c:173-175)"""
    for nm in ["berlin52", "att48", "ulysses22", "pr299", "gr96"]:
        xy, wt = instances[nm]
        g = goldens["instances"][nm]
        assert sha(oracle.dist_matrix(xy, wt)) == g["matrix_sha256"], nm
        s1, c1 = oracle.nn_tour(xy, wt, 0)
        assert sha(s1) == g["nn_sha256"] and c1 == g["nn_cost"], nm
        f1 = oracle.two_opt_fi(xy, wt, s1, c1)
        assert sha(f1[0]) == g["fi_sha256"] and f1[1] == g["fi_cost"], nm
        b1 = oracle.two_opt_bi(xy, wt, s1, want_prev=True)
        assert sha(b1[0]) == g["bi_sha256"] and b1[1] == g["bi_cost"], nm
        assert sha(b1[4]) == reference_outputs["bi_prev_sha256"][nm], nm
        if reflib_if_built:
            ref = reflib_if_built
            assert (oracle.dist_matrix(xy, wt) == ref.dist_matrix(xy, wt)).all()
            b2 = ref.two_opt_bi(xy, wt, s1, want_prev=True)
            assert (b1[0] == b2[0]).all() and b1[1] == b2[1] and (b1[4] == b2[2]).all()


def test_oracle_equals_reference_on_random_tours_and_coords(oracle, reference_outputs, reflib_if_built):
    from golden.make_reference_outputs import random_tour_cases
    cases = list(random_tour_cases())
    assert len(cases) == len(reference_outputs["random_tours"]) == 4
    for (wt, xy, succ), r in zip(cases, reference_outputs["random_tours"]):
        assert (wt, len(xy)) == (r["wt"], r["n"])
        c = oracle.succ_cost(xy, wt, succ)
        f1 = oracle.two_opt_fi(xy, wt, succ, c)
        assert sha(f1[0]) == r["fi_sha256"] and f1[1] == r["fi_cost"], wt
        b1 = oracle.two_opt_bi(xy, wt, succ)
        assert sha(b1[0]) == r["bi_sha256"] and b1[1] == r["bi_cost"], wt
        if reflib_if_built:
            f2 = reflib_if_built.two_opt_fi(xy, wt, succ, c)
            b2 = reflib_if_built.two_opt_bi(xy, wt, succ)
            assert (f1[0] == f2[0]).all() and f1[1] == f2[1] and (b1[0] == b2[0]).all() and b1[1] == b2[1]


def test_tabu_mask_restatement(oracle, reference_outputs, reflib_if_built):
    """alg_2opt_tabu with a tabu list: same tour AND same mutated list (lazy expiry, tabusearch.c:83-92)."""
    from golden.make_reference_outputs import tabu_mask_case
    xy, succ, m1 = tabu_mask_case()
    m2 = m1.copy()
    r = reference_outputs["tabu_mask"]
    b1 = oracle.two_opt_bi(xy, 0, succ, skip_edge=m1, iter_=r["iter"], tenure=r["tenure"])
    assert sha(b1[0]) == r["bi_sha256"] and b1[1] == r["bi_cost"]
    assert sha(m1) == r["mask_after_sha256"]
    if reflib_if_built:
        b2 = reflib_if_built.two_opt_bi(xy, 0, succ, skip_edge=m2, iter_=r["iter"], tenure=r["tenure"])
        assert (b1[0] == b2[0]).all() and b1[1] == b2[1] and (m1 == m2).all()


def test_synthetic_known_answers(oracle):
    """SURVEY.md §8(c): uni2000 NN 406727 -> FI 345191 (6 sweeps, 630 moves)."""
    xy = uniform_instance(2000)
    succ, cost = oracle.nn_tour(xy, 0, 0)
    assert cost == 406727
    _, fc, st, _ = oracle.two_opt_fi(xy, 0, succ, cost)
    assert fc == 345191 and st.passes == 6 and st.moves == 630 and st.evals == 11982230


def test_bi_scan_rows_mt_matches_first_move(oracle, instances):
    xy, wt = instances["pr299"]
    succ, _ = oracle.nn_tour(xy, wt, 0)
    ev, sec, key = oracle.bi_scan_rows_mt(xy, wt, succ, 0, 299, 3)
    _, _, st, log = oracle.two_opt_bi(xy, wt, succ, max_passes=1, log_cap=1)
    assert ev == 299 * 296 // 2 == st.evals
    assert [key[1], key[2], key[0]] == log[0].tolist()


def test_csv_goldens_cover_every_deterministic_column(goldens):
    """18 instances x {GREEDY, GREEDY_ITER, EXTR_MILE, 2OPT_GREEDY, 2OPT_GREEDY_ITER, 2OPT_EXTR_MIL}: every cell was re-derived
    with the compiled reference when the fixture was made (tests/golden/make_goldens.py, make_csv_goldens.py)."""
    assert len(goldens["reference_csv"]) == 18
    for nm, row in goldens["reference_csv"].items():
        assert set(row) == {"GREEDY", "GREEDY_ITER", "EXTR_MILE", "2OPT_GREEDY", "2OPT_GREEDY_ITER", "2OPT_EXTR_MIL"}, nm


def test_large_fixture_spot_check(oracle):
    """tests/golden/large.npz / goldens_large.json (decimal and 10^6-range coordinates): the cheap cells re-derived here."""
    import json
    import os
    from conftest import GOLD_DIR
    z = np.load(os.path.join(GOLD_DIR, "large.npz"))
    g = json.load(open(os.path.join(GOLD_DIR, "goldens_large.json")))["instances"]
    assert set(g) == {"fl3795", "pla7397", "usa13509", "stefano_8k"}
    xy, wt = z["fl3795__xy"], int(z["fl3795__wt"])
    succ, cost = oracle.nn_tour(xy, wt, 0)
    assert cost == g["fl3795"]["nn_cost"]
    s, obj, st, log = oracle.two_opt_bi(xy, wt, succ, max_passes=3, log_cap=8)
    assert log.tolist() == g["fl3795"]["bi_log"][:3]


def test_constructive_restatements_equal_reference_and_csv(oracle, instances, goldens, reference_outputs, reflib_if_built):
    """orc_greedy_iter / orc_extra_mileage (reference HEU_Greedy_iter, HEU_extramileage) vs the stored driver results (tour and
    cost), the compiled reference when built, and the published GREEDY_ITER / EXTR_MILE columns."""
    from golden.make_reference_outputs import tiny_extra_mileage_cases
    for nm in ("berlin52", "pr299", "att532", "ulysses22", "gr96", "eil51"):
        xy, wt = instances[nm]
        b, s, c = oracle.greedy_iter(xy, wt)
        r = reference_outputs["greedy_iter"][nm]
        assert c == r["cost"] and sha(s) == r["sha256"], nm
        if reflib_if_built:
            st, rs, rc = reflib_if_built.run_method("HEU_Greedy_iter", xy, wt)
            assert st == 0 and c == rc and (s == rs).all(), nm
        s, c = oracle.extra_mileage(xy, wt)
        r = reference_outputs["extra_mileage"][nm]
        assert c == r["cost"] and sha(s) == r["sha256"], nm
        if reflib_if_built:
            st, rs, rc = reflib_if_built.run_method("HEU_extramileage", xy, wt)
            assert st == 0 and c == rc and (s == rs).all(), nm
        if nm in goldens["reference_csv"]:
            assert c == goldens["reference_csv"][nm]["EXTR_MILE"]
    for n, xy in tiny_extra_mileage_cases():  # ties and coincident nodes
        s, c = oracle.extra_mileage(xy, 0)
        r = reference_outputs["extra_mileage"][f"ties{n}"]
        assert c == r["cost"] and sha(s) == r["sha256"], n
        if reflib_if_built:
            st, rs, rc = reflib_if_built.run_method("HEU_extramileage", xy, 0)
            assert c == rc and (s == rs).all(), n


def test_vns_kick_restatement_equals_the_reference_kick(oracle, reference_outputs, reflib_if_built):
    """oracle.vns_kick (indices handed in) against the reference's own kick() (src/vns.c:11), which draws its three indices
    from glibc random(): the draws are replayed with the restated generator.  Seeds whose largest index is n-1 are skipped —
    there the reference reads one element past its tour array."""
    from golden.make_reference_outputs import vns_kick_indices
    from tsp_optimization_b200.instances import is_tour, uniform_instance
    n = reference_outputs["vns_kick"]["n"]
    xy = uniform_instance(n)
    succ, _ = oracle.nn_tour(xy, 0, 0)
    compared = 0
    for seed in range(1, 40):
        idx = vns_kick_indices(seed, n)
        if max(idx) == n - 1:
            assert str(seed) not in reference_outputs["vns_kick"]["seeds"]
            continue
        r = reference_outputs["vns_kick"]["seeds"][str(seed)]
        s_o, c_o = oracle.vns_kick(xy, 0, succ, *idx)
        assert sha(s_o) == r["sha256"] and c_o == r["cost"] and is_tour(s_o), seed
        if reflib_if_built:
            s_ref, c_ref = reflib_if_built.vns_kick_stock(xy, 0, succ, seed)
            assert (s_ref == s_o).all() and c_ref == c_o, seed
        compared += 1
    assert compared >= 30
