"""The drop-in boundary, end to end: the reference's drivers (HEU_2opt_greedy = `-method 2OPT_GREEDY`, src/heuristics.c:572;
HEU_2opt_extramileage :596; HEU_2opt_greedy_iter :584; HEU_greedy :160) calling the product's calc_dist / alg_2opt /
alg_2opt_tabu / reverse_path / greedy / HEU_Greedy_iter / HEU_extramileage (csrc/dropin.cpp -> libtspb200.so -> CUDA) must
produce the reference's tour and objective (tests/golden/goldens.json; reference_outputs.json, provenance in its "source";
the compiled reference itself when oracle/_ref is built) and its published CSV values.
The drivers are the UNMODIFIED reference objects linked by the INTEGRATION.md §2 recipe when oracle/_ref is built from a
reference checkout, else their restatement oracle/dropin_callers.c linked against libtspb200_dropin.so."""
import hashlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.int32).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def gpulib():
    from oracle.oracle import REF_GPU_SO, DropinCallers, RefLib
    return RefLib(gpu_link=True) if os.path.exists(REF_GPU_SO) else DropinCallers()


def test_strong_symbols_come_from_the_dropin(gpulib):
    # tspb200_dropin_layout only exists in csrc/dropin.cpp: its presence next to the reference's HEU_* drivers shows
    # which definitions the link picked
    assert hasattr(gpulib.L, "tspb200_dropin_layout") and hasattr(gpulib.L, "HEU_2opt_greedy")
    # the drop-in's definitions are laid out contiguously (one object file): the weakened reference symbols greedy,
    # HEU_Greedy_iter and HEU_extramileage must resolve into that range, HEU_2opt_greedy (the caller's code) must not
    import ctypes as C
    addr = lambda nm: C.cast(getattr(gpulib.L, nm), C.c_void_p).value
    lo = min(addr(nm) for nm in ("alg_2opt", "calc_dist", "reverse_path", "tspb200_dropin_layout"))
    hi = max(addr(nm) for nm in ("alg_2opt", "calc_dist", "reverse_path", "tspb200_dropin_layout", "tspb200_dropin_reset"))
    for nm in ("greedy", "HEU_Greedy_iter", "HEU_extramileage", "alg_2opt_tabu"):
        assert lo - 4096 <= addr(nm) <= hi + 4096, nm
    assert not (lo - 4096 <= addr("HEU_2opt_greedy") <= hi + 4096)


@pytest.mark.parametrize("nm", ["berlin52", "pr299", "att532", "gr666", "dsj1000", "pr1002", "ulysses22"])
def test_reference_2opt_greedy_on_cuda_path(gpulib, instances, goldens, nm):
    xy, wt = instances[nm]
    st_g, succ_g, obj_g = gpulib.run_method("HEU_2opt_greedy", xy, wt)
    g = goldens["instances"][nm]  # the reference's alg_2opt from its greedy(inst, 0) tour
    assert st_g == 0
    assert sha(succ_g) == g["fi_sha256"] and obj_g == g["fi_cost"]
    csv = goldens["reference_csv"].get(nm)  # results/constructive_heuristics_2opt_new.csv, column 2OPT_GREEDY
    if csv:
        assert obj_g == csv["2OPT_GREEDY"]


@pytest.mark.parametrize("method,nm", [("HEU_2opt_extramileage", "lin318"), ("HEU_2opt_extramileage", "att532"),
                                       ("HEU_2opt_greedy_iter", "berlin52"), ("HEU_greedy", "gr666"),
                                       ("HEU_extramileage", "pr299"), ("HEU_2opt_greedy_iter", "gr431"),
                                       ("HEU_Greedy_iter", "dsj1000"), ("HEU_extramileage", "gr666"),
                                       ("HEU_2opt_extramileage", "dsj1000")])
def test_other_reference_drivers_on_cuda_path(gpulib, reflib_if_built, instances, reference_outputs, method, nm):
    xy, wt = instances[nm]
    st_g, succ_g, obj_g = gpulib.run_method(method, xy, wt)
    r = reference_outputs["drivers"][f"{method}:{nm}"]
    assert st_g == 0
    assert sha(succ_g) == r["sha256"] and obj_g == r["cost"]
    if reflib_if_built:
        st_r, succ_r, obj_r = reflib_if_built.run_method(method, xy, wt)
        assert st_r == 0 and (succ_g == succ_r).all() and obj_g == obj_r


def test_reference_plain_bi_through_dropin(gpulib, reflib_if_built, oracle, instances, goldens, reference_outputs):
    """alg_2opt_tabu(inst, NULL, prev, 1, 1) incl. the exported prev[] (src/tabusearch.c:173-175)."""
    xy, wt = instances["pr299"]
    g = goldens["instances"]["pr299"]
    succ0, _ = oracle.nn_tour(xy, wt, 0)
    assert sha(succ0) == g["nn_sha256"]
    s_g, o_g, p_g = gpulib.two_opt_bi(xy, wt, succ0, want_prev=True)
    assert sha(s_g) == g["bi_sha256"] and o_g == g["bi_cost"] and sha(p_g) == reference_outputs["bi_prev_sha256"]["pr299"]
    if reflib_if_built:
        s_r, o_r, p_r = reflib_if_built.two_opt_bi(xy, wt, succ0, want_prev=True)
        assert (s_g == s_r).all() and o_g == o_r and (p_g == p_r).all()


def test_reference_masked_bi_through_dropin(gpulib, reflib_if_built, oracle, instances, goldens, reference_outputs):
    """alg_2opt_tabu WITH a tabu list through the reference-named symbol: same tour, cost and mutated list."""
    from golden.make_reference_outputs import masked_bi_case
    xy, wt = instances["berlin52"]
    succ0, _ = oracle.nn_tour(xy, wt, 0)
    assert sha(succ0) == goldens["instances"]["berlin52"]["nn_sha256"]
    m_g = masked_bi_case(xy)
    m_r = m_g.copy()
    r = reference_outputs["masked_bi_berlin52"]
    s_g, o_g = gpulib.two_opt_bi(xy, wt, succ0, skip_edge=m_g, iter_=r["iter"], tenure=r["tenure"])
    assert sha(s_g) == r["bi_sha256"] and o_g == r["bi_cost"] and sha(m_g) == r["mask_after_sha256"]
    if reflib_if_built:
        s_r, o_r = reflib_if_built.two_opt_bi(xy, wt, succ0, skip_edge=m_r, iter_=r["iter"], tenure=r["tenure"])
        assert (s_g == s_r).all() and o_g == o_r and (m_g == m_r).all()
