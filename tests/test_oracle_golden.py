"""Pins the oracle (oracle/pdlp_oracle.c) against the reference's own goldens:
tests/golden/ was produced by the UNMODIFIED reference (oracle/_ref, HiGHS 1.15.1 CPU pdlp) through
Highs::run() -- iteration counts, objectives, statuses (check/TestPdlp.cpp:11-64,186-239;
check/CMakeLists.txt:321-335) and full HighsSolution vectors.  The oracle must reproduce them bit for bit."""
import numpy as np
import pytest

import recorded_reference
from conftest import (case_id, golden_lp, golden_solution, load_golden, options_to_params,
                      term_to_model_status)

CASES = load_golden()


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_oracle_reproduces_reference(oracle, case):
    lp = golden_lp(case)
    params = options_to_params(case["options"])
    warm = None
    if case["warm_from"]:
        import os
        from conftest import GOLDEN
        first = dict(np.load(os.path.join(GOLDEN, case["warm_from"])))
        warm = (first["col_value"], first["row_value"], first["row_dual"])
    res = oracle.solve(lp, warm=warm, **params)
    assert res["iters"] == case["pdlp_iteration_count"]
    status = term_to_model_status(res["term_code"], res["iters"], params.get("iter_limit", 2147483647))
    if case["model_status_code"] == 10:
        assert status == 9   # lpKktCheck upgrades kUnboundedOrInfeasible -> kUnbounded (HighsSolution.cpp:1074-1077)
    else:
        assert status == case["model_status_code"]
    if case["model_status_code"] in (7, 14):
        assert lp.objectiveValue(res["col_value"]) == pytest.approx(case["objective_function_value"], rel=1e-14, abs=1e-14)
    gold = golden_solution(case)
    if gold is not None:
        for k in ("col_value", "col_dual", "row_value", "row_dual"):
            assert np.array_equal(res[k], gold[k]), k


def test_reference_goldens_of_its_own_tests():
    """the numbers the reference's tests assert (check/TestPdlp.cpp:29,44,53-61; check/CMakeLists.txt:325)"""
    by = {(c["name"], c["tag"]): c for c in CASES}
    d = by[("distillation", "kkt1e-4")]
    assert d["pdlp_iteration_count"] == 160 and abs(d["objective_function_value"] - 31.2) < 1e-3
    l = by[("distillation", "limit80")]
    assert l["pdlp_iteration_count"] == 79 and l["model_status"] == "Iteration limit reached"
    assert by[("infeasible", "kkt1e-4")]["model_status_code"] == 9
    assert by[("unbounded", "kkt1e-4")]["model_status_code"] == 10
    assert f"{by[('avgas', 'default')]['objective_function_value']:.10e}".startswith("-7.7499999")
    assert abs(by[("boxed_row", "kkt1e-4")]["objective_function_value"] + 16) < 1e-3
    assert abs(by[("threed", "kkt1e-4")]["objective_function_value"] - 7) < 1e-3


def test_oracle_vs_live_reference(oracle):
    """fresh random LPs (equality, ranged, free rows, bounded columns, maximise) against oracle/_ref (its runs recorded in
    tests/golden/reference_runs.json)"""
    from highs_b200.lp import HighsLp, HighsSparseMatrix
    import scipy.sparse as sp
    rng = np.random.default_rng(42)
    for trial in range(4):
        m, n = int(rng.integers(8, 40)), int(rng.integers(8, 40))
        A = sp.random(m, n, density=0.3, random_state=int(rng.integers(1 << 30)), data_rvs=rng.standard_normal).tocsc()
        x0 = rng.random(n)
        ax = A @ x0
        kind = rng.integers(0, 5, size=m)
        rl = np.where(kind == 0, ax, np.where(kind == 1, ax - rng.random(m), np.where(kind == 2, -np.inf, np.where(kind == 3, ax - 1, -np.inf))))
        ru = np.where(kind == 0, ax, np.where(kind == 1, np.inf, np.where(kind == 2, ax + rng.random(m), np.where(kind == 3, ax + 1, np.inf))))
        lo = np.where(rng.random(n) < 0.8, 0.0, -np.inf)
        up = np.where(rng.random(n) < 0.3, 2.0, np.inf)
        lp = HighsLp(n, m, rng.standard_normal(n) + (1.0 if trial % 2 == 0 else 0.0), lo, up, rl, ru,
                     HighsSparseMatrix(n, m, A.indptr, A.indices, A.data), -1 if trial == 3 else 1, 0.5)
        opts = {"kkt_tolerance": 1e-4, "pdlp_iteration_limit": 20000}
        ref = recorded_reference.run_reference(lp, options=opts, want_solution=True)
        res = oracle.solve(lp, tol_primal=1e-4, tol_dual=1e-4, tol_gap=1e-4, iter_limit=20000)
        assert res["iters"] == ref["pdlp_iteration_count"]
        for k in ("col_value", "col_dual", "row_value", "row_dual"):
            assert recorded_reference.digest(res[k]) == ref[k], (trial, k)


@pytest.mark.parametrize("name", ["avgas", "afiro", "adlittle", "sctest", "chip", "boxed_row", "restart_lp"])
def test_row_side_interaction_is_equivalent(oracle, name):
    """The multi-GPU engine takes the step rule's interaction on the row side, (Ax-Ax').(y-y'), instead of the
    reference's (x-x').(A'y-A'y') -- the same number in exact arithmetic (cupdlp_step.c:259-264 computes it as
    dInteractiony).  On the CPU oracle: same termination, and the optimum agrees to the solver tolerance."""
    import os
    from conftest import GOLDEN
    from highs_b200.lp import read_b2lp
    lp = read_b2lp(os.path.join(GOLDEN, name + ".b2lp"))
    a = oracle.solve(lp)
    b = oracle.solve(lp, interaction_row_side=1)
    assert a["term_code"] == b["term_code"] == 0
    oa, ob_ = lp.objectiveValue(a["col_value"]), lp.objectiveValue(b["col_value"])
    assert abs(oa - ob_) <= 1e-6 * (1 + abs(oa))
    # rounding noise in the interaction is amplified by cancellation, so restarts can land on different checks
    assert 0.5 * a["iters"] <= b["iters"] <= 2 * a["iters"]


@pytest.mark.parametrize("name", ["80bau3b", "greenbea", "25fv47"])
def test_summation_order_sensitivity(oracle, name):
    """How far does a MERE change of summation order move a trajectory?  The oracle against itself, long sums added in blocks
    of 256 (orc_set_sum_block -- a test switch, not the reference's behaviour): after 120 iterations the iterates agree to
    1e-6 (in fact ~1e-8), after 400 they differ by more than 1e-6 on these instances.  This is why the GPU engine's
    tree-mode parity on large instances is asserted after 120 iterations (tests/test_gpu_instances.py) and at convergence
    (objective / KKT measures), not as a 400-iteration trajectory."""
    import os
    import numpy as np
    from conftest import GOLDEN
    from highs_b200.lp import read_b2lp
    lp = read_b2lp(os.path.join(GOLDEN, "instances", name + ".b2lp"))
    L = oracle.lib()
    try:
        rel = {}
        for lim in (120, 400):
            L.orc_set_sum_block(0)
            ref = oracle.solve(lp, iter_limit=lim)
            L.orc_set_sum_block(256)
            alt = oracle.solve(lp, iter_limit=lim)
            assert alt["iters"] == ref["iters"] and alt["term_code"] == ref["term_code"]
            rel[lim] = max(float(np.abs(alt[k] - ref[k]).max() / (1 + np.abs(ref[k]).max())) for k in ("col_value", "row_dual"))
    finally:
        L.orc_set_sum_block(0)
    assert rel[120] <= 1e-6, rel
    assert rel[400] > 1e-6, rel
