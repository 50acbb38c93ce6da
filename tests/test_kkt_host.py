"""The post-solve KKT assessment (highs_b200/csrc/kkt_logic.hpp + kkt_check.cu) against the reference's own lpKktCheck
(highs/lp_data/HighsSolution.cpp:1043-1327, run through oracle/_ref/ref_driver --kkt-of and recorded in
tests/golden/reference_runs.json): the HOST twin here
(no GPU); the device version is compared with both in tests/test_gpu_kkt.py.  Solutions: the committed goldens (reference
output), loose and converged oracle solutions on instances with every row / bound type, and perturbed solutions so that
every counter is exercised."""
import os

import numpy as np
import pytest

import recorded_reference
from conftest import GOLDEN, case_id, golden_lp, golden_solution, load_golden

FLOAT_FIELDS = ("objective_function_value", "primal_dual_objective_error", "max_primal_infeasibility", "sum_primal_infeasibilities",
                "max_dual_infeasibility", "sum_dual_infeasibilities", "max_relative_primal_infeasibility",
                "max_relative_dual_infeasibility", "max_primal_residual_error", "max_dual_residual_error",
                "max_relative_primal_residual_error", "max_relative_dual_residual_error", "max_complementarity_violation")
INT_FIELDS = ("num_primal_infeasibilities", "num_dual_infeasibilities", "num_complementarity_violations", "primal_solution_status",
              "dual_solution_status")


def compare(ours, ref, exact_counts=True):
    for k in FLOAT_FIELDS:
        a, b = ours[k], ref[k]
        # residual errors are differences of nearly equal numbers: the reference rounds a quad sum, we a double-double sum
        tol = 1e-9 * (1 + abs(b)) if "residual" in k else 1e-12 * (1 + abs(b))
        assert abs(a - b) <= tol, (k, a, b)
    if exact_counts:
        for k in INT_FIELDS:
            assert ours[k] == ref[k], (k, ours[k], ref[k])
    assert ours["model_status"] == ref["model_status_code"], (ours["model_status"], ref["model_status"])


CASES = [c for c in load_golden() if c["model_status_code"] in (7, 14, 15) and golden_solution(c) is not None][:24]


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_host_twin_matches_reference_on_goldens(engine_lib, case):
    from highs_b200 import engine
    lp, sol = golden_lp(case), golden_solution(case)
    tol = case["options"].get("kkt_tolerance", 0.0)
    status_in = 7 if case["model_status_code"] in (7, 15) else case["model_status_code"]
    ref = recorded_reference.reference_kkt(lp, sol, model_status_code=status_in, options=case["options"])
    ours = engine.kkt_check(lp, sol, kkt_tolerance=tol, model_status=status_in, on_device=False)
    compare(ours, ref)


@pytest.mark.parametrize("name", ["afiro", "adlittle", "e226", "boeing2", "capri", "standata", "sc105", "share2b", "stair", "scrs8"])
@pytest.mark.parametrize("tol", [1e-3, 1e-6])
def test_host_twin_matches_reference_on_instances(engine_lib, oracle, name, tol):
    from highs_b200 import engine
    from highs_b200.lp import read_b2lp
    path = os.path.join(GOLDEN, "instances", name + ".b2lp")
    if not os.path.exists(path):
        pytest.skip("instance fixture missing")
    lp = read_b2lp(path)
    sol = oracle.solve(lp, tol_primal=tol, tol_dual=tol, tol_gap=tol, iter_limit=30000)
    for status_in, kt in ((7, tol), (15, tol), (7, 0.0)):
        opts = {"kkt_tolerance": kt} if kt else {}
        ref = recorded_reference.reference_kkt(lp, sol, model_status_code=status_in, options=opts)
        ours = engine.kkt_check(lp, sol, kkt_tolerance=kt, model_status=status_in, on_device=False)
        compare(ours, ref)
    # a damaged solution: bound violations, wrong-sign duals, inconsistent activities
    rng = np.random.default_rng(1)
    bad = {k: v.copy() for k, v in sol.items() if isinstance(v, np.ndarray)}
    bad["col_value"] += 1e-2 * rng.standard_normal(lp.num_col_)
    bad["row_dual"] += 1e-2 * rng.standard_normal(lp.num_row_)
    bad["col_dual"] += 1e-3 * rng.standard_normal(lp.num_col_)
    ref = recorded_reference.reference_kkt(lp, bad, model_status_code=7)
    ours = engine.kkt_check(lp, bad, model_status=7, on_device=False)
    compare(ours, ref)
    assert ours["model_status"] == 15 and ours["num_primal_infeasibilities"] > 0
