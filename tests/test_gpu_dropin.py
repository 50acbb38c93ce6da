"""BASELINE config 1 through the real drop-in: the reference's own Highs::run() -> solveLp() with
highs_b200/csrc/highs_shim.cpp linked in place of pdlp/CupdlpWrapper.cpp (oracle/_ref/ref_driver_b200,
built by `python oracle/build_ref.py --shim`).  Everything around the boundary -- option handling,
HighsLpSolverObject, lpKktCheck, HighsInfo -- is the reference's unmodified code."""
import numpy as np
import pytest

import recorded_reference
from conftest import case_id, golden_lp, golden_solution, load_golden

pytestmark = pytest.mark.gpu
CASES = [c for c in load_golden() if c["warm_from"] is None and "synthetic" not in c
         and c["name"] in ("avgas", "afiro", "distillation", "boxed_row", "infeasible", "unbounded", "threed", "restart_lp")]


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_highs_run_with_b200_shim(oracle, case):
    if not oracle.dropin_available():
        pytest.skip("oracle/_ref/ref_driver_b200 not built")
    lp = golden_lp(case)
    res = oracle.run_reference(lp=lp, options=case["options"], want_solution=True, driver=oracle.DROPIN_DRIVER)
    assert res["model_status_code"] == case["model_status_code"], (res["model_status"], case["model_status"])
    assert res["pdlp_iteration_count"] == case["pdlp_iteration_count"]
    if case["model_status_code"] in (7, 14):
        assert res["objective_function_value"] == pytest.approx(case["objective_function_value"], rel=1e-12, abs=1e-12)
        for fld in ("max_primal_infeasibility", "max_dual_infeasibility", "primal_dual_objective_error",
                    "max_complementarity_violation"):
            assert res[fld] == pytest.approx(case[fld], rel=1e-9, abs=1e-15), fld
        gold = golden_solution(case)
        for k in ("col_value", "col_dual", "row_value", "row_dual"):
            assert np.array_equal(res[k], gold[k]), k


# ---- SURVEY.md 8(f) rank 3: the boundary sits BELOW presolve -- with presolve=choose HiGHS hands the REDUCED LP to the
# drop-in and postsolves what it returns (Highs.cpp:1554-1694, :1802-1931); then the clean-up flow of
# highs_b200/csrc/highs_pdlp_cleanup.hpp (logic checked on the CPU in tests/test_pdlp_cleanup.py) with the engine behind it
PRESOLVE_INSTANCES = ["afiro", "adlittle", "avgas", "blending", "chip", "e226", "etamacro", "standata", "scrs8", "sctest", "stair"]


@pytest.mark.parametrize("name", PRESOLVE_INSTANCES)
def test_presolved_lp_through_the_shim(oracle, name):
    """same Highs::run() with presolve on, reference CPU pdlp vs the B200 shim: the presolved LP is small (ordered mode), so
    status, iteration count and objective agree exactly"""
    import os
    from conftest import GOLDEN
    from highs_b200.lp import read_b2lp
    if not oracle.dropin_available():
        pytest.skip("oracle/_ref/ref_driver_b200 not built")
    path = os.path.join(GOLDEN, "instances", name + ".b2lp")
    if not os.path.exists(path):
        pytest.skip("instance fixture missing")
    lp = read_b2lp(path)
    opts = {"presolve": "choose", "pdlp_iteration_limit": 20000}
    ref = recorded_reference.run_reference(lp, options=opts)
    got = oracle.run_reference(lp=lp, options=opts, driver=oracle.DROPIN_DRIVER)
    assert got["model_status_code"] == ref["model_status_code"], (got["model_status"], ref["model_status"])
    assert got["pdlp_iteration_count"] == ref["pdlp_iteration_count"]
    assert got["objective_function_value"] == pytest.approx(ref["objective_function_value"], rel=1e-12, abs=1e-12)


def test_pdlp_cleanup_with_the_engine(oracle):
    """postsolve leaves kUnknown (standata, kkt 1e-4); the clean-up solve of the ORIGINAL LP runs on the GPU from the
    postsolved solution and ends kOptimal -- same decisions as with the reference's CPU solver behind the same flow"""
    import os
    from conftest import GOLDEN
    from highs_b200.lp import read_b2lp
    if not oracle.dropin_available():
        pytest.skip("oracle/_ref/ref_driver_b200 not built")
    lp = read_b2lp(os.path.join(GOLDEN, "instances", "standata.b2lp"))
    opts = {"presolve": "choose", "kkt_tolerance": 1e-4}
    ref = recorded_reference.run_reference(lp, options=opts, pdlp_cleanup=1e3, cleanup_tighten=0.1)
    got = oracle.run_reference(lp=lp, options=opts, pdlp_cleanup=1e3, cleanup_tighten=0.1, driver=oracle.DROPIN_DRIVER)
    for k in ("cleanup_considered", "cleanup_attempted", "cleanup_iteration_limit", "cleanup_first_status_code",
              "cleanup_first_pdlp_iterations", "model_status_code", "pdlp_iteration_count"):
        assert got[k] == ref[k], k
    assert got["model_status"] == "Optimal"
    assert got["objective_function_value"] == pytest.approx(ref["objective_function_value"], rel=1e-12, abs=1e-12)


# ---- solver=hipdlp through its own shim (highs_b200/csrc/highs_shim_hipdlp.cpp replaces pdlp/HiPdlpWrapper.cpp,
# HighsSolve.cpp:107-117 dispatches to it): the reference's unmodified Highs::run() with the engine's HiPDLP mode behind it
@pytest.mark.parametrize("name", ["afiro", "adlittle", "avgas", "blending", "chip", "sctest", "e226", "stair"])
def test_highs_run_hipdlp_through_the_shim(oracle, name):
    """same Highs::run(), solver=hipdlp: the reference's CPU HiPDLP vs the drop-in library -- status, iteration count and
    objective (the device mode adds the check sums in the reference's order up to 4096 rows/columns: bit-equal)"""
    import os
    from conftest import GOLDEN
    from highs_b200.lp import read_b2lp
    drv = os.path.join(os.path.dirname(oracle.DROPIN_DRIVER), "ref_driver_b200_hipdlp")
    if not os.path.exists(drv):
        pytest.skip("oracle/_ref/ref_driver_b200_hipdlp not built")
    path = os.path.join(GOLDEN, "instances", name + ".b2lp")
    if not os.path.exists(path):
        pytest.skip("instance fixture missing")
    lp = read_b2lp(path)
    opts = {"solver": "hipdlp", "presolve": "off", "pdlp_iteration_limit": 8000}
    ref = recorded_reference.run_reference(lp, options=opts)
    got = oracle.run_reference(lp=lp, options=opts, driver=drv)
    assert got["model_status_code"] == ref["model_status_code"], (got["model_status"], ref["model_status"])
    assert got["pdlp_iteration_count"] == ref["pdlp_iteration_count"]
    assert got["objective_function_value"] == pytest.approx(ref["objective_function_value"], rel=1e-12, abs=1e-12)
