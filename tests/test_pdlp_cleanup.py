"""SURVEY.md 8(f) rank 3: presolve / postsolve interplay and the PDLP clean-up after postsolve.

highs_b200/csrc/highs_pdlp_cleanup.hpp restates -- through HiGHS's public API -- the clean-up flow the reference has compiled
out (/root/reference/highs/lp_data/Highs.cpp:1940-1982, `consider_pdlp_cleanup = false`; decision rule
Highs::tryPdlpCleanup, highs/lp_data/HighsInterface.cpp:4210-4272).  The helper is solver-agnostic, so its logic is checked
HERE on the CPU against the unmodified reference library (oracle/_ref/ref_driver --pdlp-cleanup, its results recorded in
tests/golden/reference_runs.json); tests/test_gpu_dropin.py repeats the flow with the B200 engine behind solver=pdlp."""
import os

import pytest

from conftest import GOLDEN


def _lp(name):
    from highs_b200.lp import read_b2lp
    return read_b2lp(os.path.join(GOLDEN, "instances", name + ".b2lp"))


@pytest.fixture(scope="module")
def ref():
    import recorded_reference
    return recorded_reference


OPTS = {"presolve": "choose", "kkt_tolerance": 1e-4}


def test_postsolve_can_leave_unknown_and_reference_margin_rejects(ref):
    """standata at kkt 1e-4: PDLP converges on the presolved LP, postsolve magnifies the primal infeasibility to 102x the
    tolerance, lpKktCheck reports kUnknown -- and the reference's own margin (100x) then declines the clean-up"""
    lp = _lp("standata")
    plain = ref.run_reference(lp=lp, options=OPTS)
    assert plain["model_status"] == "Unknown" and plain["cleanup_considered"] == 0
    r = ref.run_reference(lp=lp, options=OPTS, pdlp_cleanup=1e2)
    assert r["cleanup_considered"] == 1 and r["cleanup_attempted"] == 0
    assert r["cleanup_first_status_code"] == 15 and r["cleanup_first_pdlp_iterations"] == plain["pdlp_iteration_count"]
    assert r["cleanup_max_relative_violation"] == pytest.approx(plain["max_relative_primal_infeasibility"] / 1e-4, rel=1e-12)
    assert r["model_status"] == "Unknown" and r["objective_function_value"] == plain["objective_function_value"]


def test_cleanup_flow_reference_tolerance_stops_at_once(ref):
    """wider margin, reference tolerance: the hot-started solve of the ORIGINAL LP runs (iteration limit max(10000, 10 %))
    but cuPDLP-C's own criteria are already met by the postsolved point -- 0 iterations, still kUnknown"""
    r = ref.run_reference(lp=_lp("standata"), options=OPTS, pdlp_cleanup=1e3)
    assert r["cleanup_attempted"] == 1 and r["cleanup_iteration_limit"] == 10000
    assert r["pdlp_iteration_count"] == 0 and r["model_status"] == "Unknown"


@pytest.mark.parametrize("name", ["standata", "standgub"])
def test_cleanup_flow_tightened_reaches_optimal(ref, name):
    """with the clean-up tolerance tightened 10x the same flow ends kOptimal with the violation back under 100x"""
    lp = _lp(name)
    r = ref.run_reference(lp=lp, options=OPTS, pdlp_cleanup=1e3, cleanup_tighten=0.1)
    assert r["cleanup_attempted"] == 1 and r["model_status"] == "Optimal"
    assert 0 < r["pdlp_iteration_count"] <= 10000
    assert r["max_relative_primal_infeasibility"] < 100 * 1e-4
    exact = ref.run_reference(lp=lp, options={"solver": "simplex", "presolve": "choose"})
    assert abs(r["objective_function_value"] - exact["objective_function_value"]) <= 2e-3 * (1 + abs(exact["objective_function_value"]))


def test_no_cleanup_when_first_run_is_conclusive(ref):
    r = ref.run_reference(lp=_lp("afiro"), options={"presolve": "choose"}, pdlp_cleanup=1e3, cleanup_tighten=0.1)
    assert r["model_status"] == "Optimal" and r["cleanup_considered"] == 0 and r["cleanup_attempted"] == 0
