"""Host-side logic that needs neither GPU nor CUDA: option mapping of the wrapper mirror, LP interchange,
the synthetic workload generator, reproducibility of the goldens."""
import os

import numpy as np
import pytest

import recorded_reference
from conftest import GOLDEN, golden_lp, load_golden


def test_option_mapping_matches_wrapper():
    """getUserParamsFromOptions, CupdlpWrapper.cpp:642-717"""
    from highs_b200 import pdlp
    o = pdlp.HighsOptions()
    p = pdlp.getUserParamsFromOptions(o, pdlp.HighsTimer())
    assert p == dict(iter_limit=2147483647, log_level=0, scaling=1, adaptive_step=1, tol_primal=1e-7, tol_dual=1e-7,
                     tol_gap=1e-7, time_limit=-1.0, restart=1)   # no limit: < 0 (0 would end the run at the first check)
    o = pdlp.HighsOptions(kkt_tolerance=1e-4, primal_feasibility_tolerance=1e-9, pdlp_iteration_limit=80,
                          pdlp_features_off=pdlp.kPdlpScalingOff | pdlp.kPdlpAdaptiveStepSizeOff, time_limit=12.5,
                          output_flag=True, log_dev_level=1)
    p = pdlp.getUserParamsFromOptions(o, pdlp.HighsTimer())
    assert (p["tol_primal"], p["tol_dual"], p["tol_gap"]) == (1e-4, 1e-4, 1e-4)     # kkt_tolerance overrides all three (:683-696)
    assert p["iter_limit"] == 80 and p["scaling"] == 0 and p["adaptive_step"] == 0 and p["restart"] == 1
    assert p["time_limit"] == 12.5 and p["log_level"] == 2
    assert pdlp.getUserParamsFromOptions(pdlp.HighsOptions(pdlp_cupdlpc_restart_method=0), pdlp.HighsTimer())["restart"] == 0
    assert pdlp.getUserParamsFromOptions(pdlp.HighsOptions(pdlp_features_off=pdlp.kPdlpRestartOff), pdlp.HighsTimer())["restart"] == 0


def test_model_status_numbering():
    """HighsModelStatus values are part of the ABI (HConst.h:201-228)"""
    from highs_b200.pdlp import HighsModelStatus as S
    assert (S.kOptimal, S.kInfeasible, S.kUnboundedOrInfeasible, S.kUnbounded, S.kTimeLimit, S.kIterationLimit, S.kUnknown,
            S.kSolveError) == (7, 8, 9, 10, 13, 14, 15, 4)


def test_b2lp_roundtrip(tmp_path):
    from highs_b200.lp import read_b2lp, synthetic_lp, write_b2lp
    lp = synthetic_lp(300, 200, 5, seed=9, dense_col_nnz=100)
    lp.sense_, lp.offset_ = -1, 3.5
    path = str(tmp_path / "x.b2lp")
    write_b2lp(path, lp)
    back = read_b2lp(path)
    assert (back.num_col_, back.num_row_, back.sense_, back.offset_) == (200, 300, -1, 3.5)
    for a, b in [(lp.col_cost_, back.col_cost_), (lp.col_upper_, back.col_upper_), (lp.row_lower_, back.row_lower_),
                 (lp.a_matrix_.start_, back.a_matrix_.start_), (lp.a_matrix_.index_, back.a_matrix_.index_),
                 (lp.a_matrix_.value_, back.a_matrix_.value_)]:
        assert np.array_equal(a, b)


def test_synthetic_generator_properties():
    """SURVEY.md 8(d): GEQ rows only, x >= 0, sorted de-duplicated columns, planted optimal pair"""
    from highs_b200.lp import synthetic_lp
    a, b = synthetic_lp(4000, 3000, 8, seed=12345), synthetic_lp(4000, 3000, 8, seed=12345)
    assert np.array_equal(a.a_matrix_.value_, b.a_matrix_.value_) and np.array_equal(a.col_cost_, b.col_cost_)   # deterministic
    A = a.a_matrix_
    assert np.all(np.isinf(a.row_upper_)) and np.all(a.col_lower_ == 0) and np.all(np.isinf(a.col_upper_))
    for j in range(0, 3000, 137):
        idx = A.index_[A.start_[j]:A.start_[j + 1]]
        assert np.all(np.diff(idx) > 0) and len(idx) <= 8
    assert 0.99 * 8 * 3000 <= A.numNz() <= 8 * 3000
    d = synthetic_lp(4000, 3000, 8, seed=1, dense_col_nnz=2000)
    assert d.a_matrix_.start_[1] - d.a_matrix_.start_[0] == 2000


def test_golden_fixture_inventory():
    cases = load_golden()
    assert len(cases) >= 35
    for c in cases:
        if "synthetic" not in c:
            assert os.path.exists(os.path.join(GOLDEN, c["name"] + ".b2lp"))
    lp = golden_lp([c for c in cases if c["name"] == "avgas"][0])
    assert (lp.num_col_, lp.num_row_, lp.a_matrix_.numNz()) == (8, 10, 30)     # check/Avgas, BASELINE config 1


def test_goldens_reproduce_from_reference():
    """the unmodified reference's runs of two committed cases (recorded in tests/golden/reference_runs.json): tests/golden/golden.json
    is what it prints"""
    for c in load_golden():
        if (c["name"], c["tag"]) in (("avgas", "default"), ("distillation", "kkt1e-4")):
            ref = recorded_reference.run_reference(golden_lp(c), options=c["options"])
            assert ref["pdlp_iteration_count"] == c["pdlp_iteration_count"]
            assert ref["objective_function_value"] == c["objective_function_value"]
            assert ref["model_status_code"] == c["model_status_code"]


def test_reference_kkt_evaluator():
    """ref_driver --kkt-of = the reference's lpKktCheck on a GIVEN solution: fed the golden solution it must return the
    golden HighsInfo (this is the yard-stick the GPU parity tests use for 'KKT residuals')"""
    from conftest import golden_solution
    c = [c for c in load_golden() if (c["name"], c["tag"]) == ("afiro", "default")][0]
    kkt = recorded_reference.reference_kkt(golden_lp(c), golden_solution(c), c["model_status_code"], c["options"])
    for k in ("max_primal_infeasibility", "max_dual_infeasibility", "primal_dual_objective_error",
              "max_complementarity_violation", "objective_function_value"):
        assert kkt[k] == c[k], k
    assert kkt["model_status_code"] == 7
