"""Pins the HiPDLP restatement (oracle/hipdlp_oracle.c -- the oracle of the engine's NEXT algorithm mode, SURVEY.md
8(a) a20 / 8(f) rank 2) against the unmodified reference's `solver=hipdlp`:
  * tests/golden/hipdlp/: 60 cases (12 of the reference's own LP instances x 5 option sets: PID and fixed primal weight,
    Ruiz/PC/L2 scaling modes, no scaling, converged and iteration-limited) generated through Highs::run()
    (make_hipdlp_golden.py) -- iteration counts and all four HighsSolution vectors bit for bit;
  * the same against the reference's runs on all 74 instances (recorded in tests/golden/reference_runs.json)."""
import glob
import json
import os

import numpy as np
import pytest

import recorded_reference
from conftest import GOLDEN

CASES = json.load(open(os.path.join(GOLDEN, "hipdlp", "golden.json")))


def _kw(options):
    kw = {}
    if "pdlp_iteration_limit" in options:
        kw["max_iterations"] = options["pdlp_iteration_limit"]
    if "kkt_tolerance" in options:
        kw["tolerance"] = options["kkt_tolerance"]
    if "pdlp_step_size_strategy" in options:
        kw["step_size_strategy"] = options["pdlp_step_size_strategy"]
    if "pdlp_scaling_mode" in options:
        kw["scaling_mode"] = options["pdlp_scaling_mode"]
    if "pdlp_ruiz_iterations" in options:
        kw["ruiz_iterations"] = options["pdlp_ruiz_iterations"]
    return kw


@pytest.mark.parametrize("case", CASES, ids=[f"{c['name']}-{c['tag']}" for c in CASES])
def test_hipdlp_oracle_reproduces_reference(oracle, case):
    from highs_b200.lp import read_b2lp
    lp = read_b2lp(os.path.join(GOLDEN, "instances", case["name"] + ".b2lp"))
    res = oracle.hipdlp_solve(lp, **_kw(case["options"]))
    assert res["iters"] == case["pdlp_iteration_count"]
    assert (res["term_name"] == "OPTIMAL") == (case["model_status"] == "Optimal")
    gold = dict(np.load(os.path.join(GOLDEN, "hipdlp", case["file"])))
    for k in ("col_value", "col_dual", "row_value", "row_dual"):
        assert np.array_equal(res[k], gold[k]), k


def test_hipdlp_goldens_cover_both_outcomes():
    assert sum(c["model_status"] == "Optimal" for c in CASES) >= 10
    assert sum(c["model_status"] != "Optimal" for c in CASES) >= 10


def test_hipdlp_oracle_vs_live_reference(oracle):
    from highs_b200.lp import read_b2lp
    variants = [{"pdlp_iteration_limit": 800}, {"pdlp_iteration_limit": 4000, "kkt_tolerance": 1e-4},
                {"pdlp_iteration_limit": 400, "pdlp_step_size_strategy": 0},
                {"pdlp_iteration_limit": 400, "pdlp_scaling_mode": 7, "pdlp_ruiz_iterations": 3},
                {"pdlp_iteration_limit": 1200, "kkt_tolerance": 1e-3, "pdlp_scaling_mode": 0}]
    n_ok = 0
    for path in sorted(glob.glob(os.path.join(GOLDEN, "instances", "*.b2lp"))):
        lp = read_b2lp(path)
        if lp.a_matrix_.numNz() > 200000:
            continue
        for opts in variants:
            ref = recorded_reference.run_reference(lp, options=dict(opts, solver="hipdlp"), want_solution=True,
                                                   keep=("pdlp_iteration_count",) + recorded_reference.VECTORS)
            res = oracle.hipdlp_solve(lp, **_kw(opts))
            assert ref["pdlp_iteration_count"] == res["iters"], (os.path.basename(path), opts)
            for k in ("col_value", "col_dual", "row_value", "row_dual"):
                assert ref[k] == recorded_reference.digest(res[k]), (os.path.basename(path), opts, k)
            n_ok += 1
    assert n_ok >= 300
