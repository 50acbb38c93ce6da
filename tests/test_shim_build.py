"""The HiGHS drop-in build (oracle/build_ref.py --shim): the reference's own objects with pdlp/CupdlpWrapper.cpp replaced
by highs_b200/csrc/highs_shim.cpp.  No GPU needed: checks the link result and that, without a device, Highs::run()
fails LOUDLY through the reference's own error path (kSolveError / HighsStatus::kError) instead of falling back."""
import os
import subprocess

import pytest

from conftest import GOLDEN, ROOT

LIB = os.path.join(ROOT, "oracle", "_ref", "libhighs_b200.so")
DRV = os.path.join(ROOT, "oracle", "_ref", "ref_driver_b200")


@pytest.mark.skipif(not os.path.exists(LIB), reason="oracle/_ref/libhighs_b200.so not built (python oracle/build_ref.py --shim)")
def test_shim_exports_the_boundary_symbols():
    syms = subprocess.check_output(["nm", "-D", "--defined-only", LIB], text=True)
    assert "_Z13solveLpCupdlpR19HighsLpSolverObject" in syms                      # CupdlpWrapper.h:92
    assert "_Z13solveLpCupdlpRK12HighsOptionsR10HighsTimerRK7HighsLp" in syms     # CupdlpWrapper.h:94-98
    assert "getCupdlpLogLevel" in syms                                            # CupdlpWrapper.h:106
    und = subprocess.check_output(["nm", "-D", "--undefined-only", LIB], text=True)
    assert "b200pdlp_solve" in und                                                # forwarded to the C ABI
    assert "formulateLP_highs" not in syms          # the reference wrapper (and its standard-form builder) is gone


@pytest.mark.skipif(not os.path.exists(DRV), reason="oracle/_ref/ref_driver_b200 not built")
def test_dropin_fails_loudly_without_gpu(engine_lib):
    from highs_b200 import engine
    if engine.device_count() > 0:
        pytest.skip("a GPU is visible")
    from oracle.binding import _parse_json_line, driver_env
    out = subprocess.run([DRV, "--lp", os.path.join(GOLDEN, "avgas.b2lp"), "--opt", "solver=pdlp", "--opt", "presolve=off"],
                         capture_output=True, text=True, env=driver_env())
    assert out.stdout.strip(), out.stderr[-2000:]
    res = _parse_json_line(out.stdout)
    assert res["run_status"] == -1 and res["model_status_code"] == 4          # HighsStatus::kError, kSolveError
    assert res["pdlp_iteration_count"] == -1


LIB3 = os.path.join(ROOT, "oracle", "_ref", "libhighs_b200_hipdlp.so")


@pytest.mark.skipif(not os.path.exists(LIB3), reason="oracle/_ref/libhighs_b200_hipdlp.so not built (python oracle/build_ref.py --shim)")
def test_hipdlp_shim_exports_the_boundary_symbols():
    """the second drop-in point, solveLpHiPdlp (HiPdlpWrapper.h; call site HighsSolve.cpp:107-117), forwarded to the C ABI"""
    syms = subprocess.check_output(["nm", "-D", "--defined-only", LIB3], text=True)
    assert "_Z13solveLpHiPdlpR19HighsLpSolverObject" in syms
    assert "_Z13solveLpCupdlpR19HighsLpSolverObject" in syms
    und = subprocess.check_output(["nm", "-D", "--undefined-only", LIB3], text=True)
    assert "b200pdlp_solve_hipdlp" in und and "b200pdlp_solve" in und
