"""ctypes binding of oracle/libpdlp_oracle.so and a runner for oracle/_ref/ref_driver.

TEST INFRASTRUCTURE ONLY (see oracle/pdlp_oracle.h).
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpdlp_oracle.so")
REF_DRIVER = os.path.join(HERE, "_ref", "ref_driver")
DROPIN_DRIVER = os.path.join(HERE, "_ref", "ref_driver_b200")   # HiGHS + highs_shim.cpp + libb200pdlp.so
TRACE_COLS = 16

TERM_NAMES = {0: "OPTIMAL", 1: "INFEASIBLE", 2: "UNBOUNDED", 3: "INFEASIBLE_OR_UNBOUNDED",
              4: "TIMELIMIT_OR_ITERLIMIT", 5: "FEASIBLE"}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class OrcLp(C.Structure):
    _fields_ = [("n", C.c_int), ("m", C.c_int), ("start", _ip), ("index", _ip), ("value", _dp),
                ("cost", _dp), ("col_lower", _dp), ("col_upper", _dp), ("row_lower", _dp), ("row_upper", _dp),
                ("sense", C.c_double), ("offset", C.c_double)]


class OrcParams(C.Structure):
    _fields_ = [("iter_limit", C.c_int), ("tol_primal", C.c_double), ("tol_dual", C.c_double),
                ("tol_gap", C.c_double), ("time_limit", C.c_double), ("scaling", C.c_int),
                ("adaptive_step", C.c_int), ("restart", C.c_int), ("interaction_row_side", C.c_int)]


class OrcForm(C.Structure):
    _fields_ = [("n", C.c_int), ("m", C.c_int), ("nnz", C.c_int), ("neq", C.c_int), ("n_orig", C.c_int),
                ("cost", _dp), ("lower", _dp), ("upper", _dp), ("rhs", _dp),
                ("cbeg", _ip), ("cidx", _ip), ("cval", _dp), ("rbeg", _ip), ("ridx", _ip), ("rval", _dp),
                ("col_scale", _dp), ("row_scale", _dp), ("row_new_idx", _ip), ("row_type", _ip),
                ("sense", C.c_double), ("offset", C.c_double), ("norm_cost", C.c_double),
                ("norm_rhs", C.c_double), ("amax", C.c_double)]


class OrcResult(C.Structure):
    _fields_ = [("col_value", _dp), ("col_dual", _dp), ("row_value", _dp), ("row_dual", _dp),
                ("value_valid", C.c_int), ("dual_valid", C.c_int), ("term_code", C.c_int),
                ("term_iterate", C.c_int), ("iters", C.c_int),
                ("pobj", C.c_double), ("dobj", C.c_double), ("pfeas", C.c_double), ("dfeas", C.c_double),
                ("gap", C.c_double), ("relgap", C.c_double),
                ("trace", _dp), ("trace_cap", C.c_int), ("trace_len", C.c_int)]


_lib = None


def build() -> str:
    subprocess.check_call(["make", "-s", "-C", HERE, "libpdlp_oracle.so"])
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        _lib = C.CDLL(LIB_PATH)
        _lib.orc_solve.argtypes = [C.POINTER(OrcLp), C.POINTER(OrcParams), C.POINTER(OrcResult)]
        _lib.orc_formulate.argtypes = [C.POINTER(OrcLp), C.POINTER(OrcForm)]
        _lib.orc_scale.argtypes = [C.POINTER(OrcForm), C.c_int]
        _lib.orc_build_csr.argtypes = [C.POINTER(OrcForm)]
        _lib.orc_form_free.argtypes = [C.POINTER(OrcForm)]
        _lib.orc_ax.argtypes = [C.POINTER(OrcForm), _dp, _dp]
        _lib.orc_aty.argtypes = [C.POINTER(OrcForm), _dp, _dp]
    return _lib


def _p(a, t):
    return a.ctypes.data_as(t)


def _mk_lp(lp):
    a = lp.a_matrix_
    keep = (a.start_, a.index_, a.value_, lp.col_cost_, lp.col_lower_, lp.col_upper_, lp.row_lower_, lp.row_upper_)
    s = OrcLp(lp.num_col_, lp.num_row_, _p(a.start_, _ip), _p(a.index_, _ip), _p(a.value_, _dp),
              _p(lp.col_cost_, _dp), _p(lp.col_lower_, _dp), _p(lp.col_upper_, _dp),
              _p(lp.row_lower_, _dp), _p(lp.row_upper_, _dp), float(lp.sense_), float(lp.offset_))
    return s, keep


def default_params(**kw) -> dict:
    """Defaults = what HiGHS passes for default options (CupdlpWrapper.cpp:642-717)."""
    p = dict(iter_limit=2147483647, tol_primal=1e-7, tol_dual=1e-7, tol_gap=1e-7, time_limit=0.0,
             scaling=1, adaptive_step=1, restart=1, interaction_row_side=0)
    p.update(kw)
    return p


def solve(lp, warm=None, trace_cap=0, **kw) -> dict:
    """Run the CPU restatement.  `warm` = (col_value, row_value, row_dual) hot start."""
    L = lib()
    p = default_params(**kw)
    clp, keep = _mk_lp(lp)
    n, m = lp.num_col_, lp.num_row_
    cv, cd, rv, rd = np.zeros(n), np.zeros(n), np.zeros(m), np.zeros(m)
    vv = dv = 0
    if warm is not None:
        cv[:] = warm[0]; rv[:] = warm[1]; rd[:] = warm[2]; vv = dv = 1
    tr = np.zeros((max(trace_cap, 1), TRACE_COLS))
    res = OrcResult(_p(cv, _dp), _p(cd, _dp), _p(rv, _dp), _p(rd, _dp), vv, dv, 0, 0, 0,
                    0, 0, 0, 0, 0, 0, _p(tr, _dp) if trace_cap else None, trace_cap, 0)
    prm = OrcParams(p["iter_limit"], p["tol_primal"], p["tol_dual"], p["tol_gap"], p["time_limit"],
                    p["scaling"], p["adaptive_step"], p["restart"], p["interaction_row_side"])
    rc = L.orc_solve(C.byref(clp), C.byref(prm), C.byref(res))
    assert rc == 0
    return dict(col_value=cv, col_dual=cd, row_value=rv, row_dual=rd, term_code=res.term_code,
                term_name=TERM_NAMES[res.term_code], term_iterate=res.term_iterate, iters=res.iters,
                pobj=res.pobj, dobj=res.dobj, pfeas=res.pfeas, dfeas=res.dfeas, gap=res.gap,
                relgap=res.relgap, trace=tr[: res.trace_len].copy())


class HipParams(C.Structure):
    _fields_ = [("tolerance", C.c_double), ("max_iterations", C.c_int), ("use_ruiz", C.c_int), ("use_pc", C.c_int),
                ("use_l2", C.c_int), ("ruiz_iterations", C.c_int), ("step_size_strategy", C.c_int)]


class HipResult(C.Structure):
    _fields_ = [("col_value", _dp), ("col_dual", _dp), ("row_value", _dp), ("row_dual", _dp),
                ("term_code", C.c_int), ("iters", C.c_int), ("pfeas", C.c_double), ("dfeas", C.c_double),
                ("pobj", C.c_double), ("dobj", C.c_double), ("relgap", C.c_double), ("primal_weight", C.c_double),
                ("op_norm_sq", C.c_double), ("trace", _dp), ("trace_cap", C.c_int), ("trace_len", C.c_int)]


def hipdlp_solve(lp, tolerance=1e-7, max_iterations=2147483647, scaling_mode=5, ruiz_iterations=10, step_size_strategy=3,
                 trace_cap=0) -> dict:
    """The HiPDLP restatement (oracle/hipdlp_oracle.c).  Arguments are the HighsOptions of the same names
    (pdlp_scaling_mode bits: 1 Ruiz, 2 L2, 4 PC; pdlp_step_size_strategy: 0 fixed, anything else PID)."""
    L = lib()
    clp, keep = _mk_lp(lp)
    n, m = lp.num_col_, lp.num_row_
    cv, cd, rv, rd = np.zeros(max(n, 1)), np.zeros(max(n, 1)), np.zeros(max(m, 1)), np.zeros(max(m, 1))
    prm = HipParams(tolerance, int(min(max_iterations, 2147483647)), int(bool(scaling_mode & 1)), int(bool(scaling_mode & 4)),
                    int(bool(scaling_mode & 2)), ruiz_iterations, 0 if step_size_strategy == 0 else 3)
    tr = np.zeros((max(trace_cap, 1), 20))
    res = HipResult(_p(cv, _dp), _p(cd, _dp), _p(rv, _dp), _p(rd, _dp), 0, 0, 0, 0, 0, 0, 0, 0, 0,
                    _p(tr, _dp) if trace_cap else None, trace_cap, 0)
    L.hip_solve.argtypes = [C.POINTER(OrcLp), C.POINTER(HipParams), C.POINTER(HipResult)]
    rc = L.hip_solve(C.byref(clp), C.byref(prm), C.byref(res))
    assert rc == 0
    return dict(col_value=cv[:n], col_dual=cd[:n], row_value=rv[:m], row_dual=rd[:m], term_code=res.term_code,
                term_name={0: "OPTIMAL", 1: "MAXITER"}[res.term_code], iters=res.iters, pfeas=res.pfeas, dfeas=res.dfeas,
                pobj=res.pobj, dobj=res.dobj, relgap=res.relgap, primal_weight=res.primal_weight, op_norm_sq=res.op_norm_sq,
                trace=tr[: res.trace_len].copy())


class HipForm(C.Structure):
    _fields_ = [("n", C.c_int), ("m", C.c_int), ("nnz", C.c_int), ("neq", C.c_int),
                ("cost", _dp), ("lower", _dp), ("upper", _dp), ("rlo", _dp), ("rup", _dp),
                ("cbeg", _ip), ("cidx", _ip), ("cval", _dp), ("col_scale", _dp), ("row_scale", _dp),
                ("new_idx", _ip), ("ctype", _ip), ("c_norm", C.c_double), ("rhs_norm", C.c_double), ("op_norm_sq", C.c_double)]


def hipdlp_form(lp, scaling_mode=5, ruiz_iterations=10) -> dict:
    """HiPDLP's processed + scaled LP and its power-method estimate (oracle/hipdlp_oracle.c::hip_form_build)."""
    L = lib()
    clp, keep = _mk_lp(lp)
    n0, m, nnz0 = lp.num_col_, lp.num_row_, lp.a_matrix_.numNz()
    nmax, zmax = n0 + m + 1, nnz0 + m + 1
    a = dict(cost=np.zeros(nmax), lower=np.zeros(nmax), upper=np.zeros(nmax), col_scale=np.zeros(nmax),
             rlo=np.zeros(m + 1), rup=np.zeros(m + 1), row_scale=np.zeros(m + 1), new_idx=np.zeros(m + 1, dtype=np.int32),
             ctype=np.zeros(m + 1, dtype=np.int32), cbeg=np.zeros(nmax + 1, dtype=np.int32), cidx=np.zeros(zmax, dtype=np.int32),
             cval=np.zeros(zmax))
    f = HipForm(0, 0, 0, 0, _p(a["cost"], _dp), _p(a["lower"], _dp), _p(a["upper"], _dp), _p(a["rlo"], _dp), _p(a["rup"], _dp),
                _p(a["cbeg"], _ip), _p(a["cidx"], _ip), _p(a["cval"], _dp), _p(a["col_scale"], _dp), _p(a["row_scale"], _dp),
                _p(a["new_idx"], _ip), _p(a["ctype"], _ip), 0.0, 0.0, 0.0)
    prm = HipParams(1e-7, 0, int(bool(scaling_mode & 1)), int(bool(scaling_mode & 4)), int(bool(scaling_mode & 2)), ruiz_iterations, 3)
    L.hip_form_build.argtypes = [C.POINTER(OrcLp), C.POINTER(HipParams), C.POINTER(HipForm)]
    assert L.hip_form_build(C.byref(clp), C.byref(prm), C.byref(f)) == 0
    n, nnz = f.n, f.nnz
    out = dict(n=n, m=m, nnz=nnz, neq=f.neq, c_norm=f.c_norm, rhs_norm=f.rhs_norm, op_norm_sq=f.op_norm_sq)
    for k in ("cost", "lower", "upper", "col_scale"):
        out[k] = a[k][:n].copy()
    for k in ("rlo", "rup", "row_scale", "new_idx", "ctype"):
        out[k] = a[k][:m].copy()
    out.update(cbeg=a["cbeg"][: n + 1].copy(), cidx=a["cidx"][:nnz].copy(), cval=a["cval"][:nnz].copy())
    return out


def formulate_and_scale(lp, scaling=1) -> dict:
    """Standard form + scaling + CSR as numpy copies (for kernel-level parity tests)."""
    L = lib()
    clp, keep = _mk_lp(lp)
    f = OrcForm()
    L.orc_formulate(C.byref(clp), C.byref(f))
    L.orc_scale(C.byref(f), scaling)
    L.orc_build_csr(C.byref(f))
    n, m, nnz = f.n, f.m, f.nnz
    arr = lambda ptr, k, dt: np.ctypeslib.as_array(ptr, shape=(max(k, 1),))[:k].astype(dt).copy()
    out = dict(n=n, m=m, nnz=nnz, neq=f.neq, n_orig=f.n_orig,
               cost=arr(f.cost, n, np.float64), lower=arr(f.lower, n, np.float64), upper=arr(f.upper, n, np.float64),
               rhs=arr(f.rhs, m, np.float64), cbeg=arr(f.cbeg, n + 1, np.int32), cidx=arr(f.cidx, nnz, np.int32),
               cval=arr(f.cval, nnz, np.float64), rbeg=arr(f.rbeg, m + 1, np.int32), ridx=arr(f.ridx, nnz, np.int32),
               rval=arr(f.rval, nnz, np.float64), col_scale=arr(f.col_scale, n, np.float64),
               row_scale=arr(f.row_scale, m, np.float64), row_new_idx=arr(f.row_new_idx, m, np.int32),
               row_type=arr(f.row_type, m, np.int32), norm_cost=f.norm_cost, norm_rhs=f.norm_rhs, amax=f.amax)
    L.orc_form_free(C.byref(f))
    return out


def _parse_json_line(text: str) -> dict:
    """ref_driver prints C doubles: map inf / nan to the spellings Python's json accepts"""
    import re
    line = text.strip().splitlines()[-1]
    line = re.sub(r"(?<![\w.])-inf(?![\w])", "-Infinity", line)
    line = re.sub(r"(?<![\w.-])inf(?![\w])", "Infinity", line)
    line = re.sub(r"(?<![\w.])-?nan(?![\w])", "NaN", line)
    return json.loads(line)


def driver_env() -> dict:
    """Environment for the ref_driver binaries: the drop-in ones load highs_b200/libb200pdlp.so of THIS tree.  Their run path
    cannot be relied on for it -- $ORIGIN resolves symlinks, so a linked or copied oracle/_ref/ no longer sits next to the
    engine -- and LD_LIBRARY_PATH is searched before a run path."""
    eng = os.path.join(os.path.dirname(HERE), "highs_b200")
    return dict(os.environ, LD_LIBRARY_PATH=os.pathsep.join(p for p in (eng, os.environ.get("LD_LIBRARY_PATH")) if p))


def ref_available() -> bool:
    return os.path.exists(REF_DRIVER)


def dropin_available() -> bool:
    return os.path.exists(DROPIN_DRIVER)


def run_reference(lp=None, mps=None, options=None, want_solution=False, warm=None, lp_path=None, timeout=None,
                  driver=None, pdlp_cleanup=None, cleanup_tighten=1.0) -> dict:
    """Run the UNMODIFIED reference (oracle/_ref) through Highs::run(); returns its JSON line.
    driver=DROPIN_DRIVER runs the same Highs::run() with the B200 shim linked in place of
    CupdlpWrapper.cpp (the drop-in integration, INTEGRATION.md)."""
    from highs_b200.lp import write_b2lp
    opts = {"solver": "pdlp", "presolve": "off"}
    opts.update(options or {})
    with tempfile.TemporaryDirectory() as td:
        cmd = [driver or REF_DRIVER]
        if mps is not None:
            cmd += ["--mps", mps]
        else:
            if lp_path is None:
                lp_path = os.path.join(td, "lp.b2lp")
                write_b2lp(lp_path, lp)
            cmd += ["--lp", lp_path]
        for k, v in opts.items():
            cmd += ["--opt", f"{k}={v}"]
        if pdlp_cleanup is not None:   # the product's clean-up flow (highs_b200/csrc/highs_pdlp_cleanup.hpp); value = margin
            cmd += ["--pdlp-cleanup", "--cleanup-margin", repr(float(pdlp_cleanup)), "--cleanup-tighten", repr(float(cleanup_tighten))]
        sol = os.path.join(td, "sol.bin")
        if want_solution:
            cmd += ["--sol", sol]
        if warm is not None:
            wp = os.path.join(td, "warm.bin")
            cv, cd, rv, rd = warm
            with open(wp, "wb") as f:
                f.write(np.array([len(cv), len(rv), 1, 1], dtype="<i8").tobytes())
                for v in (cv, cd, rv, rd):
                    f.write(np.asarray(v, dtype="<f8").tobytes())
            cmd += ["--warm", wp]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=driver_env())
        if out.returncode != 0:
            raise RuntimeError(f"ref_driver failed: {out.stderr}")
        res = _parse_json_line(out.stdout)
        if want_solution:
            raw = open(sol, "rb").read()
            n, m, vv, dv = np.frombuffer(raw[:32], dtype="<i8")
            v = np.frombuffer(raw[32:], dtype="<f8")
            res.update(col_value=v[:n].copy(), col_dual=v[n:2 * n].copy(), row_value=v[2 * n:2 * n + m].copy(),
                       row_dual=v[2 * n + m:2 * n + 2 * m].copy(), value_valid=bool(vv), dual_valid=bool(dv))
    return res


def reference_kkt(lp, solution, model_status_code=7, options=None) -> dict:
    """Evaluate a HighsSolution with the reference's own lpKktCheck (ref_driver --kkt-of).

    `solution` = dict/obj with col_value, col_dual, row_value, row_dual.  Returns the
    HighsInfo KKT fields and the model status after lpKktCheck's adjustment, exactly as
    Highs::run() would report them for that solution (Highs.cpp:1990).
    """
    from highs_b200.lp import write_b2lp
    opts = {"solver": "pdlp", "presolve": "off"}
    opts.update(options or {})
    g = (lambda k: solution[k]) if isinstance(solution, dict) else (lambda k: getattr(solution, k))
    with tempfile.TemporaryDirectory() as td:
        lp_path = os.path.join(td, "lp.b2lp")
        write_b2lp(lp_path, lp)
        sp = os.path.join(td, "sol.bin")
        cv, cd, rv, rd = (np.asarray(g(k), dtype="<f8") for k in ("col_value", "col_dual", "row_value", "row_dual"))
        with open(sp, "wb") as f:
            f.write(np.array([len(cv), len(rv), 1, 1], dtype="<i8").tobytes())
            for v in (cv, cd, rv, rd):
                f.write(v.tobytes())
        cmd = [REF_DRIVER, "--lp", lp_path, "--kkt-of", sp, "--kkt-status", str(int(model_status_code))]
        for k, v in opts.items():
            cmd += ["--opt", f"{k}={v}"]
        out = subprocess.run(cmd, capture_output=True, text=True)
        if out.returncode != 0:
            raise RuntimeError(f"ref_driver --kkt-of failed: {out.stderr}")
        return _parse_json_line(out.stdout)
