"""Every LP the reference ships for its own tests (check/instances/*.mps as read by the reference, stored in
tests/golden/instances/) through the host prologue (formulate + scale, bit for bit against the oracle) and the device
layouts of 1 and 3 ranks (host evaluation against a plain sparse product), in reference order and length-sorted; and the
oracle against the reference's runs (recorded in tests/golden/reference_runs.json; 400 iterations, bit for bit) on each of them.
usage: python tools/sweep_reference_instances.py        last line: JSON {"ok": n, "bad": [[name, what], ...]}"""
import glob, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np
import recorded_reference
from highs_b200 import engine
from highs_b200.lp import read_b2lp
from oracle import binding as ob
KEYS = ["cost", "lower", "upper", "rhs", "col_scale", "row_scale", "cbeg", "cidx", "cval", "row_new_idx", "row_type", "rbeg", "ridx", "rval"]
VECS = recorded_reference.VECTORS
bad = []; n_ok = 0; n_pinned = 0; n_hot = 0
for path in sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "instances", "*.b2lp"))):
    name = os.path.basename(path)[:-5]
    lp = read_b2lp(path)
    if lp.num_row_ == 0 or lp.a_matrix_.numNz() == 0:
        print(name, "skipped (no rows / nnz)"); continue
    try:
        a, b = engine.host_form(lp, 1), ob.formulate_and_scale(lp, 1)
        same = lambda u, v: np.array_equal(u, v, equal_nan=True) if np.asarray(u).dtype.kind == "f" else np.array_equal(u, v)
        diffs = [k for k in KEYS if not same(a[k], b[k])] + [k for k in ("n","m","nnz","neq","amax","norm_cost","norm_rhs") if not same(a[k], b[k])]
        import scipy.sparse as sp
        for w in (1, 3):
            r = engine.host_layout_eval(lp, world=w, seed=1)
            A = sp.csc_matrix((r["cval"], r["cidx"], r["cbeg"]), shape=(r["m"], r["n"]))
            sax = np.abs(A) @ np.abs(r["x"]) + 1e-300; say = np.abs(A).T @ np.abs(r["y"]) + 1e-300
            if not (np.all(np.abs(r["ax"] - A @ r["x"]) <= 1e-12 * sax) and np.all(np.abs(r["aty"] - A.T @ r["y"]) <= 1e-12 * say)):
                diffs.append(f"layout world {w}")
            r2 = engine.host_layout_eval(lp, world=w, ordered_max=-1, seed=1)
            if not (np.all(np.abs(r2["ax"] - A @ r2["x"]) <= 1e-12 * sax) and np.all(np.abs(r2["aty"] - A.T @ r2["y"]) <= 1e-12 * say)):
                diffs.append(f"sorted layout world {w}")
        # the oracle against the LIVE reference on this instance (400 iterations; 240 without restarts; to 1e-3 or 1200
        # iterations): iteration count and all four
        # solution vectors bit for bit (pins the oracle far beyond the committed goldens)
        if lp.a_matrix_.numNz() <= 200000 and not np.isnan(lp.col_cost_).any():
            for opts, prm in (({"pdlp_iteration_limit": 400}, dict(iter_limit=400)),
                              ({"pdlp_iteration_limit": 240, "pdlp_cupdlpc_restart_method": 0}, dict(iter_limit=240, restart=0)),
                              ({"pdlp_iteration_limit": 1200, "kkt_tolerance": 1e-3}, dict(iter_limit=1200, tol_primal=1e-3, tol_dual=1e-3, tol_gap=1e-3))):
                ref = recorded_reference.run_reference(lp, options=opts, want_solution=True, keep=("pdlp_iteration_count",) + VECS)
                o = ob.solve(lp, **prm)
                if ref["pdlp_iteration_count"] != o["iters"] or not all(recorded_reference.digest(o[k]) == ref[k] for k in VECS):
                    diffs.append(f"oracle vs reference {opts}: {ref['pdlp_iteration_count']} / {o['iters']} iterations")
            # hot start (PDHG_PreSolve, cupdlp_solver.c:1217-1279): restart both from the reference's own 1e-3 solution,
            # which the last option set above has just found bit-equal to the oracle's
            # (Highs::setSolution recomputes the row activities of a user solution in quad precision before the wrapper sees
            #  them -- Highs.cpp:2519-2530, calculateRowValuesQuad, HighsLpUtils.cpp:3011-3047 -- and ranged rows start
            #  their slack from them, so the oracle is given the exactly rounded A x as well)
            if lp.a_matrix_.numNz() <= 20000:
                from fractions import Fraction
                w = o
                accq = [Fraction(0)] * lp.num_row_
                Am = lp.a_matrix_
                for jc in range(lp.num_col_):
                    xj = Fraction(float(w["col_value"][jc]))
                    for pe in range(Am.start_[jc], Am.start_[jc + 1]):
                        accq[Am.index_[pe]] += xj * Fraction(float(Am.value_[pe]))
                rvq = np.array([float(a_) for a_ in accq])
                ref = recorded_reference.run_reference(lp, options={"pdlp_iteration_limit": 200}, want_solution=True,
                                                       warm=tuple(w[k] for k in VECS), keep=("pdlp_iteration_count",) + VECS)
                o = ob.solve(lp, iter_limit=200, warm=(w["col_value"], rvq, w["row_dual"]))
                if ref["pdlp_iteration_count"] != o["iters"] or not all(recorded_reference.digest(o[k]) == ref[k] for k in VECS):
                    diffs.append(f"oracle vs reference, hot start: {ref['pdlp_iteration_count']} / {o['iters']} iterations")
                n_hot += 1
            n_pinned += 1
        if diffs: bad.append((name, diffs)); print(name, "DIFF", diffs)
        else: n_ok += 1
    except Exception as e:
        bad.append((name, repr(e))); print(name, "EXC", repr(e)[:200])
import json
print(json.dumps({"ok": n_ok, "oracle_pinned_on": n_pinned, "hot_start_pinned_on": n_hot, "bad": [[k, str(v)] for k, v in bad]}))
