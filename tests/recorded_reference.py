"""What the unmodified reference (oracle/_ref: HiGHS through Highs::run(), ref_driver) returned, recorded once in
tests/golden/reference_runs.json, so that the tests that compare against it need neither the reference tree nor
oracle/_ref.

A result is found by a digest of everything the call hands the reference: the LP as written for ref_driver, the options
and flags, and for reference_kkt the solution.  A test whose inputs change finds no recorded result and fails, instead of
comparing against a result for other inputs.  Solution vectors are stored as digests of their float64 bytes (signed
zeros and NaN payloads folded), which keeps the bit-for-bit comparison at a few bytes per vector.

To record (needs oracle/_ref, built by oracle/build_ref.py), run the tests that use this module with
B200PDLP_RECORD_REFERENCE=1; every call then runs the reference and stores what it returned.
"""
import hashlib
import json
import os
import tempfile

import numpy as np
import pytest

from conftest import GOLDEN

PATH = os.path.join(GOLDEN, "reference_runs.json")
RECORD = os.environ.get("B200PDLP_RECORD_REFERENCE") == "1"
VECTORS = ("col_value", "col_dual", "row_value", "row_dual")
_runs = None


def digest(a) -> str:
    a = np.asarray(a, dtype="<f8") + 0.0      # -0.0 -> 0.0
    a = np.where(np.isnan(a), np.nan, a)
    return hashlib.sha256(a.tobytes()).hexdigest()[:32]


def _lp_digest(lp) -> str:
    from highs_b200.lp import write_b2lp
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "lp.b2lp")
        write_b2lp(p, lp)
        with open(p, "rb") as f:
            return hashlib.sha256(f.read()).hexdigest()


def _recorded(key: dict, live, keep=None):
    global _runs
    if _runs is None:
        _runs = json.load(open(PATH)) if os.path.exists(PATH) else {}
    k = hashlib.sha256(json.dumps(key, sort_keys=True).encode()).hexdigest()[:32]
    if RECORD:
        res = live()
        if keep is not None:
            res = {q: res[q] for q in keep}
        for v in VECTORS:
            if v in res:
                res[v] = digest(res[v])
        _runs[k] = res
        with open(PATH, "w") as f:
            f.write("{\n" + ",\n".join(f"{json.dumps(q)}: {json.dumps(_runs[q], sort_keys=True)}" for q in sorted(_runs)) + "\n}\n")
    if k not in _runs:
        pytest.fail(f"no recorded reference result for these inputs ({key}); record it with B200PDLP_RECORD_REFERENCE=1")
    return dict(_runs[k])


def run_reference(lp, options=None, want_solution=False, warm=None, pdlp_cleanup=None, cleanup_tighten=1.0, keep=None) -> dict:
    """oracle.binding.run_reference as recorded; with want_solution the four vectors come back as digest() strings.
    `keep` names the only fields to record (for tests that make many calls and read few fields)."""
    from oracle import binding
    key = dict(call="run_reference", lp=_lp_digest(lp), options=options, want_solution=want_solution,
               pdlp_cleanup=pdlp_cleanup, cleanup_tighten=cleanup_tighten)
    if warm is not None:
        key["warm"] = [digest(v) for v in warm]
    return _recorded(key, lambda: binding.run_reference(lp=lp, options=options, want_solution=want_solution, warm=warm,
                                                        pdlp_cleanup=pdlp_cleanup, cleanup_tighten=cleanup_tighten), keep)


def reference_kkt(lp, solution, model_status_code=7, options=None) -> dict:
    """oracle.binding.reference_kkt (the reference's lpKktCheck on a given solution) as recorded"""
    from oracle import binding
    key = dict(call="reference_kkt", lp=_lp_digest(lp), solution=[digest(solution[v]) for v in VECTORS],
               model_status_code=int(model_status_code), options=options)
    return _recorded(key, lambda: binding.reference_kkt(lp, solution, model_status_code=model_status_code, options=options))
