"""Every LP the reference ships for its own tests (check/instances/*.mps as read by the unmodified reference, stored in
tests/golden/instances/) through the product's host prologue -- formulate + Ruiz/Pock-Chambolle scaling + transposition,
bit for bit against the oracle -- and through the device layouts of 1 and 3 ranks, evaluated on the host; and the
oracle itself against the reference's runs on each of them (three option sets -- 400 iterations, 240 without restarts, to 1e-3 -- and a hot start from the reference's own 1e-3
solution: iteration count and solution vectors, bit for bit; recorded in tests/golden/reference_runs.json).
About 20 s."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_instances_through_host_prologue(engine_lib):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sweep_reference_instances.py")], capture_output=True,
                       text=True, timeout=900, cwd=ROOT)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert lines, (r.stdout[-1500:], r.stderr[-1500:])
    out = json.loads(lines[-1])
    assert out["ok"] >= 60 and out["oracle_pinned_on"] >= 60 and out["hot_start_pinned_on"] >= 50 and not out["bad"], out
