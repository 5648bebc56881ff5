"""Live pinning of the oracle: oracle/live_check.py imports the UNMODIFIED reference from PYLC_REFERENCE_ROOT
(three import-only stubs, oracle/ref_harness.py) and compares every restatement in oracle/pylc_oracle.py with
the reference function it cites, on seeded inputs other than the frozen tests/golden/ vectors.

Skipped unless PYLC_REFERENCE_ROOT names a PyLC checkout; the committed golden vectors
(tests/test_oracle_golden.py) carry the pinning without it.  A separate process keeps the
harness's chdir / sys.path changes away from the rest of the suite.
"""
import os
import subprocess
import sys

import pytest

import ref_harness

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("seed", [4242, 7])
def test_oracle_equals_reference_live(seed):
    if not ref_harness.available():
        pytest.skip("PYLC_REFERENCE_ROOT does not name a PyLC checkout: golden vectors pin the oracle instead")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "live_check.py"), "--seed", str(seed)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "0 mismatches" in r.stdout
