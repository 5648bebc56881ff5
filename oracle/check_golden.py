"""TEST INFRASTRUCTURE ONLY.  Regenerates every golden fixture from the imported reference into a scratch directory
(oracle/gen_golden.py, unchanged) and compares it, array by array, with the committed tests/golden/*.npz.
Needs a checkout of the reference:

    PYLC_REFERENCE_ROOT=<PyLC checkout> python oracle/check_golden.py   # one line per fixture, non-zero exit on any difference
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import gen_golden  # noqa: E402
import ref_harness  # noqa: E402


def main():
    if not ref_harness.available():
        print("reference not available at %s" % ref_harness.REF_ROOT)
        return 2
    committed, scratch = gen_golden.OUT, tempfile.mkdtemp(prefix="pylc_golden_")
    gen_golden.OUT = scratch
    cwd = os.getcwd()
    gen_golden.main()
    os.chdir(cwd)
    bad = 0
    for name in sorted(f for f in os.listdir(committed) if f.endswith(".npz")):
        new, old = np.load(os.path.join(scratch, name)), np.load(os.path.join(committed, name))
        same = set(new.files) == set(old.files) and all(np.array_equal(new[k], old[k]) for k in new.files)
        print("%-22s %s" % (name, "identical" if same else "DIFFERS"))
        bad += not same
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
