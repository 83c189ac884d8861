"""Generate tests/golden/reference_checks.json.xz: the REAL reference's answers to the differential checks of the kernels'
three checkers (diff_hot_path, diff_ingest, diff_online), so that tests/test_reference_differential_cpu.py compares the
checkers with the reference on machines that do not have it.

Run from the repo root where the reference is importable (tests/golden/_refshim.py):
    python -m tests.golden.gen_reference_checks
"""

import json
import lzma
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "reference_checks.json.xz")


def main():
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from tests.golden import diff_hot_path, diff_ingest, diff_online

    out = {"diff_hot_path": diff_hot_path.reference_outputs(), "diff_ingest": diff_ingest.reference_frames(),
           "diff_online": diff_online.reference_answers()}
    with lzma.open(PATH, "wt", preset=9) as fp:
        json.dump(out, fp, sort_keys=True)
    print(f"wrote {PATH}: {os.path.getsize(PATH)} bytes")
    return 0


if __name__ == "__main__":
    sys.exit(main())
