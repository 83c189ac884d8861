"""The kernels' three CHECKERS -- the batched scoring oracle, the columnar ingest oracle, the enrichment oracle -- against the
REAL reference classes on seeded random workloads.  The reference's answers are stored in tests/golden/reference_checks.json.xz
(made by tests/golden/gen_reference_checks.py); each check recomputes its side from the same seeds and compares.  The same
checks run live against the reference with `python -m tests.golden.<script>`; the other differential scripts
(`python -m tests.golden.run_diffs`, ~3 minutes) stay out of the suite."""
import importlib
import json
import lzma
import os

import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.json.xz")


@pytest.fixture(scope="module")
def reference():
    with lzma.open(GOLDEN, "rt") as fp:
        return json.load(fp)


@pytest.mark.parametrize("script,verdict", [("diff_hot_path", "the batched oracle equals the real reference"),
                                            ("diff_ingest", "ingest_columns equals the real reference"),
                                            ("diff_online", "identical on 500 random online services")])
def test_kernel_checkers_equal_the_real_reference(script, verdict, reference, capsys):
    mod = importlib.import_module(f"tests.golden.{script}")
    assert mod.check(reference[script]) == 0, capsys.readouterr().out[-1500:]
    assert verdict in capsys.readouterr().out
