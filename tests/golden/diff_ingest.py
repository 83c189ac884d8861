"""The checker of `columns_kernel` -- oracle/ingest.py `ingest_columns`, the vectorised restatement of the feature-set ingest
graph -- against the REAL reference step classes walking the frame one row at a time (storey-engine semantics: DataframeSource
emits a dict per row, every row goes through the steps' `_do_storey`, ReduceToDataFrame re-assembles; ingestion.py:38-127):
random config-5-shaped workloads (float32 columns with NaN, categorical codes with out-of-vocabulary values, counters, a
timestamp; Imputer -> MapValues(ranges, with originals) -> OneHotEncoder -> DateExtractor -> DropFeatures -> FeaturesetValidator)
at several widths and seeds.  Frames compared exactly (values, column order), violations by count.

The reference's frames are stored in tests/golden/reference_checks.json.xz (gen_reference_checks.py) as what `summary` keeps of
them: column order, a 64-bit SHA-256 digest of every column and the values of a fixed sample of rows.  The CPU suite runs `check`
against that on any machine.

    python -m tests.golden.diff_ingest      (live, needs the reference)
"""
import contextlib
import hashlib
import io
import os
import random
import sys
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402

from mlrun_b200.synthetic import ingest_workload  # noqa: E402
from oracle import ingest as oingest  # noqa: E402
from oracle import transforms as otransforms  # noqa: E402

VERDICT = "ingest_columns equals the real reference"
SAMPLE_ROWS = 16


def ref_steps():
    """the `api` object IngestWorkload.build_steps wants, over the real classes"""
    from tests.golden import api_reference as ref

    class RefSteps:
        Imputer, MapValues, OneHotEncoder, DateExtractor, DropFeatures = ref.Imputer, ref.MapValues, ref.OneHotEncoder, ref.DateExtractor, ref.DropFeatures

        @staticmethod
        def MinMaxValidator(**kw):
            return kw

        @staticmethod
        def FeaturesetValidator(validators):
            return ref.validator_step(validators, None)

    return RefSteps


def reference_rows(steps, df):
    out, printed = [], io.StringIO()
    with contextlib.redirect_stdout(printed):
        for row in df.to_dict("records"):
            body = row
            for step in steps:
                if type(step).__name__ == "FeaturesetValidator":
                    step.do(types.SimpleNamespace(body=body, key=None))
                else:
                    body = step.do(body)
            out.append(body)
    return pd.DataFrame(out, index=df.index), len([ln for ln in printed.getvalue().splitlines() if ln.strip()])


def workloads():
    rnd = random.Random(41)
    for case in range(12):
        yield case, ingest_workload(n_rows=rnd.randint(150, 400), seed=300 + case, n_f32=rnd.choice([24, 32, 48]), n_cat=rnd.choice([8, 12]),
                                    n_counter=rnd.choice([2, 5]), nan_frac=rnd.choice([0.02, 0.1, 0.3]))


def canonical(a):
    """a column in the form the comparison uses: float64 with one NaN and no negative zero; timestamps as int64 nanoseconds"""
    a = np.asarray(a)
    if a.dtype.kind == "M":
        return a.astype("datetime64[ns]").view(np.int64)
    a = a.astype(np.float64) + 0.0
    a[np.isnan(a)] = np.nan
    return a


def summary(frame, violations):
    """what the stored golden keeps of a frame: its columns, a digest of each, a fixed sample of rows, the violation count"""
    rows = np.sort(np.random.default_rng(len(frame)).choice(len(frame), size=min(SAMPLE_ROWS, len(frame)), replace=False))
    cols = [canonical(frame[c].to_numpy()) for c in frame.columns]
    return {"columns": list(frame.columns), "digests": [hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16] for a in cols],
            "rows": rows.tolist(), "sample": [a[rows].tolist() for a in cols], "violations": int(violations)}


def reference_frames():
    """the reference's row walk over every workload, kept as `summary` keeps it"""
    steps_api = ref_steps()
    return [summary(*reference_rows(wl.build_steps(steps_api), wl.df)) for _case, wl in workloads()]


def check(reference):
    """the oracle against `reference` (what reference_frames returned)"""
    rows = 0
    for (case, wl), want in zip(workloads(), reference, strict=True):
        with contextlib.redirect_stdout(io.StringIO()):
            got, violations = oingest.ingest_columns(wl.build_steps(otransforms), wl.df)
        mine = summary(got, sum(violations.values()))
        assert mine["columns"] == want["columns"], (case, mine["columns"][:8], want["columns"][:8])
        assert mine["rows"] == want["rows"], case
        for c, a, b, da, db in zip(want["columns"], mine["sample"], want["sample"], mine["digests"], want["digests"]):
            assert np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True), (case, c, a[:5], b[:5])
            assert da == db, (case, c, "values differ outside the sampled rows")
        assert mine["violations"] == want["violations"], (case, violations, want["violations"])
        rows += len(wl.df)
    print(f"{VERDICT}'s row walk on", rows, "rows of 12 random workloads")
    return 0


def main():
    return check(reference_frames())


if __name__ == "__main__":
    sys.exit(main())
