"""The statistics of the product's FeatureSet.ingest(df, infer_options=InferOptions.default(), reference_dtypes=True) against
the REAL reference: its step classes walking the frame one row at a time, then its own get_df_stats
(mlrun/data_types/infer.py:104-149) on the frame that walk produced (build container only).  The device is emulated: the
columnar kernel by tests/device_emulator.py, the statistics entry points by tests/stats_standin.py, so what this pins is the
host side of the statistics on random config-5-shaped workloads -- column kinds, quantile interpolation, histogram edges,
value types and key order; the CUDA passes are compared with the oracle in `-m gpu`.

    python -m tests.golden.diff_ingest_stats
"""
import contextlib
import io
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np  # noqa: E402

from mlrun_b200.feature_store import InferOptions  # noqa: E402
from mlrun_b200.feature_store import ingest as bingest  # noqa: E402
from mlrun_b200.feature_store import steps as bsteps  # noqa: E402
from mlrun_b200.synthetic import ingest_workload  # noqa: E402
from tests import stats_standin  # noqa: E402
from tests.golden.diff_ingest import ref_steps, reference_rows  # noqa: E402
from tests.stats_compare import assert_stats_match  # noqa: E402


class _Patch:  # monkeypatch.setattr without pytest
    def setattr(self, obj, name, value, raising=True):
        setattr(obj, name, value)


def main():
    stats_standin.install(_Patch())
    RefSteps = ref_steps()  # loads the reference in place (tests/golden/_refshim.py)
    from mlrun.data_types.infer import get_df_stats

    rnd = random.Random(47)
    rows = cols = widened = 0
    for case in range(10):
        wl = ingest_workload(n_rows=rnd.randint(2, 400), seed=500 + case, n_f32=rnd.choice([8, 24, 32]), n_cat=rnd.choice([4, 8]),
                             n_counter=rnd.choice([2, 5]), nan_frac=rnd.choice([0.0, 0.02, 0.3]))
        want_frame, _ = reference_rows(wl.build_steps(RefSteps), wl.df)
        fset = bingest.FeatureSet(f"case{case}", timestamp_key="timestamp")
        cur = fset.graph
        for st in wl.build_steps(bsteps):
            cur = cur.to(st)
        with contextlib.redirect_stdout(io.StringIO()):
            got_frame = fset.ingest(wl.df, infer_options=InferOptions.default(), reference_dtypes=True)
        # The row walk re-assembles Python floats: its float columns are float64 where the product's stay float32 (same
        # values).  Statistics describe the frame they are given, so the reference runs on its frame in the product's dtypes;
        # the columns whose statistics the float64 widening alone changes are counted (DESIGN 2).
        cast = want_frame.astype(got_frame.dtypes.to_dict())
        with np.errstate(all="ignore"):
            want = get_df_stats(cast, InferOptions.default())
            wide = get_df_stats(want_frame, InferOptions.default())
        assert_stats_match(fset.status.stats, want, got_frame.reset_index())
        widened += sum(1 for c in want if want[c] != wide[c])
        rows += len(wl.df)
        cols += len(want)
    print("ingest statistics equal the real reference's get_df_stats on", cols, "columns,", rows, "rows of 10 random workloads;",
          widened, "float columns differ only because the row walk's frame holds them as float64")
    return 0


if __name__ == "__main__":
    sys.exit(main())
