"""Feature-set statistics on the device (b2s_cols_stats_* over the columns plan's resident result) vs the CPU oracle
applied to the frame the product returns.  Exact for counts, min, max, quantiles, histogram counts and edges,
unique / top / freq, key order and value types; mean / std within the bounds of tests/stats_compare.py.  Needs a B200."""

import contextlib
import io
import json
import os

import numpy as np
import pandas as pd
import pytest

pytestmark = pytest.mark.gpu

from mlrun_b200 import _native as nat  # noqa: E402
from mlrun_b200.feature_store import InferOptions  # noqa: E402
from mlrun_b200.feature_store import columnar  # noqa: E402
from mlrun_b200.feature_store import ingest as bi  # noqa: E402
from mlrun_b200.feature_store import steps as bs  # noqa: E402
from mlrun_b200.synthetic import ingest_workload  # noqa: E402
from tests import stats_frames, stats_oracle  # noqa: E402
from tests.stats_compare import assert_stats_match, reset  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ALL = InferOptions.default()


@pytest.fixture(scope="module", autouse=True)
def _device():
    nat.init(0)
    yield


def _fset(wl, name="s", entities=None):
    fs = bi.FeatureSet(name, timestamp_key="timestamp", entities=entities)
    cur = fs.graph
    for st in wl.build_steps(bs):
        cur = cur.to(st)
    return fs


@pytest.mark.parametrize("n_rows", [1, 5, 4097, 20000, 300_000])
def test_config5_stats_match_the_oracle(n_rows):
    wl = ingest_workload(n_rows=n_rows, seed=70 + n_rows % 5)
    fs = _fset(wl)
    with contextlib.redirect_stdout(io.StringIO()):
        out = fs.ingest(wl.df, infer_options=ALL, reference_dtypes=n_rows % 2 == 1)
    with np.errstate(all="ignore"):
        want = stats_oracle.get_df_stats(out, ALL)
    assert_stats_match(fs.status.stats, want, out.reset_index())
    assert fs.get_stats_table().shape[0] == len(out.columns) + 1


def test_columnar_path_stats_match_the_oracle():
    wl = ingest_workload(n_rows=150_000, seed=8)
    src = {name: wl.df[name].to_numpy() for name in wl.df.columns}
    cols = columnar.pinned_columns(src, len(wl.df))
    for name, a in cols.items():
        a[...] = src[name]
    fs = _fset(wl, "c")
    with contextlib.redirect_stdout(io.StringIO()):
        batch = fs.ingest(cols, infer_options=ALL)
    frame = batch.to_pandas()
    with np.errstate(all="ignore"):
        want = stats_oracle.get_df_stats(frame, ALL)
    assert_stats_match(fs.status.stats, want, frame.reset_index())


def _goldens():
    with open(os.path.join(HERE, "golden", "stats_golden.json")) as fh:
        return json.load(fh)["frames"]


@pytest.mark.parametrize("g", _goldens(), ids=lambda g: g["name"])
def test_golden_frames_through_a_pass_through_feature_set(g):
    """each golden frame as the device takes it (int64 narrowed to int32, float64 columns left out: they are not device
    input) through a graph that passes every column through unchanged"""
    df = stats_frames.from_spec(g["frame"])
    keep = {}
    for name in df.columns:
        a = df[name].to_numpy()
        if a.dtype == np.int64:
            keep[name] = a.astype(np.int32)
        elif a.dtype != np.float64:
            keep[name] = a
    src = pd.DataFrame(keep, index=df.index)
    entities = None
    if not isinstance(df.index, pd.RangeIndex):
        entities = [bi.Entity(df.index.name)]
        src = src.reset_index()
    fs = bi.FeatureSet("p", entities=entities)
    fs.graph.to(bs.Imputer(mapping={}))
    out = fs.ingest(src, infer_options=g["options"])
    with np.errstate(all="ignore"):
        want = stats_oracle.get_df_stats(out, g["options"])
    assert_stats_match(fs.status.stats, want, reset(out, g["options"]))
    if not len(df):
        assert fs.status.stats == {} and fs.get_stats_table() is None


@pytest.mark.parametrize("name,df,with_nat", stats_frames.date_part_frames(), ids=lambda v: v if isinstance(v, str) else "")
def test_date_parts_bool_and_nat_kinds(name, df, with_nat):
    """DateExtractor parts: without NaT the is_* parts are bool columns (the device's ones / row-0 / unique-top-freq path,
    with ties) and the others int columns; with NaT rows every part is a float64 column with NaN (the date-part kind whose
    -1 marks a missing value)"""
    fs = bi.FeatureSet("d", timestamp_key="ts")
    fs.graph.to(bs.DateExtractor(parts=stats_frames.DATE_PARTS, timestamp_col="ts"))
    out = fs.ingest(df, infer_options=ALL)
    kinds = {out[f"ts_{p}"].dtype.kind for p in stats_frames.DATE_PARTS}
    assert kinds == ({"f"} if with_nat else {"b", "i"})
    with np.errstate(all="ignore"):
        want = stats_oracle.get_df_stats(out, ALL)
    assert_stats_match(fs.status.stats, want, out.reset_index())
    if not with_nat:
        assert fs.status.stats["ts_is_month_start"]["top"] == "True" and fs.status.stats["ts_is_month_end"]["top"] == "False"
        assert fs.status.stats["ts_is_month_start"]["freq"] == len(df) // 2


def test_finish_refuses_a_result_replaced_after_begin():
    """b2s_cols_stats_finish describes what b2s_cols_stats_begin saw: a host run of the plan in between is an error"""
    df = pd.DataFrame({"x": np.arange(1000, dtype=np.float32)})
    fs = bi.FeatureSet("g")
    fs.graph.to(bs.Imputer(mapping={}))
    fs.ingest(df)
    cplan = fs.plan.plan
    summary, _ = cplan.stats_begin([nat.STAT_F32], [fs.plan.out[0][1]], len(df))
    assert int(summary[0]["count"]) == 1000
    fs.ingest(df)
    with pytest.raises(nat.NativeError, match="run again"):
        cplan.stats_finish(np.zeros(1), np.zeros(1, np.int32), np.zeros((1, 23)), np.full((1, nat.STAT_RANKS), -1))
    out = fs.ingest(df, infer_options=ALL)  # begin + finish back to back still work
    assert fs.status.stats["x"]["max"] == 999.0 and len(out) == 1000
