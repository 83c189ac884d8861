"""Feature-set statistics (`ingest(..., infer_options=...)`) on CPU: the oracle against the reference's own get_df_stats
(tests/golden/stats_golden.json), the product's host layer (mlrun_b200/feature_store/infer.py) on a numpy stand-in for the
two device entry points against the same goldens, and the infer_options plumbing of FeatureSet.ingest on the emulated
columns plan."""

import contextlib
import io
import json
import os

import numpy as np
import pandas as pd
import pytest

from tests import stats_frames, stats_oracle
from tests.stats_compare import assert_stats_match, reset
from tests.stats_standin import StatsStandIn

HERE = os.path.dirname(os.path.abspath(__file__))


def _goldens():
    with open(os.path.join(HERE, "golden", "stats_golden.json")) as fh:
        return json.load(fh)["frames"]


GOLDENS = _goldens()


def _types(d):
    return [(k, type(v).__name__, _types(v) if isinstance(v, dict) else None) for k, v in d.items()]


@pytest.mark.parametrize("g", GOLDENS, ids=[g["name"] for g in GOLDENS])
def test_oracle_equals_the_reference_exactly(g):
    df = stats_frames.from_spec(g["frame"])
    with np.errstate(all="ignore"):
        got = stats_oracle.get_df_stats(df, g["options"])
    assert got == g["stats"]
    assert _types(got) == _types(g["stats"])  # key order and value types, not only equality


def standin_stats(df, options):
    """the product's host layer over a frame whose columns are the stand-in's result slots"""
    from mlrun_b200 import _native as nat
    from mlrun_b200.feature_store import infer

    n = len(df)
    if not n:
        return {}
    slots, cols = {}, []
    for j, name in enumerate(df.columns):
        a = df[name].to_numpy()
        if a.dtype == np.float32:
            kind, slot, what = nat.STAT_F32, a, "num"
        elif a.dtype == np.float64:  # a date part with NaT rows
            kind, slot, what = nat.STAT_I32_NAT, np.where(np.isnan(a), -1, a).astype(np.int32), "num"
        elif a.dtype == np.bool_:
            kind, slot, what = nat.STAT_BOOL, a.astype(np.int32), "bool"
        elif a.dtype.kind == "M":
            kind, slot, what = nat.STAT_DT, a.view(np.int64), "dt"
        else:
            kind, slot, what = nat.STAT_I32, a.astype(np.int32), "num"
        slots[j] = slot
        cols.append(infer._Col(name, kind, j, a.dtype, what))
    return infer.describe_columns(StatsStandIn(slots, n), cols, n, df.index, options)


@pytest.mark.parametrize("g", GOLDENS, ids=[g["name"] for g in GOLDENS])
def test_host_layer_on_the_standin_equals_the_reference(g):
    df = stats_frames.from_spec(g["frame"])
    got = standin_stats(df, g["options"])
    assert_stats_match(got, g["stats"], reset(df, g["options"]))


def test_host_layer_on_random_frames_equals_the_oracle():
    """quantile positions, ties, negative values and histogram edges at sizes the goldens do not reach"""
    rng = np.random.default_rng(5)
    for n in (2, 3, 4, 5, 17, 1000, 4097):
        df = pd.DataFrame({
            "f": (rng.normal(size=n) * 10.0 ** rng.integers(-3, 4)).astype(np.float32),
            "g": rng.integers(-3, 3, size=n).astype(np.float32),
            "i": rng.integers(-50, 50, size=n).astype(np.int32),
            "b": rng.random(n) < 0.5,
            "t": pd.to_datetime(rng.integers(1.5e18, 1.8e18, size=n)).astype("datetime64[ns]"),
        })
        want = stats_oracle.get_df_stats(df, 8 | 16 | 4)
        assert_stats_match(standin_stats(df, 8 | 16 | 4), want, df.reset_index())


# ---- FeatureSet.ingest(..., infer_options=...) on the emulated columns plan
@pytest.fixture
def emulated(monkeypatch):
    from mlrun_b200.feature_store import ingest as bi
    from tests import stats_standin

    stats_standin.install(monkeypatch)
    return bi


def _config5_fset(bi, iw, name="s"):
    from mlrun_b200.feature_store import steps as bs

    fs = bi.FeatureSet(name, timestamp_key="timestamp")
    cur = fs.graph
    for st in iw.build_steps(bs):
        cur = cur.to(st)
    return fs


def test_infer_options_on_frames_and_columns(emulated):
    from mlrun_b200.feature_store import InferOptions
    from mlrun_b200.synthetic import ingest_workload

    bi = emulated
    iw = ingest_workload(n_rows=3000, seed=3)
    with contextlib.redirect_stdout(io.StringIO()):
        fs = _config5_fset(bi, iw)
        fs.ingest(iw.df)
        assert fs.status.stats == {} and fs.get_stats_table() is None  # Null (the default) computes nothing
        out = fs.ingest(iw.df, infer_options=InferOptions.default(), reference_dtypes=True)
        want = stats_oracle.get_df_stats(out, InferOptions.default())
        assert_stats_match(fs.status.stats, want, out.reset_index())
        assert list(fs.status.stats)[0] == "index" and "hist" in fs.status.stats["index"]
        table = fs.get_stats_table()
        assert list(table.index) == list(want) and "mean" in table.columns

        cols = {name: iw.df[name].to_numpy() for name in iw.df.columns}
        fc = _config5_fset(bi, iw, "c")
        batch = fc.ingest(cols, infer_options=InferOptions.Stats)  # no histograms, no index
        frame = batch.to_pandas()
    want = stats_oracle.get_df_stats(frame, InferOptions.Stats)
    assert_stats_match(fc.status.stats, want, frame)
    assert all("hist" not in v for v in fc.status.stats.values()) and "index" not in fc.status.stats


def test_entities_are_described_on_the_host_and_come_first(emulated):
    from mlrun_b200.feature_store import InferOptions
    from mlrun_b200.feature_store import steps as bs

    bi = emulated
    df = pd.DataFrame({"id": np.array([5, 3, 9, 1], np.int32), "x": np.array([1, np.nan, 3, 4], np.float32)})
    fs = bi.FeatureSet("e", entities=[bi.Entity("id")])
    fs.graph.to(bs.Imputer(mapping={"x": 2.0}))
    out = fs.ingest(df, infer_options=InferOptions.default())
    want = stats_oracle.get_df_stats(out, InferOptions.default())
    assert list(fs.status.stats) == ["id", "x"]
    assert_stats_match(fs.status.stats, want, out.reset_index())
    got = fs.ingest({"id": df["id"].to_numpy(), "x": df["x"].to_numpy()}, infer_options=InferOptions.default())
    assert list(fs.status.stats) == ["id", "x"] and fs.status.stats["x"] == want["x"] and got.names == ["x"]


def test_empty_frame_gives_empty_stats(emulated):
    from mlrun_b200.feature_store import InferOptions
    from mlrun_b200.feature_store import steps as bs

    bi = emulated
    fs = bi.FeatureSet("z")
    fs.graph.to(bs.Imputer(mapping={"x": 2.0}))
    fs.ingest(pd.DataFrame({"x": np.array([], np.float32)}), infer_options=InferOptions.default())
    assert fs.status.stats == {} and fs.get_stats_table() is None


def test_schema_and_preview_bits_are_accepted_and_ignored(emulated):
    from mlrun_b200.feature_store import InferOptions
    from mlrun_b200.feature_store import steps as bs

    bi = emulated
    assert InferOptions.default() == InferOptions.all() == 63 and InferOptions.all_stats() == 56
    assert InferOptions.get_common_options(InferOptions.default(), InferOptions.Histogram) == 16
    fs = bi.FeatureSet("p")
    fs.graph.to(bs.Imputer(mapping={"x": 2.0}))
    fs.ingest(pd.DataFrame({"x": np.array([1, 2], np.float32)}), infer_options=InferOptions.schema() | InferOptions.Preview)
    assert fs.status.stats == {}


def test_stats_table_feeds_the_online_impute_policies(emulated):
    """FeatureVector(..., stats=fset.get_stats_table()): the $mean / $std policies of the online service read the ingested
    feature set's statistics (feature_vector.py:886-890, 935-968)"""
    from mlrun_b200.feature_store import InferOptions
    from mlrun_b200.feature_store import online as bonline
    from mlrun_b200.feature_store import steps as bs

    bi = emulated
    rng = np.random.default_rng(2)
    df = pd.DataFrame({"id": np.arange(100, dtype=np.int32), "a": rng.normal(size=100).astype(np.float32),
                       "b": rng.normal(size=100).astype(np.float32)})
    fs = bi.FeatureSet("o", entities=[bi.Entity("id")])
    fs.graph.to(bs.Imputer(mapping={"a": 0.0}))
    out = fs.ingest(df, infer_options=InferOptions.default())
    table = fs.get_stats_table()
    vec = bonline.FeatureVector("v", ["a", "b"], ["id"], out, stats=table)
    assert vec.get_stats_table() is table
    values = bonline.OnlineVectorService(vec)._resolve_policy({"a": "$mean", "b": "$std"})  # what initialize() folds in
    assert values == {"a": float(np.float32(fs.status.stats["a"]["mean"])), "b": float(np.float32(fs.status.stats["b"]["std"]))}
    assert abs(fs.status.stats["a"]["mean"] - float(out["a"].mean())) <= 1e-6


@pytest.mark.parametrize("name,df,with_nat", stats_frames.date_part_frames(), ids=lambda v: v if isinstance(v, str) else "")
def test_date_parts_bool_and_nat_kinds_on_the_emulated_plan(emulated, name, df, with_nat):
    """the body of tests/test_gpu_ingest_stats.py::test_date_parts_bool_and_nat_kinds on the emulated plan"""
    from tests import test_gpu_ingest_stats as g

    g.test_date_parts_bool_and_nat_kinds(name, df, with_nat)
