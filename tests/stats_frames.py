"""The frames the feature-set statistics are pinned on (tests/golden/stats_golden.json) and their JSON form.

Every kind of result column the device describes (float32, int32 / int64, bool, datetime64[ns], the float64-with-NaN
date parts) with NaN, +-inf, all-NaN, constant and single-row columns, bool ties, NaT, quantile positions next to
infinities, values on and next to histogram edges, and frames with and without a datetime column, with an entity index,
a RangeIndex, and empty."""

import numpy as np
import pandas as pd


def frames():
    """[(name, DataFrame, infer options)] -- options are InferOptions bits (Stats 8, Histogram 16, Index 4)"""
    rng = np.random.default_rng(20261017)
    out = []
    n = 257
    f = rng.normal(size=n).astype(np.float32) * 3 + 1
    f_nan = f.copy()
    f_nan[::7] = np.nan
    f_pinf = f.copy()
    f_pinf[5] = np.inf
    f_both = f.copy()
    f_both[3], f_both[9] = np.inf, -np.inf
    base = {
        "f": f, "f_nan": f_nan, "f_pinf": f_pinf, "f_both": f_both,
        "f_allnan": np.full(n, np.nan, np.float32), "f_const": np.full(n, 2.5, np.float32),
        "i": rng.integers(-1000, 1000, size=n).astype(np.int32), "i_const": np.full(n, 7, np.int32),
        "i64": rng.integers(-2**31, 2**31, size=n).astype(np.int64),
        "b": (rng.random(n) < 0.3), "b_const": np.zeros(n, bool),
    }
    out.append(("numeric_range_index", pd.DataFrame(base), 8 | 16 | 4))
    t = pd.to_datetime(rng.integers(1.5e18, 1.8e18, size=n)).astype("datetime64[ns]")
    t = pd.Series(t)
    t[[4, 40]] = pd.NaT
    part = pd.Series(rng.integers(1, 13, size=n).astype(np.float64))
    part[[4, 40]] = np.nan
    with_dt = dict(base, ts=t.to_numpy(), ts_month=part.to_numpy())
    out.append(("with_datetime", pd.DataFrame(with_dt), 8 | 16 | 4))
    out.append(("with_datetime_no_hist", pd.DataFrame(with_dt), 8 | 4))
    out.append(("with_datetime_no_index", pd.DataFrame(with_dt), 8 | 16))
    # bool ties: the first row decides top
    out.append(("bool_ties", pd.DataFrame({"ft": np.array([False, True]), "tf": np.array([True, False]),
                                           "x": np.array([1.0, 2.0], np.float32)}), 8 | 16 | 4))
    one_t = pd.Series(pd.to_datetime([1_600_000_000_123_456_789])).astype("datetime64[ns]").to_numpy()
    out.append(("single_row", pd.DataFrame({"f": np.array([1.5], np.float32), "i": np.array([3], np.int32),
                                            "b": np.array([True]), "t": one_t}), 8 | 16 | 4))
    # quantile positions next to infinities: n = 3 (integral 50 %), n = 5 / 6 / 8 (integral and fractional positions)
    inf = np.inf
    out.append(("inf_quantiles_3", pd.DataFrame({"x": np.array([1, 2, inf], np.float32),
                                                 "y": np.array([-inf, 2, 3], np.float32)}), 8 | 16 | 4))
    out.append(("inf_quantiles_6", pd.DataFrame({"x": np.array([1, 2, 3, 4, 5, inf], np.float32),
                                                 "y": np.array([-inf, -inf, 0, 1, inf, inf], np.float32),
                                                 "z": np.array([-inf, 0, 0, 0, 0, 1], np.float32)}), 8 | 16 | 4))
    out.append(("inf_quantiles_8", pd.DataFrame({"x": np.array([1, inf, 2, 3, inf, 4, 5, 6], np.float32),
                                                 "y": np.array([-inf, 1, 2, 3, 4, 5, 6, 7], np.float32)}), 8 | 16 | 4))
    # values on and next to the histogram edges (float32 bins for float32, float64 bins for ints)
    e32 = np.linspace(np.float32(-1.3), np.float32(2.9), 21, dtype=np.float32)
    on = np.concatenate([e32, np.nextafter(e32, np.float32(-np.inf)), np.nextafter(e32, np.float32(np.inf))])
    on = np.clip(on, e32[0], e32[-1]).astype(np.float32)
    ints = np.concatenate([np.arange(-10, 31, dtype=np.int32), np.array([-10, 30, 11, 12], np.int32)])
    m = min(len(on), len(ints))
    out.append(("hist_edges", pd.DataFrame({"f": on[:m], "i": ints[:m], "w": (np.arange(m) * 7919 % 1009).astype(np.int32)}),
                8 | 16 | 4))
    # entity index (string keys: described on the host) and an integer entity index
    idx = pd.Index([f"k{i}" for i in range(50)], name="key")
    out.append(("entity_string_index", pd.DataFrame({"f": rng.normal(size=50).astype(np.float32),
                                                     "i": rng.integers(0, 9, 50).astype(np.int32)}, index=idx), 8 | 16 | 4))
    idx2 = pd.Index(rng.integers(0, 10**6, 40).astype(np.int64), name="id")
    out.append(("entity_int_index", pd.DataFrame({"f": rng.normal(size=40).astype(np.float32)}, index=idx2), 8 | 16 | 4))
    out.append(("empty", pd.DataFrame({"f": np.array([], np.float32), "i": np.array([], np.int32)}), 8 | 16 | 4))
    return out


def to_spec(df):
    cols = []
    for name in df.columns:
        cols.append(_col(name, df[name]))
    index = None if isinstance(df.index, pd.RangeIndex) else _col(df.index.name, pd.Series(df.index))
    return {"columns": cols, "index": index, "n": len(df)}


def _col(name, s):
    dt = str(s.dtype)
    if dt.startswith("datetime64"):
        vals = [None if pd.isna(v) else int(v) for v in s.astype("int64").where(s.notna(), 0)]
        vals = [None if pd.isna(x) else v for v, x in zip(vals, s)]
    elif dt == "bool":
        vals = [bool(v) for v in s]
    elif dt in ("object", "str", "string"):
        vals = [str(v) for v in s]
        dt = "str"
    elif s.dtype.kind == "f":
        vals = [float(v) for v in s]
    else:
        vals = [int(v) for v in s]
    return {"name": name, "dtype": dt, "values": vals}


def _series(c):
    if c["dtype"].startswith("datetime64"):
        return pd.Series(pd.array([pd.NaT if v is None else pd.Timestamp(v) for v in c["values"]], dtype="datetime64[ns]"))
    if c["dtype"] == "str":
        return pd.Series(c["values"], dtype=object)
    return pd.Series(np.array(c["values"], dtype=c["dtype"]))


def from_spec(spec):
    data = {c["name"]: _series(c).to_numpy() for c in spec["columns"]}
    if spec["index"] is None:
        return pd.DataFrame(data, index=pd.RangeIndex(spec["n"]))
    idx = pd.Index(_series(spec["index"]).to_numpy(), name=spec["index"]["name"])
    return pd.DataFrame(data, index=idx)


DATE_PARTS = ["is_month_start", "is_month_end", "is_leap_year", "is_year_start", "hour", "day", "month", "day_of_week",
              "week", "day_of_year"]


def date_part_frames():
    """[(name, DataFrame with a datetime64[ns] "ts" and a float32 "x", with_nat)] for a DateExtractor over "ts": without NaT
    the is_* parts are bool columns (with ties: is_month_start alternates from True, is_month_end from False; is_leap_year
    is constant True, is_year_start constant False) and the others int columns; with NaT rows every part is a float64
    column with NaN"""
    rng = np.random.default_rng(77)
    out = []
    for n in (6, 150_002):  # the larger one spans several 64 Ki-row chunks and runs the pipelined host path
        day = np.where(np.arange(n) % 2 == 0, np.datetime64("2024-03-01", "ns"), np.datetime64("2024-03-31", "ns"))
        ts = day + rng.integers(0, 86_400 * 10**9, size=n).astype("timedelta64[ns]")
        out.append((f"bool_parts_{n}", pd.DataFrame({"ts": ts, "x": rng.normal(size=n).astype(np.float32)}), False))
    n = 20_000
    ts = pd.Series(pd.to_datetime(rng.integers(1.5e18, 1.8e18, size=n)).astype("datetime64[ns]"))
    ts[::7] = pd.NaT
    out.append(("nat_parts", pd.DataFrame({"ts": ts.to_numpy(), "x": rng.normal(size=n).astype(np.float32)}), True))
    return out
