"""Feature-set statistics of an ingested result, computed on the device (`ingest(..., infer_options=...)`).

The reference profiles what ingest produced with `get_df_stats` (mlrun/data_types/infer.py:104-149, called from
`_infer_from_static_df`, feature_store/api.py:1162-1196): `df.reset_index()` when the Index bit is set, then pandas
`describe(include="all")` per column, NaN entries dropped, plus a 20-bin `np.histogram` for numeric columns.  Here the
result columns are still resident on the GPU after the transform, so the numbers come from the `b2s_cols_stats_*` passes
(mlrun_b200/csrc/b2s_colstats.cu): counts, fp64 sums, min / max, exact order statistics (radix select), histogram counts.
This module turns them into the reference's dict: which columns are read how, the quantile interpolation (numpy's linear
method, in the frame column's dtype), the histogram edges (numpy's own, from the device's min / max), value types and the
key order pandas gives a mixed frame.  Entity (index) columns are keys, not device data: they are described on the host
with pandas.

Only Stats and Histogram (and Index) mean something here.  Entities / Features (schema inference) and Preview are accepted
and ignored.  FeatureSet.ingest defaults to `InferOptions.Null`, where the reference defaults to `InferOptions.default()`:
pass that for the reference behaviour.
"""

import math

import numpy as np

from .. import _native as nat

_QS = (0.25, 0.5, 0.75)
_NUMERIC = ("count", "mean", "std", "min", "25%", "50%", "75%", "max")
_DATETIME = ("count", "mean", "min", "25%", "50%", "75%", "max")
_BOOL = ("count", "unique", "top", "freq")


class InferOptions:
    """mlrun/data_types/data_types.py:152-184 (same bits)"""

    Null = 0
    Entities = 1
    Features = 2
    Index = 4
    Stats = 8
    Histogram = 16
    Preview = 32

    @staticmethod
    def schema():
        return InferOptions.Entities + InferOptions.Features + InferOptions.Index

    @staticmethod
    def all_stats():
        return InferOptions.Stats + InferOptions.Histogram + InferOptions.Preview

    @staticmethod
    def all():
        return InferOptions.schema() + InferOptions.Stats + InferOptions.Histogram + InferOptions.Preview

    @staticmethod
    def default():
        return InferOptions.all()

    @staticmethod
    def get_common_options(one, two):
        return one & two


def _py(val):
    """get_df_stats' conversion: floats and ints (Python bools kept) as Python scalars, anything else as its str -- numpy's
    bool_ is neither, so the `top` of a bool column is a string, 'True' or 'False'."""
    if isinstance(val, (float, np.floating)):
        return float(val)
    if isinstance(val, (int, np.integer)):
        return bool(val) if isinstance(val, bool) else int(val)
    return str(val)


def _is_nan(val):
    try:
        return val is None or val != val
    except (TypeError, ValueError):
        return False


def _quantile(a, b, n, q):
    """np.percentile's linear method for one q, given the order statistics floor(pos) and floor(pos) + 1 (clamped) as
    scalars of the column's dtype: numpy's _lerp, which reads both neighbours even at an integral position"""
    pos = (np.int64(n) - np.int64(1)) * np.float64(q)
    t = pos - np.floor(pos)
    with np.errstate(all="ignore"):
        diff = b - a
        return np.subtract(b, diff * (1 - t)) if t >= 0.5 else np.add(a, diff * t)


def _ranks(n):
    out = []
    for q in _QS:
        k = int(math.floor((n - 1) * q))
        out += [k, min(k + 1, n - 1)]
    return out


def _hist_setup(mn, mx, dtype):
    """np.histogram's uniform-bin operands for a column with these min / max (numpy/lib/_histograms_impl.py
    _get_outer_edges / _get_bin_edges): (bin kind, first_edge, last - first, edges in the bin dtype)"""
    a = np.array([mn, mx], dtype=dtype)
    if a.dtype == np.bool_:
        a = a.astype(np.uint8)  # numpy casts bool input to uint8
    first, last = a.min(), a.max()
    if first == last:
        first, last = first - 0.5, last + 0.5
    bin_type = np.result_type(first, last, a)
    if bin_type.kind in "iu":
        bin_type = np.result_type(bin_type, float)
    edges = np.linspace(first, last, nat.STAT_BINS + 1, endpoint=True, dtype=bin_type)
    dt = np.result_type(first, last)
    if dt.kind in "iu":
        den = np.subtract(np.asarray(last, dt), np.asarray(first, dt), casting="unsafe",
                          dtype=np.dtype(dt.str.replace("i", "u")))
    else:
        den = np.subtract(last, first, dtype=dt)
    kind = 1 if edges.dtype == np.float32 else 2
    return kind, float(first), float(den), edges.astype(np.float64)


class _Col:
    """one result column as the statistics see it: how the device reads its slot and what the frame holds"""

    def __init__(self, name, kind, slot, dtype, what):
        self.name, self.kind, self.slot, self.dtype, self.what = name, kind, slot, np.dtype(dtype), what


def result_columns(plan, data, counters):
    """[_Col] for the columns of an IngestPlan's result: the device kind follows the output kind and the run's counters
    (a date part with NaT rows is a float64 column with NaN; a map whose every row got an integer label is an int column)"""
    cols = []
    for name, slot, how in plan.out:
        dt = data[name].dtype
        if how == "f32":
            kind = nat.STAT_F32
        elif how == "i32":
            kind = nat.STAT_I32
        elif how == "dt":
            kind = nat.STAT_DT
        elif how[0] == "map":
            kind = nat.STAT_F32
        elif counters[how[1]]:
            kind = nat.STAT_I32_NAT
        else:
            kind = nat.STAT_BOOL if how[2] else nat.STAT_I32
        what = "dt" if kind == nat.STAT_DT else ("bool" if dt == np.bool_ else "num")
        cols.append(_Col(name, kind, slot, dt, what))
    return cols


def _decode(kind, bits):
    if kind == nat.STAT_F32:
        return np.array([bits], dtype=np.int64).astype(np.uint32).view(np.float32)[0]
    return np.int64(bits)


def device_stats(cplan, cols, n_rows, options):
    """{name: stats} of the device columns, each as (describe index before dropna, {stat: value})"""
    hist_on = bool(options & InferOptions.Histogram)
    summary, _ = cplan.stats_begin([c.kind for c in cols], [c.slot for c in cols], n_rows)
    n = len(cols)
    means = np.full(n, np.nan)
    hist_kind = np.zeros(n, dtype=np.int32)
    hist = np.zeros((n, 23))
    ranks = np.full((n, nat.STAT_RANKS), -1, dtype=np.int64)
    for i, c in enumerate(cols):
        s = summary[i]
        cnt = int(s["count"])
        if c.what != "bool" and cnt:
            ranks[i] = _ranks(cnt)
        if c.what == "num" and cnt >= 2 and not (s["pos_inf"] or s["neg_inf"]):
            means[i] = s["sum"] / cnt
        clean = cnt > 0 and s["missing"] == 0 and not (s["pos_inf"] or s["neg_inf"])
        if hist_on and c.what != "dt" and clean:
            mn, mx = _decode(c.kind, s["min_bits"]), _decode(c.kind, s["max_bits"])
            hist_kind[i], hist[i, 0], hist[i, 1], hist[i, 2:] = _hist_setup(mn, mx, c.dtype)
    m2, counts, order, _ = cplan.stats_finish(means, hist_kind, hist, ranks)
    out = {}
    for i, c in enumerate(cols):
        s = summary[i]
        cnt = int(s["count"])
        vals = {}
        if c.what == "bool":
            ones, zeros = int(s["ones"]), cnt - int(s["ones"])
            top = np.bool_(s["first_bits"] if ones == zeros else ones > zeros)  # a tie: the value of the first row
            vals = {"count": cnt, "unique": int(ones > 0) + int(zeros > 0), "top": top, "freq": max(ones, zeros)}
            index = _BOOL
        elif c.what == "dt":
            import pandas as pd

            index = _DATETIME
            vals["count"] = cnt
            if cnt:
                o = order[i]
                vals["mean"] = pd.Timestamp(int(s["sum"] / cnt))
                vals["min"] = pd.Timestamp(int(s["min_bits"]))
                for j, q in enumerate(_QS):
                    v = _quantile(np.int64(o[2 * j]), np.int64(o[2 * j + 1]), cnt, q)
                    vals[f"{int(q * 100)}%"] = pd.Timestamp(np.array([v]).astype("datetime64[ns]")[0])
                vals["max"] = pd.Timestamp(int(s["max_bits"]))
        else:
            index = _NUMERIC
            vals["count"] = float(cnt)
            if cnt:
                as_dtype = c.dtype.type
                f32 = c.dtype == np.float32
                mean = s["sum"] / cnt
                vals["mean"] = float(np.float32(mean)) if f32 else float(mean)  # pandas reduces float32 columns in float32
                if np.isfinite(means[i]):
                    std = math.sqrt(m2[i] / (cnt - 1))
                    vals["std"] = float(np.float32(std)) if f32 else std
                vals["min"] = float(as_dtype(_decode(c.kind, s["min_bits"])))
                o = order[i]
                for j, q in enumerate(_QS):
                    a, b = (as_dtype(_decode(c.kind, o[2 * j])), as_dtype(_decode(c.kind, o[2 * j + 1])))
                    v = _quantile(a, b, cnt, q)
                    # pandas returns the quantiles of a float32 column with NaN in float32
                    vals[f"{int(q * 100)}%"] = float(np.float32(v) if f32 and s["missing"] else v)
                vals["max"] = float(as_dtype(_decode(c.kind, s["max_bits"])))
        if hist_kind[i]:
            vals["hist"] = [counts[i].tolist(), hist[i, 2:].astype(np.float32 if hist_kind[i] == 1 else np.float64).tolist()]
        out[c.name] = (index, vals)
    return out


def host_stats(name, values, options):
    """an entity (index) column, described on the host with pandas exactly as get_df_stats does"""
    import pandas as pd

    frame = pd.DataFrame({name: values})
    desc = frame.describe(include="all")[name]
    vals = {k: v for k, v in desc.items()}
    if options & InferOptions.Histogram and pd.api.types.is_numeric_dtype(frame[name]):
        try:
            h, edges = np.histogram(frame[name], bins=nat.STAT_BINS)
            vals["hist"] = [h.tolist(), edges.tolist()]
        except Exception:  # noqa: BLE001 -- NaN / inf: numpy raises and get_df_stats leaves the histogram out
            pass
    return list(desc.index), vals


def assemble(described):
    """[(name, (describe index, {stat: value}))] in frame order -> get_df_stats' dict: pandas unions the stat names of the
    columns' describes, shortest first (describe(include="all")), and every column lists its non-NaN entries in that order"""
    names, seen = [], set()
    for index in sorted((idx for _n, (idx, _v) in described), key=len):
        for k in index:
            if k not in seen:
                seen.add(k)
                names.append(k)
    out = {}
    for name, (_idx, vals) in described:
        d = {k: _py(vals[k]) for k in names if k in vals and not _is_nan(vals[k])}
        if "hist" in vals:
            d["hist"] = vals["hist"]
        out[name] = d
    return out


def index_columns(index, n_rows):
    """the columns df.reset_index() puts first: [(name, values | None)], None for the row numbers 0..n-1 (described on the
    device without reading memory).  `index` is a pandas Index, or {entity: array} of a columnar batch."""
    if isinstance(index, dict):
        return [(k, np.asarray(v)) for k, v in index.items()] if index else [("index", None)]
    import pandas as pd

    if isinstance(index, pd.MultiIndex):
        return [(name if name is not None else f"level_{i}", index.get_level_values(i)) for i, name in enumerate(index.names)]
    name = index.name if index.name is not None else "index"
    if isinstance(index, pd.RangeIndex) and index.start == 0 and index.step == 1 and len(index) == n_rows:
        return [(name, None)]
    return [(name, index)]


def describe(plan, data, n_rows, index, options):
    """get_df_stats of the frame an IngestPlan run produced (its result still on the device)"""
    if not n_rows or not data:
        return {}
    return describe_columns(plan.plan, result_columns(plan, data, plan.counters), n_rows, index, options)


def describe_columns(cplan, cols, n_rows, index, options):
    """get_df_stats of a frame whose columns `cols` are result slots of `cplan` and whose index is `index`"""
    cols = list(cols)
    names, host, taken = [], {}, {c.name for c in cols}
    if options & InferOptions.Index:  # reset_index puts the index columns first
        for name, values in index_columns(index, n_rows):
            if name in taken:
                name = "level_0"  # reset_index's name when "index" is taken
            names.append(name)
            if values is None:
                cols.insert(0, _Col(name, nat.STAT_ROW, -1, np.int64, "num"))
            else:
                host[name] = host_stats(name, values, options)
    names += [c.name for c in cols if c.kind != nat.STAT_ROW]
    dev = device_stats(cplan, cols, n_rows, options)
    return assemble([(n, host[n] if n in host else dev[n]) for n in names])
