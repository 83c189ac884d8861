"""CPU oracle of the feature-set statistics: get_df_stats (mlrun/data_types/infer.py:104-149) restated per column with
numpy primitives, so that each behaviour pandas' describe(include="all") contributes is visible and named.  Pinned to the
real function by tests/golden/stats_golden.json (tests/test_ingest_stats_cpu.py); the product's device path is compared
with it in tests/test_gpu_ingest_stats.py.  Lives with the tests: nothing in mlrun_b200 imports it.

QUIRK marks a behaviour of the reference (through pandas / numpy) that a straightforward implementation would get wrong."""

import math

import numpy as np
import pandas as pd

NUM_BINS = 20  # mlrun/data_types/infer.py default_num_bins
INDEX, STATS, HISTOGRAM = 4, 8, 16
_NUMERIC = ("count", "mean", "std", "min", "25%", "50%", "75%", "max")
_DATETIME = ("count", "mean", "min", "25%", "50%", "75%", "max")
_CATEGORICAL = ("count", "unique", "top", "freq")


def _categorical(a):
    # QUIRK: pandas' top is value_counts().index[0]; value_counts sorts by count with ties in order of first appearance,
    # so [False, True] gives False and [True, False] gives True
    seen = {}
    for v in a:
        if v is None or (isinstance(v, float) and math.isnan(v)):
            continue
        seen[v] = seen.get(v, 0) + 1
    vals = {"count": sum(seen.values()), "unique": len(seen)}
    if seen:
        top = max(seen, key=lambda k: seen[k])  # max keeps the first of equal counts
        vals["top"], vals["freq"] = top, seen[top]
    return _CATEGORICAL, vals


def _numeric(s):
    a = s.to_numpy()
    v = a[~np.isnan(a)] if a.dtype.kind == "f" else a
    vals = {"count": float(len(v))}  # QUIRK: the count of a numeric column is a float
    if len(v):
        vals["mean"] = s.mean()  # pandas' own reduction (float32 columns are added pairwise in float32)
        vals["std"] = s.std()    # ddof 1; NaN (dropped) for one value or with an inf
        vals["min"], vals["max"] = np.float64(v.min()), np.float64(v.max())  # QUIRK: floats, also for int columns
        with np.errstate(all="ignore"):
            # QUIRK: numpy's linear interpolation reads both neighbours even at an integral position, so [1, 2, inf] has no
            # 50 % (2 + (inf - 2) * 0 is NaN); the difference of the neighbours is taken in the column's dtype
            qs = np.percentile(v, [25.0, 50.0, 75.0])
        if a.dtype == np.float32 and len(v) < len(a):
            qs = qs.astype(np.float32)  # QUIRK: with NaN in a float32 column pandas returns its quantiles as float32
        for q, p in zip((25, 50, 75), qs):
            vals[f"{q}%"] = p
    return _NUMERIC, vals


def _datetime(s):
    a = s.to_numpy()
    ok = ~np.isnat(a)
    v = a[ok].view(np.int64)
    vals = {"count": int(ok.sum())}  # QUIRK: an int here, where numeric columns have a float count
    if len(v):
        vals["mean"] = s.mean()
        vals["min"], vals["max"] = pd.Timestamp(int(v.min())), pd.Timestamp(int(v.max()))
        for q, p in zip((25, 50, 75), np.percentile(v, [25.0, 50.0, 75.0])):
            vals[f"{q}%"] = pd.Timestamp(np.array([p]).astype("datetime64[ns]")[0])  # float -> ns truncates
    return _DATETIME, vals


def _value(val):
    """get_df_stats' conversion: float / int / bool as Python scalars, everything else (Timestamps, strings) as str.
    QUIRK: numpy's bool_ is neither a float nor an integer type, so the `top` of a bool column is a string, 'True' or
    'False'."""
    if isinstance(val, (float, np.floating)):
        return float(val)
    if isinstance(val, (int, np.integer)):
        return bool(val) if isinstance(val, bool) else int(val)
    return str(val)


def get_df_stats(df, options):
    if df.empty:
        return {}
    if options & INDEX and df.index.names:
        df = df.reset_index()  # QUIRK: a RangeIndex becomes a column named "index" holding the row numbers
    described = []
    for name in df.columns:
        s = df[name]
        kind = s.dtype.kind
        if kind == "b" or kind == "O":
            index, vals = _categorical(s.to_numpy())
        elif kind == "M":
            index, vals = _datetime(s)
        else:
            index, vals = _numeric(s)
        if options & HISTOGRAM and kind in "biuf":
            try:
                # QUIRK: np.histogram casts bool to uint8 and uses float64 bins for integer input; any NaN or inf raises,
                # and get_df_stats then leaves the histogram out
                counts, edges = np.histogram(s.to_numpy(), bins=NUM_BINS)
                vals["hist"] = [counts.tolist(), edges.tolist()]
            except ValueError:
                pass
        described.append((name, index, vals))
    # QUIRK: describe(include="all") unions the stat names of the columns' describes, shortest list first, so a datetime
    # column moves std after max for every numeric column of the frame
    order, seen = [], set()
    for index in sorted((d[1] for d in described), key=len):
        for k in index:
            if k not in seen:
                seen.add(k)
                order.append(k)
    out = {}
    for name, _index, vals in described:
        d = {}
        for k in order:
            if k in vals and not (vals[k] is pd.NaT or (isinstance(vals[k], (float, np.floating)) and math.isnan(vals[k]))):
                d[k] = _value(vals[k])
        if "hist" in vals:
            d["hist"] = vals["hist"]
        out[name] = d
    return out
