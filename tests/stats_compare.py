"""Comparison of two get_df_stats dicts: exact for everything (key order and value types included) except mean / std,
which pandas reduces in float32 for float32 columns and in a different order: mean within 1e-5 * mean(|x|) and std within
rtol 1e-5 for float32 columns, rtol 1e-12 for the others, datetime means within 1 us."""

import numpy as np
import pandas as pd


def assert_stats_match(got, want, frame):
    """`frame` is the described frame after reset_index (for the per-column dtype and mean(|x|))"""
    assert list(got) == list(want), (list(got), list(want))
    for col in want:
        g, w = got[col], want[col]
        assert list(g) == list(w), (col, list(g), list(w))
        s = frame[col]
        for k in w:
            assert type(g[k]) is type(w[k]), (col, k, type(g[k]), type(w[k]))
            if isinstance(w[k], float) and not np.isfinite(w[k]):
                assert g[k] == w[k], (col, k, g[k], w[k])
            elif k == "mean" and s.dtype.kind == "M":
                assert abs(pd.Timestamp(g[k]) - pd.Timestamp(w[k])) <= pd.Timedelta(1, "us"), (col, g[k], w[k])
            elif k in ("mean", "std") and s.dtype == np.float32:
                a = s.to_numpy()
                scale = float(np.mean(np.abs(a[np.isfinite(a)].astype(np.float64)))) if k == "mean" else abs(w[k])
                assert abs(g[k] - w[k]) <= 1e-5 * scale + 1e-30, (col, k, g[k], w[k])
            elif k in ("mean", "std"):
                assert abs(g[k] - w[k]) <= 1e-12 * abs(w[k]) + 1e-300, (col, k, g[k], w[k])
            else:
                assert g[k] == w[k], (col, k, g[k], w[k])


def reset(df, options):
    return df.reset_index() if options & 4 and df.index.names else df
