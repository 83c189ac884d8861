"""ColumnsPlan: the lowered form of a feature-set graph over DataFrame-shaped data (thin wrapper over the
`b2s_cols_*` C-ABI, include/b200serve.h "columnar ingest").  Input and output are columnar: one contiguous
4-byte-word array per column (8-byte columns take two slots)."""

import ctypes as C

import numpy as np

from . import _native as nat

F32, I32, I64 = nat.COL_F32, nat.COL_I32, nat.COL_I64
_WORDS = {F32: 1, I32: 1, I64: 2}


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _check_args(check):
    """check = (min | None, max | None) -> (bits, cmin, cmax)"""
    if not check:
        return 0, 0.0, 0.0
    lo, hi = check
    return (1 if lo is not None else 0) | (2 if hi is not None else 0), float(lo or 0.0), float(hi or 0.0)


class ColumnsPlan:
    def __init__(self, n_in_slots):
        self._lib = nat.load()
        self.n_in = int(n_in_slots)
        self._h = C.c_void_p()
        nat.check(self._lib.b2s_cols_create(self.n_in, C.byref(self._h)))
        self.finalized = False
        self.n_out = 0
        self.n_counters = 0

    # ---- construction: every add_* returns the op's output slot(s) / counter indices
    def add_copy(self, src, kind, fill=None, keep=True, check=None):
        bits, lo, hi = _check_args(check)
        out, cnt = C.c_int32(-1), C.c_int32(-1)
        nat.check(self._lib.b2s_cols_add_copy(self._h, int(src), int(kind), 0 if fill is None else 1,
                                              0.0 if fill is None else float(fill), 1 if keep else 0, bits, lo, hi,
                                              C.byref(out), C.byref(cnt)))
        return out.value, cnt.value

    def add_range_map(self, src, kind, ranges, fill=None, check=None):
        """ranges: [(lo, hi, value)] in match order"""
        lo = _f64([r[0] for r in ranges])
        hi = _f64([r[1] for r in ranges])
        val = _f64([r[2] for r in ranges])
        bits, cmin, cmax = _check_args(check)
        out, miss, cnt = C.c_int32(-1), C.c_int32(-1), C.c_int32(-1)
        nat.check(self._lib.b2s_cols_add_range_map(
            self._h, int(src), int(kind), 0 if fill is None else 1, 0.0 if fill is None else float(fill),
            nat._p(lo, C.c_double), nat._p(hi, C.c_double), nat._p(val, C.c_double), len(lo), bits, cmin, cmax,
            C.byref(out), C.byref(miss), C.byref(cnt)))
        return out.value, miss.value, cnt.value

    def add_value_map(self, src, kind, mapping, fill=None, check=None):
        keys = _f64(list(mapping.keys()))
        vals = _f64(list(mapping.values()))
        bits, cmin, cmax = _check_args(check)
        out, miss, cnt = C.c_int32(-1), C.c_int32(-1), C.c_int32(-1)
        nat.check(self._lib.b2s_cols_add_value_map(
            self._h, int(src), int(kind), 0 if fill is None else 1, 0.0 if fill is None else float(fill),
            nat._p(keys, C.c_double), nat._p(vals, C.c_double), len(keys), bits, cmin, cmax,
            C.byref(out), C.byref(miss), C.byref(cnt)))
        return out.value, miss.value, cnt.value

    def add_onehot(self, src, kind, categories, fill=None):
        cats = _f64(list(categories))
        out, miss = C.c_int32(-1), C.c_int32(-1)
        nat.check(self._lib.b2s_cols_add_onehot(self._h, int(src), int(kind), 0 if fill is None else 1,
                                                0.0 if fill is None else float(fill), nat._p(cats, C.c_double), len(cats),
                                                C.byref(out), C.byref(miss)))
        return out.value, miss.value

    def add_date_part(self, src, part):
        out, miss = C.c_int32(-1), C.c_int32(-1)
        nat.check(self._lib.b2s_cols_add_date_part(self._h, int(src), int(part), C.byref(out), C.byref(miss)))
        return out.value, miss.value

    def finalize(self):
        nat.init()
        nat.check(self._lib.b2s_cols_finalize(self._h))
        self._read_info()
        self.finalized = True
        return self

    def _read_info(self):
        no, nc = C.c_int32(), C.c_int32()
        nat.check(self._lib.b2s_cols_info(self._h, C.byref(no), C.byref(nc)))
        self.n_out, self.n_counters = no.value, nc.value

    # ---- execution
    def run_host(self, in_slots, n_rows, out_slots, with_stats=False):
        """in_slots / out_slots: {slot: contiguous numpy array}; returns the counters (uint64 array)"""
        self._read_info()
        ins = (C.c_void_p * self.n_in)()
        for s, a in in_slots.items():
            if not a.flags["C_CONTIGUOUS"] or a.itemsize not in (4, 8) or a.shape[0] != n_rows:
                raise ValueError(f"input slot {s}: need a contiguous 4- or 8-byte array of {n_rows} rows")
            ins[s] = a.ctypes.data
        outs = (C.c_void_p * max(self.n_out, 1))()
        for s, a in out_slots.items():
            outs[s] = a.ctypes.data
        counters = np.zeros(max(self.n_counters, 1), dtype=np.uint64)
        stats = nat.Stats()
        nat.check(self._lib.b2s_cols_run_host(self._h, ins, int(n_rows), outs,
                                              counters.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(stats)))
        counters = counters[: self.n_counters]
        return (counters, stats.as_dict()) if with_stats else counters

    def run_device(self, d_in, in_stride, n_rows, d_out, out_stride, d_counters=None, stream=None):
        nat.check(self._lib.b2s_cols_run_device(self._h, d_in, int(in_stride), int(n_rows), d_out, int(out_stride), d_counters, stream))

    def time_device(self, d_in_ptrs, in_stride, n_rows, d_out, out_stride, d_counters, iters):
        arr = (C.c_void_p * len(d_in_ptrs))(*d_in_ptrs)
        ms = C.c_float()
        nat.check(self._lib.b2s_cols_time_device(self._h, arr, len(d_in_ptrs), int(in_stride), int(n_rows), d_out,
                                                 int(out_stride), d_counters, int(iters), C.byref(ms)))
        return ms.value

    # ---- feature-set statistics over the result (b2s_cols_stats_*): see feature_store/infer.py
    def stats_begin(self, kinds, slots, n_rows, d_out=None, out_stride=0):
        """pass 0 over the result columns `slots` (read as `kinds`, nat.STAT_*) of the last run_host (or of d_out):
        a structured array of nat.ColSum records, one per column, and the call's timing"""
        kinds = np.ascontiguousarray(kinds, dtype=np.int32)
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        summary = (nat.ColSum * len(kinds))()
        stats = nat.Stats()
        nat.check(self._lib.b2s_cols_stats_begin(self._h, d_out, int(out_stride), int(n_rows), nat._p(kinds, C.c_int32),
                                                 nat._p(slots, C.c_int32), len(kinds), summary, C.byref(stats)))
        return np.ctypeslib.as_array(summary).copy(), stats.as_dict()

    def stats_finish(self, means, hist_kind, hist, ranks):
        """the passes after stats_begin: (sum of squares around means, histogram counts, order statistics), timing"""
        n = len(means)
        means = np.ascontiguousarray(means, dtype=np.float64)
        hist_kind = np.ascontiguousarray(hist_kind, dtype=np.int32)
        hist = np.ascontiguousarray(hist, dtype=np.float64).reshape(n, 23)
        ranks = np.ascontiguousarray(ranks, dtype=np.int64).reshape(n, nat.STAT_RANKS)
        m2 = np.zeros(n, dtype=np.float64)
        counts = np.zeros((n, nat.STAT_BINS), dtype=np.int64)
        order = np.zeros((n, nat.STAT_RANKS), dtype=np.int64)
        stats = nat.Stats()
        i64 = C.POINTER(C.c_int64)
        nat.check(self._lib.b2s_cols_stats_finish(self._h, nat._p(means, C.c_double), nat._p(hist_kind, C.c_int32),
                                                  nat._p(hist, C.c_double), nat._p(ranks, C.c_int64), nat._p(m2, C.c_double),
                                                  counts.ctypes.data_as(i64), order.ctypes.data_as(i64), C.byref(stats)))
        return m2, counts, order, stats.as_dict()

    def stats_timing(self):
        """per pass of the last begin / finish pair: CUDA-event ms and bytes read; and the kernel launches"""
        ms = np.zeros(6, dtype=np.float32)
        nbytes = np.zeros(6, dtype=np.int64)
        n, launches = C.c_int32(), C.c_int32()
        nat.check(self._lib.b2s_cols_stats_timing(self._h, nat._p(ms, C.c_float), nbytes.ctypes.data_as(C.POINTER(C.c_int64)),
                                                  C.byref(n), C.byref(launches)))
        return {"pass_ms": ms[: n.value].tolist(), "pass_bytes": nbytes[: n.value].tolist(), "launches": launches.value}

    def close(self):
        if self._h:
            self._lib.b2s_cols_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
