"""A numpy stand-in for the two statistics entry points (b2s_cols_stats_begin / _finish) of a columns plan, tests only:
the same inputs and outputs, computed from the result slots with numpy -- including the device's histogram arithmetic
(numpy's uniform-bin index in the bin dtype) and exact order statistics -- so that the product's host layer
(mlrun_b200/feature_store/infer.py) runs end to end on CPU.  The CUDA passes are compared with the oracle in
tests/test_gpu_ingest_stats.py."""

import numpy as np

from mlrun_b200 import _native as nat


class StatsStandIn:
    """`slots` maps a result slot to its array: float32 / int32 words, or int64 for a datetime column's first slot"""

    def __init__(self, slots, n_rows):
        self.slots, self.n_rows = slots, n_rows
        self.cols = None

    def _values(self, kind, slot):
        """(non-missing values as the device reads them, missing mask, raw array)"""
        if kind == nat.STAT_ROW:
            raw = np.arange(self.n_rows, dtype=np.int64)
            return raw, np.zeros(self.n_rows, bool), raw
        raw = self.slots[slot]
        if kind == nat.STAT_F32:
            miss = np.isnan(raw)
        elif kind == nat.STAT_I32_NAT:
            miss = raw < 0
        elif kind == nat.STAT_DT:
            miss = raw == np.iinfo(np.int64).min
        else:
            miss = np.zeros(len(raw), bool)
        return raw[~miss], miss, raw

    @staticmethod
    def _bits(kind, v):
        if kind == nat.STAT_F32:
            return int(np.array([v], np.float32).view(np.uint32)[0])
        return int(v)

    def stats_begin(self, kinds, slots, n_rows):
        assert n_rows == self.n_rows
        self.cols = list(zip(kinds, slots))
        out = np.zeros(len(self.cols), dtype=np.dtype(nat.ColSum))
        for i, (kind, slot) in enumerate(self.cols):
            v, miss, raw = self._values(kind, slot)
            r = out[i]
            r["count"], r["missing"] = len(v), int(miss.sum())
            r["sum"] = float(np.sum(v.astype(np.float64)))
            if kind == nat.STAT_BOOL:
                r["ones"] = int((v == 1).sum())
            if kind == nat.STAT_F32:
                r["pos_inf"], r["neg_inf"] = int((v == np.inf).any()), int((v == -np.inf).any())
            if len(v):
                r["min_bits"], r["max_bits"] = self._bits(kind, v.min()), self._bits(kind, v.max())
            r["first_bits"], r["first_missing"] = self._bits(kind, raw[0]), int(miss[0])
        return out, {"kernels": 1}

    def stats_finish(self, means, hist_kind, hist, ranks):
        n = len(self.cols)
        m2 = np.zeros(n)
        counts = np.zeros((n, nat.STAT_BINS), dtype=np.int64)
        order = np.zeros((n, nat.STAT_RANKS), dtype=np.int64)
        for i, (kind, slot) in enumerate(self.cols):
            v, _miss, _raw = self._values(kind, slot)
            x = v.astype(np.float64)
            if np.isfinite(means[i]):
                m2[i] = float(np.sum((x - means[i]) ** 2))
            if hist_kind[i]:
                dt = np.float32 if hist_kind[i] == 1 else np.float64
                first, den, edges = dt(hist[i][0]), dt(hist[i][1]), hist[i][2:].astype(dt)
                a = v.astype(dt)
                with np.errstate(all="ignore"):
                    idx = (((a - first) / den) * dt(nat.STAT_BINS)).astype(np.intp)
                idx = np.clip(idx, 0, nat.STAT_BINS - 1)
                idx[a < edges[idx]] -= 1
                idx[(a >= edges[np.minimum(idx + 1, nat.STAT_BINS)]) & (idx != nat.STAT_BINS - 1)] += 1
                counts[i] = np.bincount(idx, minlength=nat.STAT_BINS)
            srt = np.sort(v)
            for r in range(nat.STAT_RANKS):
                if ranks[i][r] >= 0:
                    order[i][r] = self._bits(kind, srt[ranks[i][r]])
        return m2, counts, order, {"kernels": 3}


def install(monkeypatch):
    """IngestPlans built from here on run on the emulated columns plan (tests/device_emulator.py) and describe their result
    with this stand-in"""
    from tests import device_emulator

    device_emulator.install_columns(monkeypatch)
    real_run = device_emulator.EmulatedColumns.run_host

    def run_host(self, in_slots, n_rows, out_slots, with_stats=False):
        res = real_run(self, in_slots, n_rows, out_slots, with_stats)
        words = dict(out_slots)
        for _name, slot, how in self._iplan.out:  # a datetime column's first slot holds its int64 array
            if how == "dt":
                words[slot] = out_slots[slot].view(np.int64)
        self._standin = StatsStandIn(words, n_rows)
        return res

    monkeypatch.setattr(device_emulator.EmulatedColumns, "run_host", run_host)
    monkeypatch.setattr(device_emulator.EmulatedColumns, "stats_begin", lambda self, *a: self._standin.stats_begin(*a), raising=False)
    monkeypatch.setattr(device_emulator.EmulatedColumns, "stats_finish", lambda self, *a: self._standin.stats_finish(*a), raising=False)
