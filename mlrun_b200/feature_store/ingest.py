"""Feature-set ingestion on the device: DataFrame in -> transformed DataFrame out.

Plugin-API mirror of the reference's ingest caller for in-memory frames: `FeatureSet(...).graph.to(...)`,
`FeatureSet.ingest(df)` (mlrun/feature_store/feature_set.py:1004-1090) -> `init_featureset_graph`
(mlrun/feature_store/ingestion.py:38-127), which pushes the frame ROW BY ROW through the step DAG
(storey.DataframeSource, datastore/sources.py:886-895) and re-assembles a frame (ReduceToDataFrame,
datastore/targets.py:1856-1868).  Here the steps are walked symbolically over the frame's schema
(`FrameProgram`, same per-row semantics) and lowered to ONE columnar device plan (`mlrun_b200.columns`); the frame's
columns go to the GPU as they are (contiguous typed arrays) and the result columns come back the same way.

With `infer_options=InferOptions.Stats (| Histogram | Index)` ingest also profiles the result like the reference's
`_infer_from_static_df` -> get_df_stats (feature_store/api.py:1162-1196), on the device while the result is still there
(`infer.py`), into `fset.status.stats` / `get_stats_table()`.  The default here is `InferOptions.Null` (the reference's is
`InferOptions.default()`).

Out of scope (control plane / storage): targets, schema and preview inference, sources other than a DataFrame or columns.
Steps or dtypes the device cannot hold raise `LoweringError`: there is no per-row Python fallback.
"""

import math
import types

import numpy as np

from .. import _native as nat
from ..columns import F32, I32, I64, ColumnsPlan
from ..lowering import LoweringError
from ..serving.resolve import MLRunInvalidArgumentError
from . import infer
from .infer import InferOptions

_INT_DTYPES = ("int8", "int16", "int32", "uint8", "uint16", "bool")


def _short(value):
    """reports carry at most 40 characters of a violating value (mlrun/features.py:24-35)"""
    text = str(value)
    return text if len(text) <= 40 else text[:40] + "..."


class MinMaxValidator:
    """mlrun/features.py:265-321 -- range check whose only effect is a report (check_type is metadata here)"""

    kind = "minmax"

    def __init__(self, check_type=None, severity=None, min=None, max=None):
        self.check_type = check_type
        self.severity = severity
        self.min = min
        self.max = max

    def check(self, value):
        try:
            if self.min is not None and value < self.min:
                return False, {"message": "value is smaller than min", "min": self.min, "value": _short(value)}
            if self.max is not None and value > self.max:
                return False, {"message": "value is greater than max", "max": self.max, "value": _short(value)}
        except Exception as err:  # noqa: BLE001 -- the reference reports comparison errors as violations
            return False, {"message": str(err), "type": self.kind}
        return True, {}


def _num(v, what):
    if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)):
        raise LoweringError(f"{what}: {v!r} is not numeric -- string / object values are not held on the device")
    return float(v)


def _f32_exact(v, what):
    v = _num(v, what)
    if math.isfinite(v) and float(np.float32(v)) != v:
        raise LoweringError(f"{what}: {v!r} is not exactly representable in the float32 output column")
    return v


class _Col:
    """one column of the event as the steps see it"""

    __slots__ = ("name", "slot", "kind", "fill", "op", "arg", "check", "group")

    def __init__(self, name, slot, kind):
        self.name, self.slot, self.kind = name, slot, kind
        self.fill = None    # Imputer value (float sources)
        self.op = None      # None | "range" | "value" | "onehot" | "date"
        self.arg = None     # ranges / mapping / category index / date part
        self.check = None   # (min, max, validator)
        self.group = None   # one-hot group: the _Group shared by the expanded columns


class _Group:
    def __init__(self, src, cats):
        self.src, self.cats = src, cats
        self.first_out = None
        self.miss = None


def frame_schema(df):
    """[(column name, kind)] of a DataFrame, or LoweringError for dtypes the device does not take as they are"""
    schema = []
    for name in df.columns:
        dt = df[name].dtype
        s = str(dt)
        if s == "float32":
            kind = F32
        elif s in _INT_DTYPES:
            kind = I32
        elif s.startswith("datetime64"):
            kind = I64
        else:
            raise LoweringError(
                f"column {name!r} has dtype {s}: the device takes float32, (u)int8/16/32, bool and datetime64 columns; "
                "cast float64/int64 columns explicitly (a silent down-cast would change values)")
        schema.append((str(name), kind))
    return schema


class FrameProgram:
    """symbolic execution of feature-store steps over the frame's columns, with the storey engine's per-row
    semantics (feature_store/steps.py `_do_storey` methods)"""

    def __init__(self, schema):
        self.schema = list(schema)
        names = [n for n, _ in self.schema]
        if len(set(names)) != len(names):
            raise LoweringError("duplicate column names")
        self.cols, slot = [], 0
        for name, kind in self.schema:
            self.cols.append(_Col(name, slot, kind))
            slot += 2 if kind == I64 else 1
        self.n_in_slots = slot
        self.in_slot = {c.name: c.slot for c in self.cols}
        self.checked_dropped = []
        self.validators = []
        self.steps = []

    # ---- step handlers ------------------------------------------------------------------------
    def imputer(self, step):
        """Imputer._impute (steps.py:397-406): every missing value -> mapping.get(feature, default_value)"""
        mapping, default = step.mapping or {}, step.default_value
        for c in self.cols:
            fill = mapping.get(c.name, default)
            if fill is None:
                continue  # NaN -> None: still missing when the frame is re-assembled
            if c.kind == I32 or c.op in ("onehot", "date"):
                continue  # integers are never missing
            if c.kind == I64:
                raise LoweringError(f"Imputer would replace NaT in the timestamp column {c.name!r}: not held on the device")
            if c.op is not None:
                raise LoweringError(f"Imputer after MapValues on column {c.name!r} is not lowered")
            if c.fill is None:
                c.fill = _f32_exact(fill, f"Imputer fill for {c.name!r}")

    def map_values(self, step):
        """MapValues._do_storey (steps.py:203-216)"""
        mapped = []
        for c in self.cols:
            if c.name not in step.mapping:
                continue
            if c.op is not None or c.kind == I64:
                raise LoweringError(f"MapValues on the derived / timestamp column {c.name!r} is not lowered")
            fmap = step.mapping[c.name]
            m = _Col(f"{c.name}_{step.suffix}" if step.with_original_features else c.name, c.slot, c.kind)
            m.fill = c.fill
            if "ranges" in fmap:
                if len(fmap) > 1:
                    raise LoweringError("MapValues mixing ranges and value replacements is rejected by the reference")
                m.op, m.arg = "range", []
                for val, (lo, hi) in fmap["ranges"].items():
                    lo = -math.inf if lo == "-inf" else _num(lo, f"MapValues range of {c.name!r}")
                    hi = math.inf if hi == "inf" else _num(hi, f"MapValues range of {c.name!r}")
                    m.arg.append((lo, hi, _f32_exact(val, f"MapValues range label of {c.name!r}"), val))
            else:
                m.op = "value"
                m.arg = [(_num(k, f"MapValues key of {c.name!r}"), _f32_exact(v, f"MapValues value of {c.name!r}"), v)
                         for k, v in fmap.items()]
            mapped.append(m)
        # storey mode emits the mapped features first, then (optionally) the untouched event
        self.cols = mapped + (self.cols if step.with_original_features else [])

    def one_hot(self, step):
        """OneHotEncoder._do_storey (steps.py:473-478): the feature is replaced in place by one field per category"""
        new = []
        for c in self.cols:
            cats = step.mapping.get(c.name)
            if not cats:
                new.append(c)
                continue
            if c.op is not None or c.kind == I64:
                raise LoweringError(f"OneHotEncoder on the derived / timestamp column {c.name!r} is not lowered")
            if c.kind != I32:
                # a float value equal to an integer category makes the reference add a stray "<col>_<value>" field next
                # to the encoded ones (steps.py:462-470 writes encoding[f"{feature}_{value}"] for the float spelling)
                raise LoweringError(f"OneHotEncoder source {c.name!r} must be an integer column (cast the codes to int32)")
            cats = list(dict.fromkeys(cats))
            for v in cats:
                if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
                    raise LoweringError(f"OneHotEncoder categories of {c.name!r} must be integers on the device (got {v!r})")
            g = _Group(c, [float(v) for v in cats])
            for i, v in enumerate(cats):
                e = _Col(f"{c.name}_{step._sanitized_category(v)}", c.slot, c.kind)
                e.op, e.arg, e.group = "onehot", i, g
                new.append(e)
        self.cols = new

    def date_extractor(self, step):
        """DateExtractor._do_storey (steps.py:593-602)"""
        ts = next((c for c in self.cols if c.name == step.timestamp_col), None)
        if ts is None:
            raise MLRunInvalidArgumentError(f"{step.timestamp_col} does not exist in the event")
        if ts.kind != I64 or ts.op is not None:
            raise LoweringError(f"DateExtractor needs {step.timestamp_col!r} to be a datetime64 column")
        for part in step.parts:
            if part not in nat.DATE_PARTS:
                raise LoweringError(f"DateExtractor part {part!r} is not computed on the device (have {sorted(nat.DATE_PARTS)})")
            name = f"{step.timestamp_col}_{part}"
            e = _Col(name, ts.slot, I64)
            e.op, e.arg = "date", nat.DATE_PARTS[part]
            at = next((i for i, c in enumerate(self.cols) if c.name == name), None)
            if at is None:
                self.cols.append(e)
            else:
                self.cols[at] = e  # the event already had that key: overwritten in place

    def drop_features(self, step):
        """DropFeatures._do_storey (steps.py:721-729)"""
        drop = set(step.features)
        have = {c.name for c in self.cols}
        for f in step.features:
            if f not in have:
                raise MLRunInvalidArgumentError(f"The ingesting data doesn't contain a feature named '{f}'")
        for c in self.cols:
            if c.name in drop and c.check is not None:
                if c.op in ("onehot", "date"):
                    raise LoweringError(f"validated derived column {c.name!r} cannot be dropped on the device")
                self.checked_dropped.append(c)
        self.cols = [c for c in self.cols if c.name not in drop]

    def validator(self, step):
        """FeaturesetValidator._do_storey (steps.py:117-128): report only; here violations are counted"""
        for name, v in step._validators.items():
            c = next((c for c in self.cols if c.name == name), None)
            if c is None:
                continue  # `if name in body`
            if getattr(v, "kind", "minmax") != "minmax" and not hasattr(v, "min"):
                raise LoweringError(f"validator of {name!r}: only MinMaxValidator is lowered")
            if c.op in ("onehot", "date") or c.kind == I64:
                raise LoweringError(f"validator on the derived / timestamp column {name!r} is not lowered")
            if c.check is not None:
                raise LoweringError(f"column {name!r} is validated twice")
            lo = None if v.min is None else _num(v.min, f"validator min of {name!r}")
            hi = None if v.max is None else _num(v.max, f"validator max of {name!r}")
            c.check = (lo, hi, v)
        self.validators.append(step)

    def apply(self, step):
        handler = {"Imputer": self.imputer, "MapValues": self.map_values, "OneHotEncoder": self.one_hot,
                   "DateExtractor": self.date_extractor, "DropFeatures": self.drop_features,
                   "FeaturesetValidator": self.validator}.get(type(step).__name__)
        if handler is None:
            raise LoweringError(f"step {type(step).__name__} is not lowered to the columnar device plan")
        handler(step)
        self.steps.append(type(step).__name__)
        if len({c.name for c in self.cols}) != len(self.cols):
            raise LoweringError("two output columns share a name")  # a dict would keep one: not reproduced
        return self

    # ---- plan ----------------------------------------------------------------------------------
    def build(self):
        return IngestPlan(self)


class IngestPlan:
    """the device plan of a FrameProgram + the frame boundary (DataFrame columns <-> slots)"""

    def __init__(self, prog, finalize=True):
        self.prog = prog
        self.schema = prog.schema
        plan = ColumnsPlan(prog.n_in_slots)
        self.ops = []  # what was handed to the C-ABI, in order: (kind, source slot, source kind, fill, argument, check)
        self.out = []  # per output column: (name, slot, how, col)
        self.checks = []  # (counter, column name, validator)
        self.miss = []    # (counter, column name, what)
        for c in prog.cols:
            chk = None if c.check is None else c.check[:2]
            if c.op is None:
                slot, cnt = plan.add_copy(c.slot, c.kind, fill=c.fill, keep=True, check=chk)
                self.ops.append(("copy", c.slot, c.kind, c.fill, None, chk))
                how = {F32: "f32", I32: "i32", I64: "dt"}[c.kind]
            elif c.op == "range":
                slot, miss, cnt = plan.add_range_map(c.slot, c.kind, [r[:3] for r in c.arg], fill=c.fill, check=chk)
                self.ops.append(("range", c.slot, c.kind, c.fill, [r[:3] for r in c.arg], chk))
                self.miss.append((miss, c.name, "matched no range"))
                how = ("map", miss, all(isinstance(r[3], (int, np.integer)) and not isinstance(r[3], bool) for r in c.arg))
            elif c.op == "value":
                slot, miss, cnt = plan.add_value_map(c.slot, c.kind, {k: v for k, v, _ in c.arg}, fill=c.fill, check=chk)
                self.ops.append(("value", c.slot, c.kind, c.fill, {k: v for k, v, _ in c.arg}, chk))
                self.miss.append((miss, c.name, "matched no key"))
                how = ("map", miss, all(isinstance(r[2], (int, np.integer)) and not isinstance(r[2], bool) for r in c.arg))
            elif c.op == "onehot":
                g = c.group
                if g.first_out is None:
                    g.first_out, g.miss = plan.add_onehot(g.src.slot, g.src.kind, g.cats, fill=g.src.fill)
                    self.ops.append(("onehot", g.src.slot, g.src.kind, g.src.fill, list(g.cats), None))
                    self.miss.append((g.miss, g.src.name, "matched no category"))
                slot, cnt, how = g.first_out + c.arg, -1, "i32"
            else:  # date
                slot, miss = plan.add_date_part(c.slot, c.arg)
                self.ops.append(("date", c.slot, I64, None, c.arg, None))
                self.miss.append((miss, c.name, "NaT"))
                cnt, how = -1, ("date", miss, c.arg in nat.DATE_BOOL_PARTS)
            if cnt >= 0:
                self.checks.append((cnt, c.name, c.check[2]))
            self.out.append((c.name, slot, how))
        for c in prog.checked_dropped:
            chk = c.check[:2]
            if c.op is None:
                _, cnt = plan.add_copy(c.slot, c.kind, fill=c.fill, keep=False, check=chk)
                self.ops.append(("check", c.slot, c.kind, c.fill, None, chk))
            else:
                raise LoweringError(f"validated then dropped mapped column {c.name!r} is not lowered")
            self.checks.append((cnt, c.name, c.check[2]))
        self.plan = plan.finalize() if finalize else plan
        self.counters = None
        self.violations = {}
        self.unmatched = {}
        self.stats = None
        self.df_stats = None

    @property
    def out_names(self):
        return [o[0] for o in self.out]

    def _inputs(self, df):
        """the frame's columns as contiguous arrays, without copies where pandas allows it"""
        raw = self._block_columns(df)
        ins, keep = {}, []
        for name, kind in self.schema:
            a = raw[name] if raw is not None else df[name].to_numpy()
            if kind == I64:
                a = a.astype("datetime64[ns]", copy=False).view(np.int64)
            elif kind == I32 and a.dtype != np.int32:
                a = a.astype(np.int32)
            a = np.ascontiguousarray(a)
            keep.append(a)
            ins[self.prog.in_slot[name]] = a
        return ins, keep

    @staticmethod
    def _block_columns(df):
        """{column: array} taken one dtype at a time: for a consolidated frame (one block per dtype) `to_numpy()` of the
        same-dtype sub-frame is a view whose columns are contiguous, 4x cheaper than 255 `df[name]` look-ups.  Frames that
        are not consolidated (or a pandas without the block counter) use the per-column path: None."""
        nblocks = getattr(getattr(df, "_mgr", None), "nblocks", None)
        dtypes = df.dtypes
        kinds = set(dtypes)
        if nblocks is None or nblocks > len(kinds) or not df.columns.is_unique:
            return None
        out = {}
        for dt in kinds:
            sub = df.select_dtypes(include=[dt]) if len(kinds) > 1 else df  # the dtype's block(s), not a copy
            names = sub.columns
            block = sub.to_numpy()
            if block.ndim != 2 or not (block.flags["F_CONTIGUOUS"] or block.shape[1] == 1):
                return None  # pandas had to assemble it: the columns would be strided copies
            for j, name in enumerate(names):
                out[name] = block[:, j]
        return out

    def run(self, df, reference_dtypes=False, infer_options=0):
        """transform the frame; returns a new DataFrame with the same index.  `reference_dtypes=True` widens integer
        results to int64 (what a frame re-assembled from Python ints has) at the price of a host-side copy.  With the
        InferOptions.Stats bit, `self.df_stats` is get_df_stats of the returned frame (else None)."""
        import pandas as pd

        if not _same_labels_and_dtypes(df, getattr(self, "_seen", None)):  # a frame like one already checked skips the walk
            if frame_schema(df) != self.schema:
                raise ValueError("the frame does not carry the schema this plan was lowered for")
            self._seen = (df.columns, list(df.dtypes))
        n = len(df)
        ins, _keep = self._inputs(df)
        data, bufs, block, layout = self._run_arrays(ins, n, reference_dtypes)
        self._describe(data, n, df.index, infer_options)
        return self._assemble(data, bufs, block, layout, n, df.index)

    def _describe(self, data, n, index, infer_options):
        self.df_stats = infer.describe(self, data, n, index, infer_options) if infer_options & InferOptions.Stats else None

    def _run_arrays(self, ins, n, reference_dtypes=False):
        """{input slot: contiguous column array} -> ({result column: array}, landing views, their pinned block, offsets):
        the device run and the dtype rules of the result, with no DataFrame on either side"""
        # result columns live in one pinned block (fast D2H, no second copy); the frame built over them keeps the block
        # alive and it returns to the pool when the frame is collected
        specs, extra = self._landing()
        layout, off = [], 0
        for dt in [sp[2] for sp in specs] + [np.dtype(np.int32)] * len(extra):
            layout.append(off)
            off += (n * dt.itemsize + 63) // 64 * 64
        block = nat.PINNED.take(off) if n else None

        def column(i, dt):
            return np.frombuffer(block, dtype=dt, count=n, offset=layout[i]) if block is not None else np.empty(n, dtype=dt)

        bufs, outs = {}, {}
        for i, (name, slot, dt) in enumerate(specs):
            bufs[name] = outs[slot] = column(i, dt)
        # slots written by the device but not part of the result (dropped one-hot members) still need a landing buffer
        for j, s_ in enumerate(extra):
            outs[s_] = column(len(specs) + j, np.dtype(np.int32))
        self.counters, self.stats = self.plan.run_host(ins, n, outs, with_stats=True)
        data = {}
        for name, _slot, how in self.out:
            a = bufs[name]
            if how == "dt":
                a = a.view("datetime64[ns]")
            elif isinstance(how, tuple) and how[0] == "map":
                if how[2] and self.counters[how[1]] == 0:
                    a = a.astype(np.int64 if reference_dtypes else np.int32)  # every row got an integer label
            elif isinstance(how, tuple) and how[0] == "date":
                if self.counters[how[1]]:
                    a = np.where(a < 0, np.nan, a.astype(np.float64))  # NaT rows
                elif how[2]:
                    a = a.astype(np.bool_)  # the is_* parts are booleans
                elif reference_dtypes:
                    a = a.astype(np.int64)
            elif how == "i32" and reference_dtypes:
                a = a.astype(np.int64)
            data[name] = a
        self.violations = {name: int(self.counters[cnt]) for cnt, name, _v in self.checks}
        self.unmatched = {name: int(self.counters[cnt]) for cnt, name, _w in self.miss if self.counters[cnt]}
        for cnt, name, v in self.checks:
            if self.counters[cnt]:
                print(f"{v.severity}! {name} has {int(self.counters[cnt])} values outside [{v.min}, {v.max}]")
        for step in self.prog.validators:
            step.violations = getattr(step, "violations", 0) + sum(
                int(self.counters[cnt]) for cnt, name, v in self.checks if v in step._validators.values())
        return data, bufs, block, layout

    def run_columns(self, columns, reference_dtypes=False, infer_options=0, index=None):
        """columnar twin of `run` (SURVEY 8(f) #1: "Arrow/DLPack in, Arrow/Parquet-ready columns out"): `columns` maps every
        schema column to a contiguous 1-D array of its dtype (numpy, or anything `columnar.as_columns` understands: Arrow
        tables / record batches, DLPack producers); returns a `columnar.ColumnBatch` whose arrays live in one pinned block.
        No pandas object is built or taken apart; pinned inputs (`columnar.pinned_columns`) cross PCIe at full speed and
        frames of 128 Ki rows and more are pipelined in row ranges.  `index` ({entity: array}) is what the statistics of
        `infer_options` describe as the batch's index columns (none: the row numbers, as for a frame's RangeIndex)."""
        from . import columnar

        cols = columnar.as_columns(columns)
        n = None
        ins = {}
        for name, kind in self.schema:
            if name not in cols:
                raise ValueError(f"column {name!r} of the plan's schema is missing")
            a = cols[name]
            want = {F32: ("float32",), I32: _INT_DTYPES, I64: ("datetime64[ns]", "int64")}[kind]
            if a.ndim != 1 or str(a.dtype) not in want:
                raise ValueError(f"column {name!r}: expected a 1-D {' / '.join(want)} array, got {a.dtype} {a.shape}")
            if kind == I64:
                a = a.view(np.int64)
            elif kind == I32 and a.dtype != np.int32:
                a = a.astype(np.int32)
            a = np.ascontiguousarray(a)
            if n is None:
                n = len(a)
            elif len(a) != n:
                raise ValueError("columns of different lengths")
            ins[self.prog.in_slot[name]] = a
        data, _bufs, block, _layout = self._run_arrays(ins, n or 0, reference_dtypes)
        self._describe(data, n or 0, index or {}, infer_options)
        return columnar.ColumnBatch(data, n or 0, block)

    def _assemble(self, data, bufs, block, layout, n, index):
        """the result frame.  Columns that stayed in their landing buffers and sit next to each other in the result block
        with one dtype become ONE 2-D pandas block (a strided view of the block, no copy): the frame has a handful of blocks
        instead of one per column -- cheaper to build and consolidated for whatever the caller does next."""
        import pandas as pd

        names = list(data)
        if block is None or len(names) < 2:
            return pd.DataFrame(data, index=index, copy=False)
        pieces, loose, i = [], {}, 0

        def flush_loose():
            if loose:
                pieces.append(pd.DataFrame(dict(loose), index=index, copy=False))
                loose.clear()

        while i < len(names):
            a = data[names[i]]
            stride = (n * a.dtype.itemsize + 63) // 64 * 64
            j = i
            if a is bufs[names[i]]:  # untouched landing view: extend the run while dtype and spacing hold
                while (j + 1 < len(names) and data[names[j + 1]] is bufs[names[j + 1]] and data[names[j + 1]].dtype == a.dtype
                       and layout[j + 1] - layout[j] == stride):
                    j += 1
            if j > i:
                flush_loose()
                k, words = j - i + 1, stride // a.dtype.itemsize
                rows = np.frombuffer(block, dtype=a.dtype, count=(k - 1) * words + n, offset=layout[i])
                run = np.lib.stride_tricks.as_strided(rows, shape=(n, k), strides=(a.dtype.itemsize, stride), writeable=True)
                pieces.append(pd.DataFrame(run, columns=names[i:j + 1], index=index, copy=False))
            else:
                loose[names[i]] = a
            i = j + 1
        flush_loose()
        if len(pieces) == 1:
            return pieces[0]
        concat_kw = {} if int(pd.__version__.split(".")[0]) >= 3 else {"copy": False}  # pandas 3: lazy copies by default
        return pd.concat(pieces, axis=1, **concat_kw)

    def _landing(self):
        """(name, slot, dtype) of every result column + the slots the device writes that are not part of the result (dropped
        one-hot members): they still need a landing buffer.  Depends on the plan only: computed once."""
        cached = getattr(self, "_landing_cache", None)
        if cached is None:
            specs = []
            for name, slot, how in self.out:
                dt = np.int64 if how == "dt" else (np.float32 if (how == "f32" or (isinstance(how, tuple) and how[0] == "map")) else np.int32)
                specs.append((name, slot, np.dtype(dt)))
            taken = {sp[1] for sp in specs} | {slot + 1 for _n, slot, how in self.out if how == "dt"}  # + second halves
            extra = [s for s in range(self.plan.n_out) if s not in taken]
            cached = self._landing_cache = (specs, extra)
        return cached


def _same_labels_and_dtypes(df, seen):
    """seen = (columns Index, [dtypes]) of an earlier frame; Index.equals is vectorised (50 us for 255 columns where
    building a tuple key of labels and dtypes costs 1 ms)"""
    return seen is not None and df.columns.equals(seen[0]) and list(df.dtypes) == seen[1]


def lower_steps(steps, df_or_schema):
    schema = df_or_schema if isinstance(df_or_schema, list) else frame_schema(df_or_schema)
    prog = FrameProgram(schema)
    for s in steps:
        prog.apply(s)
    return prog.build()


# ------------------------------------------------------------------------------------------ FeatureSet mirror
class Entity:
    def __init__(self, name=None, value_type=None, description=None, labels=None):
        self.name, self.value_type, self.description, self.labels = name, value_type, description, labels or {}


class Feature:
    """mlrun/features.py:92-150: only what validation reads"""

    def __init__(self, value_type=None, dims=None, description=None, aggregate=None, name=None, validator=None,
                 default=None, labels=None):
        self.name, self.value_type, self.description, self.validator = name or "", value_type, description, validator
        self.default, self.labels = default, labels or {}


class FeatureSet:
    """the part of mlrun.feature_store.FeatureSet the ingest path touches (feature_set.py:319-520, 1004-1090):
    a named transformation graph (`.graph`, `.add_step`/`graph.to`), entities that become the frame's index
    (ingestion.py:84-87 `entities_to_index`) and `ingest(df)`"""

    def __init__(self, name=None, description=None, entities=None, timestamp_key=None, engine=None, label_column=None,
                 relations=None, passthrough=None):
        from ..serving.graph import RootFlowStep

        self.name = name
        self.description = description
        self.entities = [Entity(e) if isinstance(e, str) else e for e in (entities or [])]
        self.timestamp_key = timestamp_key
        self.engine = engine or "storey"
        self.label_column = label_column
        self.passthrough = passthrough
        self.features = {}
        self._graph = RootFlowStep()
        self._graph.engine = "sync"  # steps are only resolved here; the device plan replaces the executor
        self._plan = None
        self._plan_key = None
        self.status = types.SimpleNamespace(stats={})

    def get_stats_table(self):
        """feature_set.py:853-856: the statistics of the last ingest with InferOptions.Stats as a frame (one row per
        column), None when there are none"""
        import pandas as pd

        if self.status.stats:
            return pd.DataFrame.from_dict(self.status.stats, orient="index")
        return None

    @property
    def graph(self):
        return self._graph

    def __getitem__(self, name):
        return self.features[name]

    def __setitem__(self, key, item):
        self.add_feature(item, key)

    def add_feature(self, feature, name=None):
        """feature_set.py:646-656 -- `fset["bid"] = Feature(validator=MinMaxValidator(min=52, severity="info"))`"""
        name = name or feature.name
        if not name:
            raise MLRunInvalidArgumentError("feature name must be specified")
        feature.name = name
        self.features[name] = feature

    def add_step(self, *args, **kwargs):
        last = self._graph
        names = list(self._graph.steps.keys()) if hasattr(self._graph, "steps") else []
        if names:
            last = self._graph[names[-1]]
        return last.to(*args, **kwargs)

    @property
    def spec(self):
        """what the steps' `validate_args` read of a feature set (feature_set.py FeatureSetSpec)"""
        import types

        return types.SimpleNamespace(entities={e.name: e for e in self.entities}, label_column=self.label_column,
                                     timestamp_key=self.timestamp_key, graph=self._graph)

    def validate_steps(self, namespace=None):
        """ingest-time argument checks of the graph's steps (feature_set.py:508-534): every step class that has a
        `validate_args` classmethod sees the feature set and its own constructor arguments"""
        from . import transforms

        known = {k: getattr(transforms, k) for k in dir(transforms) if not k.startswith("_")}
        known.update(namespace or {})
        for step in self._graph.steps.values():
            obj = getattr(step, "_object", None)
            cls = type(obj) if obj is not None else known.get(str(step.class_name or "").rsplit(".", 1)[-1])
            check = getattr(cls, "validate_args", None)
            if check is None:
                continue
            args = dict(step.class_args or {})
            if obj is not None:  # a step added as an object: its arguments are its attributes
                args = {k: getattr(obj, k) for k in ("mapping", "features") if hasattr(obj, k)}
            check(self, **args)

    def _step_objects(self, namespace):
        from ..serving.compiler import _chain, _transform_object
        from ..serving.host import create_graph_server
        from . import transforms

        ns = {k: getattr(transforms, k) for k in dir(transforms) if not k.startswith("_")}
        ns.update(namespace or {})
        server = create_graph_server(graph=self._graph, parameters={})
        server.init_states(context=None, namespace=ns)
        server.init_object(ns)
        objs = [_transform_object(s) for s in _chain(self._graph)]
        for o in objs:
            # FeaturesetValidator.__init__ (steps.py:94-116) takes its validators from the feature set's features
            if type(o).__name__ == "FeaturesetValidator" and not o._validators and o.featureset in (".", self.name):
                o._validators = {k: f.validator for k, f in self.features.items()
                                 if f.validator is not None and (not o.columns or k in o.columns)}
        return objs

    def ingest(self, source=None, targets=None, namespace=None, return_df=True, reference_dtypes=False,
               infer_options=InferOptions.Null, **kwargs):
        """DataFrame -> transformed DataFrame through one device plan (targets are out of scope: pass none).
        `infer_options` (InferOptions bits): Stats fills `status.stats` with get_df_stats of the result, computed on the
        device; Histogram adds the 20-bin histograms; Index describes the index (entities, else the row numbers) first.
        Entities / Features / Preview (schema and preview inference) are accepted and ignored.  The default is Null:
        pass InferOptions.default() for what the reference's ingest does."""
        if targets:
            raise LoweringError("targets are storage (out of scope): ingest returns the frame")
        from . import columnar

        if columnar.is_columnar(source):
            # columnar sources (dict of arrays, Arrow table / record batch, DLPack producers): no DataFrame on either side;
            # entity columns are carried through untouched (they would be the frame's index)
            cols = columnar.as_columns(source)
            keys = [e.name for e in self.entities if e.name in cols]
            carried = {k: cols.pop(k) for k in keys}
            schema = columnar.schema_of(cols)
            if self._plan is None or self._plan_key != ("columns", schema):
                self.validate_steps(namespace)
                self._plan = lower_steps(self._step_objects(namespace), schema)
                self._plan_key = ("columns", schema)
            batch = self._plan.run_columns(cols, reference_dtypes=reference_dtypes, infer_options=infer_options, index=carried)
            batch.index = carried
            if infer_options & InferOptions.Stats:
                self.status.stats = self._plan.df_stats
            return batch if return_df else None
        if not (hasattr(source, "columns") and hasattr(source, "index")):
            raise MLRunInvalidArgumentError("illegal source")  # ingestion.py:77-78; only frames are taken here
        df = source
        keys = [e.name for e in self.entities]
        if keys and all(k in df.columns for k in keys):
            df = df.set_index(keys)
        if self._plan is None or isinstance(self._plan_key[0], str) or not _same_labels_and_dtypes(df, self._plan_key):
            self.validate_steps(namespace)
            self._plan = lower_steps(self._step_objects(namespace), df)
            self._plan_key = (df.columns, list(df.dtypes))
        out = self._plan.run(df, reference_dtypes=reference_dtypes, infer_options=infer_options)
        if infer_options & InferOptions.Stats:
            self.status.stats = self._plan.df_stats
        return out if return_df else None

    @property
    def plan(self):
        return self._plan


def ingest(featureset=None, source=None, targets=None, namespace=None, return_df=True, **kwargs):
    """module-level spelling, mlrun.feature_store.api.ingest (feature_store/api.py:404-520)"""
    return featureset.ingest(source, targets=targets, namespace=namespace, return_df=return_df, **kwargs)
