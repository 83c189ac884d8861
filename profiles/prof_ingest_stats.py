"""Feature-set statistics on the device: what each pass costs, and what `infer_options=InferOptions.default()` adds to
FeatureSet.ingest, on the config-5 workload.  Prints one JSON document and, with --out PATH, writes it there.

Run on a B200:  python profiles/prof_ingest_stats.py [n_rows] [--out PATH]   (default 1 Mi rows)

Reports the card (name, power limit, clocks), a measured HBM bandwidth (device-to-device copy of 4 GiB, read + write bytes),
each stats pass's CUDA-event time and bytes (4 B per value read; 8 B for datetimes) and its share of that bandwidth, the
launches and host synchronisations of one describe, FeatureSet.ingest through pinned columns with and without the
statistics, the host cost of describing entity columns with pandas, and the CPU oracle's time for the same statistics."""

import contextlib
import io
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mlrun_b200 import _native as nat  # noqa: E402
from mlrun_b200.feature_store import InferOptions, columnar, infer  # noqa: E402
from mlrun_b200.feature_store import ingest as bi  # noqa: E402
from mlrun_b200.feature_store import steps as bs  # noqa: E402
from mlrun_b200.synthetic import ingest_workload  # noqa: E402


def card():
    q = "name,power.limit,power.max_limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"nvidia-smi unavailable: {e}"
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if "," in out else {"query": out}


def hbm_copy_gbps():
    import torch

    x = torch.empty(1 << 30, dtype=torch.float32, device="cuda")  # 4 GiB, far beyond L2
    y = torch.empty_like(x)
    y.copy_(x)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 0.0
    for _ in range(5):
        a.record()
        y.copy_(x)
        b.record()
        b.synchronize()
        best = max(best, 2 * x.numel() * 4 / (a.elapsed_time(b) * 1e-3) / 1e9)
    del x, y
    torch.cuda.empty_cache()
    return best


def timed(fn, reps):
    with contextlib.redirect_stdout(io.StringIO()):
        fn()
        fn()
        t = time.perf_counter()
        for _ in range(reps):
            fn()
    return (time.perf_counter() - t) / reps * 1e3


def main():
    args = sys.argv[1:]
    out_path = None
    if "--out" in args:
        i = args.index("--out")
        out_path = args[i + 1]
        del args[i:i + 2]
    n = int(args[0]) if args else 1 << 20
    nat.init(0)
    res = {"n_rows": n, "card": card(), "device": nat.device_info()}
    res["hbm_copy_GBps"] = round(hbm_copy_gbps(), 1)
    wl = ingest_workload(n_rows=n, seed=5)
    src = {name: wl.df[name].to_numpy() for name in wl.df.columns}
    cols = columnar.pinned_columns(src, n)
    for name, a in cols.items():
        a[...] = src[name]
    fs = bi.FeatureSet("prof", timestamp_key="timestamp")
    cur = fs.graph
    for st in wl.build_steps(bs):
        cur = cur.to(st)
    allopt = InferOptions.default()

    plain_ms = timed(lambda: fs.ingest(cols), 10)
    stats_ms = timed(lambda: fs.ingest(cols, infer_options=allopt), 10)
    # alternate once more to see the spread between the two
    plain2 = timed(lambda: fs.ingest(cols), 10)
    stats2 = timed(lambda: fs.ingest(cols, infer_options=allopt), 10)
    res["ingest_pinned_columns_ms"] = {"without_stats": [round(plain_ms, 3), round(plain2, 3)],
                                       "with_default_infer_options": [round(stats_ms, 3), round(stats2, 3)]}
    res["stats_rate_vs_plain"] = round(min(plain_ms, plain2) / min(stats_ms, stats2), 3)

    # the passes of one describe (the last ingest above), CUDA-event timed in the library
    tm = fs.plan.plan.stats_timing()
    passes = []
    for p, (ms, nb) in enumerate(zip(tm["pass_ms"], tm["pass_bytes"])):
        if nb == 0 and p:
            continue
        gbps = nb / (ms * 1e-3) / 1e9 if ms else 0.0
        passes.append({"pass": p, "ms": round(ms, 4), "bytes": int(nb), "GBps": round(gbps, 1),
                       "share_of_measured_hbm": round(gbps / res["hbm_copy_GBps"], 3)})
    res["passes"] = passes
    res["kernel_launches_per_describe"] = tm["launches"]
    # read from the code, not measured: begin and finish each end in one cudaStreamSynchronize (their D2H copies go to
    # pageable memory, so they complete on the host by then as well)
    res["host_syncs_per_describe_from_code"] = 2
    res["columns_described"] = len(fs.plan.out) + 1  # + the row-number index

    # where the time of one describe goes: wall time of infer.describe, of the two C-ABI calls inside it (device passes,
    # copies and the syncs), and the host layer around them (kinds, ranks, edges, interpolation, the dict)
    from mlrun_b200 import columns as mcols

    spent = {"describe": [], "stats_begin": [], "stats_finish": []}

    def clock(owner, name, key):
        real = getattr(owner, name)

        def wrapped(*a, **k):
            t0 = time.perf_counter()
            try:
                return real(*a, **k)
            finally:
                spent[key].append((time.perf_counter() - t0) * 1e3)
        setattr(owner, name, wrapped)
        return real

    reals = [(infer, "describe", clock(infer, "describe", "describe")),
             (mcols.ColumnsPlan, "stats_begin", clock(mcols.ColumnsPlan, "stats_begin", "stats_begin")),
             (mcols.ColumnsPlan, "stats_finish", clock(mcols.ColumnsPlan, "stats_finish", "stats_finish"))]
    timed(lambda: fs.ingest(cols, infer_options=allopt), 10)
    for owner, name, real in reals:
        setattr(owner, name, real)
    med = {k: float(np.median(v)) for k, v in spent.items()}
    res["describe_breakdown_ms_median"] = {
        "describe_total": round(med["describe"], 3), "stats_begin_call": round(med["stats_begin"], 3),
        "stats_finish_call": round(med["stats_finish"], 3),
        "host_layer": round(med["describe"] - med["stats_begin"] - med["stats_finish"], 3)}

    # host cost of entity columns (pandas describe + histogram): an int64 key and a string key of n rows
    keys_int = np.arange(n, dtype=np.int64) * 7
    keys_str = np.array([f"k{i}" for i in range(n)], dtype=object)
    t = time.perf_counter()
    infer.host_stats("id", keys_int, allopt)
    res["entity_describe_host_ms"] = {"int64": round((time.perf_counter() - t) * 1e3, 1)}
    t = time.perf_counter()
    infer.host_stats("key", keys_str, allopt)
    res["entity_describe_host_ms"]["string"] = round((time.perf_counter() - t) * 1e3, 1)

    # the CPU oracle (pandas describe + np.histogram per column) on the frame ingest returns
    from tests import stats_oracle

    with contextlib.redirect_stdout(io.StringIO()):
        frame = fs.ingest(cols).to_pandas()
    t = time.perf_counter()
    with np.errstate(all="ignore"):
        stats_oracle.get_df_stats(frame, allopt)
    res["oracle_cpu_ms"] = round((time.perf_counter() - t) * 1e3, 1)
    text = json.dumps(res, indent=1)
    print(text)
    if out_path:
        with open(out_path, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
