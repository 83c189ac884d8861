#!/usr/bin/env python
"""bench.py -- events/sec of the serving hot path on N B200s (one process per GPU).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--batch B]

Workload (BASELINE.json `metric`): a 3-step serving graph + 4-model ensemble at 64 float32 features:
    Imputer(56 numeric cols) -> OneHotEncoder(8 categorical cols x 4) -> VotingEnsemble(4 linear models)
A "step" is one pass of the fused plan over one batch of B synthetic events already resident in HBM
(`value`), and -- for `e2e` -- the same call through the public host API with pinned HOST buffers
(H2D + kernels + D2H inside the timed region).  Other workloads: flow3_linear (configs[1]), trees_ens4 (configs[2], plus a
`wire` leg: V2 JSON body in, JSON out), ingest6 (configs[4]: feature-set ingest over DataFrame columns), enrich_ens4 (online
feature table gather + ensemble); `--gpus N` under torchrun is configs[3] (event-sharded router, fused P2P ensemble-merge or
`--merge nccl`).  Every workload prints the same JSON line (roofline of its dominant kernel, cpu_baseline, e2e) and has a
`--impl reference` arm.  See DESIGN.md "Measurement".
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BYTES_PER_EVENT = {"flow3_ens4": 260, "flow3_linear": 260, "trees_ens4": 516, "router8": 260, "dense_ens12": 260, "ingest6": 2280, "enrich_ens4": 536}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="flow3_ens4", choices=sorted(BYTES_PER_EVENT))
    ap.add_argument("--batch", type=int, default=0, help="events per step per GPU (default: 1Mi; 256Ki for trees)")
    ap.add_argument("--cpu-seconds", type=float, default=8.0, help="wall budget of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--launches-per-step", type=int, default=0,
                    help="a step = this many back-to-back launches over rotating batches (default: as many as fill ~10 ms, so "
                         "that the K timed steps hold >= 200 ms of kernels)")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config table of the default run (and the configs[3] leg)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N>1: weak = --batch events per GPU; strong = --batch events in total, split over the GPUs "
                         "(BASELINE configs[3]: --workload router8 --scaling strong --batch 65536)")
    ap.add_argument("--merge-wait", default="fused", choices=["fused", "kernel"],
                    help="p2p merge: fused = the scoring launch's last CTA waits for the completion flags itself; kernel = a "
                         "one-warp wait kernel after every launch")
    ap.add_argument("--merge-lag", type=int, default=1, choices=[0, 1],
                    help="p2p merge: 0 = every launch waits for its own completion flags (lockstep); 1 = it waits for the "
                         "previous launch's (pipelined: the merged response of a batch is complete one launch later)")
    ap.add_argument("--merge", default="p2p", choices=["p2p", "nccl"],
                    help="N>1 ensemble-merge: p2p = votes stored into every rank's buffer from the kernel epilogue over "
                         "NVLink peer memory (fused); nccl = a separate all_gather per step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed (rank 0) as DIR/<name>.npy, float32 or "
                         "float64, at most 64 MB in all (a fixed seeded sample of rows when larger): the same arguments give "
                         "the same inputs, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the device path: --impl b200")
    return args


DUMP_BYTES = 60 << 20  # of array data: the .npy headers stay within 64 MB beside it


def dump_rows(n, bytes_per_row):
    """the rows a dump keeps: all n when they fit DUMP_BYTES, else a fixed seeded sample of them (sorted)"""
    k = DUMP_BYTES // bytes_per_row
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))


def dump_arrays(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------ workloads
def make_workload(name, n_rows, seed=2):
    from mlrun_b200.synthetic import flow3_workload, ingest_workload, tree_workload

    if name == "ingest6":
        return ingest_workload(n_rows=n_rows, seed=seed + 3)

    if name == "flow3_ens4":
        return flow3_workload(n_rows=n_rows, n_num=56, n_cat=8, seed=seed, n_models=4)
    if name == "flow3_linear":
        return flow3_workload(n_rows=n_rows, n_num=56, n_cat=8, seed=seed, n_models=1)
    if name == "router8":
        return router8_workload(n_rows, seed=4)
    if name == "dense_ens12":
        return dense12_workload(n_rows, seed=6)
    return tree_cfg3_workload(n_rows, seed=3)


class Router8Workload:
    """BASELINE configs[3] (SURVEY 8(d) config 4): X (n, 64) float32 ~ N(0,1), seed 4; a VotingEnsemble router of 8 scorers over
    the 64 raw features -- 4 linear (random float64 weights, like configs[1]'s) and 4 GradientBoostingRegressor(100 trees,
    depth 6) fit on 20 000 rows (the committed fixtures tests/golden/trees_cfg4_reg.pkl.xz)"""

    def __init__(self, X, models):
        self.X, self.models, self.kind = X, models, "regression"

    def build_server(self, api, executor="array", **kw):
        fn = api.new_function("router8", kind="serving")
        graph = fn.set_topology("router", api.VotingEnsemble(vote_type="regression", executor_type=executor))
        for i, m in enumerate(self.models):
            graph.add_route(f"m{i + 1}", class_name="SKLearnModelServer", model=m, model_path="")
        return fn.to_mock_server(namespace={"SKLearnModelServer": api.SKLearnModelServer}, **kw)


def router8_workload(n_rows, seed=4):
    import lzma

    import cloudpickle
    from sklearn.linear_model import LinearRegression

    with lzma.open(os.path.join(ROOT, "tests", "golden", "trees_cfg4_reg.pkl.xz"), "rb") as fp:
        trees = cloudpickle.load(fp)
    wr = np.random.default_rng(seed + 20)
    models = []
    for i in range(4):
        lin = LinearRegression()
        lin.coef_, lin.intercept_, lin.n_features_in_ = wr.normal(size=64), float(wr.normal()), 64
        models += [lin, trees[i]]  # alternating: linear, tree, linear, tree ...
    X = np.random.default_rng(seed).normal(size=(n_rows, 64)).astype(np.float32)
    return Router8Workload(X, models)


def dense12_workload(n_rows, seed=6):
    """the dense linear-predict path the north_star puts on the tensor cores: a VotingEnsemble of 12 linear scorers over 64 raw
    float32 features (random float64 weights, like configs[1]'s) -- 12 scores per event, N = 16 on tcgen05 (csrc/b2s_dense.cu)"""
    from sklearn.linear_model import LinearRegression

    wr = np.random.default_rng(seed + 20)
    models = []
    for _ in range(12):
        lin = LinearRegression()
        lin.coef_, lin.intercept_, lin.n_features_in_ = wr.normal(size=64), float(wr.normal()), 64
        models.append(lin)
    X = np.random.default_rng(seed).normal(size=(n_rows, 64)).astype(np.float32)
    return Router8Workload(X, models)


def tree_cfg3_workload(n_rows, seed=3, kind="reg"):
    """SURVEY.md 8(d) config 3 as written: X ~ N(0,1) float32 (n_rows, 128); 4 x GradientBoosting{Regressor,Classifier}(100
    trees, depth 6, random_state 30+i) fit on 20 000 rows with every feature considered at every split.  Fitting takes
    minutes, so the fitted estimators are the committed fixtures of tests/golden/gen_trees_cfg3.py."""
    import lzma

    import cloudpickle

    from mlrun_b200.synthetic import TreeWorkload

    with lzma.open(os.path.join(ROOT, "tests", "golden", f"trees_cfg3_{kind}.pkl.xz"), "rb") as fp:
        models = cloudpickle.load(fp)
    X = np.random.default_rng(seed).normal(size=(n_rows, 128)).astype(np.float32)
    return TreeWorkload(X, models, "regression" if kind == "reg" else "classification")


def build_server(name, wl):
    """the serving graph, built with the reference's own plugin calls on mlrun_b200, and its fused plan"""
    from mlrun_b200 import api

    if name.startswith("flow3"):
        server = wl.build_server(api, engine="sync")
        names = wl.names
    else:
        server = wl.build_server(api)
        names = [f"f{i}" for i in range(wl.X.shape[1])]
    compiled = server.compile(names)
    return server, compiled.plan, names


# ------------------------------------------------------------------------------------------ CPU baseline (oracle)
def _cpu_worker(args):
    name, n_events, seed = args
    import logging

    logging.disable(logging.CRITICAL)
    try:  # one BLAS/OpenMP thread per worker process: P workers already cover the cores
        from threadpoolctl import threadpool_limits

        threadpool_limits(1)
    except Exception:
        pass
    from tests import api_oracle

    if name == "enrich_ens4":
        return _enrich_cpu_worker((n_events, seed))
    if name == "ingest6":
        import contextlib
        import io

        from oracle import ingest as oingest
        from oracle import transforms as otransforms

        wl = make_workload(name, n_events, seed)
        steps = wl.build_steps(otransforms)
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):  # the validator prints every violation
            oingest.ingest_rows(steps, wl.df)
        return n_events, time.perf_counter() - t0
    wl = make_workload(name, max(n_events, 8) if name.startswith("flow3") else 64, seed)
    if name.startswith("flow3"):
        server = wl.build_server(api_oracle)
        rows = wl.rows_as_dicts()
        path = "/" if wl.n_models == 1 else "/v2/models/infer"
        t0 = time.perf_counter()
        for row in rows[:n_events]:
            server.test(path=path, body=row)
        return n_events, time.perf_counter() - t0
    server = wl.build_server(api_oracle)
    t0 = time.perf_counter()
    for i in range(n_events):
        server.test("/v2/models/infer", body={"inputs": [wl.X[i % 64].astype(np.float64).tolist()]})
    return n_events, time.perf_counter() - t0


def _cpu_batched_worker(args):
    """SURVEY 8(d) (ii), "reference-batched": ONE event carrying all B rows in `inputs` -- what a user of the reference does to
    go fast on a router / model topology: every model sees (B, F) in one predict (V2ModelServer.do_event -> predict,
    serving/v2_serving.py:228-342), the vote runs once over (B, M) (routers.py:789-810); json-free (`server.test` with a dict)"""
    name, n_rows, seconds, seed = args
    import logging

    logging.disable(logging.CRITICAL)
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(1)
    except Exception:
        pass
    from tests import api_oracle

    wl = make_workload(name, n_rows, seed)
    server = wl.build_server(api_oracle)
    body = {"inputs": wl.X.astype(np.float64).tolist()}
    server.test("/v2/models/infer", body=body)
    reps, t0 = 0, time.perf_counter()
    while reps < 2 or time.perf_counter() - t0 < seconds:
        server.test("/v2/models/infer", body=body)
        reps += 1
    return reps * n_rows, time.perf_counter() - t0


def usable_cores():
    """host threads this process may really use: affinity mask, capped by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0))
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def cpu_baseline(name, seconds, procs=None):
    """the reference's per-event path (restated: oracle/) on all host cores: P independent worker
    processes, like nuclio's N workers (mlrun/runtimes/nuclio/serving.py:59), each pushing one
    MockEvent per row through GraphServer.run (sync engine)."""
    import multiprocessing as mp

    procs = procs or usable_cores()
    # calibrate on one process, then size the sample to the time budget
    n_cal = 300 if name.startswith("flow3") else (200 if name in ("ingest6", "enrich_ens4") else 40)
    n, dt = _cpu_worker((name, n_cal, 2))
    rate1 = n / dt
    # with P busy processes each one runs slower than alone (shared caches / SMT): budget for ~2x
    per_proc = int(max(n_cal, min(rate1 * seconds * 0.5, 200000)))
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(procs) as pool:
        res = pool.map(_cpu_worker, [(name, per_proc, 2 + i) for i in range(procs)])
    wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    if name.startswith("flow3") or name in ("ingest6", "enrich_ens4"):
        batched = ("n/a: this graph's feature steps take one dict per event (feature_store/steps.py:397-406, 453-478); only router / "
                   "model topologies accept B rows in one event")
    else:  # SURVEY 8(d) (ii): one event carrying 4 096 rows, on every core at once
        with ctx.Pool(procs) as pool:
            bres = pool.map(_cpu_batched_worker, [(name, 4096, max(1.0, seconds * 0.25), 2 + i) for i in range(procs)])
        batched = {"value": sum(r[0] for r in bres) / max(r[1] for r in bres), "unit": "events/s", "cores": procs, "rows_per_event": 4096,
                   "single_process_events_per_s": bres[0][0] / bres[0][1],
                   "how": "one MockEvent carrying 4 096 rows in `inputs` through the oracle GraphServer: every model predicts (B, F) "
                          "once, one vote over (B, M)"}
    return {
        "reference_batched": batched,
        "value": total / slowest,
        "unit": "events/s",
        "cores": procs,
        "kind": "port",
        "sample": (f"{total} rows ({per_proc}/process x {procs} processes), one dict per row through the six steps' "
                   f"_do_storey (oracle restatement of the storey ingest walk); single-process rate {rate1:.0f} rows/s; "
                   f"wall {wall:.1f}s") if name == "ingest6" else
                  f"{total} events ({per_proc}/process x {procs} processes), one MockEvent per row through the "
                  f"oracle GraphServer (sync engine); single-process rate {rate1:.0f} events/s; wall {wall:.1f}s",
        "single_process_events_per_s": rate1,
    }


def cpu_vectorised(name, wl_small):
    """upper bound of a CPU implementation: vectorised numpy / scikit-learn on one core"""
    from oracle import batch as obatch

    if name == "ingest6":
        from oracle import ingest as oingest
        from oracle import transforms as otransforms

        steps = wl_small.build_steps(otransforms)
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 1.5:
            oingest.ingest_columns(steps, wl_small.df)
            reps += 1
        return reps * len(wl_small.df) / (time.perf_counter() - t0)
    fn = obatch.flow3 if name.startswith("flow3") else obatch.tree_ensemble
    fn(wl_small)
    t0 = time.perf_counter()
    reps = 0
    while time.perf_counter() - t0 < 1.5:
        fn(wl_small)
        reps += 1
    return reps * wl_small.X.shape[0] / (time.perf_counter() - t0)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r for t, r in self.rows if (t0 is None or t >= t0) and (t1 is None or t <= t1)] or [r for _, r in self.rows]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_traffic(name, B):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture of this workload
    (profiles/traffic.json, bytes per event), scaled to this launch; None if no capture is on file"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        rec = json.load(open(p)).get(name)
        return rec["dram_bytes_per_event"] * B if rec else None
    except (OSError, ValueError, KeyError):
        return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank):
    if rank != 0:
        return
    # a step = one bounded sample of the workload through the CPU path on all usable host cores; exactly K of them are
    # timed after W untimed ones, sized so that the whole run stays within a few minutes
    steps = max(1, args.steps)
    budget = max(0.5, min(args.cpu_seconds, 150.0 / steps))
    for _ in range(max(0, args.warmup)):
        cpu_baseline(args.workload, min(budget, 1.0))
    per_step, wall, info = [], [], None
    for _ in range(steps):
        t0 = time.perf_counter()
        info = cpu_baseline(args.workload, budget)
        wall.append(time.perf_counter() - t0)
        per_step.append(info["value"])
    value = float(np.median(per_step))
    info["value"] = value
    print(json.dumps({
        "impl": "reference", "metric": "events/sec", "value": value, "unit": "events/s", "n_gpus": args.gpus,
        "steps": len(per_step), "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(wall)), "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_desc(args.workload), "engine": "sync per-event (oracle restatement of "
                   "mlrun.serving; storey/mlrun are not installable here)"},
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_desc(name):
    return {
        "flow3_ens4": "3-step flow Imputer->OneHotEncoder->VotingEnsemble(4 linear models), 64-feat f32 (56 num + 8 cat x4 -> 88)",
        "flow3_linear": "3-step flow Imputer->OneHotEncoder->linear predict, 64-feat f32 (BASELINE configs[1])",
        "router8": "router of 8 scorers (4 linear + 4 GradientBoostingRegressor(100 trees, depth 6)), 64-feat f32, sharded by events "
                   "with the fused ensemble-merge (BASELINE configs[3], SURVEY 8(d) config 4)",
        "dense_ens12": "VotingEnsemble of 12 linear scorers over 64 raw f32 features: the dense linear-predict path on the tensor "
                       "cores (tcgen05 kind::tf32, exact 3-term splits; north_star)",
        "trees_ens4": "VotingEnsemble of 4 GradientBoostingRegressor(100 trees, depth 6, fit on 20 000 rows, all features), "
                      "128-feat f32 (BASELINE configs[2], SURVEY 8(d) config 3)",
        "enrich_ens4": "real-time enrichment: entity keys -> online feature table (4 Mi keys x 64 f32, 1 GiB in HBM) -> $mean imputing "
                       "-> VotingEnsemble(4 linear models) (EnrichmentVotingEnsemble, SURVEY 8(f) #3)",
        "ingest6": "feature-set ingest, 256 four-byte slots/row (192 f32 + 62 int32 + datetime64): Imputer -> MapValues(ranges, 16 cols) "
                   "-> OneHotEncoder(8 cols x 8) -> DateExtractor(hour, day_of_week) -> DropFeatures(16) -> FeaturesetValidator(8 cols) "
                   "(BASELINE configs[4])",
    }[name]



# ------------------------------------------------------------------------------------------ per-config table
def serving_config_bench(nat, torch, name, B, min_ms=60.0, e2e_ms=250.0, seed=2):
    """one row of the `configs` table: the fused plan of workload `name` at `B` events per launch -- CUDA-event time of
    back-to-back launches over rotating batches (> L2 between re-reads), and the same batch through the public API from pinned
    host memory (H2D + kernel + D2H per call)"""
    wl = make_workload(name, min(B, 65536), seed)
    server, plan, names = build_server(name, wl)
    F = wl.X.shape[1]
    row_bytes = F * 4
    nbuf = max(2, int(np.ceil(2 * 126e6 / (B * row_bytes))) + 1)
    reps = int(np.ceil(nbuf * B / wl.X.shape[0]))
    big = torch.from_numpy(np.tile(wl.X, (reps, 1))[: nbuf * B]).cuda()
    ptrs = [big.data_ptr() + i * B * row_bytes for i in range(nbuf)]
    out = torch.empty(B * plan.out_cols, dtype=torch.float32, device="cuda")
    plan.time_device(ptrs, B, row_bytes, out.data_ptr(), 5)
    probe = plan.time_device(ptrs, B, row_bytes, out.data_ptr(), 10) / 10
    iters = int(min(20000, max(20, min_ms / max(probe, 1e-4))))
    l0 = nat.launch_count()
    ms = plan.time_device(ptrs, B, row_bytes, out.data_ptr(), iters) / iters
    launches = nat.launch_count() - l0
    peak, _src = measured_peak()
    bpe = BYTES_PER_EVENT[name]
    row = {"workload": name, "batch": B, "kernel": plan.kernel, "ms_per_launch": ms, "events_per_s": B / (ms * 1e-3),
           "algorithmic_bytes_per_event": bpe, "roofline_frac": bpe * B / (ms * 1e-3) / 1e9 / peak, "launches_timed": int(launches),
           "timed_ms": ms * iters, "input_rotation": f"{nbuf} batches, {nbuf * B * row_bytes / 1e6:.0f} MB"}
    hin = [nat.pinned_empty((B, F), np.float32) for _ in range(2)]
    src = np.tile(wl.X, (int(np.ceil(B / wl.X.shape[0])), 1))[:B]
    for j, h in enumerate(hin):
        h[:] = np.roll(src, j * 131, axis=0)
    for j in range(3):
        server.run_batch(hin[j % 2], names=names, with_status=True)
    t0 = time.perf_counter()
    server.run_batch(hin[0], names=names, with_status=True)
    one = time.perf_counter() - t0
    n = int(min(3000, max(5, e2e_ms * 1e-3 / max(one, 1e-6))))
    t0 = time.perf_counter()
    for j in range(n):
        server.run_batch(hin[j % 2], names=names, with_status=True)
    dt = time.perf_counter() - t0
    row["e2e_events_per_s"] = B * n / dt
    row["e2e_ms_per_call"] = 1e3 * dt / n
    row["e2e_calls_timed"] = n
    del big, out, hin
    return row


def ring_bench(nat, name="flow3_ens4", seconds=0.5):
    """the coalescing ring (b2s_submit / b2s_wait: the replacement of storey's emit / await_result) by itself: native
    producer threads, each emitting a few rows and awaiting them; and `GraphServer.run_events` / `emit` + `await_result`
    (the per-event Python callers of the same ring)"""
    wl = make_workload(name, 8192, 5)
    server, plan, names = build_server(name, wl)
    X = np.ascontiguousarray(wl.X)
    rows = []
    for producers, per in ((1, 1), (8, 1), (32, 1), (128, 1), (8, 16), (32, 16), (128, 16)):
        plan.ring_bench(X, producers, per, 0.1)
        rows.append(plan.ring_bench(X, producers, per, seconds))
    bodies = wl.rows_as_dicts(limit=4096)
    server.run_events(bodies[:64])
    t0 = time.perf_counter()
    reps = 0
    while time.perf_counter() - t0 < seconds:
        server.run_events(bodies)
        reps += 1
    run_events = {"events_per_s": reps * len(bodies) / (time.perf_counter() - t0), "batch": len(bodies),
                  "api": "GraphServer.run_events(list of feature dicts): pack -> one fused launch -> per-event responses"}
    lat = []
    for body in bodies[:300]:
        t0 = time.perf_counter()
        server.await_result(server.emit(body))
        lat.append((time.perf_counter() - t0) * 1e6)
    return {"how": "b2s_ring_bench: N native threads, each b2s_submit(rows) + b2s_wait(ticket) in a loop (default ring: "
                   "4 slots x 65536 rows, max_wait_us 0: a blocked caller runs its batch as soon as the stream is free, rows of other callers join meanwhile); events/s = rows served / wall",
            "native": rows, "run_events": run_events,
            "emit_await_one_caller_us": {"p50": float(np.percentile(lat[20:], 50)), "p99": float(np.percentile(lat[20:], 99)),
                                         "how": "GraphServer.emit(body) + await_result(ticket), one Python caller"}}


def config4_leg(rank, world, steps=10, timeout_s=100.0, workload_args=("--workload", "router8", "--scaling", "strong", "--batch", "65536", "--no-e2e"),
                port_shift=17):
    """BASELINE configs[3] as written -- the 8-model mixed router (4 linear + 4 tree scorers), GLOBAL batch 65 536 split over the
    GPUs (strong scaling), fused P2P ensemble-merge -- measured beside the headline workload so that the driver's 1 / 2 / 4 / 8
    runs carry its curve.  Every rank starts `bench.py --workload router8 --scaling strong --batch 65536` as a CHILD process
    (the invocation the 2-GPU lab runs used, profiles/lab/gpu18.sh); the children form their own process group (same RANK /
    WORLD_SIZE, MASTER_PORT + 17, torchrun's agent-store variables removed so that child rank 0 hosts the store).  A separate
    process, so a failure or a hang of this leg costs its own row after `timeout_s`, never the parent's line.
    `workload_args` selects another stand-alone invocation the same way (the configs[4] ingest leg).
    -> summary dict on rank 0, None elsewhere."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("TORCHELASTIC_")}
    if world > 1:
        env["MASTER_PORT"] = str(int(os.environ.get("MASTER_PORT", "29500")) + port_shift)
    cmd = [sys.executable, os.path.abspath(__file__)] + list(workload_args) + ["--gpus", str(world), "--steps", str(steps), "--warmup", "3",
                                                                     "--no-cpu-baseline", "--no-configs"]
    if os.environ.get("B2S_BENCH_CONFIG4_CMD"):  # tests: a stand-in child (tests/test_bench_config4_cpu.py)
        cmd = [sys.executable] + json.loads(os.environ["B2S_BENCH_CONFIG4_CMD"])
    t0 = time.perf_counter()
    try:
        done = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout_s)
    except subprocess.TimeoutExpired:
        return {"error": f"child did not finish within {timeout_s:.0f} s (killed)"} if rank == 0 else None
    if rank != 0:
        return None
    try:
        d = json.loads(done.stdout.strip().splitlines()[-1])
        cfg = d.get("config", {})
        lps = max(int(cfg.get("launches_per_step", 1)), 1)
        return {"workload": cfg.get("workload"), "scaling": d.get("scaling"), "n_gpus": d.get("n_gpus"), "global_batch": cfg.get("global_batch"),
                "batch_per_gpu": cfg.get("batch_per_gpu"), "events_per_s": d.get("value"), "ms_per_launch": d.get("ms_per_step", 0.0) / lps,
                "launches_timed": lps * int(d.get("steps", 0)), "parallelism": cfg.get("parallelism"), "merge_verified": cfg.get("merge_verified"),
                "kernel": cfg.get("kernel"), "roofline_frac": (d.get("roofline") or {}).get("frac"), "clocks": d.get("clocks"),
                "p50_step_latency_us": (d.get("p50_step_latency_us") or {}).get("p50"), "wall_s": round(time.perf_counter() - t0, 1),
                **({"e2e": {k: d["e2e"].get(k) for k in ("value", "unit", "batch", "steps", "h2d_bytes_per_step", "d2h_bytes_per_step", "api")}}
                   if isinstance(d.get("e2e"), dict) else {}),
                "how": "child process per rank: " + " ".join(cmd[1:])}
    except Exception as exc:  # noqa: BLE001 -- the row reports what went wrong
        return {"error": f"{type(exc).__name__}: {exc}", "rc": done.returncode, "stderr_tail": done.stderr[-400:]}


def compact_line(line):
    """a full bench line of another workload -> one row of the `configs` table"""
    r = line["roofline"]
    row = {"workload": line["config"]["workload"].split(",")[0][:60], "batch": line["config"]["batch_per_gpu"], "kernel": r["kernel"],
           "ms_per_launch": r["kernel_ms_per_launch"], "events_per_s": line["value"],
           "algorithmic_bytes_per_event": r["algorithmic_bytes_per_event"], "roofline_frac": r["frac"],
           "launches_timed": line["gpu_launches"], "p50_launch_us_at_4096": line["p50_step_latency_us"]["p50"]}
    if "e2e" in line:
        row["e2e_events_per_s"] = line["e2e"]["value"]
        row["e2e_api"] = line["e2e"]["api"][:80]
    return row

# ------------------------------------------------------------------------------------------ main (b200 arm)
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    name = args.workload
    if name == "ingest6":
        return main_ingest(args, rank, local_rank, world)
    if name == "enrich_ens4":
        return main_enrich(args, rank, local_rank, world)
    B = args.batch or (262144 if name == "trees_ens4" else (65536 if name == "router8" else 1048576))
    if args.scaling == "strong":
        B = max(64, B // world)  # the global batch is fixed; every GPU takes its share
    default_run = name == "flow3_ens4" and world == 1 and not args.batch and not args.no_configs

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(name, args.cpu_seconds)  # forks: must run before CUDA is initialised
        cpu["vectorised_numpy_events_per_s_1core"] = cpu_vectorised(name, make_workload(name, 4096))

    import torch

    from mlrun_b200 import _native as nat

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    nat.init(local_rank)
    info = nat.device_info()

    wl = make_workload(name, 65536, seed=2 + rank)
    server, plan, names = build_server(name, wl)
    F = wl.X.shape[1]
    # inputs resident in HBM: NBUF distinct batches, rotated, so that consecutive steps never re-read L2-resident rows
    row_bytes = F * 4
    nbuf = max(2, int(np.ceil(2 * 126e6 / (B * row_bytes))) + 1)
    reps = int(np.ceil(B / wl.X.shape[0]))
    base = torch.from_numpy(np.tile(wl.X, (reps, 1))[:B])
    bufs = []
    for i in range(nbuf):
        bufs.append(torch.roll(base, shifts=i * 977, dims=0).cuda())
    out = torch.empty(B * plan.out_cols, dtype=torch.float32, device="cuda")
    gathered = torch.empty(world * B * plan.out_cols, dtype=torch.float32, device="cuda") if world > 1 else None
    stream = torch.cuda.Stream()  # a real (non-NULL) stream: kernels, NCCL and the timing events all ride on it
    torch.cuda.set_stream(stream)
    merge = args.merge if world > 1 else "none"
    comm = None
    if merge == "p2p":
        # the product's communicator (mlrun_b200.sharding.MergeComm / b2s_comm_*): every rank owns the merged response rows,
        # double buffered, plus completion flags; the kernels of ALL ranks store their shard's votes into ALL of them over
        # NVLink peer mappings (CUDA IPC) and publish a flag; no collective and no host barrier run in the step
        from mlrun_b200.sharding import MergeComm, torch_exchange

        try:
            comm = MergeComm(rank, world, B, plan.out_cols, torch_exchange(dist))
            comm.set_fused_wait(args.merge_lag if args.merge_wait == "fused" else None)
            comm.attach(plan)
        except Exception as exc:  # noqa: BLE001 -- no peer access on this box: use the NCCL merge
            print(f"[rank {rank}] p2p merge unavailable ({exc}); using nccl", file=sys.stderr)
            merge = "nccl"
        flags = torch.tensor([1 if merge == "p2p" else 0], device="cuda")
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        if int(flags.item()) == 0 and merge == "p2p":
            comm.detach(plan)
            comm = None
            merge = "nccl"
    last_merged = [None]

    def launch(i):
        plan.run_device(bufs[i % nbuf].data_ptr(), B, row_bytes, out.data_ptr(), None, stream.cuda_stream)
        if merge == "nccl":  # ensemble-merge: every rank ends up with every shard's votes (4 B/event)
            dist.all_gather_into_tensor(gathered, out)
        elif merge == "p2p":  # lag 0: the step is over when this rank has seen the completion flags of all shards;
            # lag 1 (default): the wait is for the previous launch, this one's votes travel while the next is scored
            comm.wait(stream.cuda_stream, args.merge_lag)

    inner = args.launches_per_step

    def step(i):  # one step = `inner` launches, each over the next of the rotating batches
        for j in range(inner):
            launch(i * inner + j)

    def drain():  # pipelined merge: the last launch's votes have to be complete inside the timed region
        if merge == "p2p":
            last_merged[0] = comm.wait(stream.cuda_stream, 0)[0]

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if inner <= 0:  # size a step to ~10 ms of launches (the same on every rank: the probe's maximum)
        for i in range(5):
            launch(i)
        sync()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(stream)
        for i in range(10):
            launch(i)
        p1.record(stream)
        sync()
        probe = torch.tensor([p0.elapsed_time(p1) / 10], device="cuda")
        if world > 1:
            dist.all_reduce(probe, op=dist.ReduceOp.MAX)
        inner = int(max(1, min(1000, round(10.0 / max(float(probe.item()), 1e-3)))))
    for i in range(max(args.warmup, 3)):
        step(i)
    sync()
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    time.sleep(0.25)
    l0 = nat.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record(stream)
    for i in range(args.steps):
        step(i)
    drain()
    e1.record(stream)
    sync()
    t_wall1 = time.perf_counter()
    launches = nat.launch_count() - l0
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    merge_check = None
    if merge == "p2p":
        # every rank must now hold every shard: the last step's merged rows against the same launch scored locally
        comm.check()
        full = np.empty((world * comm.max_rows, plan.out_cols), dtype=np.float32)
        nat.check(nat.load().b2s_memcpy_d2h(full.ctypes.data, last_merged[0], full.nbytes))
        comm.detach(plan)  # the single-GPU measurements below write locally again
        last = inner * args.steps - 1 if inner > 0 else args.steps - 1
        plan.run_device(bufs[last % nbuf].data_ptr(), B, row_bytes, out.data_ptr(), None, stream.cuda_stream)
        torch.cuda.synchronize()
        mine = out.cpu().numpy().reshape(B, plan.out_cols)
        ok_mine = bool(np.array_equal(full[rank * comm.max_rows: rank * comm.max_rows + B], mine))
        sums = [None] * world
        dist.all_gather_object(sums, float(mine.astype(np.float64).sum()))
        got = [float(full[r * comm.max_rows: r * comm.max_rows + B].astype(np.float64).sum()) for r in range(world)]
        merge_check = ok_mine and all(abs(got[r] - sums[r]) <= 1e-9 * max(1.0, abs(got[r])) for r in range(world))
        oks = [None] * world
        dist.all_gather_object(oks, merge_check)
        merge_check = all(oks)
    if args.dump_outputs and rank == 0:
        # the last launch read rotating buffer k, the base batch shifted down by k * 977 rows: shifting its scores back puts
        # them in the base batch's row order whichever buffer that was (`inner`, hence k, is sized from a timing probe)
        scores = mine if merge == "p2p" else out.cpu().numpy().reshape(B, plan.out_cols)
        scores = np.roll(scores, -((inner * args.steps - 1) % nbuf) * 977, axis=0)
        dump_arrays(args.dump_outputs, {"outputs": scores[dump_rows(B, scores.itemsize * plan.out_cols)]})

    # kernel-only time of the dominant kernel (no collective), for the roofline
    n_k = max(args.steps * inner, 10)
    kms = plan.time_device([b.data_ptr() for b in bufs], B, row_bytes, out.data_ptr(), n_k) / n_k

    # latency at the configured serving batch (4096 events): one launch per batch, CUDA-event timed
    lat = []
    small = bufs[0].data_ptr()
    for _ in range(100):
        plan.time_device([small], 4096, row_bytes, out.data_ptr(), 1)
    for _ in range(1000):
        lat.append(plan.time_device([small], 4096, row_bytes, out.data_ptr(), 1) * 1e3)
    # end-to-end latency of one serving batch: host rows -> b2s_run_host (H2D, kernel, D2H) -> host results, wall clock
    lat_e2e = []
    h_small = nat.pinned_empty((4096, F), np.float32)
    h_small[:] = base[:4096].numpy()
    for _ in range(100):
        plan.run(h_small, with_status=True)
    for _ in range(1000):
        t0 = time.perf_counter()
        plan.run(h_small, with_status=True)
        lat_e2e.append((time.perf_counter() - t0) * 1e6)

    e2e = None
    if not args.no_e2e:
        Be = B  # the same batch as the device-timed step
        hin = [nat.pinned_empty((Be, F), np.float32) for _ in range(2)]
        for j, h in enumerate(hin):
            h[:] = np.roll(base[:Be].numpy(), j * 131, axis=0)
        for j in range(3):
            server.run_batch(hin[j % 2], names=names)
        sync()
        n_e2e = max(5, min(args.steps, 20))
        t0 = time.perf_counter()
        for j in range(n_e2e):
            res, sts = server.run_batch(hin[j % 2], names=names, with_status=True)
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": world * Be * n_e2e / dt, "unit": "events/s", "h2d_bytes_per_step": Be * row_bytes,
               "d2h_bytes_per_step": Be * (plan.out_cols + 1) * 4, "batch": Be, "steps": n_e2e,
               "api": "GraphServer.run_batch (public API) -> b2s_run_host: pinned host rows -> H2D -> fused kernel -> "
                      "D2H outputs + per-row status"}

    wire = None
    if name == "trees_ens4" and rank == 0 and not args.no_e2e:
        # wire level (SURVEY 8(f) #2): a V2 JSON body of 4096 events -> JSON response, C body codec + one fused launch;
        # beside it the reference's own decode/encode of the same body (json.loads -> np.asarray, json.dumps), model excluded
        import json as _json

        Bw = 4096
        body = _json.dumps({"inputs": wl.X[:Bw].astype(np.float64).tolist()}).encode()
        for _ in range(2):
            resp = server.run_json(body, event_id="w")
        n_w = 8
        t0 = time.perf_counter()
        for _ in range(n_w):
            resp = server.run_json(body, event_id="w")
        dt_w = (time.perf_counter() - t0) / n_w
        t0 = time.perf_counter()
        for _ in range(3):
            np.asarray(_json.loads(body)["inputs"], dtype=np.float64)
            _json.dumps({"id": "w", "model_name": "x", "outputs": [0.5] * Bw})
        dt_py = (time.perf_counter() - t0) / 3
        wire = {"value": Bw / dt_w, "unit": "events/s", "batch": Bw, "body_bytes": len(body), "response_bytes": len(resp.body),
                "api": "GraphServer.run_json: JSON body -> b2s_json_parse_inputs -> fused plan -> b2s_json_format_outputs",
                "python_json_codec_only_events_per_s": Bw / dt_py}

    cfg4 = cfg5 = None
    if name == "flow3_ens4" and not args.batch and args.scaling == "weak" and not args.no_configs:
        # BASELINE configs[3] (strong scaling of the 8-model router at a global batch of 65 536) on the same GPUs, every rank's child
        # at the same point of the run; this process keeps its buffers and is idle meanwhile
        if world > 1:
            dist.barrier()  # the children of all ranks start together
        cfg4 = config4_leg(rank, world)
        if world > 1:  # BASELINE configs[4] on all the GPUs (rows shard over the ranks, no exchange); at N = 1 it is a row of `configs`
            dist.barrier()  # (a leg that failed on one rank only must not stagger the next one)
            cfg5 = config4_leg(rank, world, steps=200, timeout_s=120.0, workload_args=("--workload", "ingest6"), port_shift=23)

    if rank == 0:
        peak, peak_src = measured_peak()
        bpe = BYTES_PER_EVENT[name]
        achieved = bpe * B / (kms * 1e-3) / 1e9
        value = world * B * inner * args.steps / (ms * 1e-3)
        line = {
            "metric": "events/sec", "value": value, "unit": "events/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32 in / f64 accumulate", "data": "synthetic",
            "config": {"workload": workload_desc(name), "batch_per_gpu": B, "global_batch": B * world,
                       "launches_per_step": inner, "events_per_step_per_gpu": B * inner, "timed_region_ms": ms,
                       "parallelism": f"event-sharded x{world}" + {"none": "", "nccl": " + NCCL all-gather of votes per step",
                                                                    "p2p": " + fused P2P ensemble-merge (votes stored to every rank over NVLink "
                                                                           "from the kernel epilogue, completion flags awaited " + ("by the launch's last CTA " if args.merge_wait == "fused" else "by a wait kernel ")
                                                                           + ("each launch)" if args.merge_lag == 0 else "one launch later: pipelined, lag 1)")}[merge],
                       "merge_verified": merge_check,
                       "l2": f"{nbuf} rotating input buffers of {B * row_bytes / 1e6:.0f} MB (> 126 MB L2 between re-reads)",
                       "device": info["name"], "kernel": plan.kernel},
            "p50_step_latency_us": {"batch": 4096, "p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)),
                                    "how": "CUDA events around one fused-kernel launch, 1000 samples after 100 warm-ups",
                                    "e2e_p50": float(np.percentile(lat_e2e, 50)), "e2e_p99": float(np.percentile(lat_e2e, 99)),
                                    "e2e_how": "wall clock of DevicePlan.run on 4096 pinned host rows (H2D + kernel + D2H + status), "
                                               "1000 samples after 100 warm-ups"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_of_nominal_8000": achieved / 8000.0,
                         "traffic": measured_traffic(name, B), "traffic_source": "from_profile: ncu --set full capture of this "
                         "kernel (profiles/traffic.json), scaled to this launch; not measured in this run",
                         "kernel": plan.kernel, "algorithmic_bytes_per_event": bpe,
                         "kernel_ms_per_launch": kms, "peak_source": peak_src},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if e2e:
            line["e2e"] = e2e
        if wire:
            line["wire"] = wire
        if cpu:
            line["cpu_baseline"] = cpu
        if cfg4:
            line["config4"] = cfg4
        if cfg5:
            line["config5"] = cfg5
        if default_run:
            # every config of BASELINE.json (and the SURVEY 8(f) callers) under the same clocks, one row each
            torch.cuda.synchronize()
            del bufs, base
            torch.cuda.empty_cache()
            rows = []
            for nm, bb in (("flow3_ens4", 4096), ("flow3_ens4", 65536), ("flow3_ens4", 1048576), ("flow3_linear", 4096),
                           ("flow3_linear", 1048576), ("trees_ens4", 16384), ("trees_ens4", 262144), ("dense_ens12", 4096),
                           ("dense_ens12", 1048576)):
                try:
                    rows.append(serving_config_bench(nat, torch, nm, bb))
                except Exception as exc:  # noqa: BLE001 -- a failing row must not hide the others
                    rows.append({"workload": nm, "batch": bb, "error": f"{type(exc).__name__}: {exc}"})
                torch.cuda.empty_cache()
            import copy

            sub = copy.copy(args)
            sub.no_cpu_baseline, sub.steps, sub.warmup, sub.batch, sub.dump_outputs = True, 200, 3, 0, None
            for nm, fn in (("ingest6", main_ingest), ("enrich_ens4", main_enrich)):
                try:
                    row = compact_line(fn(sub, 0, local_rank, 1, emit=False))
                    row["workload"] = nm
                    rows.append(row)
                except Exception as exc:  # noqa: BLE001
                    rows.append({"workload": nm, "error": f"{type(exc).__name__}: {exc}"})
                torch.cuda.empty_cache()
            line["configs"] = rows
            try:
                line["ring"] = ring_bench(nat)
            except Exception as exc:  # noqa: BLE001
                line["ring"] = {"error": f"{type(exc).__name__}: {exc}"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main_ingest(args, rank, local_rank, world, emit=True):
    """config 5: the columnar feature-set plan.  Rows shard over ranks with no exchange at all (every rank ingests its
    own partition, as the reference's N workers write their own target partitions)."""
    name = "ingest6"
    B = args.batch or 524288
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(name, args.cpu_seconds)
        cpu["vectorised_numpy_events_per_s_1core"] = cpu_vectorised(name, make_workload(name, 65536))

    import torch

    from mlrun_b200 import _native as nat
    from mlrun_b200.feature_store import ingest as bingest
    from mlrun_b200.feature_store import steps as bsteps

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    nat.init(local_rank)
    info = nat.device_info()
    wl = make_workload(name, 65536, seed=2 + rank)
    fset = bingest.FeatureSet("ingest6", timestamp_key="timestamp")
    cur = fset.graph
    for st in wl.build_steps(bsteps):
        cur = cur.to(st)
    for c, v in zip(wl.checked_cols, [bsteps.MinMaxValidator(severity="info", min=-2.5, max=2.5)] * len(wl.checked_cols)):
        fset[c] = bingest.Feature(validator=v)
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        fset.ingest(wl.df.iloc[:4096])  # lowers the graph (public API) and warms the plan
    iplan = fset.plan
    plan = iplan.plan
    stride = ((B * 4 + 255) // 256) * 256
    ins, _keep = iplan._inputs(wl.df)
    reps = int(np.ceil(B / len(wl.df)))
    nbuf = 2  # 2 x 537 MB of distinct rows: consecutive steps never re-read L2-resident data
    bufs = []
    for j in range(nbuf):
        host = np.zeros(plan.n_in * stride, dtype=np.uint8)
        for slot, a in ins.items():
            raw = np.tile(np.roll(a, j * 977), reps)[:B].view(np.uint8)
            host[slot * stride: slot * stride + raw.size] = raw
        bufs.append(torch.from_numpy(host).cuda())
        del host
    out = torch.empty(plan.n_out * stride, dtype=torch.uint8, device="cuda")
    cnt = torch.zeros(max(plan.n_counters, 1), dtype=torch.int64, device="cuda")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    def step(i):
        plan.run_device(bufs[i % nbuf].data_ptr(), stride, B, out.data_ptr(), stride, cnt.data_ptr(), stream.cuda_stream)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        step(i)
    sync()
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    time.sleep(0.25)
    l0 = nat.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record(stream)
    for i in range(args.steps):
        step(i)
    e1.record(stream)
    sync()
    t_wall1 = time.perf_counter()
    launches = nat.launch_count() - l0
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs and rank == 0:
        # every result column of the last step, as the slots hold it: float32 columns as they are, integer columns as
        # float64, timestamps as float64 seconds since the epoch
        specs, _extra = iplan._landing()
        rows = torch.from_numpy(dump_rows(B, 8 * len(specs))).cuda()
        cols = {}
        for col, slot, dt in specs:
            tdt = {np.float32: torch.float32, np.int32: torch.int32, np.int64: torch.int64}[dt.type]
            a = out[slot * stride: slot * stride + B * dt.itemsize].view(tdt)[rows].cpu().numpy()
            if dt == np.int64:
                a = (a // 10**9).astype(np.float64) + (a % 10**9) * 1e-9
            cols[col] = a if dt == np.float32 else a.astype(np.float64)
        dump_arrays(args.dump_outputs, cols)
    n_it = max(args.steps, 10)
    kms = plan.time_device([b.data_ptr() for b in bufs], stride, B, out.data_ptr(), stride, cnt.data_ptr(), n_it) / n_it
    lat = []
    for _ in range(20):
        plan.time_device([bufs[0].data_ptr()], stride, 4096, out.data_ptr(), stride, cnt.data_ptr(), 1)
    for _ in range(300):
        lat.append(plan.time_device([bufs[0].data_ptr()], stride, 4096, out.data_ptr(), stride, cnt.data_ptr(), 1) * 1e3)

    e2e = None
    if not args.no_e2e:
        frames = [wl.df, wl.df.iloc[::-1].reset_index(drop=True).copy()]  # two materialised frames, alternated
        with contextlib.redirect_stdout(io.StringIO()):
            for j in range(2):
                fset.ingest(frames[j % 2])
            n_e2e = max(3, min(args.steps, 10))
            t0 = time.perf_counter()
            for j in range(n_e2e):
                res = fset.ingest(frames[j % 2])
            dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        Be = len(wl.df)
        e2e_df = {"value": world * Be * n_e2e / dt, "unit": "events/s", "batch": Be, "steps": n_e2e, "out_columns": int(res.shape[1]),
                  "api": "FeatureSet.ingest(DataFrame): frame columns -> H2D per column -> columns_kernel -> D2H per column -> "
                         "DataFrame (pageable host memory; includes the frame (dis)assembly)"}
        # the columnar boundary (SURVEY 8(f) #1): pinned column arrays in, a ColumnBatch over a pinned block out -- no pandas
        # object on either side, the frame pipelined in row ranges (H2D of range r + 1 under kernel + D2H of range r)
        from mlrun_b200.feature_store import columnar

        Bc = 1048576
        reps_c = int(np.ceil(Bc / len(wl.df)))
        cols_in = []
        for j in range(2):
            pc = columnar.pinned_columns({n: wl.df[n].to_numpy() for n in wl.df.columns}, Bc)
            for n in wl.df.columns:
                pc[n][:] = np.tile(np.roll(wl.df[n].to_numpy(), j * 977), reps_c)[:Bc]
            cols_in.append(pc)
        fset_c = bingest.FeatureSet("ingest6c", timestamp_key="timestamp")
        cur = fset_c.graph
        for st_ in wl.build_steps(bsteps):
            cur = cur.to(st_)
        for c_, v_ in zip(wl.checked_cols, [bsteps.MinMaxValidator(severity="info", min=-2.5, max=2.5)] * len(wl.checked_cols)):
            fset_c[c_] = bingest.Feature(validator=v_)
        with contextlib.redirect_stdout(io.StringIO()):
            for j in range(2):
                batch = fset_c.ingest(cols_in[j % 2])
            n_c = max(3, min(args.steps, 6))
            t0 = time.perf_counter()
            for j in range(n_c):
                batch = fset_c.ingest(cols_in[j % 2])
            dtc = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dtc], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtc = float(t.item())
        e2e = {"value": world * Bc * n_c / dtc, "unit": "events/s", "h2d_bytes_per_step": Bc * wl.in_bytes_per_row,
               "d2h_bytes_per_step": Bc * wl.out_bytes_per_row, "batch": Bc, "steps": n_c, "out_columns": len(batch.names),
               "api": "FeatureSet.ingest(pinned column arrays) (public API, columnar boundary): H2D per column and row range -> "
                      "columns_kernel -> D2H per column into a pinned ColumnBatch; pipelined in 64 Ki-row ranges",
               "dataframe_boundary": e2e_df}
        del cols_in, batch
    if rank == 0:
        peak, peak_src = measured_peak()
        bpe = wl.in_bytes_per_row + wl.out_bytes_per_row
        achieved = bpe * B / (kms * 1e-3) / 1e9
        line = {
            "metric": "events/sec", "value": world * B * args.steps / (ms * 1e-3), "unit": "events/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 / int32 / int64 columns, fp64 compares", "data": "synthetic",
            "config": {"workload": workload_desc(name), "batch_per_gpu": B, "global_batch": B * world,
                       "parallelism": f"row-sharded x{world}, no exchange",
                       "l2": f"{nbuf} rotating columnar inputs of {B * wl.in_bytes_per_row / 1e6:.0f} MB (> 126 MB L2)",
                       "device": info["name"], "kernel": "columns_kernel (b2s_columns.cuh)",
                       "n_column_ops": len(iplan.out), "out_slots": plan.n_out},
            "p50_step_latency_us": {"batch": 4096, "p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)),
                                    "how": "CUDA events around one columns_kernel launch, 300 samples"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_of_nominal_8000": achieved / 8000.0,
                         "traffic": measured_traffic(name, B), "kernel": "columns_kernel", "algorithmic_bytes_per_event": bpe,
                         "kernel_ms_per_launch": kms, "peak_source": peak_src},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if emit:
            print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return line if rank == 0 else None


def _enrich_setup(api, n_keys, n_feat, seed):
    """the same enrichment graph on either API (product / oracle)"""
    import pandas as pd
    from sklearn.linear_model import LinearRegression

    rng = np.random.default_rng(seed)
    feat = [f"f{i}" for i in range(n_feat)]
    vals = rng.normal(size=(n_keys, n_feat)).astype(np.float32)
    vals[rng.random(vals.shape) < 0.05] = np.nan
    keys = rng.permutation(n_keys).astype(np.int64) * 7919 + 13
    coefs = np.random.default_rng(seed + 1).normal(size=(4, n_feat))
    return feat, vals, keys, coefs, pd, LinearRegression


def _enrich_cpu_worker(args):
    n_events, seed = args
    import logging

    logging.disable(logging.CRITICAL)
    from oracle import enrichment as oenr
    from tests import api_oracle

    n_keys, n_feat = 20000, 64
    feat, vals, keys, coefs, pd, LinearRegression = _enrich_setup(api_oracle, n_keys, n_feat, seed)
    table = {(int(k),): dict(zip(feat, map(float, v))) for k, v in zip(keys, vals)}
    stats = pd.DataFrame({"mean": np.nanmean(vals, axis=0).astype(np.float64)}, index=feat)
    oenr.register_feature_vector("store://bench", oenr.FeatureVector("bench", feat, ["id"], table, stats))
    fn = api_oracle.new_function("enrich", kind="serving")
    graph = fn.set_topology("router", api_oracle.EnrichmentVotingEnsemble(feature_vector_uri="store://bench", impute_policy={"*": "$mean"},
                                                                          vote_type="regression", executor_type="array"))
    for i in range(4):
        m = LinearRegression()
        m.coef_, m.intercept_, m.n_features_in_ = coefs[i], 0.0, n_feat
        graph.add_route(f"m{i}", class_name="SKLearnModelServer", model=m, model_path="")
    server = fn.to_mock_server(namespace={"SKLearnModelServer": api_oracle.SKLearnModelServer})
    ask = [int(k) for k in keys[np.random.default_rng(seed + 2).integers(0, n_keys, size=n_events)]]
    t0 = time.perf_counter()
    for k in ask:  # one event per entity, as a real-time caller sends them
        server.test("/v2/models/infer", body={"inputs": [[k]]})
    return n_events, time.perf_counter() - t0


def main_enrich(args, rank, local_rank, world, emit=True):
    """SURVEY 8(f) #3: keys -> device hash table gather (+ imputing) -> fused scoring plan; two launches per step"""
    name = "enrich_ens4"
    B = args.batch or 1048576
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(name, args.cpu_seconds)

    import torch

    from mlrun_b200 import _native as nat
    from mlrun_b200 import api

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    nat.init(local_rank)
    info = nat.device_info()
    n_keys, n_feat = 4 * 1048576, 64
    feat, vals, keys, coefs, pd, LinearRegression = _enrich_setup(api, n_keys, n_feat, 2)
    frame = pd.DataFrame(vals, columns=feat, index=pd.Index(keys, name="id"), copy=False)
    api.register_feature_vector("store://bench", api.FeatureVector("bench", feat, ["id"], frame))
    fn = api.new_function("enrich", kind="serving")
    graph = fn.set_topology("router", api.EnrichmentVotingEnsemble(feature_vector_uri="store://bench", impute_policy={"*": "$mean"},
                                                                   vote_type="regression", executor_type="array"))
    for i in range(4):
        m = LinearRegression()
        m.coef_, m.intercept_, m.n_features_in_ = coefs[i], 0.0, n_feat
        graph.add_route(f"m{i}", class_name="SKLearnModelServer", model=m, model_path="")
    server = fn.to_mock_server(namespace={"SKLearnModelServer": api.SKLearnModelServer})
    plan = server.compile().plan
    table = server.graph._object._feature_service.table
    rng = np.random.default_rng(3 + rank)
    nbuf = 3
    d_keys = [torch.from_numpy(keys[rng.integers(0, n_keys, size=B)]).cuda() for _ in range(nbuf)]
    rows = torch.empty(B * n_feat, dtype=torch.float32, device="cuda")
    out = torch.empty(B * plan.out_cols, dtype=torch.float32, device="cuda")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    # one launch when the scoring kernel can gather its own rows from the table (B2S_ENRICH_FUSED=0: gather, then score)
    fused = table.enrich_device(plan, d_keys[0].data_ptr(), 4096, out.data_ptr(), None, stream.cuda_stream)

    def step(i):
        if fused:
            table.enrich_device(plan, d_keys[i % nbuf].data_ptr(), B, out.data_ptr(), None, stream.cuda_stream)
            return
        table.lookup_device(d_keys[i % nbuf].data_ptr(), B, rows.data_ptr(), n_feat * 4, None, stream.cuda_stream)
        plan.run_device(rows.data_ptr(), B, n_feat * 4, out.data_ptr(), None, stream.cuda_stream)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        step(i)
    sync()
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    time.sleep(0.25)
    l0 = nat.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record(stream)
    for i in range(args.steps):
        step(i)
    e1.record(stream)
    sync()
    t_wall1 = time.perf_counter()
    launches = nat.launch_count() - l0
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs and rank == 0:
        scores = out.cpu().numpy().reshape(B, plan.out_cols)
        dump_arrays(args.dump_outputs, {"outputs": scores[dump_rows(B, scores.itemsize * plan.out_cols)]})
    n_it = max(args.steps, 10)
    lat = []
    if fused:  # the step IS the kernel: time it alone, and one 4096-key launch for the latency figure
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record(stream)
        for i in range(n_it):
            step(i)
        k1.record(stream)
        sync()
        kms = k0.elapsed_time(k1) / n_it
        for j in range(320):
            k0.record(stream)
            table.enrich_device(plan, d_keys[0].data_ptr(), 4096, out.data_ptr(), None, stream.cuda_stream)
            k1.record(stream)
            k1.synchronize()
            if j >= 20:
                lat.append(k0.elapsed_time(k1) * 1e3)
    else:
        kms = table.time_device([k.data_ptr() for k in d_keys], B, rows.data_ptr(), n_feat * 4, n_it) / n_it
        for _ in range(20):
            table.time_device([d_keys[0].data_ptr()], 4096, rows.data_ptr(), n_feat * 4, 1)
        for _ in range(300):
            lat.append(table.time_device([d_keys[0].data_ptr()], 4096, rows.data_ptr(), n_feat * 4, 1) * 1e3)
    e2e = None
    if not args.no_e2e:
        Be = B  # the same batch as the device-timed step
        hk = [nat.pinned_empty((Be,), np.int64) for _ in range(2)]  # the step's inputs wait in pinned host memory
        for h in hk:
            h[:] = keys[rng.integers(0, n_keys, size=Be)]
        for j in range(2):
            server.run_enriched(hk[j % 2])
        n_e2e = max(5, min(args.steps, 20))
        t0 = time.perf_counter()
        for j in range(n_e2e):
            res = server.run_enriched(hk[j % 2], with_status=True)
        dt = time.perf_counter() - t0
        e2e = {"value": world * Be * n_e2e / dt, "unit": "events/s", "h2d_bytes_per_step": Be * 8, "d2h_bytes_per_step": Be * 8,
               "batch": Be, "steps": n_e2e, "api": "GraphServer.run_enriched(keys) (public API) -> b2s_table_enrich_host: host int64 keys -> H2D -> "
               "gather kernel -> fused scoring plan -> D2H votes + status (pinned result block)"}
        del res
    if rank == 0:
        peak, peak_src = measured_peak()
        # fused: key 8 + slot 16 + row 4F + vote 4 (the gathered rows never reach HBM); else the gather kernel alone
        bpe = 8 + 16 + 4 * n_feat + 4 * plan.out_cols if fused else BYTES_PER_EVENT[name]
        top = f"{plan.kernel.split(' ')[0]} with the gather loader" if fused else "table_lookup_kernel"
        achieved = bpe * B / (kms * 1e-3) / 1e9
        line = {
            "metric": "events/sec", "value": world * B * args.steps / (ms * 1e-3), "unit": "events/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 rows / int64 keys, f64 accumulate", "data": "synthetic",
            "config": {"workload": workload_desc(name), "batch_per_gpu": B, "global_batch": B * world,
                       "parallelism": f"event-sharded x{world} (table replicated), no exchange",
                       "l2": "uniformly random keys over a 1 GiB table + 256 MiB of slots (> 126 MB L2)", "device": info["name"],
                       "kernel": f"{plan.kernel}, rows gathered from the table by its loader (one launch)" if fused
                       else f"table_lookup_kernel + {plan.kernel}"},
            "p50_step_latency_us": {"batch": 4096, "p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)),
                                    "how": f"CUDA events around one launch ({top}), 300 samples"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_of_nominal_8000": achieved / 8000.0,
                         "traffic": None if fused else measured_traffic(name, B), "kernel": top,
                         "algorithmic_bytes_per_event": bpe, "kernel_ms_per_launch": kms, "peak_source": peak_src},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if emit:
            print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return line if rank == 0 else None


if __name__ == "__main__":
    main()
