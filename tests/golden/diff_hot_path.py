"""The checker of the CUDA kernels -- oracle/batch.py, the vectorised float64 restatement -- against the REAL reference running
the hot path one event at a time: seeded random metric-shaped workloads (Imputer -> OneHotEncoder -> 1..6 linear models -> mean
vote; 4..24 numeric and 0..6 categorical columns, different seeds, NaN and out-of-vocabulary rates) through the reference's sync
flow, one MockEvent per row; and tree-ensemble routers (regression: mean vote, classification: majority vote; 2..5 models) with
one event carrying the batch.  rtol 1e-12 for regression (the per-event path adds the same float64 terms in a different
association), exact for labels.  The reference's answers are stored in tests/golden/reference_checks.json.xz
(gen_reference_checks.py), so the CPU suite runs `check` against them on any machine.

    python -m tests.golden.diff_hot_path      (live, needs the reference)
"""
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np  # noqa: E402

from mlrun_b200.synthetic import flow3_workload, tree_workload  # noqa: E402
from oracle import batch as obatch  # noqa: E402

VERDICT = "the batched oracle equals the real reference"


def workloads():
    """the 64 seeded workloads, in order: ("flow3", case, workload) x 40, then ("trees", case, workload) x 24"""
    rnd = random.Random(31)
    for case in range(40):
        n_models = rnd.choice([1, 1, 2, 4, 6])
        yield "flow3", case, flow3_workload(n_rows=rnd.randint(20, 60), n_num=rnd.randint(4, 24), n_cat=rnd.randint(0, 6), seed=100 + case,
                                            n_models=n_models)
    for case in range(24):
        kind = rnd.choice(["regression", "classification"])
        yield "trees", case, tree_workload(n_rows=rnd.randint(16, 80), n_feat=rnd.randint(4, 24), n_models=rnd.randint(2, 5),
                                           n_trees=rnd.randint(3, 12), depth=rnd.randint(2, 5), seed=200 + case, kind=kind, n_fit=400)


def reference_outputs():
    """the reference's answer to every workload: one output per event (flow3), the router's outputs for the batch (trees)"""
    from tests.golden import api_reference as ref

    res = []
    for what, _case, wl in workloads():
        if what == "flow3":
            server = wl.build_server(ref, engine="sync")
            path = "/" if wl.n_models == 1 else "/v2/models/infer"
            got = []
            for row in wl.rows_as_dicts():
                out = server.test(path=path, body=row)["outputs"]
                got.append(float(out[0] if isinstance(out, list) else out))
            res.append(got)
        else:
            server = wl.build_server(ref)
            out = server.test("/v2/models/infer", body={"inputs": wl.X.astype(np.float64).tolist()})["outputs"]
            res.append(np.asarray(out).tolist())
    return res


def check(reference):
    """the oracle against `reference` (what reference_outputs returned)"""
    n_events = 0
    for (what, case, wl), got in zip(workloads(), reference, strict=True):
        if what == "flow3":
            want = obatch.flow3(wl)["out"]
            np.testing.assert_allclose(np.asarray(got, dtype=np.float64), want, rtol=1e-12, atol=1e-12, err_msg=f"flow3 case {case}")
        else:
            want = obatch.tree_ensemble(wl)["out"]
            if wl.kind == "regression":
                np.testing.assert_allclose(np.asarray(got, dtype=np.float64), want, rtol=1e-12, atol=1e-12, err_msg=f"trees case {case}")
            else:
                assert list(got) == want.tolist(), f"trees case {case}: labels differ"
        n_events += len(got)
    print(f"{VERDICT}'s per-event path on", n_events, "events of 64 random workloads")
    return 0


def main():
    return check(reference_outputs())


if __name__ == "__main__":
    sys.exit(main())
