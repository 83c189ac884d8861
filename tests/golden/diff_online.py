"""The checker of the enrichment path -- oracle/enrichment.py's OnlineVectorService restatement -- against the REAL
OnlineVectorService (feature_store/feature_vector.py:903-1067; the online-store read is the same dict stub under both, as in
the `online_service_logic` scenario): random tables (floats, ints, nan, +-inf, None, missing features, all-zero rows), random
impute policies ("*" and per-feature constants and $mean / $min / $max / $std / $count statistics, unknown and label features),
with and without label column / index columns, single and composite keys; lookups as lists, dicts, a single dict, unknown keys,
extra columns, malformed asks.  Results, impute tables and exceptions compared.  The reference's answers are stored in
tests/golden/reference_checks.json.xz (gen_reference_checks.py), so the CPU suite runs `check` against them on any machine.

    python -m tests.golden.diff_online      (live, needs the reference)
"""
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import pandas as pd  # noqa: E402

from tests import api_oracle as ora  # noqa: E402
from tests.scenarios import _first_line  # noqa: E402

VERDICT = "identical on 500 random online services"


def norm(v):
    if isinstance(v, float) and v != v:
        return "nan"
    if isinstance(v, float) and v in (float("inf"), float("-inf")):
        return repr(v)
    if isinstance(v, dict):
        return {k: norm(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [norm(x) for x in v]
    return v.item() if hasattr(v, "item") else v


def attempt(fn):
    try:
        return norm(fn())
    except Exception as exc:  # noqa: BLE001
        return {"raised": type(exc).__name__, "message": _first_line(str(exc))}


def services():
    """the 500 seeded cases: (feats, index, table, stats, label, with_idx, policy, composite, asks)"""
    rnd = random.Random(23)
    for _case in range(500):
        nf = rnd.randint(1, 6)
        feats = [f"f{i}" for i in range(nf)]
        label = rnd.choice([None, feats[-1]]) if nf > 1 else None
        composite = rnd.random() < 0.2
        index = ["a", "b"] if composite else ["k"]
        val = lambda: rnd.choice([rnd.uniform(-5, 5), rnd.randint(-3, 3), float("nan"), float("inf"), float("-inf"), None, 0.0, 0])  # noqa: E731
        table = {}
        for i in range(rnd.randint(1, 6)):
            key = (f"k{i}", i) if composite else (f"k{i}",)
            row = {f: val() for f in feats if rnd.random() < 0.85}
            if rnd.random() < 0.1:
                row = {f: 0.0 for f in feats}
            table[key] = row
        stats = pd.DataFrame({c: [rnd.uniform(-3, 3) for _ in feats] for c in ("mean", "min", "max", "std", "count")}, index=feats)
        policy = None
        if rnd.random() < 0.75:
            policy = {}
            if rnd.random() < 0.6:
                policy["*"] = rnd.choice(["$mean", "$min", "$max", "$std", "$count", 0, 0.5, -1])
            for f in feats:
                if rnd.random() < 0.3:
                    policy[f] = rnd.choice(["$mean", "$max", 7, -2.5, 0])
            if rnd.random() < 0.08:
                policy["ghost"] = 1
        with_idx = rnd.random() < 0.3
        keys = list(table) + [("nobody", 9) if composite else ("nobody",)]
        asks = [list(rnd.choice(keys)) for _ in range(rnd.randint(1, 4))]
        yield feats, index, table, stats, label, with_idx, policy, composite, asks


def answers(api):
    """repr of everything `api`'s OnlineVectorService answers, per case"""
    out = []
    for feats, index, table, stats, label, with_idx, policy, composite, asks in services():
        def go():
            svc = api.online_service(feats, index, table, stats, label, with_idx, policy)
            res = {"impute": norm(dict(svc._impute_values)),
                   "lists": attempt(lambda: svc.get(asks, as_list=True)),
                   "dicts": attempt(lambda: svc.get([dict(zip(index, a)) for a in asks])),
                   "one": attempt(lambda: svc.get(dict(zip(index, asks[0])))),
                   "extra": attempt(lambda: svc.get([{**dict(zip(index, asks[0])), "note": 1}])),
                   "short": attempt(lambda: svc.get([asks[0][:1]])) if composite else None,
                   "empty": attempt(lambda: svc.get([])), "string": attempt(lambda: svc.get("k0"))}
            return res
        out.append(repr(attempt(go)))
    return out


def reference_answers():
    from tests.golden import api_reference as ref

    return answers(ref)


def check(reference):
    """the oracle against `reference` (what reference_answers returned)"""
    mine = answers(ora)
    assert len(mine) == len(reference)
    for case, (want, got, args) in enumerate(zip(reference, mine, services())):
        if want != got:
            feats, index, table, _stats, label, with_idx, policy, _composite, asks = args
            print("DIFF", case, feats, label, index, table, policy, with_idx, asks)
            print("  ref :", want[:1200])
            print("  mine:", got[:1200])
            return 1
    print(VERDICT)
    return 0


def main():
    return check(reference_answers())


if __name__ == "__main__":
    sys.exit(main())
