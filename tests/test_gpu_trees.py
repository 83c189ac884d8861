"""Round-2 tree path (csrc/b2s_trees3.cuh) vs the CPU oracles, through the C-ABI.  Needs a B200: `-m gpu`.

Scores rtol 1e-5 (+ atol 1e-5, the north_star's bound); labels, votes and status words exact.
Oracles: scikit-learn's own predict() (oracle/batch.py) for sklearn estimators -- at BASELINE configs[2]'s full size from
the committed fixtures tests/golden/trees_cfg3_*.pkl.xz -- and oracle/tree_libs.py for xgboost / LightGBM documents."""

import json
import lzma
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from mlrun_b200 import _native as nat  # noqa: E402
from mlrun_b200 import packing, tree_formats  # noqa: E402
from mlrun_b200.feature_store.steps import Imputer  # noqa: E402
from mlrun_b200.lowering import ColumnProgram  # noqa: E402
from mlrun_b200.synthetic import tree_workload  # noqa: E402
from oracle import batch as obatch  # noqa: E402
from oracle import tree_libs  # noqa: E402
from tests import tree_fixtures as fx  # noqa: E402

RTOL, ATOL = 1e-5, 1e-5
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module", autouse=True)
def _device():
    nat.init(0)
    yield


def names(n):
    return [f"f{i}" for i in range(n)]


def cfg3_models(kind):
    import cloudpickle

    with lzma.open(os.path.join(GOLDEN, f"trees_cfg3_{kind}.pkl.xz"), "rb") as fp:
        return cloudpickle.load(fp)


# ------------------------------------------------------------------------------------------ configs[2] at its size
def test_config3_regression_at_size():
    """16 384 x 128 float32, VotingEnsemble(mean) of 4 x GradientBoostingRegressor(100 trees, depth 6) fit on 20 000 rows"""
    models = cfg3_models("reg")
    X = np.random.default_rng(3).normal(size=(16384, 128)).astype(np.float32)
    packed = [packing.pack_model(m) for m in models]
    plan = ColumnProgram(names(128)).build_plan(packed, vote=(nat.VOTE_MEAN, [0.25] * 4))
    assert "trees3_kernel<D=6" in plan.kernel and "4 parts" in plan.kernel, plan.kernel
    out, status = plan.run(X, with_status=True)
    per = np.stack([m.predict(X.astype(np.float64)) for m in models], axis=1)
    np.testing.assert_allclose(out[:, 0], obatch.mean_vote(per, [0.25] * 4), rtol=RTOL, atol=ATOL)
    assert not status.any()
    np.testing.assert_allclose(ColumnProgram(names(128)).build_plan(packed).run(X), per, rtol=RTOL, atol=ATOL)


def test_config3_classification_at_size_is_exact():
    """the 3-class variant: 4 x GradientBoostingClassifier = 4 x 300 trees -> 12 parts (one per model and class), majority vote"""
    models = cfg3_models("cls")
    X = np.random.default_rng(4).normal(size=(16384, 128)).astype(np.float32)
    packed = [packing.pack_model(m) for m in models]
    plan = ColumnProgram(names(128)).build_plan(packed, vote=(nat.VOTE_MAJORITY, [0.25] * 4))
    assert "trees3_kernel<D=6" in plan.kernel and "12 parts" in plan.kernel, plan.kernel
    out = plan.run(X)
    per = np.stack([m.predict(X.astype(np.float64)) for m in models], axis=1)
    labels = ColumnProgram(names(128)).build_plan(packed).run(X)
    # a label may only differ where the two best class scores tie to ~1e-12 (summation order); none do on this workload
    assert np.array_equal(labels, per)
    assert np.array_equal(out[:, 0], obatch.majority_vote(per, [0.25] * 4))


# ------------------------------------------------------------------------------------------ shapes the loader must cover
@pytest.mark.parametrize("n_feat,n_rows", [(128, 1), (128, 63), (128, 65), (32, 4097), (20, 777), (6, 130), (33, 64)])
def test_row_and_feature_shapes(n_feat, n_rows):
    """TMA boxes (features a multiple of 32), cp.async 16 B (a multiple of 4) and 4 B loaders; ragged last tiles"""
    wl = tree_workload(n_rows=n_rows, n_feat=n_feat, n_models=3, n_trees=9, depth=4, seed=n_feat + n_rows, n_fit=600)
    packed = [packing.pack_model(m) for m in wl.models]
    plan = ColumnProgram(names(n_feat)).build_plan(packed, vote=(nat.VOTE_MEAN, [1 / 3] * 3))
    assert "trees3_kernel" in plan.kernel
    out, status = plan.run(wl.X, with_status=True)
    np.testing.assert_allclose(out[:, 0], obatch.tree_ensemble(wl)["out"], rtol=RTOL, atol=ATOL)
    assert not status.any()


@pytest.mark.parametrize("depth,n_trees", [(1, 30), (2, 30), (3, 25), (7, 12), (8, 6)])
def test_depths(depth, n_trees):
    wl = tree_workload(n_rows=1500, n_feat=16, n_models=2, n_trees=n_trees, depth=depth, seed=40 + depth, n_fit=3000)
    packed = [packing.pack_model(m) for m in wl.models]
    plan = ColumnProgram(names(16)).build_plan(packed)
    assert f"trees3_kernel<D={max(depth, 2)}" in plan.kernel, plan.kernel
    np.testing.assert_allclose(plan.run(wl.X), obatch.tree_ensemble(wl)["per_model"], rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("depth,routes_nan", [(3, False), (6, False), (5, True)])
def test_walk_levels_match_the_oracle(depth, routes_nan):
    """the top two levels of every tree are read with warp-uniform loads, the rest node by node: both against predict(),
    with and without NaN routing"""
    if routes_nan:
        from sklearn.ensemble import RandomForestRegressor

        rng = np.random.default_rng(70)
        Xf = rng.normal(size=(3000, 16)).astype(np.float32)
        Xf[rng.random(Xf.shape) < 0.1] = np.nan
        yf = np.nan_to_num(Xf[:, 0]) * 2 + np.nan_to_num(Xf[:, 3]) + rng.normal(size=3000) * 0.1
        models = [RandomForestRegressor(n_estimators=20, max_depth=depth, random_state=i).fit(Xf, yf) for i in range(2)]
        X = rng.normal(size=(1500, 16)).astype(np.float32)
        X[rng.random(X.shape) < 0.1] = np.nan
    else:
        wl = tree_workload(n_rows=1500, n_feat=16, n_models=2, n_trees=20, depth=depth, seed=60 + depth, n_fit=3000)
        models, X = wl.models, wl.X
    plan = ColumnProgram(names(16)).build_plan([packing.pack_model(m) for m in models])
    assert f"trees3_kernel<D={depth},{'NaN routing' if routes_nan else 'floats'}>" in plan.kernel, plan.kernel
    np.testing.assert_allclose(plan.run(X), np.stack([m.predict(X.astype(np.float64)) for m in models], axis=1), rtol=RTOL, atol=ATOL)


def test_rows_too_wide_for_the_parts_kernel_take_the_generic_tree_kernel():
    """432 columns: two transposed 64-row tiles fill a CTA's shared memory, so no part fits next to them and the plan runs on
    the generic rows_kernel<TREES>"""
    wl = tree_workload(n_rows=3000, n_feat=432, n_models=4, n_trees=10, depth=2, seed=12, n_fit=600)
    packed = [packing.pack_model(m) for m in wl.models]
    ref = obatch.tree_ensemble(wl)
    plan = ColumnProgram(names(432)).build_plan(packed, vote=(nat.VOTE_MEAN, [0.25] * 4))
    assert plan.kernel.startswith("rows_kernel<TREES"), plan.kernel
    out, status = plan.run(wl.X, with_status=True)
    np.testing.assert_allclose(out[:, 0], ref["out"], rtol=RTOL, atol=ATOL)
    assert not status.any()
    np.testing.assert_allclose(ColumnProgram(names(432)).build_plan(packed).run(wl.X), ref["per_model"], rtol=RTOL, atol=ATOL)


def test_a_model_larger_than_one_cta_is_split_into_parts():
    """600 depth-6 trees do not fit one CTA's shared memory: the model becomes several parts whose partial sums are added
    in a fixed order"""
    from sklearn.ensemble import RandomForestRegressor

    rng = np.random.default_rng(7)
    Xf = rng.normal(size=(3000, 16)).astype(np.float32)
    y = 2 * Xf[:, 0] + np.sin(Xf[:, 1]) + Xf[:, 2] * Xf[:, 3]
    model = RandomForestRegressor(n_estimators=600, max_depth=6, random_state=0, n_jobs=4).fit(Xf, y)
    X = rng.normal(size=(5000, 16)).astype(np.float32)
    plan = ColumnProgram(names(16)).build_plan([packing.pack_model(model)])
    assert "trees3_kernel<D=6" in plan.kernel and "1 parts" not in plan.kernel, plan.kernel
    np.testing.assert_allclose(plan.run(X)[:, 0], model.predict(X.astype(np.float64)), rtol=RTOL, atol=ATOL)
    again = plan.run(X)
    np.testing.assert_array_equal(plan.run(X), again)  # deterministic


def test_mixed_linear_and_tree_ensemble():
    """BASELINE configs[3]'s router: linear and tree scorers behind one VotingEnsemble, one launch"""
    from sklearn.ensemble import GradientBoostingRegressor
    from sklearn.linear_model import LinearRegression, Ridge

    rng = np.random.default_rng(8)
    Xf = rng.normal(size=(4000, 64)).astype(np.float32)
    y = 2 * Xf[:, 0] + np.sin(Xf[:, 1]) + Xf[:, 2] * Xf[:, 3] + 0.1 * rng.normal(size=4000)
    models = []
    for i in range(8):
        if i % 2 == 0:
            models.append(GradientBoostingRegressor(n_estimators=30, max_depth=6, random_state=i, subsample=0.5).fit(Xf, y))
        else:
            models.append((Ridge(alpha=i) if i % 4 == 1 else LinearRegression()).fit(Xf + 0.01 * i, y))
    X = rng.normal(size=(10000, 64)).astype(np.float32)
    X[5, 3] = np.nan
    X[9, 60] = np.inf
    w = list(rng.random(8))
    plan = ColumnProgram(names(64)).build_plan([packing.pack_model(m) for m in models], vote=(nat.VOTE_MEAN, w))
    assert "trees3_kernel" in plan.kernel and "5 parts" in plan.kernel, plan.kernel
    out, status = plan.run(X, with_status=True)
    ok = np.isfinite(X).all(axis=1)
    per = np.stack([m.predict(X[ok].astype(np.float64)) for m in models], axis=1)
    np.testing.assert_allclose(out[ok, 0], obatch.mean_vote(per, w), rtol=RTOL, atol=ATOL)
    assert np.array_equal(status != 0, ~ok)


def test_imputer_in_front_of_a_tree_ensemble():
    wl = tree_workload(n_rows=3000, n_feat=32, n_models=2, n_trees=15, depth=5, seed=9, n_fit=1500)
    X = wl.X.copy()
    X[np.random.default_rng(10).random(X.shape) < 0.05] = np.nan
    prog = ColumnProgram(names(32))
    mapping = {f"f{i}": float(i) / 10 for i in range(0, 32, 2)}  # odd columns are not imputed: their NaN rows are errors
    prog.apply(Imputer(mapping=mapping))
    plan = prog.build_plan([packing.pack_model(m) for m in wl.models])
    assert "trees3_kernel" in plan.kernel
    out, status = plan.run(X, with_status=True)
    Xi = obatch.impute(X, names(32), mapping)
    ok = np.isfinite(Xi).all(axis=1)
    assert np.array_equal(status != 0, ~ok) and ok.any() and (~ok).any()
    want = np.stack([m.predict(Xi[ok]) for m in wl.models], axis=1)
    np.testing.assert_allclose(out[ok], want, rtol=RTOL, atol=ATOL)


# ------------------------------------------------------------------------------------------ missing values / other libraries
def test_sklearn_forests_route_nan_on_the_device():
    from sklearn.ensemble import RandomForestClassifier, RandomForestRegressor
    from sklearn.tree import DecisionTreeRegressor

    rng = np.random.default_rng(51)
    Xf = rng.normal(size=(2000, 12)).astype(np.float32)
    Xn = Xf.copy()
    Xn[rng.random(Xf.shape) < 0.1] = np.nan
    y = Xf[:, 0] * 2 + Xf[:, 1] * Xf[:, 2]
    Xt = fx.grid_inputs(5000, 12, seed=52, with_inf=True)
    ok = ~np.isinf(Xt).any(axis=1)
    for model in (DecisionTreeRegressor(max_depth=6, random_state=0).fit(Xn, y),
                  RandomForestRegressor(n_estimators=20, max_depth=6, random_state=0).fit(Xn, y),
                  RandomForestClassifier(n_estimators=15, max_depth=5, random_state=0).fit(Xn, (y > 0).astype(int) + (y > 1))):
        plan = ColumnProgram(names(12)).build_plan([packing.pack_model(model)])
        assert "NaN routing" in plan.kernel, plan.kernel
        out, status = plan.run(Xt, with_status=True)
        assert np.array_equal(status != 0, ~ok)  # NaN is data for these estimators, Inf is not
        np.testing.assert_allclose(out[ok, 0], model.predict(Xt[ok].astype(np.float64)), rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("objective,num_class", [("reg:squarederror", 0), ("binary:logistic", 0), ("multi:softprob", 3)])
def test_xgboost_documents_on_the_device(objective, num_class):
    doc = fx.random_xgb_model(n_trees=25, depth=6, n_feat=24, seed=61, objective=objective, num_class=num_class, base_score=0.4)
    X = fx.grid_inputs(3000, 24, seed=62)
    plan = ColumnProgram(names(24)).build_plan([("trees", tree_formats.pack_xgboost_json(json.dumps(doc)))])
    assert "NaN routing" in plan.kernel, plan.kernel
    out, status = plan.run(X, with_status=True)
    want = tree_libs.xgboost_predict(doc, X[:600])
    assert not status.any()
    if objective == "reg:squarederror":
        np.testing.assert_allclose(out[:600, 0], want, rtol=RTOL, atol=ATOL)
    else:
        assert np.array_equal(out[:600, 0], want)
    # the whole batch against the numpy emulation of the same packed model (the oracle above is a per-row Python loop)
    from tests import device_emulator as emu

    full = emu.trees_predict(tree_formats.pack_xgboost_json(doc), X)
    if objective == "reg:squarederror":
        np.testing.assert_allclose(out[:, 0], full, rtol=RTOL, atol=ATOL)
    else:
        assert np.array_equal(out[:, 0], full)


def test_lightgbm_documents_on_the_device():
    dump = fx.random_lgbm_dump(n_trees=20, depth=6, n_feat=16, seed=71)
    X = fx.grid_inputs(800, 16, seed=72)
    plan = ColumnProgram(names(16)).build_plan([("trees", tree_formats.pack_lightgbm_dump(dump))])
    out, status = plan.run(X, with_status=True)
    np.testing.assert_allclose(out[:, 0], tree_libs.lightgbm_predict(dump, X), rtol=RTOL, atol=ATOL)
    assert not status.any()


def test_xgboost_ensemble_served_through_the_router():
    """VotingEnsemble over XGBoostModelServer routes (frameworks/xgboost/__init__.py:30), models given as save_model documents"""
    from mlrun_b200 import api

    docs = [fx.random_xgb_model(n_trees=10, depth=5, n_feat=10, seed=80 + i) for i in range(4)]
    fn = api.new_function("xgb", kind="serving")
    graph = fn.set_topology("router", api.VotingEnsemble(vote_type="regression"))
    for i, d in enumerate(docs):
        graph.add_route(f"m{i + 1}", class_name="XGBoostModelServer", model=d, model_path="")
    server = fn.to_mock_server(namespace={"XGBoostModelServer": api.XGBoostModelServer})
    X = fx.grid_inputs(512, 10, seed=90)
    out, status = server.run_batch(X, with_status=True)
    want = np.mean([tree_libs.xgboost_predict(d, X) for d in docs], axis=0)
    np.testing.assert_allclose(out[:, 0], want, rtol=RTOL, atol=ATOL)
    assert not status.any()
    one = server.test(path="/v2/models/infer", body={"inputs": np.nan_to_num(X[:3]).astype(np.float64).tolist()})
    np.testing.assert_allclose(one["outputs"], np.mean([tree_libs.xgboost_predict(d, np.nan_to_num(X[:3])) for d in docs], axis=0),
                               rtol=RTOL, atol=ATOL)
