"""Host side of the forest path (no GPU): the random numbers drawn per tree and the wrapping of
node arrays into scikit-learn trees; plus the pin that the reference's own `_build_trees`
yields scikit-learn's trees (so sklearn's RandomForestClassifier is a valid oracle), on the trees
it built as stored in tests/golden/reference_pins.npz."""
import os

import numpy as np
import pytest
from sklearn.ensemble import RandomForestClassifier

from skdist_b200.distribute.ensemble import MAX_RAND_SEED, _make_sklearn_tree, _tree_inputs

PINS = os.path.join(os.path.dirname(__file__), "golden", "reference_pins.npz")


def lattice(n, d, seed, levels=16):
    rng = np.random.default_rng(seed)
    X = rng.integers(0, levels, size=(n, d)).astype(np.float32)
    y = ((X[:, 0] + X[:, 1] * 0.5 + rng.standard_normal(n) * 3) > levels * 0.75).astype(np.int64)
    return X, y


def test_tree_inputs_match_sklearn_sample_weights():
    X, y = lattice(500, 5, 1)
    rf = RandomForestClassifier(n_estimators=3, random_state=7).fit(X, y)
    states = np.random.RandomState(7).randint(MAX_RAND_SEED, size=3)
    for s, t in zip(states, rf.estimators_):
        assert t.random_state == s
        counts, rstate = _tree_inputs(s, 500, True)
        # weighted_n_node_samples of the root = n; number of distinct rows = n_node_samples of the root
        assert counts.sum() == 500 and (counts > 0).sum() == t.tree_.n_node_samples[0]


def test_wrapping_roundtrip():
    X, y = lattice(800, 6, 2)
    rf = RandomForestClassifier(n_estimators=2, random_state=3).fit(X, y)
    t = rf.estimators_[0].tree_
    arrays = {"left": t.children_left.astype(np.int32), "right": t.children_right.astype(np.int32),
              "feature": t.feature.astype(np.int32), "threshold": t.threshold.copy(), "impurity": t.impurity.copy(),
              "n_node_samples": t.n_node_samples.astype(np.int32),
              "weighted_n_node_samples": t.weighted_n_node_samples.copy(),
              "missing_go_to_left": np.zeros(t.node_count, np.uint8), "value": t.value[:, 0, :].copy(),
              "max_depth": t.max_depth}
    est = _make_sklearn_tree({"max_features": "sqrt"}, 11, arrays, 6, 2, 2)
    np.testing.assert_array_equal(est.predict_proba(X), rf.estimators_[0].predict_proba(X))
    np.testing.assert_array_equal(est.apply(X), rf.estimators_[0].apply(X))


def test_reference_build_trees_equals_sklearn():
    gold = np.load(PINS)
    X, y = lattice(1500, 8, 3)
    ref = RandomForestClassifier(n_estimators=3, random_state=5).fit(X, y)
    for i, t in enumerate(ref.estimators_):
        np.testing.assert_array_equal(gold["build_trees_threshold_%d" % i], t.tree_.threshold)
        np.testing.assert_array_equal(gold["build_trees_children_left_%d" % i], t.tree_.children_left)


def test_native_bootstrap_counts_equal_numpy():
    """csrc/bootstrap.cu (host threads, no GPU) vs the numpy form of the reference's per-tree draw
    (ref ensemble.py:51-55; `_tree_inputs`): bit-identical counts and splitter seeds, edge sizes included."""
    from skdist_b200.bootstrap import bootstrap_counts
    from skdist_b200.distribute.ensemble import _tree_inputs
    rng = np.random.RandomState(3)
    for n in (1, 2, 5, 255, 4097, 65536, 65537, 300_000):
        seeds = list(rng.randint(np.iinfo(np.int32).max, size=5)) + [0, 1, 2 ** 31 - 2]
        counts, rand_r = bootstrap_counts(seeds, n, n_threads=3)
        for i, s in enumerate(seeds):
            cw, rw = _tree_inputs(s, n, True)
            np.testing.assert_array_equal(counts[i], cw)
            assert rand_r[i] == rw
        c0, r0 = bootstrap_counts(seeds, n, bootstrap=False)
        assert c0 is None
        np.testing.assert_array_equal(r0, rand_r)


@pytest.mark.filterwarnings("ignore")
@pytest.mark.parametrize("kind", ["rf", "et", "rfr"])
def test_forest_fit_pipeline_on_engine_double(fake_engine, kind, monkeypatch):
    """The whole host pipeline of the forest fit (seed draw, chunked bootstrap counts from the native
    helper, wrapping into scikit-learn trees) on an engine double whose trees are scikit-learn's own:
    the fitted forest must equal scikit-learn's forest tree for tree."""
    from sklearn.ensemble import ExtraTreesClassifier, RandomForestClassifier, RandomForestRegressor
    from sklearn.utils import check_random_state
    from skdist.distribute.ensemble import (DistExtraTreesClassifier, DistRandomForestClassifier,
                                            DistRandomForestRegressor)
    from skdist_b200.distribute.ensemble import MAX_RAND_SEED, _tree_inputs
    from skdist_b200.datasets import make_multiclass
    monkeypatch.setenv("SKDIST_B200_FOREST_CHUNK", "3")          # several chunks -> the pipelined path
    X, y = make_multiclass(400, 6, 3, seed=2)
    Xq = np.round(X * 8).astype(np.float32)
    n_trees, rs = 7, 11
    states = check_random_state(rs).randint(MAX_RAND_SEED, size=n_trees)
    from skdist_b200.engine import get_engine
    get_engine().seed_of_rand_r = {int(_tree_inputs(s, len(y), False)[1]): int(s) for s in states}
    if kind == "rf":
        ours = DistRandomForestClassifier(n_estimators=n_trees, random_state=rs).fit(Xq, y)
        ref = RandomForestClassifier(n_estimators=n_trees, random_state=rs).fit(Xq, y)
    elif kind == "et":
        ours = DistExtraTreesClassifier(n_estimators=n_trees, random_state=rs).fit(Xq, y)
        ref = ExtraTreesClassifier(n_estimators=n_trees, random_state=rs).fit(Xq, y)
    else:
        yr = (Xq[:, 0] * 2 + Xq[:, 1]).astype(np.float64)
        ours = DistRandomForestRegressor(n_estimators=n_trees, random_state=rs).fit(Xq, yr)
        ref = RandomForestRegressor(n_estimators=n_trees, random_state=rs).fit(Xq, yr)
    assert len(ours.estimators_) == n_trees
    for a, b in zip(ours.estimators_, ref.estimators_):
        np.testing.assert_array_equal(a.tree_.threshold, b.tree_.threshold)
        np.testing.assert_array_equal(a.tree_.children_left, b.tree_.children_left)
        np.testing.assert_array_equal(a.tree_.value, b.tree_.value)
    np.testing.assert_array_equal(ours.predict(Xq), ref.predict(Xq))


def test_warm_start_adds_the_trees_a_cold_fit_would_have(fake_engine):
    """ref ensemble.py:250-272: with warm_start the fitted trees are kept, the random state is drawn
    past their seeds and only the additional trees are built -- the forest equals a cold fit with the
    larger n_estimators (and scikit-learn's warm-started RandomForestClassifier)."""
    from sklearn.ensemble import RandomForestClassifier
    from skdist.distribute.ensemble import DistRandomForestClassifier
    rng = np.random.default_rng(3)
    X = rng.integers(0, 16, size=(400, 6)).astype(np.float32)
    y = (X[:, 0] + X[:, 1] > 14).astype(int)
    from sklearn.utils import check_random_state
    from skdist.distribute.ensemble import MAX_RAND_SEED, _tree_inputs
    from skdist_b200.engine import get_engine
    states = check_random_state(9).randint(MAX_RAND_SEED, size=7)
    get_engine().seed_of_rand_r = {int(_tree_inputs(s, len(y), False)[1]): int(s) for s in states}
    warm = DistRandomForestClassifier(n_estimators=3, random_state=9, warm_start=True).fit(X, y)
    warm.sc = None
    warm.set_params(n_estimators=7)
    warm.fit(X, y)
    cold = DistRandomForestClassifier(n_estimators=7, random_state=9).fit(X, y)
    ref = RandomForestClassifier(n_estimators=7, random_state=9).fit(X, y)
    assert len(warm.estimators_) == 7
    for a, b, c in zip(warm.estimators_, cold.estimators_, ref.estimators_):
        np.testing.assert_array_equal(a.tree_.threshold, b.tree_.threshold)
        np.testing.assert_array_equal(a.tree_.threshold, c.tree_.threshold)
        np.testing.assert_array_equal(a.tree_.value, c.tree_.value)
    with pytest.raises(ValueError):
        warm.set_params(n_estimators=5)
        warm.fit(X, y)


@pytest.mark.parametrize("kind", ["rf", "et"])
def test_histogram_mode_for_continuous_features(fake_engine, monkeypatch, kind):
    """SKDIST_B200_FOREST_MAX_BINS: features with more distinct values than the bins are replaced by equal-count
    bin codes; the fitted trees are scikit-learn's trees on the coded matrix with the thresholds moved back to
    raw units, so they route raw rows exactly as the coded trees route coded rows -- training rows and new
    rows alike (a new row's code is found with the same edges)."""
    from sklearn.ensemble import ExtraTreesClassifier, RandomForestClassifier
    from sklearn.utils import check_random_state
    from skdist.distribute.ensemble import DistExtraTreesClassifier, DistRandomForestClassifier
    from skdist_b200.distribute.ensemble import MAX_RAND_SEED, _quantile_codes, _tree_inputs
    from skdist_b200.engine import get_engine
    rng = np.random.default_rng(5)
    n, d, bins = 900, 5, 16
    X = rng.standard_normal((n, d)).astype(np.float32)
    X[:, 3] = rng.integers(0, 6, n)                      # a low-cardinality feature stays as it is
    X[::7, 1] = X[0, 1]                                  # heavy ties inside a continuous feature
    y = ((X[:, 0] + 0.5 * X[:, 1] * X[:, 2] + 0.3 * X[:, 3]) > 0.4).astype(int)
    Xc, table = _quantile_codes(X, bins)
    assert np.isnan(table[3]).all() and not np.isnan(table[0, 0])
    assert np.array_equal(Xc[:, 3], X[:, 3]) and Xc[:, 0].max() <= bins - 1
    for f in (0, 1, 2, 4):                               # the raw thresholds reproduce the coding: x <= thr[c]  <=>  code <= c
        nb = int(Xc[:, f].max())
        for c in range(nb):
            assert np.array_equal(X[:, f] <= table[f, c], Xc[:, f] <= c)
    n_trees, rs = 5, 3
    states = check_random_state(rs).randint(MAX_RAND_SEED, size=n_trees)
    get_engine().seed_of_rand_r = {int(_tree_inputs(s, n, False)[1]): int(s) for s in states}
    monkeypatch.setenv("SKDIST_B200_FOREST_MAX_BINS", str(bins))
    if kind == "rf":
        ours = DistRandomForestClassifier(n_estimators=n_trees, random_state=rs).fit(X, y)
        ref = RandomForestClassifier(n_estimators=n_trees, random_state=rs).fit(Xc, y)
    else:
        ours = DistExtraTreesClassifier(n_estimators=n_trees, random_state=rs).fit(X, y)
        ref = ExtraTreesClassifier(n_estimators=n_trees, random_state=rs).fit(Xc, y)
    for a, b in zip(ours.estimators_, ref.estimators_):
        np.testing.assert_array_equal(a.tree_.feature, b.tree_.feature)
        np.testing.assert_array_equal(a.tree_.children_left, b.tree_.children_left)
        np.testing.assert_array_equal(a.tree_.value, b.tree_.value)
        on3 = a.tree_.feature == 3
        np.testing.assert_array_equal(a.tree_.threshold[on3], b.tree_.threshold[on3])
    np.testing.assert_array_equal(ours.predict_proba(X), ref.predict_proba(Xc))
    # new rows: coded with the training edges (searchsorted on the raw thresholds), same routing
    Xn = rng.standard_normal((300, d)).astype(np.float32)
    Xn[:, 3] = rng.integers(0, 6, 300)
    Xnc = Xn.copy()
    for f in (0, 1, 2, 4):
        thr = table[f][~np.isnan(table[f])]
        Xnc[:, f] = np.searchsorted(thr, Xn[:, f].astype(np.float64), side="left")
    np.testing.assert_array_equal(ours.predict_proba(Xn), ref.predict_proba(Xnc))
    assert ours.score(X, y) > 0.9


def test_remap_thresholds_on_node_records():
    """The library hands back scikit-learn node records (one structured array): the remap writes through the
    field views and leaves leaves / uncoded features alone."""
    from sklearn.tree._tree import NODE_DTYPE
    from skdist_b200.distribute.ensemble import _remap_thresholds
    nodes = np.zeros(6, dtype=NODE_DTYPE)
    nodes["feature"] = [0, 2, -2, 0, 1, -2]
    nodes["threshold"] = [1.5, 3.0, -2.0, 0.25, 7.5, -2.0]
    table = np.full((3, 8), np.nan)
    table[0, :4] = [-0.7, -0.1, 0.4, 1.9]
    table[2, :5] = [10.0, 20.0, 30.0, 40.0, 50.0]
    out = _remap_thresholds({"nodes": nodes, "left": nodes["left_child"]}, table)
    np.testing.assert_array_equal(out["nodes"]["threshold"], [-0.1, 40.0, -2.0, -0.7, 7.5, -2.0])


def test_random_trees_embedding_matches_sklearn_and_the_reference_test(fake_engine):
    """DistRandomTreesEmbedding (ref ensemble.py:619-708): the reference's own test case
    (skdist/distribute/tests/test_ensemble.py:61-66: shape (3, 30)) and scikit-learn's RandomTreesEmbedding with the
    same random_state on a larger lattice, leaf for leaf."""
    from sklearn.base import clone
    from sklearn.ensemble import RandomTreesEmbedding
    from sklearn.utils import check_random_state
    from skdist.distribute.ensemble import DistRandomTreesEmbedding
    from skdist_b200.engine import get_engine

    def seeds(rs, n_trees, n):
        st = check_random_state(rs).randint(MAX_RAND_SEED, size=n_trees)
        get_engine().seed_of_rand_r = {int(_tree_inputs(s, n, False)[1]): int(s) for s in st}

    X = np.array([[0, 1, 0, 1], [0, 0, 0, 1], [1, 0, 1, 0]])
    seeds(5, 10, 3)
    rte = DistRandomTreesEmbedding(n_estimators=10, random_state=5)
    rte.fit(X, y=None)
    assert rte.transform(X).shape == (3, 30)
    Xl, _ = lattice(600, 7, 4)
    seeds(11, 6, 600)
    ours = DistRandomTreesEmbedding(None, "auto", 6, max_depth=4, random_state=11)
    got = ours.fit_transform(Xl)
    ref = RandomTreesEmbedding(n_estimators=6, max_depth=4, random_state=11)
    want = ref.fit_transform(Xl)
    assert got.shape == want.shape and (got != want).nnz == 0
    assert (ours.transform(Xl[:50]) != ref.transform(Xl[:50])).nnz == 0
    assert clone(ours).get_params()["max_depth"] == 4 and not hasattr(ours, "sc")


def test_out_of_fold_helpers():
    """get_oof / get_single_oof (ref ensemble.py:112-151) against the reference's own functions."""
    from sklearn.linear_model import LogisticRegression
    from skdist.distribute.ensemble import get_oof, get_single_oof
    X, y = lattice(300, 4, 6)
    clf, oof = get_oof(LogisticRegression(), X, y, n_splits=3)
    assert oof.shape == (300, 2) and np.allclose(oof.sum(1), 1.0) and hasattr(clf, "coef_")
    idx, p = get_single_oof(LogisticRegression(), X, y, np.arange(100, 300), np.arange(100))
    np.testing.assert_allclose(p, oof[:100], rtol=1e-12)
    np.testing.assert_array_equal(oof, np.load(PINS)["get_oof"])
