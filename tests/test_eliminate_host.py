"""DistFeatureEliminator host logic on the test-double engine, pinned against the UNMODIFIED
reference class (joblib branch, ref eliminate.py:163-184) through the scores it computed,
stored in tests/golden/reference_pins.npz."""
import os

import numpy as np
import pytest
from sklearn.linear_model import LogisticRegression

from skdist.distribute.eliminate import DistFeatureEliminator
from skdist_b200.datasets import make_g1_classification

# (step, cv, min_features_to_select) of the reference pin
ELIMINATOR_CASES = ((2, 3, 7), (3, 4, 3))


def _data():
    X, y = make_g1_classification(600, 10, seed=13)
    rng = np.random.default_rng(0)
    X = np.hstack([X, rng.standard_normal((600, 4)).astype(np.float32)])     # 4 pure-noise features
    return X, y


def feature_sets(X, y, step, min_keep):
    """The feature sets dropped in turn, built as eliminate.py:131-154 builds them."""
    d = X.shape[1]
    coefs = LogisticRegression(C=0.3).fit(X, y).coef_
    ranks = np.ravel(np.argsort((coefs ** 2).sum(axis=0)))[: d - min_keep]
    sets, k = [np.array([])], 0
    while k < d - min_keep:
        k += step
        sets.append(ranks[:k])
    return sets


@pytest.mark.filterwarnings("ignore")
def test_eliminator_matches_reference_task_function(fake_engine):
    """The reference class itself cannot run under scikit-learn 1.9 (`check_cv` is called with three
    positional arguments, eliminate.py:125), so the pin is on what every task executes: the
    UNMODIFIED `_fit_and_score_one` / `_drop_col` (eliminate.py:22-38) for each (feature set, fold),
    with the feature sets built as eliminate.py:131-154 builds them."""
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_pins.npz"))
    X, y = _data()
    d = X.shape[1]
    for i, (step, n_cv, min_keep) in enumerate(ELIMINATOR_CASES):
        base = LogisticRegression(C=0.3)
        ours = DistFeatureEliminator(base, None, step=step, cv=n_cv, min_features_to_select=min_keep).fit(X, y)
        sets = feature_sets(X, y, step, min_keep)
        ref_scores = gold["eliminator_scores_%d" % i]
        assert len(ref_scores) == len(sets)
        np.testing.assert_allclose(ours.scores_, ref_scores, atol=1e-12)
        best = int(np.argmax(ref_scores))
        exp_keep = np.delete(range(d), sets[best].astype(int)) if len(sets[best]) else np.arange(d)
        assert list(ours.best_features_) == list(exp_keep)
        ref_final = LogisticRegression(C=0.3).fit(X[:, exp_keep], y)
        np.testing.assert_allclose(ours.best_estimator_.coef_, ref_final.coef_, atol=1e-5)
        np.testing.assert_array_equal(ours.predict(X), ref_final.predict(X[:, exp_keep]))
    assert not hasattr(ours, "sc")


@pytest.mark.filterwarnings("ignore")
def test_eliminator_restatement_and_errors(fake_engine):
    """Same algorithm written out with scikit-learn on the CPU (runs everywhere)."""
    from sklearn.model_selection import StratifiedKFold
    X, y = _data()
    fe = DistFeatureEliminator(LogisticRegression(), None, step=3, cv=3, min_features_to_select=4).fit(X, y)
    d = X.shape[1]
    ranks = np.argsort(LogisticRegression().fit(X, y).coef_[0].astype(np.float64) ** 2)[: d - 4]
    sets, k = [np.array([], int)], 0
    while k < d - 4:
        k += 3
        sets.append(ranks[:k])
    exp = []
    for rm in sets:
        keep = np.setdiff1d(np.arange(d), rm)
        exp.append(np.mean([LogisticRegression().fit(X[tr][:, keep], y[tr]).score(X[te][:, keep], y[te])
                            for tr, te in StratifiedKFold(3).split(X, y)]))
    np.testing.assert_allclose(fe.scores_, exp, atol=1e-12)
    assert fe.n_features_ == d - len(sets[int(np.argmax(exp))])
    assert fe.predict_proba(X[:4]).shape == (4, 2) and 0.5 < fe.score(X, y) <= 1.0
    with pytest.raises(ValueError):
        DistFeatureEliminator(LogisticRegression(), step=0).fit(X, y)
    from sklearn.svm import LinearSVC
    with pytest.raises(NotImplementedError):
        DistFeatureEliminator(LinearSVC()).fit(X, y)


@pytest.mark.filterwarnings("ignore")
def test_eliminator_roc_auc(fake_engine):
    """scoring="roc_auc" as in the reference's examples/eliminate/basic_usage.py."""
    from sklearn.metrics import roc_auc_score
    from sklearn.model_selection import StratifiedKFold
    X, y = _data()
    fe = DistFeatureEliminator(LogisticRegression(), None, step=4, cv=3, min_features_to_select=4,
                               scoring="roc_auc").fit(X, y)
    d = X.shape[1]
    ranks = np.argsort(LogisticRegression().fit(X, y).coef_[0].astype(np.float64) ** 2)[: d - 4]
    sets, k = [np.array([], int)], 0
    while k < d - 4:
        k += 4
        sets.append(ranks[:k])
    exp = []
    for rm in sets:
        keep = np.setdiff1d(np.arange(d), rm)
        exp.append(np.mean([roc_auc_score(y[te], LogisticRegression().fit(X[tr][:, keep], y[tr])
                                          .decision_function(X[te][:, keep]))
                            for tr, te in StratifiedKFold(3).split(X, y)]))
    np.testing.assert_allclose(fe.scores_, exp, atol=1e-6)


@pytest.mark.filterwarnings("ignore")
def test_eliminator_multiclass(fake_engine):
    """Multiclass target: multinomial fits, ranking by the squared coefficients summed over the class rows
    (ref eliminate.py:153-154), written out with scikit-learn on the CPU."""
    from sklearn.model_selection import StratifiedKFold
    from skdist_b200.datasets import make_multiclass
    X, y = make_multiclass(500, 8, 3, seed=4)
    rng = np.random.default_rng(1)
    X = np.hstack([X, rng.standard_normal((500, 3)).astype(np.float32)])
    d = X.shape[1]
    base = LogisticRegression(C=0.5, max_iter=60)
    fe = DistFeatureEliminator(base, None, step=2, cv=3, min_features_to_select=5).fit(X, y)
    coefs = LogisticRegression(C=0.5, max_iter=60).fit(X, y).coef_.astype(np.float64)
    ranks = np.argsort((coefs ** 2).sum(axis=0))[: d - 5]
    sets, k = [np.array([], int)], 0
    while k < d - 5:
        k += 2
        sets.append(ranks[:k])
    exp = []
    for rm in sets:
        keep = np.setdiff1d(np.arange(d), rm)
        exp.append(np.mean([LogisticRegression(C=0.5, max_iter=60).fit(X[tr][:, keep], y[tr]).score(X[te][:, keep], y[te])
                            for tr, te in StratifiedKFold(3).split(X, y)]))
    np.testing.assert_allclose(fe.scores_, exp, atol=1e-12)
    keep = np.setdiff1d(np.arange(d), sets[int(np.argmax(exp))])
    assert list(fe.best_features_) == list(keep)
    ref = LogisticRegression(C=0.5, max_iter=60).fit(X[:, keep], y)
    assert fe.best_estimator_.coef_.shape == (3, len(keep))
    np.testing.assert_array_equal(fe.best_estimator_.coef_, ref.coef_)
    np.testing.assert_array_equal(fe.predict(X), ref.predict(X[:, keep]))
