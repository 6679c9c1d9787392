"""DistOneVsRestClassifier host logic (no GPU) against scikit-learn's OneVsRestClassifier, which the
reference's DistOneVsRestClassifier equals bit for bit when run unmodified with sc=None
(SURVEY.md section 8c; checked in test_reference_ovr_equals_sklearn on the coefficients the reference
computed, stored in tests/golden/reference_pins.npz)."""
import os
import pickle
import warnings

import numpy as np
import pytest
from sklearn.linear_model import LogisticRegression, SGDClassifier
from sklearn.multiclass import OneVsRestClassifier

from oracle import sgd_oracle
from skdist.distribute.multiclass import DistOneVsRestClassifier
from skdist_b200.datasets import make_multiclass

PINS = os.path.join(os.path.dirname(__file__), "golden", "reference_pins.npz")
# (max_negatives, method, random_state) of the reference's _negatives_mask pin
NEGATIVES_CASES = [(mn, method, rs) for mn, method in [(300, "ratio"), (0.2, "ratio"), (2, "multiplier"),
                                                       (1.5, "multiplier"), (10 ** 6, "ratio")] for rs in (0, 7)]


def negatives_input():
    rng = np.random.default_rng(0)
    n = 5000
    X = np.arange(n, dtype=np.float64)[:, None]
    y = (rng.random(n) < 0.07).astype(int)
    return X, y


def test_ovr_logreg_matches_sklearn(fake_engine):
    X, y = make_multiclass(1200, 10, 5, seed=4)
    ovr = DistOneVsRestClassifier(LogisticRegression(C=0.5), None).fit(X, y)
    ref = OneVsRestClassifier(LogisticRegression(C=0.5)).fit(X, y)
    assert list(ovr.classes_) == list(ref.classes_) and len(ovr.estimators_) == 5
    for a, b in zip(ovr.estimators_, ref.estimators_):
        np.testing.assert_array_equal(a.coef_, b.coef_)
        np.testing.assert_array_equal(a.intercept_, b.intercept_)
        assert a.coef_.dtype == b.coef_.dtype and list(a.classes_) == list(b.classes_)
        assert a.get_params() == b.get_params() and a is not ovr.estimators_[0] or a is ovr.estimators_[0]
    assert len({id(e) for e in ovr.estimators_}) == 5          # independent clones of the template
    np.testing.assert_array_equal(ovr.predict(X), ref.predict(X))
    np.testing.assert_allclose(ovr.predict_proba(X[:20]).sum(1) > 0, True)
    assert not hasattr(ovr, "sc")
    pickle.loads(pickle.dumps(ovr))


def test_reference_toy_case(fake_engine):
    """ref skdist/distribute/tests/test_multiclass.py:23-38 (lbfgs instead of liblinear)."""
    X = np.array([[0, 0, 1, 1], [1, 1, 0, 0], [-1, -1, -1, -1]] * 100)
    y = np.array([0, 1, 2] * 100)
    ovr = DistOneVsRestClassifier(LogisticRegression()).fit(X, y)
    assert np.allclose(ovr.predict(X[:3]), np.array([0, 1, 2]))


@pytest.mark.filterwarnings("ignore")
def test_sgd_oracle_is_bit_identical_to_sklearn():
    X, y = make_multiclass(400, 7, 3, seed=6)
    for loss in ("hinge", "log_loss"):
        for shuffle in (True, False):
            yk = (y == 1).astype(int)
            m = SGDClassifier(loss=loss, random_state=3, shuffle=shuffle).fit(X, yk)
            w, b, it, t = sgd_oracle.fit_binary_sgd(X, np.where(yk == 1, 1, -1), loss=loss, shuffle=shuffle,
                                                    random_state=3)
            # hinge has no transcendental functions; log_loss goes through libm's exp/log/log1p
            # (math.*), the same ones sklearn's Cython code calls: both are bit-exact
            assert np.array_equal(w, m.coef_[0]) and b == m.intercept_[0]
            assert it == m.n_iter_ and t == m.t_


@pytest.mark.filterwarnings("ignore")
def test_ovr_sgd_matches_sklearn(fake_engine):
    X, y = make_multiclass(300, 6, 3, seed=7)
    ovr = DistOneVsRestClassifier(SGDClassifier(random_state=0)).fit(X, y)
    ref = OneVsRestClassifier(SGDClassifier(random_state=0)).fit(X, y)
    for a, b in zip(ovr.estimators_, ref.estimators_):
        np.testing.assert_array_equal(a.coef_, b.coef_)
        np.testing.assert_array_equal(a.intercept_, b.intercept_)
        assert a.n_iter_ == b.n_iter_ and a.t_ == b.t_
    np.testing.assert_array_equal(ovr.predict(X), ref.predict(X))


@pytest.mark.filterwarnings("ignore")
def test_reference_ovr_equals_sklearn():
    """Pin of the oracle choice: the UNMODIFIED reference DistOneVsRestClassifier (sc=None)
    equals sklearn's OneVsRestClassifier coefficient for coefficient."""
    want = np.load(PINS)["ovr_sgd_coef"]
    X, y = make_multiclass(500, 6, 4, seed=8)
    s = OneVsRestClassifier(SGDClassifier(random_state=0)).fit(X, y)
    assert len(s.estimators_) == len(want)
    for a, b in zip(want, s.estimators_):
        np.testing.assert_array_equal(a, b.coef_[0])


@pytest.mark.filterwarnings("ignore")
def test_ovo_logreg_matches_sklearn(fake_engine):
    """DistOneVsOneClassifier host logic (pair order, label mapping, voting) on the test-double engine."""
    from sklearn.multiclass import OneVsOneClassifier
    from skdist.distribute.multiclass import DistOneVsOneClassifier
    X, y = make_multiclass(400, 6, 4, seed=8)
    labels = np.array(["d", "a", "c", "b"])[y]
    ovo = DistOneVsOneClassifier(LogisticRegression(), None).fit(X, labels)
    ref = OneVsOneClassifier(LogisticRegression()).fit(X, labels)
    assert len(ovo.estimators_) == 6 and not hasattr(ovo, "sc")
    for a, b in zip(ovo.estimators_, ref.estimators_):
        np.testing.assert_allclose(a.coef_, b.coef_, rtol=0, atol=1e-6)
        np.testing.assert_allclose(a.intercept_, b.intercept_, rtol=0, atol=1e-6)
    np.testing.assert_array_equal(ovo.predict(X), ref.predict(X))
    np.testing.assert_allclose(ovo.decision_function(X), ref.decision_function(X), atol=1e-5)
    with pytest.raises(ValueError):
        DistOneVsOneClassifier(LogisticRegression()).fit(X, np.zeros(len(X)))


@pytest.mark.filterwarnings("ignore")
def test_string_labels_and_pandas_inputs(fake_engine):
    """String class labels and pandas containers through one-vs-rest and one-vs-one."""
    import pandas as pd
    from sklearn.multiclass import OneVsOneClassifier
    from skdist.distribute.multiclass import DistOneVsOneClassifier
    X, y = make_multiclass(700, 10, 4, seed=6)
    names = np.array(["delta", "alpha", "charlie", "bravo"])[y]
    ovr = DistOneVsRestClassifier(LogisticRegression(C=0.3), None).fit(pd.DataFrame(X), pd.Series(names))
    ref = OneVsRestClassifier(LogisticRegression(C=0.3)).fit(X, names)
    assert list(ovr.classes_) == list(ref.classes_) == ["alpha", "bravo", "charlie", "delta"]
    for a, b in zip(ovr.estimators_, ref.estimators_):
        np.testing.assert_array_equal(a.coef_, b.coef_)
    np.testing.assert_array_equal(ovr.predict(X), ref.predict(X))
    ovo = DistOneVsOneClassifier(LogisticRegression(C=0.3), None).fit(X, names)
    refo = OneVsOneClassifier(LogisticRegression(C=0.3)).fit(X, names)
    np.testing.assert_array_equal(ovo.predict(X), refo.predict(X))


def test_negatives_rows_match_reference():
    """`max_negatives` down-sampling: the training rows of a label column equal the rows the
    reference's `_negatives_mask` (ref multiclass.py:76-106) keeps, for every method / type of
    `max_negatives` / random_state."""
    from skdist_b200.distribute.multiclass import _negatives_rows
    gold = np.load(PINS)
    _, y = negatives_input()
    for i, (mn, method, rs) in enumerate(NEGATIVES_CASES):
        rows = gold["negatives_rows_%d" % i]
        np.testing.assert_array_equal(rows, np.flatnonzero(_negatives_rows(y == 1, mn, rs, method)))
        assert y[rows].sum() == y.sum()


def test_ovr_max_negatives_and_multilabel_host(fake_engine):
    """Host logic of the per-column row sets: with the engine double doing each column's fit the way the
    reference's `_fit_binary` does (lbfgs on the kept rows), DistOneVsRestClassifier equals a loop over
    scikit-learn fits on `_negatives_rows` / on the columns of a multilabel indicator matrix."""
    from skdist_b200.distribute.multiclass import _negatives_rows
    X, y = make_multiclass(1500, 8, 4, seed=9)
    ovr = DistOneVsRestClassifier(LogisticRegression(), None, max_negatives=200, random_state=3).fit(X, y)
    for k, est in enumerate(ovr.estimators_):
        m = _negatives_rows(y == k, 200, 3, "ratio")
        ref = LogisticRegression().fit(X[m], (y[m] == k).astype(int))
        np.testing.assert_allclose(est.coef_, ref.coef_, rtol=0, atol=2e-4 * np.abs(ref.coef_).max())
        assert m.sum() == (y == k).sum() + 200
    # multilabel: indicator matrix and sequences of labels (MultiLabelBinarizer, ref :267-274)
    rng = np.random.default_rng(1)
    Y = (rng.random((1500, 3)) < 0.3).astype(int)
    Y[:, 0] |= (X[:, 0] > 0.5)
    ml = DistOneVsRestClassifier(LogisticRegression(), None).fit(X, Y)
    assert len(ml.estimators_) == 3 and ml.label_binarizer_.y_type_ == "multilabel-indicator"
    for k, est in enumerate(ml.estimators_):
        ref = LogisticRegression().fit(X, Y[:, k])
        np.testing.assert_allclose(est.coef_, ref.coef_, rtol=0, atol=2e-4 * np.abs(ref.coef_).max())
    np.testing.assert_array_equal(ml.predict(X[:50]).shape, (50, 3))
    seqs = [tuple(np.flatnonzero(r)) for r in Y]
    ml2 = DistOneVsRestClassifier(LogisticRegression(), None).fit(X, seqs)
    assert hasattr(ml2, "mlb") and len(ml2.estimators_) == 3
    for a, b in zip(ml.estimators_, ml2.estimators_):
        np.testing.assert_array_equal(a.coef_, b.coef_)
    with pytest.raises(NotImplementedError):
        DistOneVsRestClassifier(SGDClassifier(), None, max_negatives=100).fit(X, y)


@pytest.mark.filterwarnings("ignore")
def test_ovo_sgd_matches_sklearn(fake_engine):
    """DistOneVsOneClassifier(SGDClassifier): one exact-order fit per class pair on the pair's rows (ref
    `_fit_ovo_binary`, multiclass.py:155-173) -- the estimators scikit-learn's OneVsOneClassifier fits."""
    from sklearn.linear_model import SGDClassifier
    from sklearn.multiclass import OneVsOneClassifier
    from skdist.distribute.multiclass import DistOneVsOneClassifier
    from skdist_b200.datasets import make_multiclass
    X, y = make_multiclass(1200, 9, 4, seed=6)
    labels = np.array(["a", "b", "c", "d"])[y]                       # string labels: pairs are formed on class indices
    ours = DistOneVsOneClassifier(SGDClassifier(random_state=0), None).fit(X, labels)
    ref = OneVsOneClassifier(SGDClassifier(random_state=0)).fit(X, labels)
    assert len(ours.estimators_) == 6
    for a, b in zip(ours.estimators_, ref.estimators_):
        np.testing.assert_array_equal(a.coef_, b.coef_)
        np.testing.assert_array_equal(a.intercept_, b.intercept_)
        assert a.n_iter_ == b.n_iter_ and a.t_ == b.t_
    np.testing.assert_array_equal(ours.predict(X), ref.predict(X))
    np.testing.assert_array_equal(ours.decision_function(X), ref.decision_function(X))
