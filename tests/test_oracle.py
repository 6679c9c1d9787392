"""The oracle against (a) the committed golden fixtures produced by the reference's own
_fit_and_score (tests/golden/make_golden.py) and (b) installed scikit-learn."""
import os

import numpy as np
import pytest
from sklearn.datasets import load_digits
from sklearn.linear_model import LogisticRegression
from sklearn.model_selection import ParameterGrid

from oracle import logreg_oracle as lo
from oracle import search_oracle
from skdist_b200.datasets import make_g1_classification

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _case(name):
    if name == "search_logreg_g1_4000x16":
        X, y = make_g1_classification(4000, 16, seed=3)
        return X, y, 3
    if name == "search_logreg_digits3":
        dg = load_digits()
        return dg.data.astype(np.float32), (dg.target == 3).astype(np.int64), 3
    X, y = make_g1_classification(20000, 64, seed=4)
    return X, y, 5


@pytest.mark.parametrize("name", ["search_logreg_g1_4000x16", "search_logreg_digits3"])
@pytest.mark.filterwarnings("ignore")
def test_search_oracle_matches_golden(name):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    X, y, cv = _case(name)
    cands = [{"C": float(c)} for c in g["C"]]
    ora = search_oracle.search_cv(LogisticRegression(), cands, X, y, cv=cv, iid=True)
    for i in range(cv):
        k = "split%d_test_score" % i
        np.testing.assert_array_equal(ora["cv_results_"][k], g[k])
    np.testing.assert_array_equal(ora["cv_results_"]["mean_test_score"], g["mean_test_score"])
    np.testing.assert_array_equal(ora["cv_results_"]["rank_test_score"], g["rank_test_score"])
    assert ora["best_index_"] == int(g["best_index"])


@pytest.mark.filterwarnings("ignore")
def test_logreg_restatement_is_bit_identical_to_sklearn():
    X, y = make_g1_classification(5000, 20, seed=7)
    yf = y.astype(np.float32)
    for C in [0.01, 1.0, 100.0]:
        for fi in [True, False]:
            coef, b, it = lo.fit_binary_lbfgs(X, yf, C=C, fit_intercept=fi)
            m = LogisticRegression(C=C, fit_intercept=fi).fit(X, y)
            assert np.array_equal(coef, m.coef_[0]) and it == m.n_iter_[0]
            if fi:
                assert b == m.intercept_[0]
            assert lo.accuracy(X, yf, coef, b) == m.score(X, y)


@pytest.mark.filterwarnings("ignore")
def test_oracle_task_equals_reference_task():
    """Pin: reference _fit_and_score (search.py:180-288), as stored in reference_pins.*, vs oracle.fit_and_score."""
    import json
    X, y = make_g1_classification(1500, 8, seed=5)
    cands = list(ParameterGrid({"C": [0.1, 10.0]}))
    b = search_oracle.search_cv(LogisticRegression(), cands, X, y, cv=3)
    np.testing.assert_array_equal(np.load(os.path.join(GOLD, "reference_pins.npz"))["task_mean_test_score"],
                                  b["cv_results_"]["mean_test_score"])
    with open(os.path.join(GOLD, "reference_pins.json")) as f:
        assert json.load(f)["task_best_params"] == b["best_params_"]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_multinomial_restatement_is_sklearn(dtype):
    """fit_multinomial_lbfgs vs LogisticRegression.fit on a multiclass target: bit-identical for
    fp32 inputs (the device path's input type); fp64 differs only by numpy-vs-libm exp/log ulps."""
    import warnings
    from sklearn.linear_model import LogisticRegression
    dg = load_digits()
    X, y = (dg.data / 16).astype(dtype), dg.target
    for C in (0.1, 10.0):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            est = LogisticRegression(C=C, max_iter=40).fit(X, y)
        W, b, it = lo.fit_multinomial_lbfgs(X, y, 10, C=C, max_iter=40)
        assert it == est.n_iter_[0]
        if dtype == np.float32:
            np.testing.assert_array_equal(W, est.coef_)
            np.testing.assert_array_equal(b, est.intercept_)
        else:
            np.testing.assert_allclose(W, est.coef_, rtol=0, atol=1e-7)
            np.testing.assert_allclose(b, est.intercept_, rtol=0, atol=1e-7)


@pytest.mark.parametrize("name", ["search_logreg_digits10_scaled", "search_logreg_digits10_raw"])
@pytest.mark.filterwarnings("ignore")
def test_multinomial_oracle_matches_golden(name):
    """BASELINE config 1 (10-class digits, 4 C x 3 folds): the fixtures hold the scores of the reference's
    unmodified `_fit_and_score` (tests/golden/make_golden.py --multinomial-only).  The oracle's driver loop
    reproduces them exactly; on fp32 inputs the restated multinomial solve reproduces the stored
    coefficients bit for bit."""
    g = np.load(os.path.join(GOLD, name + ".npz"))
    dg = load_digits()
    X = (dg.data / 16).astype(np.float32) if name.endswith("scaled") else dg.data
    y = dg.target
    est = LogisticRegression(max_iter=int(g["max_iter"]))
    cands = [{"C": float(c)} for c in g["C"]]
    ora = search_oracle.search_cv(est, cands, X, y, cv=3, iid=True)
    for k in ("split0_test_score", "split1_test_score", "split2_test_score", "mean_test_score", "rank_test_score"):
        np.testing.assert_array_equal(ora["cv_results_"][k], g[k], err_msg=k)
    assert ora["best_index_"] == int(g["best_index"])
    if name.endswith("scaled"):
        from sklearn.model_selection import StratifiedKFold
        splits = list(StratifiedKFold(3).split(X, y))
        for ci, fi in ((0, 0), (2, 1), (3, 2)):
            tr = splits[fi][0]
            W, b, it = lo.fit_multinomial_lbfgs(X[tr], y[tr], 10, C=float(g["C"][ci]), max_iter=int(g["max_iter"]))
            np.testing.assert_array_equal(W, g["coef"][ci, fi, :, :64])
            np.testing.assert_array_equal(b, g["coef"][ci, fi, :, 64])
            assert it == g["n_iter"][ci, fi]
