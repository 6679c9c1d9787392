"""Host-side logic of DistGridSearchCV / DistRandomizedSearchCV (no GPU): cv_results_
assembly, best selection and refit must equal the oracle restatement of the reference's
driver loop (oracle/search_oracle.py <- ref search.py:315-571)."""
import pickle

import numpy as np
import pytest
from sklearn.base import clone
from sklearn.linear_model import LogisticRegression
from sklearn.model_selection import ParameterGrid

from oracle import search_oracle
from skdist.distribute.search import DistGridSearchCV, DistRandomizedSearchCV
from skdist_b200.datasets import make_g1_classification


def test_grid_matches_oracle(fake_engine):
    X, y = make_g1_classification(3000, 12, seed=1)
    grid = {"C": [0.01, 0.1, 1.0, 10.0]}
    gs = DistGridSearchCV(LogisticRegression(), grid, None, cv=3, return_train_score=True)
    gs.fit(X, y)
    ora = search_oracle.search_cv(LogisticRegression(), ParameterGrid(grid), X, y, cv=3,
                                  iid=True, return_train_score=True)
    for k in ["split0_test_score", "split1_test_score", "split2_test_score", "mean_test_score",
              "std_test_score", "rank_test_score", "mean_train_score"]:
        np.testing.assert_array_equal(gs.cv_results_[k], ora["cv_results_"][k], err_msg=k)
    assert gs.best_index_ == ora["best_index_"]
    assert gs.best_params_ == ora["best_params_"]
    assert gs.best_score_ == ora["best_score_"]
    assert gs.n_splits_ == 3
    np.testing.assert_array_equal(gs.best_estimator_.coef_, ora["best_estimator_"].coef_)
    np.testing.assert_array_equal(gs.predict(X[:50]), ora["best_estimator_"].predict(X[:50]))
    assert list(gs.cv_results_["params"]) == list(ParameterGrid(grid))
    assert not hasattr(gs, "sc")              # ref search.py:568
    pickle.loads(pickle.dumps(gs))            # fitted object pickles (examples/search/basic_usage.py:113)
    assert gs.get_params()["sc"] is None


def test_reference_toy_case(fake_engine):
    """ref skdist/distribute/tests/test_search.py:37-56 (same data, lbfgs instead of liblinear)."""
    X = np.array([[1, 1, 1], [0, 0, 0], [-1, -1, -1]] * 100)
    y = np.array([0, 0, 1] * 100)
    gs = DistGridSearchCV(LogisticRegression(), {"C": [0.1, 1.0]}, cv=3)
    gs.fit(X, y)
    assert np.allclose(gs.predict(X[:3]), np.array([0, 0, 1]))
    rs = DistRandomizedSearchCV(LogisticRegression(), {"C": [0.1, 1.0]}, cv=3, n_iter=2)
    rs.fit(X, y)
    assert np.allclose(rs.predict(X[:3]), np.array([0, 0, 1]))


def test_preds_and_unsupported(fake_engine):
    X, y = make_g1_classification(600, 5, seed=2)
    gs = DistGridSearchCV(LogisticRegression(), {"C": [1.0]}, cv=3, preds=True).fit(X, y)
    assert gs.get_preds().shape == (600, 2)
    np.testing.assert_allclose(gs.get_preds().sum(1), 1.0)
    gs.drop_preds()
    assert gs.get_preds() is None
    from sklearn.naive_bayes import GaussianNB
    with pytest.raises(NotImplementedError):
        DistGridSearchCV(GaussianNB(), {"var_smoothing": [1e-9]}, cv=3).fit(X, y)
    with pytest.raises(NotImplementedError):
        DistGridSearchCV(LogisticRegression(solver="liblinear"), {"C": [1.0]}, cv=3).fit(X, y)


def test_ridge_randomized_matches_oracle(fake_engine):
    """Config 5 shape in miniature: DistRandomizedSearchCV(Ridge) over loguniform alpha."""
    from scipy.stats import loguniform
    from sklearn.linear_model import Ridge
    from sklearn.model_selection import ParameterSampler
    from skdist_b200.datasets import make_g1_regression
    X, y = make_g1_regression(2000, 10, seed=3)
    dist = {"alpha": loguniform(1e-3, 1e3)}
    rs = DistRandomizedSearchCV(Ridge(), dist, None, n_iter=6, cv=4, random_state=0,
                                return_train_score=True).fit(X, y)
    cands = list(ParameterSampler(dist, 6, random_state=0))
    ora = search_oracle.search_cv(Ridge(), cands, X, y, cv=4, iid=True, return_train_score=True)
    assert rs.cv_results_["params"] == cands
    np.testing.assert_allclose(rs.cv_results_["mean_test_score"], ora["cv_results_"]["mean_test_score"],
                               rtol=1e-6)
    np.testing.assert_allclose(rs.cv_results_["mean_train_score"], ora["cv_results_"]["mean_train_score"],
                               rtol=1e-6)
    assert rs.best_index_ == ora["best_index_"]
    np.testing.assert_allclose(rs.best_estimator_.coef_, ora["best_estimator_"].coef_, rtol=1e-5)
    np.testing.assert_allclose(rs.predict(X[:20]), ora["best_estimator_"].predict(X[:20]), rtol=1e-5)
    pickle.loads(pickle.dumps(rs))


@pytest.mark.filterwarnings("ignore")
def test_multi_model_search_matches_reference_semantics(fake_engine):
    """DistMultiModelSearch: per-model ParameterSampler draws with the shared random_state, plain
    fold means, arg-max over all (model, params) rows (ref search.py:60-177, 800-866).  The expected
    values come from the same loops written with scikit-learn estimators on the CPU."""
    from scipy.stats import loguniform
    from sklearn.model_selection import ParameterSampler, StratifiedKFold
    from skdist.distribute.search import DistMultiModelSearch
    from skdist_b200.datasets import make_g1_classification
    X, y = make_g1_classification(500, 6, seed=2)
    models = [("lr_small", LogisticRegression(), {"C": loguniform(1e-3, 1e-1)}),
              ("lr_big", LogisticRegression(max_iter=50), {"C": [1.0, 10.0, 100.0], "fit_intercept": [True, False]})]
    ms = DistMultiModelSearch(models, None, n=3, cv=3, random_state=4).fit(X, y)
    exp_scores, exp_rows = [], []
    for mi, (_, est, dist) in enumerate(models):
        for params in ParameterSampler(dist, n_iter=3, random_state=4):
            fold_scores = []
            for tr, te in StratifiedKFold(3).split(X, y):
                e = clone(est).set_params(**params).fit(X[tr], y[tr])
                fold_scores.append(e.score(X[te], y[te]))
            exp_scores.append(np.mean(fold_scores))
            exp_rows.append((mi, params))
    np.testing.assert_allclose(ms.cv_results_["mean_test_score"], exp_scores, atol=1e-12)
    assert ms.cv_results_["model_index"] == [r[0] for r in exp_rows]
    assert ms.cv_results_["params"] == [r[1] for r in exp_rows]
    b = int(np.argmax(exp_scores))
    assert ms.best_model_index_ == exp_rows[b][0] and ms.best_params_ == exp_rows[b][1]
    assert ms.best_model_name_ == models[exp_rows[b][0]][0]
    assert ms.predict(X[:5]).shape == (5,) and not hasattr(ms, "sc")
    with pytest.raises(ValueError):
        DistMultiModelSearch([("a__b", LogisticRegression(), {"C": [1]})]).fit(X, y)
    with pytest.raises(ValueError):
        DistMultiModelSearch([("n", LogisticRegression(), {"C": [1]})]).fit(X, y)     # clashes with ctor arg `n`


@pytest.mark.filterwarnings("ignore")
def test_multi_model_search_against_reference_functions(fake_engine):
    """Pin against the UNMODIFIED reference: its `_raw_sampler`, `_fit_one_fold` and
    `_get_results` (ref search.py:71-177) on the same inputs must give our cv_results_.  (The reference's own
    `DistMultiModelSearch.fit` raises NameError whenever random_state is set — `i` is undefined at
    search.py:810 — so the pin is on the functions it calls.)  What they returned is stored in
    tests/golden/reference_pins.* (tests/golden/make_golden.py --reference-pins).

    The Spark branch of `_fit_batch` (search.py:137-146) ships a pickled COPY of every
    (fold, param_set) task to `_fit_one_fold`; its joblib branch passes the same dict object for
    every fold, so each fold overwrites the previous fold's "score" (search.py:109-111) and the
    "mean" becomes the last fold's score.  The Spark semantics are the intended ones: the stored
    results emulate them."""
    import json
    import os
    from skdist_b200.distribute.search import DistMultiModelSearch
    gold = os.path.join(os.path.dirname(__file__), "golden", "reference_pins")
    with open(gold + ".json") as f:
        results = json.load(f)["multi_model"]
    score = np.load(gold + ".npz")["multi_model_score"]
    X, y = make_g1_classification(400, 5, seed=6)
    models = [("a", LogisticRegression(), {"C": [0.01, 0.1, 1.0, 10.0]}),
              ("b", LogisticRegression(fit_intercept=False), {"C": [0.5, 5.0], "tol": [1e-4, 1e-3]})]
    ms = DistMultiModelSearch(models, None, n=3, cv=4, random_state=11).fit(X, y)
    assert ms.cv_results_["params"] == results["param_set"]
    assert ms.cv_results_["model_index"] == results["model_index"]
    np.testing.assert_allclose(ms.cv_results_["mean_test_score"], score, atol=1e-12)
    assert ms.best_params_ == results["param_set"][int(np.argmax(score))]


@pytest.mark.filterwarnings("ignore")
def test_multimetric_scoring_matches_sklearn(fake_engine):
    """Multi-metric search (ref search.py:336-358, 512-541): every supported scorer is a function of the
    per-column confusion counts (classifiers) or of (SSE, n) (regressors); cv_results_ must carry the same
    keys and values scikit-learn's GridSearchCV produces."""
    from sklearn.linear_model import Ridge
    from sklearn.model_selection import GridSearchCV
    from skdist_b200.datasets import make_g1_regression
    X, y = make_g1_classification(600, 6, seed=5)
    scoring = ["accuracy", "f1", "precision", "recall", "balanced_accuracy"]
    grid = {"C": [0.001, 0.05, 1.0]}
    ours = DistGridSearchCV(LogisticRegression(), grid, None, cv=3, scoring=scoring, refit="f1",
                            return_train_score=True).fit(X, y)
    ref = GridSearchCV(LogisticRegression(), grid, cv=3, scoring=scoring, refit="f1", return_train_score=True).fit(X, y)
    for m in scoring:
        for k in ["split0_test_%s" % m, "split2_test_%s" % m, "mean_test_%s" % m, "mean_train_%s" % m]:
            np.testing.assert_allclose(ours.cv_results_[k], ref.cv_results_[k], rtol=0, atol=1e-12, err_msg=k)
        np.testing.assert_array_equal(ours.cv_results_["rank_test_%s" % m], ref.cv_results_["rank_test_%s" % m])
    assert ours.best_params_ == ref.best_params_ and ours.multimetric_ and set(ours.scorer_) == set(scoring)
    assert ours.best_score_ == pytest.approx(ref.best_score_, abs=1e-12)
    with pytest.raises(ValueError):      # multi-metric needs refit=<scorer name> or False
        DistGridSearchCV(LogisticRegression(), grid, None, cv=3, scoring=scoring).fit(X, y)
    nr = DistGridSearchCV(LogisticRegression(), grid, None, cv=3, scoring=scoring, refit=False).fit(X, y)
    assert not hasattr(nr, "best_index_")
    with pytest.raises(NotImplementedError):
        DistGridSearchCV(LogisticRegression(), grid, None, cv=3, scoring="average_precision").fit(X, y)
    Xr, yr = make_g1_regression(500, 5, seed=2)
    rs = ["r2", "neg_mean_squared_error", "neg_root_mean_squared_error"]
    ours = DistGridSearchCV(Ridge(), {"alpha": [0.1, 10.0]}, None, cv=3, scoring=rs, refit="r2").fit(Xr, yr)
    ref = GridSearchCV(Ridge(), {"alpha": [0.1, 10.0]}, cv=3, scoring=rs, refit="r2").fit(Xr, yr)
    for m in rs:      # per split: the reference weights the mean by fold size (iid), scikit-learn 1.9 does not
        for k in ("split0_test_%s" % m, "split1_test_%s" % m, "split2_test_%s" % m):
            np.testing.assert_allclose(ours.cv_results_[k], ref.cv_results_[k], rtol=2e-5, atol=1e-6, err_msg=k)


def test_fast_fold_ids_equal_sklearn_splitters():
    """The direct restatement of unshuffled StratifiedKFold / KFold must give scikit-learn's folds."""
    from sklearn.model_selection import GroupKFold, KFold, StratifiedKFold
    from skdist_b200.distribute.folds import _cv_fold_ids, _fold_ids
    rng = np.random.RandomState(3)
    for n, k, ymaker in [(1000, 5, lambda: rng.randint(0, 2, 1000)), (1003, 7, lambda: rng.randint(0, 4, 1003)),
                         (50, 3, lambda: np.r_[np.zeros(40, int), np.ones(10, int)]),
                         (997, 4, lambda: (rng.rand(997) < 0.03).astype(np.int64) * 5 - 2),
                         (300, 3, lambda: rng.rand(300) < 0.5)]:
        y = ymaker()
        X = np.zeros((n, 1))
        for cv in (StratifiedKFold(k), KFold(k)):
            want = _fold_ids(list(cv.split(X, y)), n)
            got, ks = _cv_fold_ids(cv, X, y, None, n)
            assert ks == k and got.dtype == np.int8
            np.testing.assert_array_equal(got, want)
    # anything else goes through cv.split
    y = rng.randint(0, 2, 60)
    g = np.repeat(np.arange(12), 5)
    got, ks = _cv_fold_ids(GroupKFold(3), np.zeros((60, 1)), y, g, 60)
    np.testing.assert_array_equal(got, _fold_ids(list(GroupKFold(3).split(np.zeros((60, 1)), y, g)), 60))
    got, _ = _cv_fold_ids(StratifiedKFold(3, shuffle=True, random_state=0), np.zeros((60, 1)), y, None, 60)
    np.testing.assert_array_equal(got, _fold_ids(list(StratifiedKFold(3, shuffle=True, random_state=0).split(np.zeros((60, 1)), y)), 60))


def test_config1_digits_multinomial_matches_oracle(fake_engine):
    """BASELINE config 1: DistGridSearchCV(LogisticRegression) 4 params x 3 folds on sklearn digits
    (10 classes -> multinomial lbfgs, SK/linear_model/_logistic.py:523-547).  The host logic on the
    oracle-backed engine double must reproduce the reference's driver loop exactly (fp32 pixels:
    the restated solve is bit-identical to scikit-learn's there)."""
    from sklearn.datasets import load_digits
    dg = load_digits()
    X, y = (dg.data / 16).astype(np.float32), dg.target
    grid = {"C": [0.01, 0.1, 1.0, 10.0]}
    est = LogisticRegression(max_iter=30)
    gs = DistGridSearchCV(est, grid, None, cv=3, return_train_score=True, preds=True).fit(X, y)
    ora = search_oracle.search_cv(est, ParameterGrid(grid), X, y, cv=3, iid=True, return_train_score=True)
    for k in ["split0_test_score", "split1_test_score", "split2_test_score", "mean_test_score",
              "std_test_score", "rank_test_score", "mean_train_score"]:
        np.testing.assert_array_equal(gs.cv_results_[k], ora["cv_results_"][k], err_msg=k)
    assert gs.best_params_ == ora["best_params_"] and gs.best_index_ == ora["best_index_"]
    be = gs.best_estimator_
    assert be.coef_.shape == (10, 64) and be.intercept_.shape == (10,) and be.n_iter_.shape == (1,)
    np.testing.assert_array_equal(be.coef_, ora["best_estimator_"].coef_)
    np.testing.assert_array_equal(be.intercept_, ora["best_estimator_"].intercept_)
    np.testing.assert_array_equal(gs.predict(X[:200]), ora["best_estimator_"].predict(X[:200]))
    np.testing.assert_allclose(gs.predict_proba(X[:20]), ora["best_estimator_"].predict_proba(X[:20]), rtol=1e-4)
    assert gs.get_preds().shape == (len(y), 10)
    np.testing.assert_allclose(gs.get_preds().sum(1), 1.0, rtol=1e-6)
    with pytest.raises(NotImplementedError):
        DistGridSearchCV(est, grid, cv=3, scoring="roc_auc_ovr").fit(X, y)


def test_confusion_metrics_are_sklearns():
    """precision / recall / f1 (micro, macro, weighted), accuracy and balanced accuracy from a
    confusion matrix, including classes missing from y_true, from y_pred or from both."""
    import warnings
    from sklearn import metrics as M
    from skdist_b200.distribute.logreg_family import _metric_from_confusion
    rng = np.random.default_rng(0)
    K = 6
    for trial in range(8):
        yt = rng.integers(0, K - 1 - (trial % 2), 300)          # the last class(es) never occur in y_true
        yp = rng.integers(0 if trial < 6 else 1, K - (trial % 3), 300)
        conf = np.zeros((K, K), np.int64)
        np.add.at(conf, (yt, yp), 1)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            assert _metric_from_confusion("accuracy", None, conf) == M.accuracy_score(yt, yp)
            np.testing.assert_allclose(_metric_from_confusion("balanced_accuracy", None, conf),
                                       M.balanced_accuracy_score(yt, yp), rtol=1e-15)
            for avg in ("micro", "macro", "weighted"):
                for kind, f in (("f1", M.f1_score), ("precision", M.precision_score), ("recall", M.recall_score)):
                    np.testing.assert_allclose(_metric_from_confusion(kind, avg, conf), f(yt, yp, average=avg),
                                               rtol=1e-14, err_msg="%s %s" % (kind, avg))


def test_multiclass_f1_weighted_search_matches_oracle(fake_engine):
    """The reference's examples/search/hand_written_digits.py scoring ("f1_weighted") plus a second
    scorer, on 10-class digits."""
    from sklearn.datasets import load_digits
    dg = load_digits()
    X, y = (dg.data / 16).astype(np.float32), dg.target
    grid = {"C": [0.05, 5.0]}
    est = LogisticRegression(max_iter=25)
    scoring = {"f1w": "f1_weighted", "bal": "balanced_accuracy", "pm": "precision_macro"}
    gs = DistGridSearchCV(est, grid, None, cv=3, scoring=scoring, refit="f1w", return_train_score=True).fit(X, y)
    # equal-sized folds (599 rows each): the reference's test-size weighting == scikit-learn's plain mean
    from sklearn.model_selection import GridSearchCV
    sk = GridSearchCV(est, grid, cv=3, scoring=scoring, refit="f1w", return_train_score=True).fit(X, y)
    for k in ["mean_test_f1w", "mean_test_bal", "mean_test_pm", "split1_test_f1w", "mean_train_pm", "rank_test_f1w"]:
        np.testing.assert_allclose(gs.cv_results_[k], sk.cv_results_[k], rtol=1e-12, err_msg=k)
    assert gs.best_params_ == sk.best_params_


def test_binary_averaged_scorers_match_oracle(fake_engine):
    X, y = make_g1_classification(1500, 8, seed=9)
    grid = {"C": [0.1, 10.0]}
    scoring = {"f1m": "f1_macro", "rw": "recall_weighted", "pmi": "precision_micro", "f1": "f1"}
    gs = DistGridSearchCV(LogisticRegression(), grid, None, cv=3, scoring=scoring, refit="f1m").fit(X, y)
    from sklearn.model_selection import GridSearchCV
    sk = GridSearchCV(LogisticRegression(), grid, cv=3, scoring=scoring, refit="f1m").fit(X, y)
    for k in ["mean_test_f1m", "mean_test_rw", "mean_test_pmi", "mean_test_f1"]:
        np.testing.assert_allclose(gs.cv_results_[k], sk.cv_results_[k], rtol=1e-12, err_msg=k)


def test_roc_auc_search_matches_sklearn(fake_engine):
    """scoring="roc_auc" as in the reference's examples/search/basic_usage.py:89-100."""
    from sklearn.model_selection import GridSearchCV
    X, y = make_g1_classification(1500, 8, seed=11)
    grid = {"C": [0.01, 1.0, 100.0]}
    gs = DistGridSearchCV(LogisticRegression(), grid, None, cv=3, scoring="roc_auc", return_train_score=True).fit(X, y)
    sk = GridSearchCV(LogisticRegression(), grid, cv=3, scoring="roc_auc", return_train_score=True).fit(X, y)
    for k in ["mean_test_score", "split2_test_score", "mean_train_score", "rank_test_score"]:
        np.testing.assert_allclose(gs.cv_results_[k], sk.cv_results_[k], rtol=1e-6, err_msg=k)
    assert gs.best_params_ == sk.best_params_
    both = DistGridSearchCV(LogisticRegression(), grid, None, cv=3, scoring={"auc": "roc_auc", "acc": "accuracy"},
                            refit="auc").fit(X, y)
    np.testing.assert_allclose(both.cv_results_["mean_test_auc"], sk.cv_results_["mean_test_score"], rtol=1e-6)


def test_neg_log_loss_search_matches_sklearn(fake_engine):
    from sklearn.datasets import load_digits
    from sklearn.model_selection import GridSearchCV
    X, y = make_g1_classification(1200, 6, seed=12)
    grid = {"C": [0.01, 1.0]}
    gs = DistGridSearchCV(LogisticRegression(), grid, None, cv=3, scoring="neg_log_loss").fit(X, y)
    sk = GridSearchCV(LogisticRegression(), grid, cv=3, scoring="neg_log_loss").fit(X, y)
    np.testing.assert_allclose(gs.cv_results_["mean_test_score"], sk.cv_results_["mean_test_score"], rtol=1e-6)
    dg = load_digits()
    Xd, yd = (dg.data / 16).astype(np.float32), dg.target
    est = LogisticRegression(max_iter=20)
    gm = DistGridSearchCV(est, grid, None, cv=3, scoring={"nll": "neg_log_loss", "acc": "accuracy"}, refit="nll").fit(Xd, yd)
    sm = GridSearchCV(est, grid, cv=3, scoring={"nll": "neg_log_loss", "acc": "accuracy"}, refit="nll").fit(Xd, yd)
    np.testing.assert_allclose(gm.cv_results_["mean_test_nll"], sm.cv_results_["mean_test_nll"], rtol=1e-6)
    np.testing.assert_array_equal(gm.cv_results_["mean_test_acc"], sm.cv_results_["mean_test_acc"])


@pytest.mark.filterwarnings("ignore")
def test_odd_inputs_match_sklearn(fake_engine):
    """Inputs a drop-in user passes: string labels, bool labels, float labels, pandas containers,
    Fortran-ordered / float64 X, a single candidate, two folds."""
    import pandas as pd
    from sklearn.model_selection import GridSearchCV
    X, y = make_g1_classification(600, 6, seed=21)
    grid = {"C": [0.1, 1.0]}

    def check(Xi, yi, g=grid, cv=3, **kw):
        gs = DistGridSearchCV(LogisticRegression(), g, None, cv=cv, **kw).fit(Xi, yi)
        sk = GridSearchCV(LogisticRegression(), g, cv=cv, **kw).fit(np.asarray(Xi, dtype=np.float32), yi)
        np.testing.assert_allclose(gs.cv_results_["mean_test_score"], sk.cv_results_["mean_test_score"], rtol=1e-12)
        assert gs.best_params_ == sk.best_params_
        np.testing.assert_array_equal(gs.predict(np.asarray(Xi)[:40]), sk.predict(np.asarray(Xi, dtype=np.float32)[:40]))
        return gs

    gs = check(X, np.where(y == 1, "spam", "ham"))
    assert list(gs.classes_) == ["ham", "spam"]
    check(X, y.astype(bool))
    check(X, y.astype(np.float64))
    check(pd.DataFrame(X), pd.Series(y))
    check(np.asfortranarray(X), y)
    check(X, y, g={"C": [0.5]}, cv=2)
    ym = (np.arange(600) % 3 == 0).astype(int) + 2 * (np.arange(600) % 5 == 0)      # 4 classes, strings below
    check(X, np.array(["a", "b", "c", "d"])[ym])


@pytest.mark.parametrize("cvname", ["shuffle", "repeated", "predefined"])
def test_cross_validators_with_overlapping_test_sets(fake_engine, cvname):
    """Any splitter whose train sets are the complements of its test sets (ref search.py:334,379 take
    whatever `check_cv` returns): the splits are grouped into fold-id layouts of disjoint test sets
    (folds._cv_fold_groups); cv_results_ equal scikit-learn's GridSearchCV on the same splitter."""
    from sklearn.model_selection import GridSearchCV, PredefinedSplit, RepeatedStratifiedKFold, ShuffleSplit
    X, y = make_g1_classification(900, 8, seed=11)
    if cvname == "shuffle":
        cv = ShuffleSplit(n_splits=4, test_size=0.3, random_state=2)
    elif cvname == "repeated":
        cv = RepeatedStratifiedKFold(n_splits=3, n_repeats=2, random_state=5)
    else:
        tf = np.random.RandomState(0).randint(-1, 3, size=len(y))      # -1: always in the training set
        cv = PredefinedSplit(tf)
    grid = {"C": [0.01, 0.1, 1.0]}
    gs = DistGridSearchCV(LogisticRegression(), grid, None, cv=cv).fit(X, y)
    ref = GridSearchCV(LogisticRegression(), grid, cv=cv).fit(X, y)
    n_splits = cv.get_n_splits(X, y)
    assert gs.n_splits_ == n_splits
    for i in range(n_splits):
        np.testing.assert_allclose(gs.cv_results_["split%d_test_score" % i], ref.cv_results_["split%d_test_score" % i],
                                   rtol=0, atol=1e-12)
    assert gs.best_params_ == ref.best_params_


def test_time_series_split_has_no_device_path(fake_engine):
    from sklearn.model_selection import TimeSeriesSplit
    X, y = make_g1_classification(300, 5, seed=1)
    with pytest.raises(NotImplementedError):
        DistGridSearchCV(LogisticRegression(), {"C": [1.0]}, None, cv=TimeSeriesSplit(3)).fit(X, y)
