"""Generate tests/golden/*.npz by running the UNMODIFIED reference per-task functions
(skdist/distribute/search.py:_fit_and_score of sk-dist) under oracle/refshim.py.

Needs a source tree of the reference (oracle/refshim.py, SKDIST_REFERENCE_ROOT):
    python tests/golden/make_golden.py
    python tests/golden/make_golden.py --reference-pins
The fixtures pin (i) the oracle restatement oracle/search_oracle.py against the reference
and (ii) the CUDA path against both (tests/test_gpu_parity.py); reference_pins.{npz,json} hold
what the reference's own classes and helpers return on the inputs of the host tests that are pinned
to it, so that those tests run without the reference.  Inputs are regenerated from seeds by
skdist_b200.datasets, so only outputs are stored.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from sklearn.datasets import load_digits  # noqa: E402
from sklearn.linear_model import LogisticRegression  # noqa: E402
from sklearn.model_selection import ParameterGrid  # noqa: E402

from oracle import refshim, search_oracle  # noqa: E402
from skdist_b200.datasets import make_g1_classification  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def reference_task(ref_search):
    def task(estimator, X, y, scorer, train, test, params):
        # exactly the call DistBaseSearchCV.fit makes (ref search.py:391-406)
        return ref_search._fit_and_score(
            estimator, X, y, {"score": scorer}, train, test, 0, params, fit_params={},
            return_train_score=False, return_n_test_samples=True, return_times=True,
            return_parameters=False, error_score="raise")
    return task


def run_case(name, X, y, grid, cv, ref_search, variants=12):
    est = LogisticRegression()
    cands = list(ParameterGrid(grid))
    ref = search_oracle.search_cv(est, cands, X, y, cv=cv, iid=True, task_fn=reference_task(ref_search))
    ora = search_oracle.search_cv(est, cands, X, y, cv=cv, iid=True)
    n_splits = ref["n_splits_"]
    keys = ["split%d_test_score" % i for i in range(n_splits)] + ["mean_test_score", "std_test_score",
                                                                  "rank_test_score"]
    for k in keys:
        assert np.array_equal(ref["cv_results_"][k], ora["cv_results_"][k]), (name, k)
    assert ref["best_index_"] == ora["best_index_"]
    # per-(candidate, fold) coefficients from the same sklearn fit the task runs
    from sklearn.model_selection import check_cv
    splits = list(check_cv(cv, y, classifier=True).split(X, y))
    d = X.shape[1]
    coef = np.zeros((len(cands), n_splits, d + 1), np.float32)
    n_iter = np.zeros((len(cands), n_splits), np.int32)
    for ci, p in enumerate(cands):
        for fi, (tr, te) in enumerate(splits):
            m = LogisticRegression(**p).fit(X[tr], y[tr])
            coef[ci, fi, :d] = m.coef_[0]
            coef[ci, fi, d] = m.intercept_[0]
            n_iter[ci, fi] = m.n_iter_[0]
    # The reference's own sensitivity to floating-point summation order: the same sklearn fits
    # with 1 BLAS thread / all BLAS threads / permuted training-row order.  Columns that stop on
    # max_iter before converging amplify 1-ulp differences (DESIGN.md "Parity"); the envelope is
    # stored so that the CUDA path is held to the reference's own reproducibility, no looser.
    from threadpoolctl import threadpool_limits
    rng = np.random.default_rng(12345)
    noise_flips = np.zeros((len(cands), n_splits), np.int64)
    noise_coef = np.zeros((len(cands), n_splits))
    for variant in range(variants):  # 1 thread, default threads, then row permutations
        for ci, p in enumerate(cands):
            for fi, (tr, te) in enumerate(splits):
                trv = tr if variant < 2 else tr[rng.permutation(len(tr))]
                with threadpool_limits(limits=1 if variant == 0 else None):
                    m = LogisticRegression(**p).fit(X[trv], y[trv])
                base_correct = int(round(ref["cv_results_"]["split%d_test_score" % fi][ci] * len(te)))
                fl = abs(int((m.predict(X[te]) == y[te]).sum()) - base_correct)
                w = np.r_[m.coef_[0], m.intercept_]
                noise_flips[ci, fi] = max(noise_flips[ci, fi], fl)
                noise_coef[ci, fi] = max(noise_coef[ci, fi],
                                         np.abs(w - coef[ci, fi]).max() / np.abs(coef[ci, fi]).max())
    out = {k: ref["cv_results_"][k] for k in keys}
    out.update(noise_flips=noise_flips, noise_coef=noise_coef)
    out.update(best_index=ref["best_index_"], coef=coef, n_iter=n_iter,
               refit_coef=np.r_[ref["best_estimator_"].coef_[0], ref["best_estimator_"].intercept_],
               C=np.array([p["C"] for p in cands]))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "noise_flips", noise_flips.ravel(), "\n  noise_coef", np.round(noise_coef.ravel(), 5))
    print(name, "mean_test_score", ref["cv_results_"]["mean_test_score"], "n_iter", n_iter.ravel())


def run_ridge_case(name, X, y, alphas, cv, ref_search):
    from sklearn.linear_model import Ridge
    from sklearn.model_selection import KFold
    est = Ridge()
    cands = [{"alpha": float(a)} for a in alphas]
    ref = search_oracle.search_cv(est, cands, X, y, cv=cv, iid=True, task_fn=reference_task(ref_search))
    ora = search_oracle.search_cv(est, cands, X, y, cv=cv, iid=True)
    keys = ["split%d_test_score" % i for i in range(cv)] + ["mean_test_score", "rank_test_score"]
    for k in keys:
        assert np.array_equal(ref["cv_results_"][k], ora["cv_results_"][k]), (name, k)
    d = X.shape[1]
    coef = np.zeros((len(cands), cv, d + 1), np.float32)
    coef64 = np.zeros((len(cands), cv, d + 1))      # same fit in float64: the fp32 reference's own error bar
    X64, y64 = X.astype(np.float64), y.astype(np.float64)
    for ci, p in enumerate(cands):
        for fi, (tr, te) in enumerate(KFold(cv).split(X)):
            m = Ridge(**p).fit(X[tr], y[tr])
            coef[ci, fi, :d] = m.coef_
            coef[ci, fi, d] = m.intercept_
            m = Ridge(**p).fit(X64[tr], y64[tr])
            coef64[ci, fi, :d] = m.coef_
            coef64[ci, fi, d] = m.intercept_
    out = {k: ref["cv_results_"][k] for k in keys}
    out.update(best_index=ref["best_index_"], coef=coef, coef64=coef64, alpha=np.asarray(alphas, float),
               refit_coef=np.r_[ref["best_estimator_"].coef_, ref["best_estimator_"].intercept_])
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "mean_test_score", ref["cv_results_"]["mean_test_score"])


def run_multinomial_case(name, X, y, grid, cv, max_iter, ref_search):
    """BASELINE config 1 shape: multiclass target -> multinomial lbfgs (SK/linear_model/_logistic.py:523-547).
    Scores from the reference's unmodified `_fit_and_score`; per-(candidate, fold) coefficients from the same
    scikit-learn fit, checked bit for bit against the oracle's restatement when X is float32."""
    import warnings
    from sklearn.model_selection import check_cv
    from threadpoolctl import threadpool_limits
    from oracle import logreg_oracle
    warnings.simplefilter("ignore")
    est = LogisticRegression(max_iter=max_iter)
    cands = list(ParameterGrid(grid))
    ref = search_oracle.search_cv(est, cands, X, y, cv=cv, iid=True, task_fn=reference_task(ref_search))
    ora = search_oracle.search_cv(est, cands, X, y, cv=cv, iid=True)
    n_splits = ref["n_splits_"]
    keys = ["split%d_test_score" % i for i in range(n_splits)] + ["mean_test_score", "std_test_score",
                                                                  "rank_test_score"]
    for k in keys:
        assert np.array_equal(ref["cv_results_"][k], ora["cv_results_"][k]), (name, k)
    splits = list(check_cv(cv, y, classifier=True).split(X, y))
    K, d = len(np.unique(y)), X.shape[1]
    coef = np.zeros((len(cands), n_splits, K, d + 1), X.dtype)
    n_iter = np.zeros((len(cands), n_splits), np.int32)
    for ci, p in enumerate(cands):
        for fi, (tr, te) in enumerate(splits):
            m = LogisticRegression(max_iter=max_iter, **p).fit(X[tr], y[tr])
            coef[ci, fi, :, :d] = m.coef_
            coef[ci, fi, :, d] = m.intercept_
            n_iter[ci, fi] = m.n_iter_[0]
            if X.dtype == np.float32:
                W, b, it = logreg_oracle.fit_multinomial_lbfgs(X[tr], y[tr], K, C=p["C"], max_iter=max_iter)
                assert np.array_equal(W, m.coef_) and np.array_equal(b, m.intercept_) and it == m.n_iter_[0]
    rng = np.random.default_rng(4321)
    noise_flips = np.zeros((len(cands), n_splits), np.int64)
    noise_coef = np.zeros((len(cands), n_splits))
    for variant in range(8):        # 1 thread, default threads, then 6 row permutations
        for ci, p in enumerate(cands):
            for fi, (tr, te) in enumerate(splits):
                trv = tr if variant < 2 else tr[rng.permutation(len(tr))]
                with threadpool_limits(limits=1 if variant == 0 else None):
                    m = LogisticRegression(max_iter=max_iter, **p).fit(X[trv], y[trv])
                base_correct = int(round(ref["cv_results_"]["split%d_test_score" % fi][ci] * len(te)))
                noise_flips[ci, fi] = max(noise_flips[ci, fi], abs(int((m.predict(X[te]) == y[te]).sum()) - base_correct))
                w = np.c_[m.coef_, m.intercept_]
                noise_coef[ci, fi] = max(noise_coef[ci, fi], np.abs(w - coef[ci, fi]).max() / np.abs(coef[ci, fi]).max())
    out = {k: ref["cv_results_"][k] for k in keys}
    out.update(noise_flips=noise_flips, noise_coef=noise_coef, best_index=ref["best_index_"], coef=coef, n_iter=n_iter,
               C=np.array([p["C"] for p in cands]), max_iter=max_iter)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "mean_test_score", ref["cv_results_"]["mean_test_score"], "n_iter", n_iter.ravel())
    print(name, "noise_flips", noise_flips.ravel(), "\n  noise_coef", np.round(noise_coef.ravel(), 5))


def reference_pins():
    """What the tests that pin the drop-in against the reference's own code compare with: the outputs of
    the UNMODIFIED reference functions and classes on the tests' inputs, stored as
    reference_pins.npz (arrays) and reference_pins.json (signatures, parameter sets)."""
    import copy
    import json
    import warnings
    from itertools import product
    from sklearn.linear_model import SGDClassifier
    from sklearn.metrics import check_scoring
    from sklearn.model_selection import StratifiedKFold
    from sklearn.tree import DecisionTreeClassifier
    from skdist_b200.datasets import make_multiclass
    from skdist_b200.distribute.ensemble import MAX_RAND_SEED
    from tests.test_boundary_host import CLASSES, _params
    from tests.test_eliminate_host import ELIMINATOR_CASES, _data, feature_sets
    from tests.test_forest_host import lattice
    from tests.test_multiclass_host import NEGATIVES_CASES, negatives_input
    warnings.simplefilter("ignore")
    ref_search, ref_mc, ref_ens = refshim.load()
    arrays, meta = {}, {}

    # constructor signatures and public names of every Dist* class (tests/test_boundary_host.py)
    meta["surface"] = {}
    for module, names in CLASSES.items():
        mod = refshim.load_module("skdist.distribute." + module)
        meta["surface"][module] = {n: {"params": _params(getattr(mod, n)),
                                       "public": sorted(a for a in dir(getattr(mod, n)) if not a.startswith("_"))}
                                   for n in names}

    # per-task function of the search: mean_test_score and best_params_ (tests/test_oracle.py)
    X, y = make_g1_classification(1500, 8, seed=5)
    cands = list(ParameterGrid({"C": [0.1, 10.0]}))
    a = search_oracle.search_cv(LogisticRegression(), cands, X, y, cv=3, task_fn=reference_task(ref_search))
    arrays["task_mean_test_score"] = a["cv_results_"]["mean_test_score"]
    meta["task_best_params"] = a["best_params_"]

    # the multi-model search's _raw_sampler / _fit_one_fold / _get_results (tests/test_search_host.py); the
    # Spark branch's copy of each (fold, param_set) task is emulated with deepcopy (see the test)
    X, y = make_g1_classification(400, 5, seed=6)
    models = [("a", LogisticRegression(), {"C": [0.01, 0.1, 1.0, 10.0]}),
              ("b", LogisticRegression(fit_intercept=False), {"C": [0.5, 5.0], "tol": [1e-4, 1e-3]})]
    folds = list(StratifiedKFold(4).split(X, y))
    param_sets = ref_search._raw_sampler(models, n=3, random_state=11)
    scores = [ref_search._fit_one_fold((f, copy.deepcopy(ps)), models, X, y, None, {})
              for f, ps in product(folds, param_sets)]
    results = ref_search._get_results(scores)
    meta["multi_model"] = {"param_set": list(results["param_set"]),
                           "model_index": [int(i) for i in results["model_index"]]}
    arrays["multi_model_score"] = results["score"].values.astype(np.float64)

    # the feature eliminator's _fit_and_score_one per feature set (tests/test_eliminate_host.py)
    ref_elim = refshim.load_module("skdist.distribute.eliminate")
    X, y = _data()
    for i, (step, n_cv, min_keep) in enumerate(ELIMINATOR_CASES):
        base = LogisticRegression(C=0.3)
        scorer = check_scoring(base, scoring=None)
        arrays["eliminator_scores_%d" % i] = np.array(
            [np.mean([ref_elim._fit_and_score_one(idx, base, X, y, scorer, tr, te, False, {})
                      for tr, te in StratifiedKFold(n_cv).split(X, y)])
             for idx in feature_sets(X, y, step, min_keep)])

    # the forest's _build_trees (tests/test_forest_host.py)
    X, y = lattice(1500, 8, 3)
    for i, s in enumerate(np.random.RandomState(5).randint(MAX_RAND_SEED, size=3)):
        tr = ref_ens._build_trees(DecisionTreeClassifier(max_features="sqrt"), (), {}, X,
                                  y.astype(np.float64)[:, None], None, s, 3, bootstrap=True)
        arrays["build_trees_threshold_%d" % i] = tr.tree_.threshold
        arrays["build_trees_children_left_%d" % i] = tr.tree_.children_left.astype(np.int32)
    X, y = lattice(300, 4, 6)
    arrays["get_oof"] = ref_ens.get_oof(LogisticRegression(), X, y, n_splits=3)[1]

    # one-vs-rest with sc=None, and the max_negatives down-sampling (tests/test_multiclass_host.py)
    X, y = make_multiclass(500, 6, 4, seed=8)
    r = ref_mc.DistOneVsRestClassifier(SGDClassifier(random_state=0)).fit(X, y)
    arrays["ovr_sgd_coef"] = np.stack([e.coef_[0] for e in r.estimators_])
    X, y = negatives_input()
    for i, (mn, method, rs) in enumerate(NEGATIVES_CASES):
        Xr, yr = ref_mc._negatives_mask(X, y, max_negatives=mn, random_state=rs, method=method)
        arrays["negatives_rows_%d" % i] = np.sort(Xr[:, 0].astype(np.int32))
        assert yr.sum() == y.sum()

    np.savez_compressed(os.path.join(HERE, "reference_pins.npz"), **arrays)
    with open(os.path.join(HERE, "reference_pins.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
        f.write("\n")
    print("reference_pins:", sorted(arrays))


def main():
    ref_search, _, _ = refshim.load()
    if "--reference-pins" in sys.argv:
        reference_pins()
        return
    if "--multinomial-only" in sys.argv:
        dg = load_digits()
        grid = {"C": [0.01, 0.1, 1.0, 10.0]}
        # config 1 of BASELINE.json as stated (raw 0..16 pixels, float64, default max_iter) and on scaled
        # float32 pixels with enough iterations to converge (the reproducible variant)
        run_multinomial_case("search_logreg_digits10_raw", dg.data, dg.target, grid, 3, 100, ref_search)
        run_multinomial_case("search_logreg_digits10_scaled", (dg.data / 16).astype(np.float32), dg.target, grid, 3,
                             300, ref_search)
        return
    if "--mid-only" in sys.argv:
        # mid-size pin of the headline workload's generator and shape class (d = 256, tcgen05-eligible):
        # G1 200 000 x 256, 32 C x 5 folds = 160 fits of the reference's unmodified _fit_and_score;
        # envelope from 1 BLAS thread, all threads and 2 row permutations (about 40 minutes on 8 cores)
        X, y = make_g1_classification(200000, 256, seed=7)
        run_case("search_logreg_g1_200000x256", X, y, {"C": list(np.logspace(-4, 4, 32))}, 5, ref_search, variants=4)
        return
    if "--ridge-only" in sys.argv:
        from skdist_b200.datasets import make_g1_regression
        X, y = make_g1_regression(6000, 40, seed=5)
        run_ridge_case("search_ridge_g1_6000x40", X, y, [1e-3, 1e-1, 1.0, 10.0, 1e3], 4, ref_search)
        return
    X, y = make_g1_classification(4000, 16, seed=3)
    run_case("search_logreg_g1_4000x16", X, y, {"C": [1e-3, 1e-2, 1e-1, 1.0, 10.0, 100.0]}, 3, ref_search)
    X, y = make_g1_classification(20000, 64, seed=4)
    run_case("search_logreg_g1_20000x64", X, y, {"C": [1e-4, 1e-2, 1.0, 100.0]}, 5, ref_search)
    # config 1 of BASELINE.json, binarised (digit 3 vs rest), float32 as the device path computes
    dg = load_digits()
    Xd = dg.data.astype(np.float32)
    yd = (dg.target == 3).astype(np.int64)
    run_case("search_logreg_digits3", Xd, yd, {"C": [0.01, 0.1, 1.0, 10.0]}, 3, ref_search)


if __name__ == "__main__":
    main()
