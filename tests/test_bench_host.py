"""bench.py's checker pieces on the CPU: the task sample of the CPU leg and the `parity` block that compares its
scores with cv_results_ at the same (candidate, fold) -- on an engine double whose fits are scikit-learn's, so the
block must report no difference."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def test_cpu_tasks_are_whole_candidates_spread_over_the_grid():
    import bench
    tasks = bench.cpu_tasks(512, 5, 40)
    assert len(tasks) == 40
    cands = sorted({c for c, _ in tasks})
    assert cands[0] == 0 and cands[-1] == 511 and len(cands) == 8
    assert all(sorted(f for c, f in tasks if c == ci) == list(range(5)) for ci in cands)
    assert len(bench.cpu_tasks(512, 5, 3)) == 3


def test_parity_block_against_the_cpu_leg(fake_engine):
    import bench
    from sklearn.linear_model import LogisticRegression
    from skdist.distribute.search import DistGridSearchCV
    from skdist_b200.datasets import make_g1_classification
    X, y = make_g1_classification(3000, 12, seed=2)
    Cs = np.logspace(-3, 2, 6)
    fold = bench.fold_ids(y, 3)
    gs = DistGridSearchCV(LogisticRegression(), {"C": list(Cs)}, None, cv=3).fit(X, y)
    tasks = bench.cpu_tasks(len(Cs), 3, 9)
    fps, dt, scores, n_jobs, inner = bench.cpu_fits_per_sec(X, y, fold, Cs, tasks, n_jobs=1)
    assert fps > 0 and len(scores) == len(tasks) == 9
    blk = bench.parity_block(gs.cv_results_, tasks, scores, fold, Cs, 3)
    assert blk["n_compared"] == 9 and blk["max_flips_per_fold"] == 0 and blk["max_abs_dscore"] < 1e-12
    assert blk["best_C_equal_on_subgrid"] and blk["best_C_tied"]
    assert blk["test_rows_per_fold"] == 1000
    # a device result that differs by 3 test rows in one fold is reported as such
    bad = {k: np.array(v, dtype=float).copy() if k.startswith(("split", "mean_test")) else v for k, v in gs.cv_results_.items()}
    ci, f = tasks[4]
    bad["split%d_test_score" % f][ci] -= 3 / 1000
    assert bench.parity_block(bad, tasks, scores, fold, Cs, 3)["max_flips_per_fold"] == 3


def test_dump_outputs_in_column_order_and_capped(tmp_path, monkeypatch):
    """--dump-outputs: rows go back to column order whatever the dealing, every file is float32 / float64, and
    above the size cap the same seeded sample of columns is written on every run."""
    import bench
    n_cols, d = 40, 5
    order = np.random.default_rng(3).permutation(n_cols)       # the order the columns were fitted in
    res = {"coef": (order[:, None] * 10.0 + np.arange(d + 1)).astype(np.float32), "n_iter": order.astype(np.int32),
           "status": np.zeros(n_cols, np.int32), "loss": order * 0.5, "n_evals": order.astype(np.int32) + 1}
    correct, count = order.astype(np.int64), np.full(n_cols, 7, np.int64)
    bench.dump_outputs(str(tmp_path / "all"), res, correct, count, n_cols, 0, 1, order, None)
    got = {p.stem: np.load(p) for p in (tmp_path / "all").iterdir()}
    assert set(got) == {"column", "coef", "n_iter", "status", "loss", "n_evals", "correct", "count"}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    np.testing.assert_array_equal(got["column"], np.arange(n_cols))
    np.testing.assert_array_equal(got["coef"][:, 0], np.arange(n_cols) * 10.0)
    np.testing.assert_array_equal(got["n_evals"], np.arange(n_cols) + 1)
    row_bytes = 8 + 4 * (d + 1) + 8 * 6
    monkeypatch.setattr(bench, "DUMP_LIMIT", 10 * row_bytes)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), res, correct, count, n_cols, 0, 1, order, None)
    cols = np.load(tmp_path / "a" / "column.npy")
    assert len(cols) == 10 and np.array_equal(cols, np.load(tmp_path / "b" / "column.npy"))
    assert sum(p.stat().st_size - 128 for p in (tmp_path / "a").iterdir()) <= 10 * row_bytes
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "correct.npy"), cols)
