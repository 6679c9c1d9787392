"""oracle/ -- CPU restatement of the reference's hot path.  TEST INFRASTRUCTURE ONLY.

Nothing under ``skdist_b200/`` (the product) may import, call or link this
package.  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs use it, and only as the checker /
the CPU arm that is timed beside the GPU arm.

Pinning status (see DESIGN.md "Oracle"):

* The reference (Ibotta/sk-dist @ v0.1.9) is pure Python; every FLOP of the hot
  path is executed by its third-party dependency scikit-learn (reference pins
  ``>=0.20,<0.23.2`` in setup.py:30-31; this image and the GPU box carry 1.9.0)
  and scipy 1.18.1 (L-BFGS-B, LAPACK).  The oracle therefore restates the
  reference's *driver loops* (search.py:315-571, multiclass.py:288-335,
  ensemble.py:177-336) and per-task functions (search.py:180-288) in numpy and
  calls the same installed scikit-learn estimators the reference calls.
* The restatement is pinned against the reference's own per-task functions,
  imported unmodified from /root/reference under a 3-line in-memory shim
  (``oracle/refshim.py``), by ``tests/golden/make_golden.py``; its outputs are
  committed as ``tests/golden/*.npz`` and re-checked by ``tests/test_oracle.py``.
* BASELINE config 1 (10-class digits, multinomial lbfgs) is pinned the same way:
  ``tests/golden/search_logreg_digits10_{raw,scaled}.npz`` hold the scores of the reference's
  unmodified ``_fit_and_score`` plus its own run-to-run envelope; ``logreg_oracle.fit_multinomial_lbfgs``
  reproduces the stored fp32 coefficients bit for bit (``tests/test_oracle.py``).
* Pins on what the reference's own code returns, recorded by ``tests/golden/make_golden.py
  --reference-pins`` into ``tests/golden/reference_pins.{npz,json}``: the multi-model search
  against the reference's ``_raw_sampler`` / ``_fit_one_fold`` / ``_get_results``
  (``tests/test_search_host.py``), the feature eliminator against its ``_fit_and_score_one`` /
  ``_drop_col`` (``tests/test_eliminate_host.py``), and the constructor signatures and public
  names of every Dist* class (``tests/test_boundary_host.py``).
* The SGD (``sgd_oracle.py``), logistic (``logreg_oracle.py``) and ridge (``ridge_oracle.py``)
  restatements are bit-identical to the installed scikit-learn estimators (``tests/test_oracle.py``,
  ``tests/test_multiclass_host.py``); trees are checked against scikit-learn directly, which the
  reference's ``_build_trees`` equals tree for tree (``tests/test_forest_host.py``).
* The reference's own tests pin only toy predictions
  (skdist/distribute/tests/test_search.py:37-56, test_multiclass.py:23-38, test_ensemble.py:25-58);
  those cases are reproduced in ``tests/test_search_host.py``, ``tests/test_multiclass_host.py``,
  ``tests/test_forest_gpu.py`` (incl. the golden regressor predictions [0.15, 0.18, 0.12]).
"""
