"""The Python drop-in boundary (SURVEY section 8b): constructor signatures (names, order, defaults) and the
public method surface of every Dist* class against the reference's own classes, as recorded from the
unmodified reference in tests/golden/reference_pins.json (tests/golden/make_golden.py --reference-pins)."""
import inspect
import json
import os

import pytest

PINS = os.path.join(os.path.dirname(__file__), "golden", "reference_pins.json")

CLASSES = {
    "search": ["DistGridSearchCV", "DistRandomizedSearchCV", "DistMultiModelSearch"],
    "multiclass": ["DistOneVsRestClassifier", "DistOneVsOneClassifier"],
    "ensemble": ["DistRandomForestClassifier", "DistRandomForestRegressor", "DistExtraTreesClassifier",
                 "DistExtraTreesRegressor", "DistRandomTreesEmbedding"],
    "eliminate": ["DistFeatureEliminator"],
}
# The reference's one-vs-rest / one-vs-one constructors end in **kwargs, forwarded to scikit-learn's
# OneVsRestClassifier / OneVsOneClassifier, whose only parameter besides `estimator` is n_jobs: spelled out here.
KWARGS_AS = {"DistOneVsRestClassifier": ("n_jobs", None), "DistOneVsOneClassifier": ("n_jobs", None)}
# delegating methods the reference exposes only when the wrapped estimator has them (if_delegate_has_method):
# absent from the class attribute listing here for the same reason (sklearn's available_if)
CONDITIONAL = {"transform", "inverse_transform"}


def _params(cls):
    out = []
    for k, v in inspect.signature(cls.__init__).parameters.items():
        if k == "self":
            continue
        out.append((k, v.kind == v.VAR_KEYWORD, None if v.default is inspect._empty else repr(v.default)))
    return out


@pytest.mark.parametrize("module", sorted(CLASSES))
def test_constructors_and_public_surface_match_the_reference(module):
    import importlib
    ours = importlib.import_module("skdist.distribute." + module)
    with open(PINS) as f:
        surface = json.load(f)["surface"][module]
    for name in CLASSES[module]:
        ref = surface[name]
        want, got = [tuple(p) for p in ref["params"]], _params(getattr(ours, name))
        if name in KWARGS_AS:
            assert want[-1][1], "the reference constructor no longer ends in **kwargs"
            k, d = KWARGS_AS[name]
            want = want[:-1] + [(k, False, repr(d))]
        assert got == want, name
        missing = set(ref["public"]) - {n for n in dir(getattr(ours, name)) if not n.startswith("_")} - CONDITIONAL
        assert not missing, (name, sorted(missing))


def test_conditional_delegates_follow_the_estimator(fake_engine):
    from sklearn.linear_model import LogisticRegression
    from skdist.distribute.eliminate import DistFeatureEliminator
    from skdist.distribute.search import DistMultiModelSearch
    assert not hasattr(DistFeatureEliminator(LogisticRegression()), "transform")
    m = DistMultiModelSearch([("lr", LogisticRegression(), {"C": [1.0]})])
    assert not hasattr(m, "transform") and not hasattr(m, "inverse_transform")

    class _T:
        def transform(self, X):
            return X
    m.best_estimator_ = _T()
    assert hasattr(m, "transform") and not hasattr(m, "inverse_transform")
