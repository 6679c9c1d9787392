"""Import the UNMODIFIED reference (``/root/reference/skdist``) under sklearn 1.9.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Works only where a source tree of the
reference exists; used by tests/golden/make_golden.py to produce the committed
fixtures, which the tests compare against without the reference.

The reference targets sklearn<0.23.2.  Three in-memory patches make its
hot-path modules importable without touching any file (SURVEY.md section 8c):
  * ``np.int`` alias (search.py:510, multiclass.py:159),
  * ``sklearn.utils.metaestimators.if_delegate_has_method`` (search.py:23),
  * ``sklearn.ensemble.forest`` module alias (ensemble.py:11).
"""
import os
import sys

REFERENCE_ROOT = os.environ.get("SKDIST_REFERENCE_ROOT", "/root/reference")


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "skdist", "distribute"))


def _patch():
    import numpy as np
    import sklearn.utils.metaestimators as _m
    from sklearn.utils.metaestimators import available_if

    if not hasattr(np, "int"):
        np.int = int
    if not hasattr(_m, "if_delegate_has_method"):
        def if_delegate_has_method(delegate):
            names = tuple(delegate) if isinstance(delegate, (list, tuple)) else (delegate,)
            return available_if(lambda self: any(hasattr(self, n) for n in names))
        _m.if_delegate_has_method = if_delegate_has_method
    if "sklearn.ensemble.forest" not in sys.modules:
        import sklearn.ensemble._forest as _f
        sys.modules["sklearn.ensemble.forest"] = _f


def _import_reference(names):
    """Import reference modules by dotted name ('skdist.distribute.search', ...).  Our own drop-in
    alias package is also called ``skdist``: the reference's copy is imported under that name only
    for the duration of the call and the previous ``sys.modules`` entries are restored afterwards."""
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    _patch()
    import importlib
    import importlib.util
    saved = {k: v for k, v in sys.modules.items() if k == "skdist" or k.startswith("skdist.")}
    for k in saved:
        del sys.modules[k]
    try:
        spec = importlib.util.spec_from_file_location(
            "skdist", os.path.join(REFERENCE_ROOT, "skdist", "__init__.py"),
            submodule_search_locations=[os.path.join(REFERENCE_ROOT, "skdist")])
        pkg = importlib.util.module_from_spec(spec)
        sys.modules["skdist"] = pkg
        spec.loader.exec_module(pkg)
        mods = [importlib.import_module(n) for n in names]
    finally:
        ref_mods = {k: v for k, v in sys.modules.items() if k == "skdist" or k.startswith("skdist.")}
        for k in ref_mods:
            del sys.modules[k]
        sys.modules.update(saved)
    return mods


def load():
    """Return the reference's (search, multiclass, ensemble) modules."""
    return tuple(_import_reference(["skdist.distribute.search", "skdist.distribute.multiclass",
                                    "skdist.distribute.ensemble"]))


def load_module(name):
    """Return one more reference module, e.g. 'skdist.distribute.eliminate'."""
    return _import_reference([name])[0]
