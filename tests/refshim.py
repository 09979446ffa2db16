"""Import harness for the upstream reference (test infrastructure only).

The reference (a checkout of utiasSTARS/tightly-coupled-SfM named by the
environment variable ``TCSFM_REFERENCE_ROOT``) is pure Python/PyTorch but
imports a few packages that need not be installed (``liegroups``,
``pykitti``, ``matplotlib``) from modules the hot path never touches.  This
harness registers empty stand-ins for them and returns the reference's own
modules so that golden vectors can be generated from, and the oracle pinned
against, the real thing.  Without that checkout the tests that need it skip;
nothing marked ``gpu``, ``smoke()`` or ``bench.py`` may call it.
"""
import os
import sys
import types

REF_ROOT = os.environ.get("TCSFM_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "models", "stn.py"))


def _stub(name, **attrs):
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    sys.modules.setdefault(name, mod)
    return sys.modules[name]


def load_reference():
    """Returns a namespace with the reference modules ``stn``, ``losses``,
    ``train_mono``, ``optimizer``, ``helpers`` and ``learning_helpers``."""
    if not reference_available():
        raise RuntimeError("reference tree not found: set TCSFM_REFERENCE_ROOT to a checkout of the reference")
    dummy = type("Dummy", (), {})
    _stub("liegroups", SE3=dummy, SO3=dummy)
    _stub("liegroups.torch", SE3=dummy, SO3=dummy)
    _stub("pykitti")
    mpl = _stub("matplotlib", use=lambda *a, **k: None)
    plt = _stub("matplotlib.pyplot")
    mpl.pyplot = plt
    _stub("matplotlib.cm")
    _stub("imageio")
    for p in (os.path.join(REF_ROOT, "optimization_experiments"), REF_ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    # The reference has top-level modules called ``losses``/``models``/``utils``;
    # import them under their own names (they import each other that way).
    import importlib
    ns = types.SimpleNamespace()
    ns.stn = importlib.import_module("models.stn")
    ns.learning_helpers = importlib.import_module("utils.learning_helpers")
    ns.losses = importlib.import_module("losses")
    ns.geometry_helpers = importlib.import_module("utils.geometry_helpers")
    try:
        ns.train_mono = importlib.import_module("train_mono")
    except Exception as e:  # data loaders need cv2/scipy; report, don't hide
        ns.train_mono = None
        ns.train_mono_error = e
    try:
        ns.optimizer = importlib.import_module("optimizer")
        ns.helpers = importlib.import_module("helpers")
    except Exception as e:
        ns.optimizer = None
        ns.helpers = None
        ns.optimizer_error = e
    return ns
