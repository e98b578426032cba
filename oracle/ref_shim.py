"""Run the reference's OWN estimator / utils / OneEuroFilter, unchanged, from a checkout of the reference project.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Only usable where the environment variable VNECT_REFERENCE_ROOT names a
checkout of XinArkh/VNect; it is what ``tests/golden/make_golden.py`` uses to mint the committed fixtures, and what the
live comparisons of the test suite use when the reference tree is present.

``src/estimator.py`` imports ``tensorflow`` (not installable here) and ``src/utils.py`` imports matplotlib (not
installed).  Both are replaced by stubs *in sys.modules only*: the stub ``tf.Session.run`` hands the fed batch to a
``forward`` callable supplied by the caller (``oracle.forward.OracleNet`` or a synthetic-map generator).  Every line of
the reference's pre-processing, multi-scale averaging, argmax, gather and filtering runs as written.
"""
import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("VNECT_REFERENCE_ROOT", "")
TENSOR_NAMES = ("split_2:0", "split_2:1", "split_2:2", "split_2:3")


def reference_available():
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "src", "estimator.py"))


class _Forward:
    fn = None


def _install_stubs():
    if "tensorflow" not in sys.modules or not getattr(sys.modules["tensorflow"], "_vnect_stub", False):
        tf = types.ModuleType("tensorflow")
        tf._vnect_stub = True

        class Session:
            def run(self, fetches, feed_dict):
                (batch,) = feed_dict.values()
                outs = _Forward.fn(batch)
                return [outs[TENSOR_NAMES.index(f)] for f in fetches]

        class _Saver:
            def restore(self, sess, path):
                pass

        class _Graph:
            def get_tensor_by_name(self, name):
                return name

        tf.Session = Session
        tf.train = types.SimpleNamespace(import_meta_graph=lambda p: _Saver(), latest_checkpoint=lambda p: p)
        tf.get_default_graph = lambda: _Graph()
        sys.modules["tensorflow"] = tf
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.animation", "mpl_toolkits", "mpl_toolkits.mplot3d"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m._vnect_stub = True
            sys.modules[name] = m
    sys.modules["matplotlib.animation"].FuncAnimation = object
    sys.modules["mpl_toolkits"].mplot3d = sys.modules["mpl_toolkits.mplot3d"]
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]


def load_reference_modules():
    """Import (utils, OneEuroFilter, estimator) from the reference tree, unchanged."""
    if not reference_available():
        raise RuntimeError("reference tree not found: set VNECT_REFERENCE_ROOT to a checkout of XinArkh/VNect")
    _install_stubs()
    src = os.path.join(REFERENCE_ROOT, "src")
    if src not in sys.path:
        sys.path.insert(0, src)
    mods = []
    for name in ("utils", "OneEuroFilter", "estimator"):
        mods.append(importlib.import_module(name))
    return tuple(mods)


class ScriptedClock:
    """Stands in for the ``time`` module inside the reference estimator: returns the scripted values in order."""

    def __init__(self, values):
        self.values = list(values)
        self.i = 0

    def time(self):
        v = self.values[self.i]
        self.i += 1
        return v


def frame_clock(t2d, t3d):
    """The four time.time() calls of one frame (estimator.py:98, :84 twice via joint_filter, :141)."""
    return [t2d - 1e-3, t2d, t3d, t3d + 1e-3]


def make_reference_estimator(forward, scales=None):
    """Instantiate the reference VNectEstimator with ``forward`` behind its TF session."""
    utils, oef, est_mod = load_reference_modules()
    _Forward.fn = forward
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        est = est_mod.VNectEstimator()
    if scales is not None:
        est.scales = list(scales)
    return est, est_mod


def run_reference(est, est_mod, img, t2d, t3d):
    """One reference __call__ with scripted timestamps; returns (joints_2d, joints_3d)."""
    import contextlib
    import io
    real_time = est_mod.time
    est_mod.time = ScriptedClock(frame_clock(t2d, t3d))
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            j2, j3 = est(img)
    finally:
        est_mod.time = real_time
    return j2, j3
