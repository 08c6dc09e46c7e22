"""Import the UNMODIFIED reference, wvangansbeke/LaneDetection_End2End (TEST INFRASTRUCTURE).

``install()`` (called by ``__graft_entry__.build()``) byte-compiles the reference's hot-path modules from a checkout of
the original project into ``oracle/_ref/`` (git-ignored): sourceless ``.pyc`` modules that import from the tree wherever
it is copied, without the checkout.  The checkout is ``DEFAULT_SOURCE`` unless the environment variable
``LANEFIT_REFERENCE`` names another one.  ``import_reference()`` loads, in this order: the checkout LANEFIT_REFERENCE
names (so ``oracle/make_golden.py`` regenerates the goldens from exactly that checkout), the install, the default
checkout.  Nothing under ``-m gpu`` or ``smoke()`` calls this; ``bench.py`` uses it for the reference arm /
cpu_baseline only (kind "reference").
Recipe = SURVEY.md Appendix A: the reference modules use top-level
``import Networks`` and need ``matplotlib`` at import time
(Backprojection_Loss/Networks/utils.py:17-21), which this image lacks -> stub it.
"""
import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INSTALLED_ROOT = os.path.join(_REPO, "oracle", "_ref")
DEFAULT_SOURCE = "/root/reference"
_EXPLICIT_SOURCE = os.environ.get("LANEFIT_REFERENCE") or None
SOURCE_ROOT = _EXPLICIT_SOURCE or DEFAULT_SOURCE
_HOT_PATH_FILES = ["Networks/__init__.py", "Networks/ERFNet.py", "Networks/LSQ_layer.py", "Networks/gels.py",
                   "Networks/utils.py", "Loss_crit.py"]


def _has_reference(r):
    return r is not None and os.path.isdir(os.path.join(r, "Backprojection_Loss", "Networks"))


def _root():
    for r in (_EXPLICIT_SOURCE, INSTALLED_ROOT, DEFAULT_SOURCE):
        if _has_reference(r):
            return r
    return None


REFERENCE_ROOT = _root() or INSTALLED_ROOT


def available():
    return _root() is not None


def install(src=SOURCE_ROOT, dst=INSTALLED_ROOT):
    """Byte-compile the reference's hot-path modules (both variants) from the checkout `src` into `dst` (oracle/_ref),
    replacing whatever an earlier install left there.  No-op (False), leaving `dst` as it is, when `src` holds no
    reference.

    Bytecode rather than a copy of the files: `dst` lies inside the working tree, and keeping the original project's
    source text out of it means no copy of that source can be committed or shipped with the tree.  A .pyc only loads
    in the interpreter version that wrote it; every build() rewrites the install with the interpreter that runs it,
    and the benchmark reports the "port" kind (with the import error on stderr) if the install does not load."""
    import py_compile
    import shutil
    if not _has_reference(src):
        return False
    shutil.rmtree(dst, ignore_errors=True)
    for variant in ("Backprojection_Loss", "Birds_Eye_View_Loss"):
        for rel in _HOT_PATH_FILES:
            s = os.path.join(src, variant, rel)
            if os.path.exists(s):
                d = os.path.join(dst, variant, rel + "c")
                os.makedirs(os.path.dirname(d), exist_ok=True)
                py_compile.compile(s, cfile=d, dfile=os.path.join(variant, rel), doraise=True)
    for extra in ("LICENSE.txt",):
        if os.path.exists(os.path.join(src, extra)):
            shutil.copyfile(os.path.join(src, extra), os.path.join(dst, extra))
    return True


def _stub_matplotlib():
    if "matplotlib" in sys.modules:
        return
    try:
        import matplotlib  # noqa: F401
        return
    except Exception:
        pass
    m = types.ModuleType("matplotlib")
    m.use = lambda *a, **k: None
    p = types.ModuleType("matplotlib.pyplot")
    p.rcParams = {}
    m.pyplot = p
    sys.modules["matplotlib"] = m
    sys.modules["matplotlib.pyplot"] = p


def purge():
    for k in list(sys.modules):
        if k == "Networks" or k.startswith("Networks.") or k in ("Loss_crit",):
            del sys.modules[k]
    roots = [r for r in (_EXPLICIT_SOURCE, INSTALLED_ROOT, DEFAULT_SOURCE) if r]
    sys.path[:] = [p for p in sys.path if not any(p.startswith(r) for r in roots)]


def import_reference(variant="Backprojection_Loss"):
    """Returns a namespace with the reference's Net, define_args, define_init_weights,
    backprojection_loss / Area_Loss, get_homography, Weighted_least_squares,
    ProjectiveGridGenerator, GELS for the given variant directory."""
    root = _root()
    if root is None:
        raise RuntimeError("reference not installed under %s and no checkout at %s (set LANEFIT_REFERENCE)"
                           % (INSTALLED_ROOT, SOURCE_ROOT))
    _stub_matplotlib()
    purge()
    sys.path.insert(0, os.path.join(root, variant))
    ns = types.SimpleNamespace()
    import Networks  # noqa: F401
    from Networks import LSQ_layer, ERFNet, utils
    import Loss_crit
    ns.Networks = Networks
    ns.LSQ_layer = LSQ_layer
    ns.ERFNet = ERFNet
    ns.utils = utils
    ns.Loss_crit = Loss_crit
    if variant == "Backprojection_Loss":
        from Networks import gels
        ns.gels = gels
    return ns


def make_args(ns, extra=(), no_cuda=True):
    """argparse Namespace the reference's ``Net(args)`` consumes (utils.py:24-99)."""
    argv = ["--image_dir", "x", "--gt_dir", "y"] + (["--no_cuda"] if no_cuda else []) + list(extra)
    return ns.utils.define_args().parse_args(argv)
