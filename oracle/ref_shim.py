"""TEST INFRASTRUCTURE ONLY -- load-time shim that EXECUTES the reference's own sources.

Nothing is copied: the Python-2 files under ``/root/reference`` are read at run time,
passed through a handful of mechanical py2->py3 regex rewrites (SURVEY.md section 8(c)) and
``exec``-ed into fresh module objects.  It exists so that

  * ``tests/golden/make_golden*.py`` can freeze golden input/output vectors of the real
    reference (``gp.py``, ``GPEIOptChooser.py``, ``GPEIperSecChooser.py``, ``GPEIChooser.py``,
    the spearmint-lite controller).

The reference tree is not part of this repository, so no test, ``__graft_entry__.smoke()``
or ``bench.py`` may depend on this file at run time.
The product package ``spearmint_b200`` never imports anything from ``oracle/``.
"""
import os
import re
import sys
import types

REF_ROOT = os.environ.get("SPEARMINT_REFERENCE", "/root/reference")
REF_PKG = os.path.join(REF_ROOT, "spearmint", "spearmint")


def available():
    return os.path.isfile(os.path.join(REF_PKG, "gp.py"))


_PRINT_RE = re.compile(r"^(\s*)print\s+(?!\()(.*)$", re.M)


def _py3(src):
    """The ~10 mechanical rewrites listed in SURVEY.md section 8(c)."""
    src = src.replace("\t", "        ")
    src = _PRINT_RE.sub(lambda m: "%sprint(%s)" % (m.group(1), m.group(2).rstrip().rstrip(",")), src)
    src = src.replace("xrange", "range")
    src = src.replace("import cPickle", "import pickle as cPickle")
    src = re.sub(r"^import scipy\.weave\s*$", "", src, flags=re.M)
    src = re.sub(r"(\w+(?:\.\w+)*)\.has_key\(([^)]+)\)", r"(\2 in \1)", src)
    src = src.replace("ordering = range(dims)", "ordering = list(range(dims))")
    src = src.replace("NamedTemporaryFile(mode='w'", "NamedTemporaryFile(mode='wb'")
    src = src.replace("open(self.state_pkl, 'r')", "open(self.state_pkl, 'rb')")
    src = re.sub(r",\s*disp=0", "", src)
    # py2 `map` returned a list; util.unpack_args feeds it to dict() which is fine in py3.
    return src


def _exec_module(name, path, extra_globals=None):
    with open(path, "r") as fh:
        src = _py3(fh.read())
    mod = types.ModuleType(name)
    mod.__file__ = path
    if extra_globals:
        mod.__dict__.update(extra_globals)
    sys.modules[name] = mod
    exec(compile(src, path, "exec"), mod.__dict__)
    return mod


_loaded = {}


def load():
    """Returns a dict of the reference modules: gp, util, Locker, OPT, PSEC, GPEI, sobol_lib."""
    if _loaded:
        return _loaded
    if not available():
        raise RuntimeError("reference tree not present at %s" % REF_ROOT)

    # Stubs (SURVEY 8c): real helpers.py imports a stale generated protobuf module.
    helpers = types.ModuleType("helpers")
    helpers.log = lambda *a: None
    helpers.__all__ = ["log"]
    sys.modules["helpers"] = helpers
    if "imp" not in sys.modules:
        sys.modules["imp"] = types.ModuleType("imp")

    pkg = types.ModuleType("spearmint")
    pkg.__path__ = []
    sys.modules["spearmint"] = pkg

    gp = _exec_module("spearmint.gp", os.path.join(REF_PKG, "gp.py"))
    util = _exec_module("spearmint.util", os.path.join(REF_PKG, "util.py"))
    pkg.gp, pkg.util = gp, util
    sys.modules["gp"], sys.modules["util"] = gp, util
    locker = _exec_module("Locker", os.path.join(REF_PKG, "Locker.py"))
    sobol = _exec_module("sobol_lib", os.path.join(REF_PKG, "sobol_lib.py"))

    chooser_pkg = types.ModuleType("chooser")
    chooser_pkg.__path__ = []
    sys.modules["chooser"] = chooser_pkg
    cdir = os.path.join(REF_PKG, "chooser")
    opt = _exec_module("chooser.GPEIOptChooser", os.path.join(cdir, "GPEIOptChooser.py"))
    psec = _exec_module("chooser.GPEIperSecChooser", os.path.join(cdir, "GPEIperSecChooser.py"))
    gpei = _exec_module("chooser.GPEIChooser", os.path.join(cdir, "GPEIChooser.py"))

    _loaded.update(gp=gp, util=util, Locker=locker, sobol_lib=sobol,
                   OPT=opt, PSEC=psec, GPEI=gpei)
    return _loaded


def load_lite():
    """The reference's spearmint-lite controller (spearmint-lite/spearmint-lite.py) with its own ExperimentGrid,
    executed under the same py3 rewrites.  Returns the module (main_controller, GridMap...)."""
    load()
    lite_dir = os.path.join(REF_ROOT, "spearmint-lite")
    if "ExperimentGrid" not in sys.modules or not getattr(sys.modules["ExperimentGrid"], "_lite", False):
        sys.modules["sobol_lib"] = _exec_module("sobol_lib", os.path.join(lite_dir, "sobol_lib.py"))
        eg = _exec_module("ExperimentGrid", os.path.join(lite_dir, "ExperimentGrid.py"))
        eg._lite = True
    return _exec_module("spearmint_lite", os.path.join(lite_dir, "spearmint-lite.py"))
