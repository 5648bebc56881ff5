"""
TEST INFRASTRUCTURE ONLY -- never imported by the product (pylc_b200/).

Harness that imports the *unmodified* PyLC reference from the checkout named by the
PYLC_REFERENCE_ROOT environment variable (default: oracle/_ref/, ignored by git) so that
(a) the oracle restatements in oracle/pylc_oracle.py can be validated against it and
(b) golden input/output vectors can be generated (oracle/gen_golden.py -> tests/golden/).

The reference is not part of this repository, so everything here is guarded by `available()`;
without it the committed golden vectors carry the pinning.

Recipe (SURVEY.md Appendix B):
  * stub modules for h5py / seaborn / matplotlib (import-only dependencies of
    db/database.py:17, utils/metrics.py:15-16 that are not installed here),
  * cwd must contain ./schemas (config.py:108,296-298) and a writable ./data
    (utils/evaluate.py:59-62),
  * TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD=1 for Model.load (models/model.py:100).
"""
import contextlib
import os
import shutil
import sys
import tempfile
import types

REF_ROOT = os.environ.get("PYLC_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))

_state = {"loaded": False, "workdir": None}


def available():
    return os.path.isfile(os.path.join(REF_ROOT, "utils", "tools.py"))


def _install_stubs():
    if "h5py" not in sys.modules:
        try:
            import h5py  # noqa: F401
        except Exception:
            sys.modules["h5py"] = types.ModuleType("h5py")
    try:
        import seaborn  # noqa: F401
    except Exception:
        sb = types.ModuleType("seaborn")

        class _Fig:
            def savefig(self, *a, **k):
                pass

        class _Ax:
            def get_figure(self):
                return _Fig()

        sb.set = lambda *a, **k: None
        sb.heatmap = lambda *a, **k: _Ax()
        sys.modules["seaborn"] = sb
    try:
        import matplotlib.pyplot  # noqa: F401
    except Exception:
        mpl = types.ModuleType("matplotlib")
        plt = types.ModuleType("matplotlib.pyplot")
        for name in ("ylabel", "xlabel", "clf", "rc", "figure", "show"):
            setattr(plt, name, lambda *a, **k: None)
        mpl.pyplot = plt
        sys.modules["matplotlib"] = mpl
        sys.modules["matplotlib.pyplot"] = plt


def load():
    """Import the reference modules. Returns a namespace with the modules we drive."""
    if not available():
        raise RuntimeError("reference not available at %s" % REF_ROOT)
    if not _state["loaded"]:
        os.environ.setdefault("TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD", "1")
        _install_stubs()
        wd = tempfile.mkdtemp(prefix="pylc_ref_")
        shutil.copytree(os.path.join(REF_ROOT, "schemas"), os.path.join(wd, "schemas"))
        for d in ("db", "save", "models", "outputs"):
            os.makedirs(os.path.join(wd, "data", d), exist_ok=True)
        _state["workdir"] = wd
        _state["prev_cwd"] = os.getcwd()
        os.chdir(wd)
        # The reference is a flat script directory whose top-level module names
        # (config, utils, db, models) must win over anything else on sys.path.
        for name in list(sys.modules):
            if name in ("config", "utils", "db", "models") or name.split(".")[0] in ("utils", "db", "models"):
                mod = sys.modules[name]
                if not getattr(mod, "__file__", "") or not str(getattr(mod, "__file__", "")).startswith(REF_ROOT):
                    del sys.modules[name]
        sys.path.insert(0, REF_ROOT)
        _state["loaded"] = True
    import config as ref_config
    import utils.tools as ref_tools
    import utils.extract as ref_extract
    import utils.profile as ref_profile
    import utils.metrics as ref_metrics
    import utils.evaluate as ref_evaluate
    import models.modules.loss as ref_loss
    import db.dataset as ref_dataset
    ns = types.SimpleNamespace(
        config=ref_config, tools=ref_tools, extract=ref_extract, profile=ref_profile,
        metrics=ref_metrics, evaluate=ref_evaluate, loss=ref_loss, dataset=ref_dataset,
        workdir=_state["workdir"])
    return ns


@contextlib.contextmanager
def in_workdir():
    """Run a block with cwd = the scratch dir holding ./schemas and ./data."""
    prev = os.getcwd()
    os.chdir(_state["workdir"])
    try:
        yield _state["workdir"]
    finally:
        os.chdir(prev)


def load_model_modules():
    load()
    import models.model as ref_model
    import models.architectures.deeplab as ref_deeplab
    return types.SimpleNamespace(model=ref_model, deeplab=ref_deeplab)


@contextlib.contextmanager
def quiet():
    """Silence the reference's print() chatter."""
    with open(os.devnull, "w") as dn, contextlib.redirect_stdout(dn):
        yield
