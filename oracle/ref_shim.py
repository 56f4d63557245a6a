"""TEST INFRASTRUCTURE — import shim for the UNMODIFIED reference: a checkout of marcemq/crowdmod-ddpm-4D at
oracle/_ref/ (git-ignored) or wherever $CROWDMOD_REFERENCE points.

Only usable where such a checkout exists; the repository does not ship one.  Used by
oracle/make_golden.py to generate tests/golden/* and by the `not gpu` tests that pin the oracle
restatement against the live reference.  Never imported by the product package.

The reference imports wheels that are absent here (torchmetrics, matplotlib, scikit-image,
easydict, imageio, ...); none of them is on the hot path, so they are replaced by inert stubs
before importing `models.diffusion.ddpm`.
"""
import importlib
import os
import sys
import types

REF_ROOT = os.environ.get("CROWDMOD_REFERENCE", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))
MISSING = f"no checkout of the original project at {REF_ROOT} (set CROWDMOD_REFERENCE to its path)"


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "models", "diffusion"))


class _Anything(types.ModuleType):
    """Module whose every attribute is a harmless callable/class."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        obj = type(name, (), {"__init__": lambda self, *a, **k: None,
                              "__call__": lambda self, *a, **k: None})
        setattr(self, name, obj)
        return obj


class EasyDict(dict):
    """Minimal stand-in for easydict.EasyDict (attribute access, recursive)."""

    def __init__(self, d=None, **kw):
        super().__init__()
        d = dict(d or {}, **kw)
        for k, v in d.items():
            self[k] = v

    def __setitem__(self, k, v):
        if isinstance(v, dict) and not isinstance(v, EasyDict):
            v = EasyDict(v)
        elif isinstance(v, (list, tuple)):
            v = type(v)(EasyDict(x) if isinstance(x, dict) else x for x in v)
        super().__setitem__(k, v)

    __setattr__ = __setitem__

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)


class _MeanMetric:
    def __init__(self):
        self.s, self.n = 0.0, 0

    def update(self, v):
        self.s += float(v)
        self.n += 1

    def compute(self):
        import torch
        return torch.tensor(self.s / max(self.n, 1))


_STUB_ROOTS = ("matplotlib", "mpl_toolkits", "skimage", "imageio", "torchsummary", "seaborn",
               "cv2", "PIL", "wandb", "sklearn_extra")


class _StubFinder:
    """meta-path finder: any (sub)module of a stub root that cannot be imported for real
    becomes an inert _Anything package."""

    def find_spec(self, fullname, path=None, target=None):
        if fullname.split(".")[0] not in _STUB_ROOTS:
            return None
        import importlib.machinery

        class _Loader:
            def create_module(self, spec):
                m = _Anything(spec.name)
                m.__path__ = []
                return m

            def exec_module(self, module):
                pass

        return importlib.machinery.ModuleSpec(fullname, _Loader(), is_package=True)


def _install_stubs():
    if not any(isinstance(f, _StubFinder) for f in sys.meta_path):
        sys.meta_path.append(_StubFinder())     # appended: real packages still win
    if "torchmetrics" not in sys.modules:
        try:
            importlib.import_module("torchmetrics")
        except Exception:
            m = _Anything("torchmetrics")
            m.MeanMetric = _MeanMetric
            sys.modules["torchmetrics"] = m
    if "easydict" not in sys.modules:
        try:
            importlib.import_module("easydict")
        except Exception:
            m = types.ModuleType("easydict")
            m.EasyDict = EasyDict
            sys.modules["easydict"] = m


def load():
    """Returns a namespace with the reference's hot-path classes, imported from REF_ROOT."""
    if not available():
        raise RuntimeError(f"reference not found at {REF_ROOT}")
    _install_stubs()
    # The reference uses top-level package names `models` / `utils`; make sure ours (if the
    # product directory is on sys.path) do not shadow them while importing.
    saved = {k: sys.modules.pop(k) for k in list(sys.modules)
             if k == "models" or k.startswith("models.") or k == "utils" or k.startswith("utils.")}
    sys.path.insert(0, REF_ROOT)
    try:
        ns = types.SimpleNamespace()
        ns.unet = importlib.import_module("models.backbones.unet")
        ns.layers = importlib.import_module("models.backbones.layers")
        ns.embeddings = importlib.import_module("models.backbones.embeddings")
        ns.forward = importlib.import_module("models.diffusion.forward")
        ns.ddpm = importlib.import_module("models.diffusion.ddpm")
        ns.guidance = importlib.import_module("models.guidance")
        ns.UNet = ns.unet.UNet
        ns.ForwardSampler = ns.forward.ForwardSampler
        ns.DDPM = ns.ddpm.DDPM
        ns.DDPM_model = ns.ddpm.DDPM_model
        ns.EasyDict = sys.modules["easydict"].EasyDict
        try:
            ns.dit = importlib.import_module("models.backbones.DiT4D_V4")
            ns.DiT4D_V4 = ns.dit.DiT4D_V4
        except Exception as e:  # noqa: BLE001 - optional: only the f2 pins need it
            ns.dit, ns.DiT4D_V4, ns.dit_error = None, None, repr(e)
        # the callers either side of the path (SURVEY.md section 8 f3 / f4): CPU metrics tail, windowed dataset
        try:
            ns.metrics = importlib.import_module("utils.metrics.metricsGenerator")
            ns.MetricsGenerator = ns.metrics.MetricsGenerator
        except Exception as e:  # noqa: BLE001 - optional: only the f3 pins need it
            ns.metrics, ns.MetricsGenerator, ns.metrics_error = None, None, repr(e)
        try:
            ns.dataset = importlib.import_module("utils.dataset")
            ns.MacropropsDataset = ns.dataset.MacropropsDataset
        except Exception as e:  # noqa: BLE001
            ns.dataset, ns.MacropropsDataset, ns.dataset_error = None, None, repr(e)
        return ns
    finally:
        sys.path.remove(REF_ROOT)
        # leave the reference modules registered under private names only
        for k in list(sys.modules):
            if k == "models" or k.startswith("models.") or k == "utils" or k.startswith("utils."):
                sys.modules["_crowdmod_ref." + k] = sys.modules.pop(k)
        sys.modules.update(saved)
