"""Import the UNMODIFIED reference model (BlockBasedImgCompLossyNetv9) in this container.

TEST INFRASTRUCTURE ONLY; needs a checkout of the reference repository, which is not part of this one:
LBIC_REFERENCE_ROOT names its directory.  Only fixture generation (tests/golden/make_golden*.py) and the
`needs_reference` tests use it; those tests skip where the variable is not set.

The reference's package __init__ files import every sibling module (graphs/layers/__init__.py:6-10,
utils/__init__.py:6-10) and so drag in matplotlib/easydict/bjontegaard/compressai, none of which
is installed.  We therefore register bare namespace packages and load the few files the codec path
needs BY PATH, with oracle/ref_shim/compressai standing in for CompressAI.
"""
import importlib.util
import os
import sys
import types

REF = os.environ.get("LBIC_REFERENCE_ROOT", "")
_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(os.path.dirname(_HERE))


def available() -> bool:
    return bool(REF) and os.path.isfile(os.path.join(REF, "graphs/models/BlockBasedImgCompLossy_net.py"))


def _load(name, relpath):
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, relpath))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def _ns(name):
    if name not in sys.modules:
        m = types.ModuleType(name)
        m.__path__ = []
        sys.modules[name] = m
    return sys.modules[name]


def load():
    """Returns the reference module graphs.models.BlockBasedImgCompLossy_net."""
    if not available():
        raise FileNotFoundError(f"reference tree not found at LBIC_REFERENCE_ROOT={REF!r}")
    for p in (_REPO, _HERE):
        if p not in sys.path:
            sys.path.insert(0, p)
    import compressai  # the stand-in in this directory

    assert os.path.dirname(compressai.__file__) == os.path.join(_HERE, "compressai"), compressai.__file__
    _ns("utils")
    bound_ops = _load("utils.bound_ops", "utils/bound_ops.py")
    _load("utils.parametrizers", "utils/parametrizers.py")
    ops = types.ModuleType("compressai.ops")
    ops.LowerBound = bound_ops.LowerBound
    sys.modules["compressai.ops"] = ops
    compressai.ops = ops
    _ns("graphs"); _ns("graphs.layers"); _ns("graphs.models")
    gdn = _load("graphs.layers.gdn_compressai", "graphs/layers/gdn_compressai.py")
    layers = types.ModuleType("compressai.layers")
    layers.GDN, layers.GDN1 = gdn.GDN, gdn.GDN1
    sys.modules["compressai.layers"] = layers
    compressai.layers = layers
    ent = _load("graphs.layers.entropy_layers_cai", "graphs/layers/entropy_layers_cai.py")
    em = types.ModuleType("compressai.entropy_models")
    em.GaussianConditional, em.EntropyBottleneck, em.EntropyModel = (
        ent.GaussianConditional, ent.EntropyBottleneck, ent.EntropyModel)
    sys.modules["compressai.entropy_models"] = em
    compressai.entropy_models = em
    _load("graphs.layers.masked_conv2d", "graphs/layers/masked_conv2d.py")
    return _load("graphs.models.BlockBasedImgCompLossy_net", "graphs/models/BlockBasedImgCompLossy_net.py")


class EasyDict(dict):
    """Minimal stand-in for easydict.EasyDict (attribute access on a dict), enough for utils/config.py and the agent."""

    def __init__(self, d=None, **kw):
        super().__init__()
        for k, v in dict(d or {}, **kw).items():
            self[k] = v

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v


def load_agent():
    """Returns the reference module agents.blkbsdimgcomp_agent (class BlockBasedImgCompLossyAgent), UNMODIFIED, with
    stand-ins for the packages it imports that are not installed here: easydict, matplotlib (display only),
    bjontegaard, ptflops, torchsummary, and pytorch_msssim (-> lbic_b200.codec.ms_ssim, a restatement: MS-SSIM values
    printed by a run through this loader are NOT a pin of that package)."""
    load()
    import torch

    def stub(name, **attrs):
        m = sys.modules.get(name) or types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    stub("easydict", EasyDict=EasyDict)
    mpl = stub("matplotlib")
    mpl.__path__ = []
    mpl.pyplot = stub("matplotlib.pyplot")
    stub("bjontegaard")
    stub("ptflops", get_model_complexity_info=lambda *a, **k: (0, 0))
    stub("torchsummary", summary=lambda *a, **k: None)
    from lbic_b200 import codec as _codec

    class _MS(torch.nn.Module):                       # MS_SSIM / SSIM module forms (training losses only)
        def __init__(self, *a, data_range=1.0, **k):
            super().__init__()
            self.data_range = data_range

        def forward(self, x, y):
            return _codec.ms_ssim(x, y, data_range=self.data_range)

    stub("pytorch_msssim", ms_ssim=lambda x, y, data_range=1.0, **k: _codec.ms_ssim(x, y, data_range=data_range),
         MS_SSIM=_MS, SSIM=_MS, ssim=lambda *a, **k: (_ for _ in ()).throw(NotImplementedError("ssim stub")))
    # the reference was written against an older torch: ReduceLROnPlateau(verbose=...) no longer exists (torch >= 2.7);
    # accept and drop the argument (an environment stand-in, the reference file itself stays untouched)
    import inspect
    _RLP = torch.optim.lr_scheduler.ReduceLROnPlateau
    if "verbose" not in inspect.signature(_RLP.__init__).parameters and not getattr(_RLP, "_lbic_compat", False):
        class ReduceLROnPlateau(_RLP):
            _lbic_compat = True

            def __init__(self, *a, verbose=False, **k):
                super().__init__(*a, **k)

        torch.optim.lr_scheduler.ReduceLROnPlateau = ReduceLROnPlateau
    for pkg in ("agents", "dataloaders", "loggers", "graphs.losses"):
        _ns(pkg)
    _load("utils.image_plots", "utils/image_plots.py")
    _load("graphs.losses.rate_dist", "graphs/losses/rate_dist.py")
    _load("dataloaders.image_dl_ACL", "dataloaders/image_dl_ACL.py")
    _load("loggers.rate", "loggers/rate.py")
    _load("agents.base", "agents/base.py")
    return _load("agents.blkbsdimgcomp_agent", "agents/blkbsdimgcomp_agent.py")
