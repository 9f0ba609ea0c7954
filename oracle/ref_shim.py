"""Import shim for the *live* reference modules (test infrastructure, NOT product code).

Only usable where IGN_REFERENCE_ROOT names a checkout of the reference
(InterpretGatedNetwork); the repository does not carry it.  Nothing under tests/ -m gpu,
smoke() or bench.py imports this file: it exists so that tests/golden/make_golden.py can
run the unmodified reference (model/Shapelet.py, model/InterpGN.py) and freeze its outputs
into tests/golden/*.npz, and so that `-m "not gpu"` tests can cross-check the oracle
restatement against the real thing when that checkout is given.

The reference's directories are `model/` and `data_factory/` but its imports say
`models.` / `data_provider.`; plotting dependencies are absent here.  We alias/stub
exactly those names and touch no reference file.  The reference is loaded under
PRIVATE module names so it cannot shadow this repo's own `models` / `utils` packages.
"""
import importlib.util
import os
import sys
import types

REF_ROOT = os.environ.get("IGN_REFERENCE_ROOT", "")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "model", "Shapelet.py"))


def _load(private_name, relpath):
    spec = importlib.util.spec_from_file_location(private_name, os.path.join(REF_ROOT, relpath))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[private_name] = mod
    spec.loader.exec_module(mod)
    return mod


_cache = {}


def load_reference():
    """Returns a namespace with the reference's Shapelet / InterpGN / FCN classes."""
    if "ns" in _cache:
        return _cache["ns"]
    if not available():
        raise RuntimeError("no reference checkout at IGN_REFERENCE_ROOT=%r" % REF_ROOT)
    saved = {k: sys.modules.get(k) for k in (
        "utils", "utils.shapelet_util", "models", "models.Shapelet", "models.FullyConvNet",
        "models.PatchTST", "models.TimesNet", "models.Transformer", "models.ResNet",
        "seaborn", "matplotlib", "matplotlib.colors", "matplotlib.pyplot", "sklearn.manifold",
        "layers", "layers.Embed", "layers.SelfAttention_Family", "layers.Transformer_EncDec", "utils.masking",
        "reformer_pytorch")}
    try:
        # stubs for absent plotting deps pulled in by utils/shapelet_util.py:8-11
        for n in ("seaborn", "matplotlib", "matplotlib.colors", "matplotlib.pyplot"):
            sys.modules[n] = types.ModuleType(n)
        sys.modules["matplotlib.colors"].TABLEAU_COLORS = {"tab:blue": "#1f77b4"}
        sys.modules["matplotlib"].colors = sys.modules["matplotlib.colors"]
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
        util = _load("_ignref_shapelet_util", "utils/shapelet_util.py")
        upkg = types.ModuleType("utils")
        upkg.shapelet_util = util
        sys.modules["utils"] = upkg
        sys.modules["utils.shapelet_util"] = util
        shp = _load("_ignref_Shapelet", "model/Shapelet.py")
        fcn = _load("_ignref_FCN", "model/FullyConvNet.py")
        # InterpGN.py imports five deep experts; only FCN is needed for the oracle,
        # the others get inert placeholders (their layers need reformer_pytorch etc.).
        mpkg = types.ModuleType("models")
        sys.modules["models"] = mpkg
        sys.modules["models.Shapelet"] = shp
        sys.modules["models.FullyConvNet"] = fcn
        for n in ("PatchTST", "TimesNet", "ResNet"):
            ph = types.ModuleType("models." + n)
            ph.Model = type("Unavailable" + n, (), {})
            sys.modules["models." + n] = ph
        # the Transformer expert: its layers import reformer_pytorch (absent) for an unused attention variant
        rp = types.ModuleType("reformer_pytorch")
        rp.LSHSelfAttention = object
        sys.modules["reformer_pytorch"] = rp
        upkg.masking = _load("utils.masking", "utils/masking.py")
        lpkg = types.ModuleType("layers")
        sys.modules["layers"] = lpkg
        for n in ("Embed", "SelfAttention_Family", "Transformer_EncDec"):
            setattr(lpkg, n, _load("layers." + n, "layers/%s.py" % n))
        trf = _load("_ignref_Transformer", "model/Transformer.py")
        sys.modules["models.Transformer"] = trf
        ign = _load("_ignref_InterpGN", "model/InterpGN.py")
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    ns = types.SimpleNamespace(
        Shapelet=shp.Shapelet, DistThresholdShapelet=shp.DistThresholdShapelet,
        ShapeBottleneckModel=shp.ShapeBottleneckModel, DistThresholdSBM=shp.DistThresholdSBM,
        ShapeletDistanceFunc=shp.ShapeletDistanceFunc, pearson_corrcoef=shp.pearson_corrcoef,
        InterpGN=ign.InterpGN, FullyConvNetwork=fcn.FullyConvNetwork, Transformer=trf.Model,
        ModelInfo=util.ModelInfo)
    _cache["ns"] = ns
    return ns
