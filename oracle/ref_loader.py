"""Import the UNMODIFIED reference tokenizer from a checkout of the original project: oracle/_ref/ (git-ignored,
not part of this repository) or the directory named by P3TOK_REFERENCE_ROOT.

TEST INFRASTRUCTURE - not product code.  Only `tests/`, `tests/golden/make_golden.py`
and ad-hoc probes may use this.  Where there is no checkout nothing may call `load()`;
use `available()` to gate.

The reference package imports `timm` and `h5py` at package-import time
(src/models/__init__.py:1 -> vit.py:1, src/data/__init__.py:1 -> scanobjectnn.py:2);
neither is installed in this image and neither is touched by the tokenizer classes,
so they are replaced with inert stub modules before import.
"""
import os
import sys
import types

REF_ROOT = os.environ.get("P3TOK_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "src", "models", "apf.py"))


def _install_stubs():
    import torch.nn as nn

    def _mod(name, **attrs):
        m = sys.modules.get(name)
        if m is None:
            m = types.ModuleType(name)
            sys.modules[name] = m
        for k, v in attrs.items():
            setattr(m, k, v)
        return m

    class DropPath(nn.Module):
        def __init__(self, p=0.0):
            super().__init__()

        def forward(self, x):
            return x

    class Mlp(nn.Module):
        def __init__(self, in_features, hidden_features=None, out_features=None, **kw):
            super().__init__()
            hidden_features = hidden_features or in_features
            out_features = out_features or in_features
            self.fc1 = nn.Linear(in_features, hidden_features)
            self.act = nn.GELU()
            self.fc2 = nn.Linear(hidden_features, out_features)

        def forward(self, x):
            return self.fc2(self.act(self.fc1(x)))

    def _no_timm(*a, **k):
        raise RuntimeError("timm is not installed in this image (stub)")

    try:
        import timm  # noqa: F401
    except Exception:
        _mod("timm", create_model=_no_timm)
        _mod("timm.models")
        _mod("timm.models.layers", DropPath=DropPath, Mlp=Mlp)
        _mod("timm.scheduler", CosineLRScheduler=object)
    try:
        import h5py  # noqa: F401
    except Exception:
        _mod("h5py")


_cache = None


def load():
    """Returns a namespace with the reference's hot-path callables."""
    global _cache
    if _cache is not None:
        return _cache
    if not available():
        raise FileNotFoundError(f"reference tree not found at {REF_ROOT}")
    _install_stubs()
    src = os.path.join(REF_ROOT, "src")
    if src not in sys.path:
        sys.path.insert(0, src)
    import models.apf as apf
    import models.pix4point as p4p
    import models.apf_utils as apf_utils
    import data.sampler as sampler

    ns = types.SimpleNamespace(
        apf=apf, p4p=p4p, apf_utils=apf_utils, sampler=sampler,
        furthest_point_sample=sampler.furthest_point_sample,
        fps=sampler.fps,
        knn_point=sampler.knn_point,
        square_distance=sampler._square_distance,
        index_points=sampler.index_points,
        farthest_point_sampling=p4p.farthest_point_sampling,
        group_knn=p4p.group_knn,
        Group=apf.Group, Encoder=apf.Encoder, PointNet=apf.PointNet,
        P3Embed=p4p.P3Embed,
        MortonEncoder=apf_utils.MortonEncoder,
    )
    _cache = ns
    return ns
