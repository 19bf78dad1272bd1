"""B200-native Neighbourhood Feature Pooling (NFP).

Hand-written sm_100a CUDA kernels behind a C ABI (``include/nfp_b200.h``,
``lib/libnfp_b200.so``) and, above it, drop-in ``nn.Module`` classes with the
reference's interfaces:

    from neighbour_feature_pooling_b200 import NFPPooling, nfp_pooling

or, to run the reference's own model zoo / heads unchanged:

    import neighbour_feature_pooling_b200 as nfpb
    nfpb.install_dropin()            # before `import models.texture_pooling`
    from models.NFP_Pooling import nfp_pooling   # -> the B200 implementation

There is no CPU or PyTorch fallback: without the built library every op raises.
"""
from __future__ import annotations

import sys
import types

from . import _capi, functional
from .functional import NFPConfig, nfp_gap_pair, nfp_multi_radius, nfp_pooled_similarity, nfp_similarity
from .modules import (EnhancedNFPPooling, MultiRadiusNFP, NFPPooling, fuse_multi_radius, fuse_pooled_nfp, nfp_pooling,
                      unfuse_multi_radius, unfuse_pooled_nfp)

__version__ = "0.1.0"

# the reference import paths this package can stand in for (SURVEY.md section 8 row b1)
_DROPIN_MODULES = {
    "models.pooling.nfp": {"NFPPooling": NFPPooling},                      # models/pooling/nfp.py
    "models.NFP_Pooling": {"nfp_pooling": nfp_pooling, "NFPPooling": NFPPooling},  # models/NFP_Pooling.py
    "models.pooling.enhanced_nfp": {"EnhancedNFPPooling": EnhancedNFPPooling},     # missing upstream
}


def install_dropin(force: bool = True):
    """Register this implementation under the reference's import paths.

    Only the three leaf modules are injected into ``sys.modules``; the rest of
    the reference's ``models`` package (``texture_pooling``, ``nfp_heads``,
    ``resnet18`` ...) is imported from wherever it lives on ``sys.path`` and
    picks these up through its own ``from models.pooling.nfp import NFPPooling``
    statements.  Returns the list of module names installed."""
    done = []
    for name, symbols in _DROPIN_MODULES.items():
        if name in sys.modules and not force:
            continue
        mod = types.ModuleType(name)
        mod.__doc__ = f"neighbour_feature_pooling_b200 drop-in for the reference module {name}"
        mod.__dict__.update(symbols)
        mod.__nfpb200_dropin__ = True
        sys.modules[name] = mod
        done.append(name)
    return done


def uninstall_dropin():
    for name in _DROPIN_MODULES:
        mod = sys.modules.get(name)
        if mod is not None and getattr(mod, "__nfpb200_dropin__", False):
            del sys.modules[name]


def library_path() -> str:
    return _capi.library_path()


__all__ = ["NFPPooling", "EnhancedNFPPooling", "nfp_pooling", "NFPConfig", "nfp_similarity", "nfp_gap_pair",
           "nfp_multi_radius", "nfp_pooled_similarity", "MultiRadiusNFP", "fuse_multi_radius", "unfuse_multi_radius",
           "fuse_pooled_nfp", "unfuse_pooled_nfp",
           "install_dropin", "uninstall_dropin", "library_path", "functional"]
