"""TEST INFRASTRUCTURE ONLY -- import the *unmodified* reference modules.

The original Neighbour_Feature_Pooling project is not part of this repository.
It is read from the checkout named by ``NFP_REFERENCE_ROOT``, else from a copy
of its files inside the tree (git-ignored): ``oracle/_ref/``, where
``__graft_entry__.build()`` stages them, or ``baseline/_ref/``, where earlier
builds did.  Such a copy travels with the working tree to a machine that has no
checkout.  The reference imports ``matplotlib.pyplot`` without using it
(``models/pooling/nfp.py:12``); if that package is not installed, an empty stub
is injected before import.
"""
from __future__ import annotations

import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGED_ROOTS = (os.path.join(_REPO, "oracle", "_ref"), os.path.join(_REPO, "baseline", "_ref"))
# the operator files, and the heads module that tests/test_modules_contract.py runs on the drop-in
OPERATOR_FILES = ("models/__init__.py", "models/pooling/nfp.py", "models/NFP_Pooling.py", "models/nfp_heads.py")


def _has_reference(root: str) -> bool:
    return bool(root) and os.path.isfile(os.path.join(root, "models", "pooling", "nfp.py"))


REFERENCE_ROOT = os.environ.get("NFP_REFERENCE_ROOT") or next(
    (r for r in STAGED_ROOTS if _has_reference(r)), STAGED_ROOTS[0])


def reference_available() -> bool:
    return _has_reference(REFERENCE_ROOT)


def stage_reference(src_root: str = os.environ.get("NFP_REFERENCE_ROOT", "")) -> bool:
    """Copy OPERATOR_FILES, unmodified, from the checkout `src_root` to oracle/_ref/ so that bench.py's CPU arm and the
    reference tests can use them where that checkout is absent.  Returns whether a copy is in the tree."""
    import shutil
    if _has_reference(src_root) and os.path.abspath(src_root) != STAGED_ROOTS[0]:
        for rel in OPERATOR_FILES:
            src, dst = os.path.join(src_root, rel), os.path.join(STAGED_ROOTS[0], rel)
            os.makedirs(os.path.dirname(dst), exist_ok=True)
            if os.path.isfile(src):
                shutil.copyfile(src, dst)
            elif rel.endswith("__init__.py"):
                open(dst, "w").close()
    return any(_has_reference(r) for r in STAGED_ROOTS)


def load_reference():
    """Return ``(NFPPooling, nfp_pooling)`` classes of the reference."""
    if not reference_available():
        raise RuntimeError(f"reference not found at {REFERENCE_ROOT} (set NFP_REFERENCE_ROOT to a checkout of it)")
    for name in ("matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            try:
                __import__(name)
            except ImportError:
                sys.modules[name] = types.ModuleType(name)
    if getattr(sys.modules.get("matplotlib"), "pyplot", None) is None:
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    # The drop-in package may have registered itself under the reference's import
    # paths (neighbour_feature_pooling_b200.install_dropin); make sure we get the
    # real reference here.
    saved = {k: sys.modules.pop(k) for k in list(sys.modules)
             if k == "models" or k.startswith("models.")}
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        from models.pooling.nfp import NFPPooling  # type: ignore
        from models.NFP_Pooling import nfp_pooling  # type: ignore
    finally:
        sys.path.remove(REFERENCE_ROOT)
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
            sys.modules.pop(k)
        sys.modules.update(saved)
    return NFPPooling, nfp_pooling
