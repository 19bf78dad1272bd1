"""CPU: the host side of the second-order entry points (nfpb200_jvp, nfpb200_backward_backward).

Symbols and op codes (7, 8) through the query entry points, the problems they refuse, and each pointer refused with
NFPB200_EALIGN one step below its documented alignment -- all before any CUDA call (invalid descriptors on purpose:
an accepted pointer set ends in NFPB200_EINVAL, never in a launch).
"""
import ctypes
import os
import re

import pytest

from neighbour_feature_pooling_b200 import _capi

EALIGN, EINVAL, EUNSUPPORTED, EWORKSPACE = -7, -1, -5, -4
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _desc(dtype=_capi.F32, B=2, C=8, H=7, W=7, R=1, stride=1, padding=1, dilation=1, mode="reflect",
          measure="cosine", **kw):
    return _capi.make_desc(dtype, B, C, H, W, R, stride, padding, dilation, mode, measure, True, False, 1e-6, 1, 1e-6,
                           **kw)


def test_symbols_and_op_codes():
    lib = _capi.load()
    assert hasattr(lib, "nfpb200_jvp") and hasattr(lib, "nfpb200_backward_backward")
    assert "nfpb200_jvp" in _capi.EXPORTS and "nfpb200_backward_backward" in _capi.EXPORTS
    assert (_capi.OP_JVP, _capi.OP_BACKWARD_BACKWARD) == (7, 8)
    assert (_capi.JVP_FORWARD_AD, _capi.JVP_REVERSE) == (0, 1)
    assert lib.nfpb200_abi_version() == 5


@pytest.mark.parametrize("dtype", [_capi.F32, _capi.BF16, _capi.F16])
@pytest.mark.parametrize("geom", [dict(), dict(R=2, padding=2), dict(stride=2, dilation=2, padding=0, H=11, W=9),
                                  dict(mode="circular"), dict(mode="zeros", padding=3), dict(H=112, W=112, C=16)])
def test_queries(dtype, geom):
    for path in ("auto", "generic", "fused"):
        d = _desc(dtype, path=path, **geom)
        assert _capi.describe_path(d, _capi.OP_JVP) == "second/jvp"
        assert _capi.describe_path(d, _capi.OP_BACKWARD_BACKWARD) == "second/pairs"
        assert _capi.launch_count(d, _capi.OP_JVP) == 1
        assert _capi.launch_count(d, _capi.OP_BACKWARD_BACKWARD) == 2
        assert _capi.workspace_bytes(d, _capi.OP_JVP) == 0
        Ho, Wo = _capi.output_shape(d)
        K = (2 * d.R + 1) ** 2 - 1
        n = _capi.workspace_bytes(d, _capi.OP_BACKWARD_BACKWARD)
        assert n >= 6 * 4 * d.B * K * Ho * Wo and n % 256 == 0


def test_unsupported_problems():
    lib = _capi.load()
    n = ctypes.c_size_t()
    buf = ctypes.create_string_buffer(64)
    k = ctypes.c_int32()
    for d in (_desc(measure="norm"), _desc(measure="dot"), _desc(dtype=_capi.BF16, layout=_capi.LAYOUT_NHWC),
              _desc(R=2, padding=2, inner_R=1)):
        for op in (_capi.OP_JVP, _capi.OP_BACKWARD_BACKWARD):
            assert lib.nfpb200_workspace_bytes(ctypes.byref(d), op, ctypes.byref(n)) == EUNSUPPORTED
            assert lib.nfpb200_describe_path(ctypes.byref(d), op, buf, 64) == EUNSUPPORTED
            assert lib.nfpb200_launch_count(ctypes.byref(d), op, ctypes.byref(k)) == EUNSUPPORTED
        p = 0x7F0000100000
        assert lib.nfpb200_jvp(ctypes.byref(d), p, p, p, _capi.JVP_REVERSE, None, 0, None) == EUNSUPPORTED
        assert lib.nfpb200_backward_backward(ctypes.byref(d), p, p, p, p, None, 0, None) == EUNSUPPORTED
    for op in (6, 9):
        assert lib.nfpb200_workspace_bytes(ctypes.byref(_desc()), op, ctypes.byref(n)) == EINVAL
        assert lib.nfpb200_launch_count(ctypes.byref(_desc()), op, ctypes.byref(k)) == EINVAL


def test_unknown_rule_and_missing_workspace():
    lib = _capi.load()
    p = 0x7F0000100000
    for rule in (-1, 2, 7):
        assert lib.nfpb200_jvp(ctypes.byref(_desc()), p, p, p, rule, None, 0, None) == EINVAL
    d = _desc()
    need = _capi.workspace_bytes(d, _capi.OP_BACKWARD_BACKWARD)
    assert lib.nfpb200_backward_backward(ctypes.byref(d), p, p, p, p, None, need, None) == EWORKSPACE
    assert lib.nfpb200_backward_backward(ctypes.byref(d), p, p, p, p, p + 0x100000, need - 1, None) == EWORKSPACE
    assert lib.nfpb200_jvp(ctypes.byref(d), None, p, p, _capi.JVP_REVERSE, None, 0, None) == EINVAL
    assert lib.nfpb200_backward_backward(ctypes.byref(d), p, p, None, p, p, need, None) == EINVAL


SIGNATURES = {"jvp": ("x", "v", "ydot", "ws"), "backward_backward": ("x", "gy", "v", "gx2", "ws")}


def _call(entry, desc, ptrs):
    args = []
    for n in SIGNATURES[entry]:
        args.append(ptrs[n])
        if n == "ws":
            args.append(1 << 20)
        if entry == "jvp" and n == "ydot":
            args.append(_capi.JVP_REVERSE)
    return getattr(_capi.load(), f"nfpb200_{entry}")(ctypes.byref(desc), *args, None)


@pytest.mark.parametrize("entry", list(SIGNATURES))
def test_each_pointer_is_refused_below_its_alignment(entry):
    bad = _desc()
    bad.struct_bytes = 0
    names = SIGNATURES[entry]
    base = {n: 0x7F0000000000 + 0x100000 * (i + 1) for i, n in enumerate(names)}
    assert _call(entry, bad, base) == EINVAL
    for n in names:
        assert _call(entry, bad, dict(base, **{n: base[n] + 16})) == EINVAL, n
        assert _call(entry, bad, dict(base, **{n: base[n] + 8})) == EALIGN, n


def test_header_documents_every_pointer_alignment():
    with open(os.path.join(ROOT, "include", "nfp_b200.h")) as f:
        header = f.read()
    for entry, names in SIGNATURES.items():
        doc = header[:header.index(f"int nfpb200_{entry}(")].rsplit("Alignment:", 1)[1].split("*/")[0]
        for n in names:
            word = "workspace" if n == "ws" else n
            assert re.search(rf"\b{word}\b[^;.]*?16 bytes", doc), (entry, n, doc)
    for name in ("NFPB200_OP_JVP = 7", "NFPB200_OP_BACKWARD_BACKWARD = 8", "NFPB200_JVP_FORWARD_AD = 0",
                 "NFPB200_JVP_REVERSE = 1"):
        assert name in header
