"""CPU: the pieces of the C-ABI contract test that need no GPU.

* the guard checker (tests/_util.py, Guarded) flags each way a kernel can break the memory contract;
* the grid of tests/test_abi_contract_gpu.py reaches every (family, entry point) cell and all six ring-kernel
  instantiations, by the host-only path and launch-count queries;
* every pointer of every entry point is refused with NFPB200_EALIGN one step below its documented alignment and
  accepted at it, and bad batch strides and workspaces are refused -- all before any CUDA call.  The descriptors of the
  alignment checks are invalid on purpose, so an accepted pointer ends in NFPB200_EINVAL, never in a launch.
"""
import ctypes
import re

import pytest
import torch

from neighbour_feature_pooling_b200 import _capi

import test_abi_contract_gpu as G
from _util import SENTINEL, Guarded, bits, fill_bits

EALIGN, EINVAL, EWORKSPACE = -7, -1, -4


# ---- the guard checker ----------------------------------------------------------------------------------------------
def _written_output(dtype=torch.float32, n=49, **kw):
    g = Guarded(n, dtype, "cpu", "output", **kw)
    if g.written is None:
        g.body.copy_(torch.arange(n, dtype=dtype))
    else:
        g.body[g.written] = 1.0
    return g


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_guard_checker_passes_a_clean_call(dtype):
    out = _written_output(dtype, n=49)   # 98 bytes in bf16: a body that is not a multiple of 16
    inp = Guarded(49, dtype, "cpu", "input", data=torch.randn(49), place=4)
    assert out.ptr() % 512 == 16 and inp.ptr() % 512 == 4
    assert out.lo >= 256 * 1024 and out.raw.numel() - out.hi >= 256 * 1024
    assert not out.problems("y") and not inp.problems("x")
    assert bool(torch.isnan(inp.raw[:inp.lo].view(dtype)).all()) and bool(torch.isnan(inp.raw[inp.hi:][:64].view(dtype)).all())
    want = torch.empty(1, dtype=dtype)
    fill_bits(want, SENTINEL[dtype])
    assert bool((bits(out.raw[:out.lo].view(dtype)) == bits(want)).all())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_guard_checker_flags_a_write_past_the_body(dtype):
    g = _written_output(dtype)
    g.raw[g.hi:g.hi + 2] = 0
    assert any("tail guard" in m for m in g.problems("y"))


def test_guard_checker_flags_a_write_before_the_body():
    g = _written_output()
    g.raw[g.lo - 16:g.lo] = 0
    assert any("lead guard" in m for m in g.problems("y"))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_guard_checker_flags_an_element_never_written(dtype):
    g = Guarded(49, dtype, "cpu", "output")
    g.body[:48] = 2.0
    assert any("never written" in m for m in g.problems("y"))


def test_guard_checker_flags_a_changed_input_byte():
    g = Guarded(49, torch.bfloat16, "cpu", "input", data=torch.randn(49))
    g.raw[g.lo + 5] ^= 1
    assert any("input body written" in m for m in g.problems("x"))
    h = Guarded(49, torch.float32, "cpu", "input", data=torch.randn(49), place=4)
    h.raw[h.lo - 1] ^= 1
    assert any("lead guard" in m for m in h.problems("x"))


def test_guard_checker_flags_a_write_between_nhwc_images():
    dense, stride, B = 7 * 7 * 8, 7 * 7 * 8 + 64, 3
    mask = torch.zeros((B - 1) * stride + dense, dtype=torch.bool)
    for b in range(B):
        mask[b * stride:b * stride + dense] = True
    g = _written_output(torch.bfloat16, n=mask.numel(), written=mask)
    assert not g.problems("gx")
    g.body[dense + 3] = 0.5   # in the gap after image 0
    assert any("outside the output" in m for m in g.problems("gx"))


def test_guard_checker_accepts_a_scribbled_workspace():
    w = Guarded(1000, torch.uint8, "cpu", "workspace")
    w.body.fill_(0)
    assert not w.problems("workspace")
    w.raw[w.hi] = 0
    assert w.problems("workspace")


# ---- the GPU grid reaches every cell --------------------------------------------------------------------------------
EXPECTED_ENTRIES = {
    "stream": set(G.ENTRIES), "token": set(G.ENTRIES), "split": set(G.ENTRIES[:6]), "generic": set(G.ENTRIES[:6]),
    "band": {"forward", "backward", "pooled_map_forward", "pooled_map_backward"}, "table": {"forward", "backward"},
}


def test_grid_reaches_every_cell():
    lib = _capi.load()
    seen = {}
    for c in G.GRID:
        p = G.Problem(c)
        path = p.path()
        assert path.startswith(G.FAMILIES[c.family][0]), (G.cell_id(c), path)
        assert p.launch_count() >= 1, G.cell_id(c)
        if p.head:
            assert lib.nfpb200_head_supported(ctypes.byref(p.desc)) == 0, G.cell_id(c)
        seen.setdefault(c.family, set()).add(c.entry)
    assert seen == EXPECTED_ENTRIES
    ids = [G.cell_id(c) for c in G.GRID]
    assert len(ids) == len(set(ids))
    # all six ring-kernel instantiations, in both dtypes, on every entry point
    inst = {(G.Problem(c).path(), c.dtype, c.entry) for c in G.GRID if c.family == "stream"}
    names = {re.sub(r"^fused/stream_", "", n) for n, _, _ in inst}
    assert names == {"7x7_r1", "7x7_r2", "14x14_r1", "14x14_r2", "2x2_r1", "4x4_r1"}, names
    for n in names:
        for dt in (torch.float32, torch.bfloat16):
            assert {e for m, d, e in inst if m.endswith(n) and d == dt} == set(G.ENTRIES), (n, dt)
    # the options the issue of each family needs
    opts = {(c.family, k, v) for c in G.GRID for k, v in c.opts}
    for want in [("stream", "hint", 1), ("stream", "yf32", 1), ("stream", "inner", 1), ("band", "inner", 1),
                 ("token", "inner", 1), ("token", "xbs", "vit"), ("token", "xbs", "pad8"), ("token", "gxbs", "pad64"),
                 ("token", "gxbs", "pad8"), ("generic", "measure", "attention"), ("generic", "measure", "scs"),
                 ("generic", "mode", "circular")]:
        assert want in opts, want
    # every x / gx batch stride pair on the token backward
    pairs = {(dict(c.opts)["xbs"], dict(c.opts)["gxbs"]) for c in G.GRID if c.family == "token" and c.entry == "backward"
             and c.shape == (3, 64, 14, 14, 1)}
    assert len(pairs) == 9
    # one stream-test case per (family, entry point)
    assert {(c.family, c.entry) for c in G.STREAM_CELLS} == {(f, e) for f, es in EXPECTED_ENTRIES.items() for e in es}


def test_grid_launch_counts_cover_multi_launch_paths():
    """The graph node count check is only worth something where a call issues more than one launch."""
    multi = {(c.family, c.entry) for c in G.GRID if G.Problem(c).launch_count() > 1}
    for want in [("stream", "pooled_map_backward"), ("token", "pooled_map_backward"), ("band", "pooled_map_forward"),
                 ("table", "forward"), ("table", "backward"), ("generic", "forward"), ("generic", "backward")]:
        assert want in multi, want


# ---- alignment and argument checks before any CUDA call ----------------------------------------------------------
# entry point -> its pointer arguments in order; "ws" is the workspace (followed by its size in the call)
SIGNATURES = {
    "forward": ("x", "y", "ws"),
    "backward": ("x", "gy", "gx", "ws"),
    "pool_forward": ("x", "gap_x", "gap_nfp", "ws"),
    "pool_backward": ("x", "g_gap_x", "g_gap_nfp", "gx", "ws"),
    "pooled_map_forward": ("x", "gap_nfp", "ws"),
    "pooled_map_backward": ("x", "g_gap_nfp", "gx", "ws"),
    "head_forward": ("x", "proj_w", "proj_b", "out", "gap_x", "gap_nfp"),
    "head_backward": ("x", "proj_w", "proj_b", "gap_x", "gap_nfp", "g_out", "gx"),
}
ALIGN = {n: 4 for n in G.F32_VECTORS}   # everything else: 16 bytes


def _call(entry, desc, ptrs):
    lib = _capi.load()
    args = []
    for n in SIGNATURES[entry]:
        args.append(ptrs[n])
        if n == "ws":
            args.append(1 << 20)
    args.append(None)   # stream
    return getattr(lib, f"nfpb200_{entry}")(ctypes.byref(desc), *args)


def _bad_desc():
    d = _capi.make_desc(_capi.F32, 2, 8, 7, 7, 1, 1, 1, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6)
    d.struct_bytes = 0   # invalid: an accepted pointer set returns NFPB200_EINVAL, nothing is launched
    return d


@pytest.mark.parametrize("entry", list(SIGNATURES))
def test_each_pointer_is_refused_below_its_alignment(entry):
    names = SIGNATURES[entry]
    base = {n: 0x7F0000000000 + 0x100000 * (i + 1) for i, n in enumerate(names)}
    assert _call(entry, _bad_desc(), base) == EINVAL
    for n in names:
        a = ALIGN.get(n, 16)
        at = dict(base, **{n: base[n] + a})           # exactly the documented alignment: accepted
        below = dict(base, **{n: base[n] + a // 2})   # one step below it: refused
        assert _call(entry, _bad_desc(), at) == EINVAL, (n, a)
        assert _call(entry, _bad_desc(), below) == EALIGN, (n, a)
    if "proj_b" in names:   # no bias
        assert _call(entry, _bad_desc(), dict(base, proj_b=None)) == EINVAL
    if "ws" in names:       # no workspace
        assert _call(entry, _bad_desc(), dict(base, ws=None)) == EINVAL


def test_header_documents_every_pointer_alignment():
    import os
    with open(os.path.join(G.ROOT, "include", "nfp_b200.h")) as f:
        header = f.read()
    for entry, names in SIGNATURES.items():
        # the last "Alignment:" sentence before the declaration (the head's block documents both directions)
        doc = header[:header.index(f"int nfpb200_{entry}(")].rsplit("Alignment:", 1)[1].split("*/")[0]
        for n in names:
            word = "workspace" if n == "ws" else n
            a = ALIGN.get(n, 16)
            assert re.search(rf"\b{word}\b[^;.]*?{a} bytes", doc), (entry, n, doc)
    assert "nothing is written between images" in header


def _token_desc(**kw):
    return _capi.make_desc(_capi.BF16, 3, 64, 14, 14, 1, 1, 1, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6,
                           layout=_capi.LAYOUT_NHWC, **kw)


def test_bad_batch_strides():
    lib = _capi.load()
    n = ctypes.c_size_t()
    dense = 14 * 14 * 64
    for kw, rc in [(dict(gx_batch_stride=dense - 8), EINVAL), (dict(gx_batch_stride=dense + 4), EALIGN),
                   (dict(gx_batch_stride=-8), EINVAL), (dict(x_batch_stride=dense - 8), EINVAL),
                   (dict(x_batch_stride=197 * 64 + 2), EALIGN), (dict(gx_batch_stride=dense + 8), 0),
                   (dict(x_batch_stride=197 * 64, gx_batch_stride=dense + 64), 0)]:
        assert lib.nfpb200_workspace_bytes(ctypes.byref(_token_desc(**kw)), _capi.OP_BACKWARD, ctypes.byref(n)) == rc, kw
    # refused by the compute entry points too, before any CUDA call
    p = 0x7F0000100000
    assert lib.nfpb200_backward(ctypes.byref(_token_desc(gx_batch_stride=dense + 4)), p, p, p, None, 0, None) == EALIGN
    assert lib.nfpb200_backward(ctypes.byref(_token_desc(gx_batch_stride=dense - 8)), p, p, p, None, 0, None) == EINVAL


def test_workspace_missing_or_short():
    """NFPB200_EWORKSPACE comes from the host-only checks, before the device is queried."""
    lib = _capi.load()
    d = _capi.make_desc(_capi.F32, 3, 5, 9, 11, 1, 1, 1, 1, "reflect", "attention", True, False, 1e-6, 1, 1e-6)
    need = _capi.workspace_bytes(d, _capi.OP_BACKWARD)
    assert need > 0
    p = 0x7F0000100000
    assert lib.nfpb200_backward(ctypes.byref(d), p, p, p, None, need, None) == EWORKSPACE
    assert lib.nfpb200_backward(ctypes.byref(d), p, p, p, p + 0x100000, need - 1, None) == EWORKSPACE
    pm = _capi.make_desc(_capi.F32, 3, 64, 7, 7, 1, 1, 1, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6)
    assert _capi.workspace_bytes(pm, _capi.OP_POOLED_MAP_BACKWARD) >= 3 * 64 * 4   # the zero g_gap_x rows
    assert lib.nfpb200_pooled_map_backward(ctypes.byref(pm), p, p, p, None, 0, None) == EWORKSPACE


def test_x_pointer_is_image_zero_for_every_batch_stride():
    """The pointer the GPU tests pass as x is image 0's first pixel, and image b starts x_batch_stride elements on,
    also in the ViT token view, where the buffer starts one (class) token earlier."""
    for c in G.GRID:
        if c.family != "token" or c.entry != "forward":
            continue
        p = G.Problem(c)
        flat = p.inputs["x"][0].to(c.dtype)   # as the kernels get it
        bufs = {"x": flat}
        off = (G._ptrs(p, bufs)["x"] - flat.data_ptr()) // flat.element_size()
        stride = p.xbs or p.H * p.W * p.C
        for b in range(p.B):
            img = flat[off + b * stride:off + b * stride + p.H * p.W * p.C].view(p.H, p.W, p.C).permute(2, 0, 1)
            assert torch.equal(img.double(), p.x[b]), (G.cell_id(c), b)
        assert bool(torch.isnan(flat[:off]).all()), G.cell_id(c)   # the class token (vit) is NaN
