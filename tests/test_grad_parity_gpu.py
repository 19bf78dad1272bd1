"""GPU: input-gradient parity of every cosine kernel family against the fp64 oracle, with nothing masked.

Grid: kernel family x padding mode {reflect, zeros, replicate} x similarity {sim, dist} x dtype {fp32, bf16} (the
tensor-core token kernels: bf16 channels-last only).  Every case runs two inputs:

* clean -- randn (ReLU'd for some channel counts), no pixel norm below 0.1;
* degenerate -- one image entirely zero, and pixels of norm {0, 1e-9, 0.5 eps, 0.99 eps, 1.01 eps, 4 eps} at the four
  corners, on each edge and in the interior (two adjacent sub-eps pixels there), in the first and the last image.

y, pooled vectors and projection gradients are scored with rel_err; input gradients with grad_errs (tests/_util.py):
each image and each pixel-norm region on its own scale, so the 1e6-sized gradients of the degenerate pixels cannot
hide an error anywhere else.  Each case asserts the kernel path it ran, so a dispatch change cannot move it to another
kernel unnoticed.  tests/test_grad_metric.py checks on the CPU that this grid reaches every cell, and that grad_errs
flags the kernel bugs this file is meant to catch.
"""
import ctypes
from collections import namedtuple

import numpy as np
import pytest
import torch

import neighbour_feature_pooling_b200 as nfpb
from neighbour_feature_pooling_b200 import NFPPooling, _capi, functional as NF, nfp_pooling
from oracle import nfp_oracle as O

from _util import REGION_NAMES, grad_errs, rel_err, worst

pytestmark = pytest.mark.gpu

EPS = 1e-6
TOL = {torch.float32: 1e-5, torch.bfloat16: 2e-2}
MODES = ("reflect", "zeros", "replicate")
SIMS = (True, False)
BOTH = (torch.float32, torch.bfloat16)
BF16 = (torch.bfloat16,)
DEG_NORMS = (0.0, 1e-9, 0.5 * EPS, 0.99 * EPS, 1.01 * EPS, 4 * EPS)
KINDS = ("clean", "degenerate")

# family -> (path prefix, layout, cfg.path)
FAMILIES = {
    "stream": ("fused/stream_", _capi.LAYOUT_NCHW, "auto"),
    "split": ("fused/split_", _capi.LAYOUT_NCHW, "split"),
    "band": ("planar/band", _capi.LAYOUT_NCHW, "auto"),
    "table": ("planar/table", _capi.LAYOUT_NCHW, "auto"),
    "token": ("fused/token_", _capi.LAYOUT_NHWC, "auto"),
}
# op: "map" (nfp_similarity), "pooled" (nfp_gap_pair), "head" (nfp_pooling, one launch each way),
#     "multi" (radii 1 + 2 in one launch; shape R is the outer radius)
Case = namedtuple("Case", "family op shape mode sim dtype")

STREAM_SHAPES = [(5, 64, 7, 7, 1), (3, 512, 7, 7, 2), (3, 256, 14, 14, 1), (6, 512, 2, 2, 1), (300, 16, 7, 7, 1),
                 (300, 512, 7, 7, 1)]   # more images than resident CTAs at full width: the resident-image backward
SPLIT_SHAPES = STREAM_SHAPES[:-1]
BAND_SHAPES = [(2, 16, 112, 112, 1), (2, 24, 56, 56, 1), (1, 4, 5, 8, 2), (2, 8, 4, 12, 1)]
TABLE_SHAPES = [(3, 33, 7, 7, 1), (2, 5, 3, 3, 1), (2, 10, 5, 9, 2)]
TOKEN_SHAPES = [(5, 64, 7, 7, 1), (3, 128, 7, 7, 2), (2, 64, 14, 14, 2), (300, 64, 7, 7, 1)]
HEAD_SHAPES = [(5, 64, 7, 7, 1), (3, 128, 7, 7, 2)]
MULTI_SHAPES = {"stream": (3, 512, 7, 7, 2), "band": (2, 16, 28, 28, 2), "token": (5, 64, 7, 7, 2)}


def _cases(family, op, shapes, dtypes):
    return [Case(family, op, s, m, sim, dt) for s in shapes for m in MODES for sim in SIMS for dt in dtypes]


GRID = (_cases("stream", "map", STREAM_SHAPES, BOTH) + _cases("split", "map", SPLIT_SHAPES, BOTH)
        + _cases("stream", "pooled", SPLIT_SHAPES, BOTH) + _cases("split", "pooled", SPLIT_SHAPES, BOTH)
        + _cases("band", "map", BAND_SHAPES, BOTH) + _cases("table", "map", TABLE_SHAPES, BOTH)
        + _cases("token", "map", TOKEN_SHAPES, BF16) + _cases("token", "pooled", TOKEN_SHAPES, BF16)
        + _cases("stream", "head", HEAD_SHAPES, BOTH) + _cases("token", "head", HEAD_SHAPES, BF16)
        + [c for f, s in MULTI_SHAPES.items() for c in _cases(f, "multi", [s], BF16 if f == "token" else BOTH)])


def case_id(c):
    dt = "fp32" if c.dtype == torch.float32 else "bf16"
    return f'{c.family}-{c.op}-{"x".join(map(str, c.shape[:4]))}_r{c.shape[4]}-{c.mode}-{"sim" if c.sim else "dist"}-{dt}'


def case_cfg(c):
    B, C, H, W, R = c.shape
    return NF.replace(NFPPooling(C, R=R, measure="cosine", padding=R, padding_mode=c.mode, similarity=c.sim).config,
                      path=FAMILIES[c.family][2])


def case_paths(c):
    """Host-only: the kernel path each launch of the case takes, from nfpb200_describe_path (no GPU needed)."""
    B, C, H, W, R = c.shape
    cfg = case_cfg(c)
    desc = _capi.make_desc(_capi.F32 if c.dtype == torch.float32 else _capi.BF16, B, C, H, W, R, 1, R, 1, c.mode,
                           "cosine", c.sim, False, EPS, 1, 1e-6, cfg.path, layout=FAMILIES[c.family][1],
                           inner_R=1 if c.op == "multi" else 0)
    if c.op == "head" and _capi.load().nfpb200_head_supported(ctypes.byref(desc)) != 0:
        return ["head not supported"]
    ops = (_capi.OP_FORWARD, _capi.OP_BACKWARD) if c.op in ("map", "multi") else \
        (_capi.OP_POOL_FORWARD, _capi.OP_POOL_BACKWARD)
    return [_capi.describe_path(desc, op) for op in ops]


def make_inputs(kind, shape, dtype, seed):
    """(x, rows): x as the kernels see it (bf16-rounded for bf16) and the images the oracle is run on."""
    B, C, H, W, R = shape
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, H, W, generator=gen)
    if C % 3 == 0 or C % 128 == 0:
        x = x.relu()
    r = torch.randn(B, C, H, W, generator=gen).abs()
    low = x.norm(dim=1, keepdim=True) < 0.1   # clean: no pixel norm below 0.1
    x = torch.where(low, 0.5 * r / r.norm(dim=1, keepdim=True), x)
    if kind == "degenerate":
        x0 = x.clone()   # the direction of every planted pixel (spots coincide on the smallest maps)
        zero = B - 2 if B >= 3 else (1 if B == 2 else None)
        imgs = [b for b in dict.fromkeys((0, B - 1)) if b != zero]
        if zero is not None:
            x[zero] = 0.0
        h2, w2 = H // 2, W // 2
        spots = [(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1),            # corners
                 (0, w2), (H - 1, w2), (h2, 0), (h2, W - 1)]                 # edges
        for j, b in enumerate(imgs):
            norms = [DEG_NORMS[(i + 3 * j) % len(DEG_NORMS)] for i in range(len(spots))]
            # the interior: two adjacent sub-eps pixels (on maps this small they may land on an edge)
            spots_b = spots + [(h2, w2), (h2, max(w2 - 1, 0))]
            norms += [0.5 * EPS, 0.99 * EPS] if j == 0 else [1e-9, 0.0]
            for (h, w), nv in zip(spots_b, norms):
                v = x0[b, :, h, w]
                x[b, :, h, w] = v * (nv / v.norm())
    if dtype == torch.bfloat16:
        x = x.bfloat16().float()
    rows = list(range(B)) if B <= 32 else [0, 1] + list(range(B - 4, B))   # the resident-image loop: first and last
    return x, rows


def _to_device(x, c, dev):
    xd = x.to(dev, c.dtype)
    if FAMILIES[c.family][1] == _capi.LAYOUT_NHWC:
        xd = xd.contiguous(memory_format=torch.channels_last)
    return xd.requires_grad_(True)


def _traced(fn):
    NF.PATH_TRACE = set()
    try:
        out = fn()
        return out, set(NF.PATH_TRACE)
    finally:
        NF.PATH_TRACE = None


def _check_gx(got, want, x, c, kind, record):
    errs = grad_errs(got, want, x)
    for name in REGION_NAMES:
        vals = [e for (b, r), e in errs.items() if r == name]
        if vals:
            record(f"gx_{kind}_{name}", f"{max(vals):.3e}")
    assert max(errs.values()) < TOL[c.dtype], (kind, worst(errs))


def _gap_ref(x, g1, g2, R, mode, sim):
    """GAP(x), GAP(NFP(x)) and the input gradient of <g1, GAP(x)> + <g2, GAP(NFP(x))>, fp64 oracle."""
    B, C, H, W = x.shape
    K = g2.shape[1]
    gy = (g2.double() / (H * W))[:, :, None, None].expand(B, K, H, W).contiguous()
    y_map, gx_map = O.nfp_forward_backward(x.double(), gy, R=R, measure="cosine", padding=R, padding_mode=mode,
                                           similarity=sim)
    gx = torch.as_tensor(np.asarray(gx_map)) + (g1.double() / (H * W))[:, :, None, None]
    return x.double().mean((2, 3)), torch.as_tensor(np.asarray(y_map)).mean((2, 3)), gx


def _multi_ref(x, g, mode, sim):
    """cat([NFP_1(x), NFP_2(x)], dim=1) and its input gradient, layer by layer as the reference composes them."""
    kw = dict(measure="cosine", padding_mode=mode, similarity=sim)
    y1, gx1 = O.nfp_forward_backward(x.double(), g[:, :8].double().contiguous(), R=1, padding=1, **kw)
    y2, gx2 = O.nfp_forward_backward(x.double(), g[:, 8:].double().contiguous(), R=2, padding=2, **kw)
    return torch.cat([torch.as_tensor(np.asarray(y1)), torch.as_tensor(np.asarray(y2))], dim=1), \
        torch.as_tensor(np.asarray(gx1)) + torch.as_tensor(np.asarray(gx2))


def _seed(c, kind):
    B, C, H, W, R = c.shape
    return 7919 * B + 131 * C + 17 * H + W + R + MODES.index(c.mode) + 3 * c.sim + 5 * KINDS.index(kind)


def _check_trace(c, trace, what):
    prefix = FAMILIES[c.family][0]
    assert trace and all(t.startswith(prefix) and what in t for t in trace), (c, trace)


def _case_params(op):
    return [pytest.param(c, id=case_id(c)) for c in GRID if c.op == op]


@pytest.mark.parametrize("c", _case_params("map"))
def test_map_gradient(c, cuda_device, record_property):
    """nfp_similarity forward and backward: y and d y / d x."""
    B, C, H, W, R = c.shape
    K = (2 * R + 1) ** 2 - 1
    paths = case_paths(c)
    assert all(p.startswith(FAMILIES[c.family][0]) for p in paths), paths
    cfg = case_cfg(c)
    tol = TOL[c.dtype]
    for kind in KINDS:
        x, rows = make_inputs(kind, c.shape, c.dtype, _seed(c, kind))
        gen = torch.Generator().manual_seed(_seed(c, kind) + 1)
        g = torch.randn(B, K, H, W, generator=gen).to(c.dtype).float()
        y_ref, gx_ref = O.nfp_forward_backward(x[rows].double(), g[rows].double(), R=R, measure="cosine", padding=R,
                                               padding_mode=c.mode, similarity=c.sim)
        xd = _to_device(x, c, cuda_device)
        y, trace = _traced(lambda: NF.nfp_similarity(xd, cfg))
        _check_trace(c, trace, "map")
        y.backward(g.to(cuda_device, y.dtype))
        assert rel_err(y.detach().float().cpu()[rows], y_ref) < tol, kind
        _check_gx(xd.grad.float().cpu()[rows], gx_ref, x[rows], c, kind, record_property)


@pytest.mark.parametrize("c", _case_params("pooled"))
def test_pooled_gradient(c, cuda_device, record_property):
    """nfp_gap_pair (nfpb200_pool_forward / _backward): GAP(x), GAP(NFP(x)) and the input gradient."""
    B, C, H, W, R = c.shape
    K = (2 * R + 1) ** 2 - 1
    paths = case_paths(c)
    assert all(p.startswith(FAMILIES[c.family][0]) for p in paths), paths
    cfg = case_cfg(c)
    tol = TOL[c.dtype]
    for kind in KINDS:
        x, rows = make_inputs(kind, c.shape, c.dtype, _seed(c, kind))
        gen = torch.Generator().manual_seed(_seed(c, kind) + 2)
        g1, g2 = torch.randn(B, C, generator=gen), torch.randn(B, K, generator=gen)
        gap_x_ref, gap_n_ref, gx_ref = _gap_ref(x[rows], g1[rows], g2[rows], R, c.mode, c.sim)
        xd = _to_device(x, c, cuda_device)
        (a, n), trace = _traced(lambda: NF.nfp_gap_pair(xd, cfg))
        _check_trace(c, trace, "pooled head")
        ((a.float() * g1.to(cuda_device)).sum() + (n.float() * g2.to(cuda_device)).sum()).backward()
        assert rel_err(a.detach().float().cpu()[rows], gap_x_ref) < tol, kind
        assert rel_err(n.detach().float().cpu()[rows], gap_n_ref) < tol, kind
        _check_gx(xd.grad.float().cpu()[rows], gx_ref, x[rows], c, kind, record_property)


@pytest.mark.parametrize("c", _case_params("head"))
def test_head_gradient(c, cuda_device, record_property):
    """The fused nfp_pooling head, GAP(x) * (W GAP(NFP(x)) + b): output, and the gradients of x, W and b."""
    B, C, H, W, R = c.shape
    paths = case_paths(c)
    assert all(p.startswith(FAMILIES[c.family][0]) for p in paths), paths
    tol = TOL[c.dtype]
    params = {"num_ftrs": {"m": C}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 3}}
    layer = NFPPooling(C, R=R, measure="cosine", padding=R, padding_mode=c.mode, similarity=c.sim)
    torch.manual_seed(_seed(c, "clean"))
    head = nfp_pooling(nfp_layer=layer, Params=params).to(cuda_device)
    Wp, bp = head.nfp_proj.weight.detach().cpu().double(), head.nfp_proj.bias.detach().cpu().double()
    for kind in KINDS:
        x, rows = make_inputs(kind, c.shape, c.dtype, _seed(c, kind))
        g = torch.randn(B, C, generator=torch.Generator().manual_seed(_seed(c, kind) + 3))
        xr = x.double()
        y_map = torch.as_tensor(np.asarray(O.nfp_forward(xr, R=R, measure="cosine", padding=R, padding_mode=c.mode,
                                                         similarity=c.sim)))
        gap_n, gap_x = y_map.mean((2, 3)), xr.mean((2, 3))
        proj = gap_n @ Wp.t() + bp
        t = g.double() * gap_x
        _, _, gx_ref = _gap_ref(x, g.double() * proj, t @ Wp, R, c.mode, c.sim)
        head.zero_grad()
        xd = _to_device(x, c, cuda_device)
        out, trace = _traced(lambda: head(xd))
        assert len(trace) == 1 and "fused head" in next(iter(trace)), trace
        _check_trace(c, trace, "fused head")
        out.backward(g.to(cuda_device, out.dtype))
        assert rel_err(out.detach().float().cpu(), gap_x * proj) < tol, kind
        assert rel_err(head.nfp_proj.weight.grad.cpu(), t.t() @ gap_n) < tol, kind
        assert rel_err(head.nfp_proj.bias.grad.cpu(), t.sum(0)) < tol, kind
        _check_gx(xd.grad.float().cpu(), gx_ref, x, c, kind, record_property)


@pytest.mark.parametrize("c", _case_params("multi"))
def test_multi_radius_gradient(c, cuda_device, record_property):
    """Radii 1 and 2 from one launch each way (MultiRadiusNFP) against the reference's two layers + torch.cat."""
    B, C, H, W, R = c.shape
    paths = case_paths(c)
    assert all(p.startswith(FAMILIES[c.family][0]) for p in paths), paths
    tol = TOL[c.dtype]
    blocks = nfpb.MultiRadiusNFP(C, padding_mode=c.mode, similarity=c.sim).to(cuda_device)
    assert NF.multi_radius_fusable([b.config for b in blocks.nfp_blocks])
    for kind in KINDS:
        x, rows = make_inputs(kind, c.shape, c.dtype, _seed(c, kind))
        g = torch.randn(B, 32, H, W, generator=torch.Generator().manual_seed(_seed(c, kind) + 4)).to(c.dtype).float()
        y_ref, gx_ref = _multi_ref(x[rows], g[rows], c.mode, c.sim)
        xd = _to_device(x, c, cuda_device)
        y, trace = _traced(lambda: blocks(xd))
        _check_trace(c, trace, "radii 1+2 in one launch")
        y.backward(g.to(cuda_device, y.dtype))
        assert rel_err(y.detach().float().cpu()[rows], y_ref) < tol, kind
        _check_gx(xd.grad.float().cpu()[rows], gx_ref, x[rows], c, kind, record_property)
