"""GPU: nfp_pooled_similarity (GAP(NFP(x)) without the map, nfpb200_pooled_map_*) against the fp64 oracle, on every
path it takes -- the row-band kernels' pooled mode, the ring and token kernels' pooled modes and the generic kernels --
and fuse_pooled_nfp under a stand-in of the reference's multi-stage head (models/texture_pooling.py:211-268).

Every case runs a clean and a degenerate input (the recipe of test_grad_parity_gpu.make_inputs: one all-zero image,
pixels of norm {0, 1e-9, 0.5, 0.99, 1.01, 4} eps at corners, edges and in the interior), scores gap_nfp with rel_err
and the input gradient with grad_errs (each image and pixel-norm region on its own scale), asserts the kernel path, and
checks that a rerun gives identical bits."""
from collections import namedtuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import neighbour_feature_pooling_b200 as nfpb
from neighbour_feature_pooling_b200 import NFPPooling, _capi, functional as NF
from oracle import nfp_oracle as O

from _util import grad_errs, rel_err, worst
from test_grad_parity_gpu import make_inputs

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-5, torch.bfloat16: 2e-2}
KINDS = ("clean", "degenerate")
MODES = ("reflect", "zeros", "replicate")
BOTH = (torch.float32, torch.bfloat16)
MAPS = [(2, 16, 112, 112, 1), (2, 24, 56, 56, 1), (2, 40, 28, 28, 1), (2, 112, 14, 14, 1), (2, 960, 7, 7, 1)]

# family -> (path prefix, layout, cfg.path)
FAMILIES = {
    "band": ("planar/band", _capi.LAYOUT_NCHW, "auto"),
    "stream": ("fused/stream_", _capi.LAYOUT_NCHW, "auto"),
    "token": ("fused/token_", _capi.LAYOUT_NHWC, "auto"),
    "generic": ("generic/pairs", _capi.LAYOUT_NCHW, "auto"),
    "forced": ("generic/pairs", _capi.LAYOUT_NCHW, "generic"),
}
Case = namedtuple("Case", "family shape mode sim dtype")

BAND_EDGES = [(1, 4, 5, 8, 2),      # every pixel is a border pixel
              (2, 8, 4, 12, 1),
              (2, 12, 21, 24, 1),   # H = 21 is not a multiple of the band height
              (2, 8, 12, 4, 1),     # W < 4R: no interior columns in the backward
              (2, 16, 28, 28, 2)]
BAND_WIDE = [(2, 256, 28, 28, 1),   # the band shrinks to one row granule
             (300, 16, 28, 28, 1),  # more images than CTAs per wave
             (2, 72, 28, 28, 1)]    # fp32: a 49 072-byte slab, under 48 KB alone but not with the static shared memory


def _grid():
    g = []
    for s in BAND_EDGES:
        g += [Case("band", s, m, sim, dt) for m in MODES for sim in (True, False) for dt in BOTH]
    for s in BAND_WIDE + MAPS[:3]:
        g += [Case("band", s, m, sim, dt) for m, sim in (("reflect", True), ("zeros", False)) for dt in BOTH]
    for s in MAPS[3:] + [(3, 512, 7, 7, 2)]:
        g += [Case("stream", s, m, sim, dt) for m, sim in (("reflect", True), ("replicate", False)) for dt in BOTH]
    for s in [(2, 960, 7, 7, 1), (3, 128, 7, 7, 2)]:
        g += [Case("token", s, m, sim, torch.bfloat16) for m, sim in (("reflect", True), ("zeros", False))]
    for s in [(3, 20, 9, 6, 1), (2, 400, 28, 28, 1)]:   # unaligned planes; too wide for one band slab
        g += [Case("generic", s, "reflect", True, dt) for dt in BOTH]
    g += [Case("forced", (2, 16, 28, 28, 1), "zeros", False, dt) for dt in BOTH]
    return g


GRID = _grid()


def case_id(c):
    dt = "fp32" if c.dtype == torch.float32 else "bf16"
    return f'{c.family}-{"x".join(map(str, c.shape[:4]))}_r{c.shape[4]}-{c.mode}-{"sim" if c.sim else "dist"}-{dt}'


def case_cfg(c):
    B, C, H, W, R = c.shape
    return NF.replace(NFPPooling(C, R=R, measure="cosine", padding=R, padding_mode=c.mode, similarity=c.sim).config,
                      path=FAMILIES[c.family][2])


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


def _oracle(x, g, R, mode, sim):
    """GAP(NFP(x)) and the input gradient of <g, GAP(NFP(x))> in fp64: the map gradient g / (H' W') expanded."""
    B, C, H, W = x.shape
    gy = (g.double() / (H * W))[:, :, None, None].expand(B, g.shape[1], H, W).contiguous()
    y, gx = O.nfp_forward_backward(x.double(), gy, R=R, measure="cosine", padding=R, padding_mode=mode, similarity=sim)
    return torch.as_tensor(np.asarray(y)).mean((2, 3)), torch.as_tensor(np.asarray(gx))


def _run(xd, cfg, g):
    xd.grad = None
    gn, trace = _traced(lambda: NF.nfp_pooled_similarity(xd, cfg))
    (gn.float() * g).sum().backward()
    return gn.detach().clone(), xd.grad.detach().clone(), trace


@pytest.mark.parametrize("c", [pytest.param(c, id=case_id(c)) for c in GRID])
def test_pooled_map_vs_oracle(c, cuda_device, record_property):
    B, C, H, W, R = c.shape
    K = (2 * R + 1) ** 2 - 1
    prefix, layout, _ = FAMILIES[c.family]
    cfg = case_cfg(c)
    for op in (_capi.OP_POOLED_MAP_FORWARD, _capi.OP_POOLED_MAP_BACKWARD):
        assert NF.describe((B, C, H, W), c.dtype, cfg, op, layout).startswith(prefix), (op, c)
    tol = TOL[c.dtype]
    for kind in KINDS:
        seed = 7919 * B + 131 * C + 17 * H + W + R + MODES.index(c.mode) + 3 * c.sim + 5 * KINDS.index(kind)
        x, rows = make_inputs(kind, c.shape, c.dtype, seed)
        g = torch.randn(B, K, generator=torch.Generator().manual_seed(seed + 9))
        gn_ref, gx_ref = _oracle(x[rows], g[rows], R, c.mode, c.sim)
        xd = _to_device(x, c, cuda_device)
        gd = g.to(cuda_device)
        gn, gx, trace = _run(xd, cfg, gd)
        assert trace and all(t.startswith(prefix) and t.endswith("pooled map") for t in trace), trace
        assert gn.dtype == c.dtype and gn.shape == (B, K)
        assert gx.dtype == c.dtype and gx.is_contiguous(memory_format=torch.channels_last) == (layout == 1)
        e = rel_err(gn.float().cpu()[rows], gn_ref)
        record_property(f"gap_{kind}", f"{e:.3e}")
        assert e < tol, (kind, e)
        errs = grad_errs(gx.float().cpu()[rows], gx_ref, x[rows])
        record_property(f"gx_{kind}", f"{max(errs.values()):.3e}")
        assert max(errs.values()) < tol, (kind, worst(errs))
        gn2, gx2, _ = _run(xd, cfg, gd)
        assert torch.equal(gn, gn2) and torch.equal(gx, gx2), "rerun changed bits"


@pytest.mark.parametrize("shape,dtype,layout", [((3, 112, 14, 14, 1), torch.float32, 0), ((3, 960, 7, 7, 1), torch.bfloat16, 0),
                                                ((3, 512, 7, 7, 2), torch.float32, 0), ((4, 960, 7, 7, 1), torch.bfloat16, 1)])
def test_ring_and_token_equal_gap_pair(shape, dtype, layout, cuda_device):
    """Same kernel as nfp_gap_pair's pooled mode: gap_nfp is bit for bit its second output."""
    B, C, H, W, R = shape
    cfg = NFPPooling(C, R=R, measure="cosine", padding=R).config
    x = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(1)).to(cuda_device, dtype)
    if layout:
        x = x.contiguous(memory_format=torch.channels_last)
    with torch.no_grad():
        gn = NF.nfp_pooled_similarity(x, cfg)
        _, want = NF.nfp_gap_pair(x, cfg)
    assert torch.equal(gn, want)


@pytest.mark.parametrize("dtype", BOTH)
@pytest.mark.parametrize("shape", [s for s in MAPS[:3]] + [(2, 16, 28, 28, 2)], ids=lambda s: "x".join(map(str, s)))
def test_band_agrees_with_pooled_map(shape, dtype, cuda_device):
    """The composition it replaces, adaptive_avg_pool2d(nfp_similarity(x), 1), within the dtype bound (the map is
    rounded to the dtype before the pool there, the pooled kernels sum in fp32)."""
    B, C, H, W, R = shape
    cfg = NFPPooling(C, R=R, measure="cosine", padding=R).config
    x = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(2)).to(cuda_device, dtype)
    with torch.no_grad():
        gn = NF.nfp_pooled_similarity(x, cfg)
        want = F.adaptive_avg_pool2d(NF.nfp_similarity(x, cfg), 1).flatten(1)
    assert gn.dtype == want.dtype
    assert rel_err(gn.float().cpu(), want.float().cpu()) < TOL[dtype]


def test_dtypes_and_autocast(cuda_device):
    cfg = NFPPooling(24, R=1, measure="cosine", padding=1).config
    x = torch.randn(2, 24, 56, 56, device=cuda_device)
    for dt in (torch.float32, torch.bfloat16, torch.float16):   # fp16: widened to fp32 by the kernels, fp16 out
        xd = x.to(dt).detach().requires_grad_(True)
        y = NF.nfp_pooled_similarity(xd, cfg)
        assert y.dtype == dt and y.shape == (2, 8)
        y.float().sum().backward()
        assert xd.grad.dtype == dt
    with torch.autocast("cuda", dtype=torch.bfloat16):
        for dt in (torch.float32, torch.bfloat16):
            y = NF.nfp_pooled_similarity(x.to(dt), cfg)
            want = F.adaptive_avg_pool2d(NF.nfp_similarity(x.to(dt), cfg), 1).flatten(1)
            assert y.dtype == want.dtype == torch.float32
    # channels-last bf16 is consumed in place by the token kernels, and its gradient comes back channels-last
    cfg7 = NFPPooling(960, R=1, measure="cosine", padding=1).config
    xt = torch.randn(2, 960, 7, 7, device=cuda_device, dtype=torch.bfloat16).contiguous(
        memory_format=torch.channels_last).requires_grad_(True)
    y, trace = _traced(lambda: NF.nfp_pooled_similarity(xt, cfg7))
    assert all(t.startswith("fused/token_7x7_r1") and "channels-last" in t for t in trace), trace
    y.float().sum().backward()
    assert xt.grad.dtype == torch.bfloat16 and xt.grad.is_contiguous(memory_format=torch.channels_last)


# ---- the multi-stage head, unmodified, with fuse_pooled_nfp ------------------------------------------------------------

HEAD_MAPS = [(16, 112, 112), (24, 56, 56), (40, 28, 28), (112, 14, 14), (960, 7, 7)]


class _MultiStageStandIn(torch.nn.Module):
    """What MobileNetV3_MultiStageNFP does with its five feature maps (texture_pooling.py:249-268)."""

    def __init__(self):
        super().__init__()
        self.nfp = torch.nn.ModuleList([NFPPooling(c, R=1, measure="cosine", padding=1) for c, _, _ in HEAD_MAPS])
        self.fc = torch.nn.Linear(40, 64)

    def forward(self, feats):
        pooled = []
        for layer, f in zip(self.nfp, feats):
            y = F.adaptive_avg_pool2d(layer(f), (1, 1))
            pooled.append(y.view(y.size(0), -1))
        return self.fc(torch.cat(pooled, dim=1))


def _head_ref(xs, Wl, bl, t):
    """fp64: out = fc(cat(GAP(NFP(x_i)))), and the gradients of <t, out> w.r.t. every x_i, W and b."""
    feats = []
    for x in xs:
        y = torch.as_tensor(np.asarray(O.nfp_forward(x.double(), R=1, measure="cosine", padding=1)))
        feats.append(y.mean((2, 3)))
    f = torch.cat(feats, 1)
    out = f @ Wl.t() + bl
    gf = t @ Wl
    gxs, o = [], 0
    for x in xs:
        gxs.append(_oracle(x, gf[:, o:o + 8], 1, "reflect", True)[1])
        o += 8
    return out, gxs, t.t() @ f, t.sum(0)


@pytest.mark.parametrize("variant", ["fp32", "bf16-autocast-channels-last"])
def test_multistage_head_fused(variant, cuda_device):
    B = 4
    torch.manual_seed(0)
    head = _MultiStageStandIn().to(cuda_device)
    gen = torch.Generator().manual_seed(3)
    xs = [torch.randn(B, c, h, w, generator=gen) for c, h, w in HEAD_MAPS]
    t = torch.randn(B, 64, generator=gen)
    amp = variant != "fp32"
    if amp:
        xs = [x.bfloat16().float() for x in xs]
    Wl, bl = head.fc.weight.detach().cpu().double(), head.fc.bias.detach().cpu().double()
    out_ref, gx_ref, gw_ref, gb_ref = _head_ref(xs, Wl, bl, t.double())
    tol = TOL[torch.bfloat16 if amp else torch.float32]

    def run():
        head.zero_grad()
        xd = [x.to(cuda_device, torch.bfloat16 if amp else torch.float32) for x in xs]
        if amp:
            xd = [x.contiguous(memory_format=torch.channels_last) for x in xd]
        xd = [x.requires_grad_(True) for x in xd]
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            out, trace = _traced(lambda: head(xd))
        (out.float() * t.to(cuda_device)).sum().backward()
        return out.detach().float().cpu(), [x.grad.float().cpu() for x in xd], trace

    results = {}
    for fused in (False, True):
        if fused:
            assert all(nfpb.fuse_pooled_nfp(layer) for layer in head.nfp)
        out, gxs, trace = run()
        results[fused] = out
        if fused:
            assert trace and all(e.endswith("pooled map") for e in trace), trace
        else:
            assert trace and all(e.endswith(" map") and "pooled" not in e for e in trace), trace
        assert rel_err(out, out_ref) < tol, fused
        for gx, want, x in zip(gxs, gx_ref, xs):
            errs = grad_errs(gx, want, x)
            assert max(errs.values()) < tol, (fused, worst(errs))
        assert rel_err(head.fc.weight.grad.cpu(), gw_ref) < tol, fused
        assert rel_err(head.fc.bias.grad.cpu(), gb_ref) < tol, fused
    for layer in head.nfp:
        nfpb.unfuse_pooled_nfp(layer)
    assert rel_err(results[True], results[False]) < tol
