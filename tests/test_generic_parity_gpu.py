"""GPU: the generic kernels (csrc/nfp_generic.cu, path generic/pairs) against the fp64 oracle, for every measure, in map
mode (nfp_similarity) and pooled mode (nfp_gap_pair), fp32 and bf16, with nothing masked.

Grid: every measure spelling (SPELLINGS: the 17 measures, plus 'Norm' / 'RMSE', whose capital letter turns the
difference taps off, and 'sharpened_cosine') x every geometry (GEOMS of tests/test_parity_gpu.py, and EDGE_GEOMS: the
limits of each padding rule's fold in the gather backward, 1-pixel rows and columns, pixels no tap reaches,
Ho = Wo = 1, C = 1).  Thinned where the oracle's CPU time requires it:
* the similarity flag alternates over the grid (case_sim) instead of doubling it: every measure and every geometry
  sees both values;
* the 112x112 map runs the hot measures (cosine, norm, dot) in map mode on the clean input only (the fp64 cosine
  oracle takes ~3 s there).
Every case runs the whole batch (scs couples the images) and two inputs: clean (randn) and conditioned (make_inputs:
the elements that make some measure ill-conditioned, at corners, on edges and in the interior).

Checks per case, op, dtype and input: y or both GAP vectors with rel_err; the input gradient with elem_grad_errs
(tests/_util.py): structural zeros exact, the other elements in magnitude buckets each on its own scale; the kernel
path (PATH_TRACE and describe_path); the same bits on a second run.  tests/test_generic_grad_metric.py derives the fp32
bounds below from ATen's own fp32 error, shows that they flag the bugs this file is meant to catch, and checks on the
CPU that every cell of this grid takes generic/pairs.
"""
import zlib

import numpy as np
import pytest
import torch

from neighbour_feature_pooling_b200 import NFPPooling, functional as NF, nfp_pooling
from oracle import nfp_oracle as O

from _util import elem_grad_errs, rel_err, worst
from test_parity_gpu import GEOMS, LOOSE

pytestmark = pytest.mark.gpu

EPS = 1e-6
EDGE_GEOMS = [  # (B, C, H, W, R, stride, padding, dilation, mode)
    (2, 6, 5, 7, 1, 1, 4, 1, "reflect"),      # reflect at pad = min(H, W) - 1
    (2, 6, 5, 6, 1, 1, 5, 1, "circular"),     # circular at pad = H: wraps exactly once
    (2, 6, 3, 4, 1, 1, 6, 1, "replicate"),    # replicate with pad > H, W
    (2, 6, 1, 9, 1, 1, 1, 1, "zeros"),        # H = 1
    (2, 6, 9, 1, 1, 1, 1, 1, "replicate"),    # W = 1
    (2, 6, 1, 9, 1, 1, 1, 1, "circular"),     # H = 1, wrapping onto itself
    (2, 6, 6, 6, 1, 1, 4, 1, "zeros"),        # output centres in the padding
    (2, 6, 11, 10, 1, 4, 1, 1, "reflect"),    # stride > dilation * 2R + 1: pixels no tap reaches
    (1, 1, 7, 7, 1, 1, 1, 1, "reflect"),      # C = 1
    (2, 6, 6, 6, 1, 1, 3, 3, "circular"),     # dilated window wrapping
    (2, 6, 5, 5, 2, 1, 0, 1, "reflect"),      # Ho = Wo = 1
    (2, 4, 8, 8, 3, 2, 3, 1, "replicate"),    # 7x7 window, stride 2
    (2, 6, 7, 7, 1, 3, 0, 3, "zeros"),        # stride = dilation, pad 0
]
ALL_GEOMS = GEOMS + EDGE_GEOMS
SPELLINGS = O.MEASURES + ("Norm", "RMSE", "sharpened_cosine")
P = {"norm": 1, "Norm": 2, "scs": 2}          # norm's default p = 1 and p = 2; scs sharpened with p = 2 and 1
HOT = ("cosine", "norm", "dot")
BIG = 4096                                     # H*W above which only HOT runs (the 112x112 map)
OPS = ("map", "pooled")
DTYPES = (torch.float32, torch.bfloat16)
KINDS = ("clean", "conditioned")

# Bounds, from ATen's own fp32 evaluation of the oracle against its fp64 evaluation on the same input (aten_fp32).
# ATEN_FP32[m]: ATen's largest error over this grid (y, GAP vectors, every elem_grad_errs bucket, both ops and inputs)
# in the cells where it stays below LOOSE[m] / FP32_MULT; tests/test_generic_grad_metric.py measures it again and
# prints it beside the bound.  The fp32 bound of measure m is FP32_MULT x ATEN_FP32[m], at least 1e-5: never above
# the LOOSE bound (tests/test_parity_gpu.py) it replaces.
#
# In the remaining cells the fp32 evaluation is ill-conditioned by construction: the gradient of an element is a
# cancellation of terms far larger than itself, so every fp32 evaluation is off by ~1e-7 of those terms.  Examples:
# C = 1, where cosine and gfc are +-1 and their gradient is 0 up to rounding; canberra's sgn(c-n)/s - |c-n| sgn(c)/s^2
# = eps/s^2 for c, n of opposite signs; attention's softmax saturated by a 1e3-scaled pixel.  There each bucket is
# allowed FP32_MULT x ATen's error in that very cell and bucket (allowed()), and tests/test_generic_grad_metric.py
# lists every such cell with ATen's number.
# geman is the exception the other way: ATen differentiates d / (d + eps) as 1/(d + eps) - d/(d + eps)^2, two ~1
# terms for an eps-sized result, and is ~1e-2 off everywhere (printed by the metric test); the kernel evaluates
# 2 d eps / (d^2 + eps)^2 directly, so geman's input gradient is held to
# its bound with no per-cell allowance.
ATEN_FP32 = {
    "norm": 4.4e-07, "cosine": 8.4e-07, "dot": 6.0e-07, "rmse": 7.7e-07, "geman": 9.3e-06, "attention": 5.0e-06,
    "emd": 2.6e-07, "canberra": 8.7e-06, "hellinger": 9.7e-06, "chisquared1": 7.6e-07, "chisquared2": 7.9e-06,
    "gfc": 1.6e-06, "pearson": 4.0e-06, "jeffrey": 1.2e-05, "squaredchord": 8.8e-06, "smith": 1.9e-06,
    "scs": 7.7e-06,
}
FP32_MULT = 8
BF16_TOL = 2e-2
NO_CELL_ALLOWANCE = ("geman",)


def fp32_bound(measure):
    m = O.canonical_measure(measure)
    return min(LOOSE.get(m, 1e-5), max(1e-5, FP32_MULT * ATEN_FP32[m]))


def tol(measure, dtype):
    return fp32_bound(measure) if dtype == torch.float32 else BF16_TOL


def aten_fp32(op, x, gs, kw):
    """ATen's fp32 evaluation of the oracle against its fp64 evaluation, on the same input and upstream gradients:
    ([rel_err of y] or [rel_err of GAP(x), of GAP(NFP(x))], elem_grad_errs of the input gradient)."""
    B, C, H, W = x.shape
    geo = O.geometry(H, W, kw["R"], kw["stride"], kw["padding"], kw["dilation"], kw["padding_mode"])
    if op == "map":
        y64, gx64 = oracle_map(x, gs[0], kw)
        y32, gx32 = O.nfp_forward_backward(x.float(), gs[0].float(), **kw)
        outs = [rel_err(y32, y64)]
    else:
        a64, n64, gx64 = oracle_pooled(x, gs[0], gs[1], kw)
        gy = (gs[1].float() / (geo.Ho * geo.Wo))[:, :, None, None].expand(B, gs[1].shape[1], geo.Ho, geo.Wo)
        y32, gx32 = O.nfp_forward_backward(x.float(), gy.contiguous(), **kw)
        gx32 = gx32 + (gs[0].float() / (H * W))[:, :, None, None]
        outs = [rel_err(x.float().mean((2, 3)), a64), rel_err(y32.mean((2, 3)), n64)]
    return outs, elem_grad_errs(gx32, gx64, geo)


def allowed(measure, dtype, aten):
    """(bound of y / the GAP vectors, {elem_grad_errs key: bound}) of one cell, given aten_fp32 on its input: the
    measure's bound, or FP32_MULT x ATen's own error where that is larger (the ill-conditioned cells)."""
    t = tol(measure, dtype)
    outs, gx = aten
    t_out = max([t] + [FP32_MULT * e for e in outs])
    if O.canonical_measure(measure) in NO_CELL_ALLOWANCE:
        return t_out, {k: t for k in gx}
    return t_out, {k: max(t, FP32_MULT * e) for k, e in gx.items()}


def geom_id(g):
    return "x".join(map(str, g[:8])) + g[8]


def case_sim(measure, geom):
    """The similarity flag alternates over the grid: both values for every measure and for every geometry."""
    return (SPELLINGS.index(measure) + ALL_GEOMS.index(geom)) % 2 == 0


def case_kw(measure, geom):
    B, C, H, W, R, s, pad, d, mode = geom
    return dict(R=R, measure=measure, p=P.get(measure, 1), stride=s, padding=pad, dilation=d, padding_mode=mode,
                similarity=case_sim(measure, geom))


def case_geo(geom):
    B, C, H, W, R, s, pad, d, mode = geom
    return O.geometry(H, W, R, s, pad, d, mode)


def runs(measure, geom):
    """(op, dtype, kind) checked for this case."""
    if geom[2] * geom[3] > BIG:
        return [("map", dt, "clean") for dt in DTYPES]
    return [(op, dt, k) for op in OPS for dt in DTYPES for k in KINDS]


GRID = [(m, g) for g in ALL_GEOMS for m in SPELLINGS if g[2] * g[3] <= BIG or m in HOT]


def seed(*parts):
    """A stable seed of a case (Python salts str hashes per process)."""
    return zlib.crc32(repr(parts).encode())


def spots(H, W):
    """Corners, edge midpoints and the centre of an H x W map, without repeats."""
    h2, w2 = H // 2, W // 2
    return list(dict.fromkeys([(0, 0), (H - 1, W - 1), (0, W - 1), (H - 1, 0), (0, w2), (h2, 0), (H - 1, w2),
                               (h2, W - 1), (h2, w2)]))


# what the conditioned input plants, per measure family (make_inputs)
SMALL_CHANNELS = ("canberra", "chisquared1", "chisquared2", "jeffrey", "squaredchord", "hellinger")
BIG_PIXEL = ("attention", "geman")


def make_inputs(kind, geom, dtype, s, measure="norm"):
    """x as the kernels see it (bf16-rounded for bf16).

    clean: randn.  conditioned: randn with, at the corners, the edge midpoints and the centre of every image, what
    makes `measure` ill-conditioned:
    * SMALL_CHANNELS: a few channels of the pixel and of its next pixel set to +-{0.3 .. 3} eps, so that
      |c| + |n| + eps (|c| + eps for chisquared2) is a few eps;
    * BIG_PIXEL: the pixel scaled by 1e3 (attention's softmax saturates, geman's d / (d + eps) flattens);
    * the others: the whole pixel scaled to a norm of {0.5, 1, 2} eps (the eps clamps of cosine, gfc, pearson, scs;
      tiny values for the rest).
    No two pixels are made equal, so no difference is exactly 0 (the NaN footprint of rmse / hellinger / norm at a zero
    difference is not part of the contract, DESIGN.md section 2)."""
    B, C, H, W = geom[:4]
    gen = torch.Generator().manual_seed(s)
    x = torch.randn(B, C, H, W, generator=gen)
    m = O.canonical_measure(measure)
    if kind == "conditioned":
        small = torch.tensor([0.3, -1.0, 2.0, -3.0, 0.5, 1.5])
        for b in range(B):
            for i, (h, w) in enumerate(spots(H, W)):
                what = 0 if m in SMALL_CHANNELS else (2 if m in BIG_PIXEL else 1)
                if what == 2 and (i + b) % 3:
                    continue   # one pixel in three: a saturated softmax everywhere would leave nothing to check
                if what == 0:
                    hn, wn = next((u, v) for u, v in ((h, w + 1), (h + 1, w), (h, w - 1), (h - 1, w))
                                  if 0 <= u < H and 0 <= v < W)
                    k = min(C, 3)
                    x[b, :k, h, w] = small[:k] * EPS
                    x[b, :k, hn, wn] = -small[3:3 + k] * EPS
                elif what == 1:
                    x[b, :, h, w] *= (0.5, 1.0, 2.0)[(i // 3 + b) % 3] * EPS / x[b, :, h, w].norm()
                else:
                    x[b, :, h, w] *= 1e3
    if dtype == torch.bfloat16:
        x = x.bfloat16().float()
    return x


def grads(op, geom, measure, kind, dtype):
    """The upstream gradients of a run: g (map) or (g1, g2) (pooled), rounded to the kernel dtype."""
    B, C, H, W = geom[:4]
    geo = case_geo(geom)
    K = (2 * geom[4] + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(seed(measure, geom, kind, op, "g"))
    shapes = [(B, K, geo.Ho, geo.Wo)] if op == "map" else [(B, C), (B, K)]
    return [torch.randn(*s, generator=gen).to(dtype).float() for s in shapes]


def oracle_map(x, g, kw):
    y, gx = O.nfp_forward_backward(x.double(), g.double(), **kw)
    return torch.as_tensor(np.asarray(y)), torch.as_tensor(np.asarray(gx))


def oracle_pooled(x, g1, g2, kw, gap_div=None):
    """GAP(x), GAP(NFP(x)) and the gradient of <g1, GAP(x)> + <g2, GAP(NFP(x))>.  gap_div: what the map's gradient is
    divided by (Ho*Wo; another value only to build a wrong reference in tests/test_generic_grad_metric.py)."""
    B, C, H, W = x.shape
    geo = O.geometry(H, W, kw["R"], kw["stride"], kw["padding"], kw["dilation"], kw["padding_mode"])
    div = geo.Ho * geo.Wo if gap_div is None else gap_div
    gy = (g2.double() / div)[:, :, None, None].expand(B, g2.shape[1], geo.Ho, geo.Wo).contiguous()
    y, gx = oracle_map(x, gy, kw)
    return x.double().mean((2, 3)), y.mean((2, 3)), gx + (g1.double() / (H * W))[:, :, None, None]


def config(measure, geom):
    kw = case_kw(measure, geom)
    C = geom[1]
    return NF.replace(NFPPooling(C, **kw).config, path="generic")


def _traced(fn):
    NF.PATH_TRACE = set()
    try:
        out = fn()
        return out, set(NF.PATH_TRACE)
    finally:
        NF.PATH_TRACE = None


def _run(op, x, gs, cfg, dtype, dev):
    """One forward + backward on the GPU -> (outputs, gx, trace), all as fp32 CPU tensors."""
    xd = x.to(dev, dtype).requires_grad_(True)
    if op == "map":
        y, trace = _traced(lambda: NF.nfp_similarity(xd, cfg))
        y.backward(gs[0].to(dev, y.dtype))
        outs = [y]
    else:
        (a, n), trace = _traced(lambda: NF.nfp_gap_pair(xd, cfg))
        ((a.float() * gs[0].to(dev)).sum() + (n.float() * gs[1].to(dev)).sum()).backward()
        outs = [a, n]
    return [o.detach().float().cpu() for o in outs], xd.grad.float().cpu(), trace


def _bits(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.parametrize("measure,geom", [pytest.param(m, g, id=f"{m}-{geom_id(g)}") for m, g in GRID])
def test_generic_gradient(measure, geom, cuda_device, record_property):
    cfg = config(measure, geom)
    kw = case_kw(measure, geom)
    geo = case_geo(geom)
    for op, dtype, kind in runs(measure, geom):
        what = (op, "fp32" if dtype == torch.float32 else "bf16", kind)
        x = make_inputs(kind, geom, dtype, seed(measure, geom, kind), measure)
        gs = grads(op, geom, measure, kind, dtype)
        if op == "map":
            y_ref, gx_ref = oracle_map(x, gs[0], kw)
            refs = [y_ref]
        else:
            gap_x, gap_n, gx_ref = oracle_pooled(x, gs[0], gs[1], kw)
            refs = [gap_x, gap_n]
        outs, gx, trace = _run(op, x, gs, cfg, dtype, cuda_device)
        assert trace and all(t.startswith("generic/pairs") for t in trace), (what, trace)
        fb = (0, 1) if op == "map" else (2, 3)
        assert all(NF.describe(tuple(x.shape), dtype, cfg, op=o) == "generic/pairs" for o in fb), what
        t_out, t_gx = allowed(measure, dtype, aten_fp32(op, x, gs, kw))
        for o, r in zip(outs, refs):
            assert rel_err(o, r) < t_out, (what, rel_err(o, r), t_out)
        errs = elem_grad_errs(gx, gx_ref, geo, dtype)
        for b in ("struct", "bulk", "high", "spike"):
            vals = [e for (_, k), e in errs.items() if k == b]
            if vals:
                record_property(f"gx_{'_'.join(what)}_{b}", f"{max(vals):.3e}")
        over = {k: (e, t_gx[k]) for k, e in errs.items() if not e < t_gx[k]}
        assert not over, (what, over)
        outs2, gx2, _ = _run(op, x, gs, cfg, dtype, cuda_device)
        assert all(torch.equal(_bits(a), _bits(b)) for a, b in zip(outs + [gx], outs2 + [gx2])), what


@pytest.mark.parametrize("measure", ["norm", "chisquared2"])
def test_nfp_pooling_module(measure, cuda_device):
    """An nfp_pooling head around NFPPooling(C) (its default measure 'norm', and chisquared2): GAP(x) *
    (W GAP(NFP(x)) + b) through nfp_gap_pair on the generic kernels, and the gradients of x, W and b, against fp64
    autograd through oracle.nfp_pooling_forward."""
    B, C, H, W = 3, 24, 7, 7
    layer = NFPPooling(C) if measure == "norm" else NFPPooling(C, measure=measure)
    params = {"num_ftrs": {"m": C}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 3}}
    torch.manual_seed(seed("module", measure))
    head = nfp_pooling(nfp_layer=layer, Params=params).to(cuda_device)
    geom = (B, C, H, W, 1, 1, 0, 1, "reflect")
    for kind in KINDS:
        x = make_inputs(kind, geom, torch.float32, seed("module", measure, kind), measure)
        g = torch.randn(B, C, generator=torch.Generator().manual_seed(seed("module", measure, kind, "g")))
        xr = x.double().requires_grad_(True)
        Wr = head.nfp_proj.weight.detach().cpu().double().requires_grad_(True)
        br = head.nfp_proj.bias.detach().cpu().double().requires_grad_(True)
        c = layer.config
        out_ref = O.nfp_pooling_forward(xr, Wr, br, R=c.R, measure=measure, p=c.p, stride=c.stride,
                                        padding=c.padding, dilation=c.dilation, padding_mode=c.padding_mode,
                                        similarity=c.similarity)
        gx_ref, gW_ref, gb_ref = torch.autograd.grad(out_ref, (xr, Wr, br), g.double())
        head.zero_grad()
        xd = x.to(cuda_device).requires_grad_(True)
        out, trace = _traced(lambda: head(xd))
        assert trace == {"generic/pairs f32 nchw pooled head"}, trace
        out.backward(g.to(cuda_device))
        t = fp32_bound(measure)
        assert rel_err(out.detach().cpu(), out_ref.detach()) < t, kind
        assert rel_err(head.nfp_proj.weight.grad.cpu(), gW_ref) < t, kind
        assert rel_err(head.nfp_proj.bias.grad.cpu(), gb_ref) < t, kind
        errs = elem_grad_errs(xd.grad.cpu(), gx_ref, case_geo(geom))
        assert max(errs.values(), default=0.0) < t, (kind, worst(errs))
