"""GPU: parity of the CUDA path (through the C ABI) with the reference.

* every golden case generated from the unmodified reference (tests/golden/, oracle/make_golden.py):
  all 17 measures + spelling quirks, 3x3 / 5x5, stride / dilation / pad != R, reflect / zeros;
* seeded random inputs against the oracle over a geometry x measure grid (generic kernels) and over
  the fused-kernel shapes;
* size-independent properties at BASELINE.json's full sizes (B=256, 512x7x7 / 256x14x14).

Tolerances (BASELINE.json north_star): fp32 <= 1e-5 relative (max-norm), bf16 <= 2e-2 against the
fp32/fp64 reference evaluated on the bf16-rounded input.  Input gradients are scored with grad_err (tests/_util.py):
each image and each pixel-norm region (||x|| <= 2 eps, small, ordinary) on its own scale, so that the 1e6-sized
gradients of the planted degenerate pixels do not set the scale for all the others.
"""
import numpy as np
import pytest
import torch

import neighbour_feature_pooling_b200 as nfpb
from neighbour_feature_pooling_b200 import NFPPooling, nfp_pooling, functional as NF
from oracle import nfp_oracle as O

from _util import (case_id, case_kwargs, grad_err, grad_errs, load_measure_cases, load_multi_radius_cases,
                   load_wrapper_cases, rel_err, worst)

pytestmark = pytest.mark.gpu

INDEX, ARR = load_measure_cases()
FP32_TOL = 1e-5
BF16_TOL = 2e-2
# measures whose fp32 evaluation is ill-conditioned by construction (log / sqrt of eps-shifted values,
# divisions by eps-sized denominators): the reference's own fp32 run is not 1e-5-close to its fp64 run.
LOOSE = {"jeffrey": 2e-4, "hellinger": 1e-4, "squaredchord": 1e-4, "canberra": 1e-4, "chisquared1": 1e-4,
         "chisquared2": 1e-4, "geman": 1e-4, "pearson": 5e-5, "scs": 1e-4, "sharpened_cosine": 1e-4,
         "smith": 5e-5, "rmse": 5e-5, "norm": 5e-5, "gfc": 2e-5, "attention": 5e-5}


def _run(x, g, kw, dev, dtype=torch.float32, path="auto"):
    layer = NFPPooling(x.shape[1], **kw).to(dev)
    layer._cfg = NF.replace(layer._cfg, path=path)
    xd = x.to(dev, dtype).requires_grad_(True)
    y = layer(xd)
    y.backward(g.to(dev, dtype))
    return y.detach().float().cpu(), xd.grad.float().cpu()


@pytest.mark.parametrize("c", INDEX, ids=case_id)
def test_golden_fp32(c, cuda_device):
    x = torch.from_numpy(ARR[c["key"] + "_x"])
    g = torch.from_numpy(ARR[c["key"] + "_g"])
    tol = LOOSE.get(c["measure"].lower(), FP32_TOL)
    for path in ("auto", "generic"):
        y, gx = _run(x, g, case_kwargs(c), cuda_device, path=path)
        gtol = FP32_TOL if c["measure"].lower() == "cosine" else max(tol, 2e-5)
        assert rel_err(y, ARR[c["key"] + "_y_f64"]) < tol, path
        # per region over the (1-3 image) batch: the fixtures pin each measure's semantics; the per-image scale is for
        # the batched kernels' tests, and Geman's own fp32 evaluation is too ill-conditioned for it (0.66 of the bound)
        errs = grad_errs(gx, ARR[c["key"] + "_gx_f64"], x, per_image=False)
        assert max(errs.values()) < gtol, (path, worst(errs))


@pytest.mark.parametrize("c", [c for c in INDEX if c["measure"] in ("cosine", "dot", "gfc", "emd")], ids=case_id)
def test_golden_bf16(c, cuda_device):
    x = torch.from_numpy(ARR[c["key"] + "_x"]).bfloat16().float()   # the bf16-rounded input
    g = torch.from_numpy(ARR[c["key"] + "_g"]).bfloat16().float()
    y_ref, gx_ref = O.nfp_forward_backward(x.double(), g.double(), **case_kwargs(c))
    y, gx = _run(x, g, case_kwargs(c), cuda_device, dtype=torch.bfloat16)
    assert rel_err(y, y_ref) < BF16_TOL
    assert grad_err(gx, gx_ref, x, per_image=False) < BF16_TOL


GEOMS = [  # (B, C, H, W, R, stride, padding, dilation, mode)
    (3, 20, 7, 7, 1, 1, 1, 1, "reflect"),
    (2, 12, 9, 6, 2, 1, 2, 1, "reflect"),
    (2, 8, 6, 6, 1, 1, 2, 1, "reflect"),
    (2, 8, 9, 8, 1, 2, 1, 1, "replicate"),
    (2, 8, 9, 9, 1, 1, 2, 2, "circular"),
    (2, 8, 7, 7, 1, 2, 3, 2, "zeros"),
    (1, 5, 11, 13, 3, 1, 3, 1, "reflect"),     # 7x7 window, odd channel count
    (2, 16, 112, 112, 1, 1, 1, 1, "reflect"),  # multi-stage MobileNetV3 stem map: large HxW, small C
]


@pytest.mark.parametrize("measure", O.MEASURES)
@pytest.mark.parametrize("geom", GEOMS, ids=lambda g: "x".join(map(str, g[:8])) + g[8])
def test_random_vs_oracle_generic(measure, geom, cuda_device):
    B, C, H, W, R, s, pad, d, mode = geom
    if H * W > 4096 and measure not in ("cosine", "norm", "dot"):
        pytest.skip("large map checked for the hot measures only")
    gen = torch.Generator().manual_seed(hash((measure, geom)) % (2 ** 31))
    x = torch.randn(B, C, H, W, generator=gen)
    kw = dict(R=R, measure=measure, p=2 if measure in ("norm", "scs") else 1, stride=s, padding=pad,
              dilation=d, padding_mode=mode)
    y_ref = O.nfp_forward(x.double(), **kw)
    g = torch.randn(y_ref.shape, generator=gen)
    y_ref, gx_ref = O.nfp_forward_backward(x.double(), g.double(), **kw)
    y, gx = _run(x, g, kw, cuda_device, path="generic")
    tol = LOOSE.get(measure, FP32_TOL)
    assert rel_err(y, y_ref) < tol
    assert rel_err(gx, gx_ref) < max(tol, 2e-5)
    # the generic backward gathers through the inverse index map in a fixed order (no atomics): same bits every time
    y2, gx2 = _run(x, g, kw, cuda_device, path="generic")
    assert torch.equal(y.view(torch.int32), y2.view(torch.int32))
    assert torch.equal(gx.view(torch.int32), gx2.view(torch.int32))


FUSED_SHAPES = [(5, 64, 7, 7, 1), (3, 512, 7, 7, 1), (2, 960, 7, 7, 1), (3, 256, 14, 14, 1), (2, 192, 14, 14, 1),
                (6, 512, 2, 2, 1), (4, 32, 4, 4, 1), (3, 24, 7, 7, 1), (300, 16, 7, 7, 1),
                (3, 128, 7, 7, 2), (2, 512, 7, 7, 2), (2, 64, 14, 14, 2), (2, 256, 14, 14, 2),
                (300, 512, 7, 7, 1)]   # more images than resident CTAs at full width: the resident-image backward (8 ring slots,
                                       # two-round table publish, double-buffered gradient), some CTAs with a second image


PLANAR_SHAPES = [(2, 16, 112, 112, 1), (2, 24, 56, 56, 1), (3, 40, 28, 28, 1), (2, 7, 9, 13, 1), (2, 5, 3, 3, 1),
                 (2, 12, 28, 28, 2), (1, 6, 11, 13, 3), (3, 33, 7, 7, 1), (2, 10, 5, 9, 2),
                 (2, 5, 8, 6, 1), (70, 3, 12, 8, 1), (1, 4, 16, 20, 2),   # row granule 2 / many images
                 # the band kernels' interior / border split at its corners: no interior rows, no interior columns,
                 # a one-row last band, a 5x5 window on a map narrower than its backward margin
                 (2, 8, 4, 12, 1), (2, 4, 20, 4, 1), (3, 6, 33, 16, 1), (1, 4, 5, 8, 2)]
PLANAR_BAND = {(16, 112, 112), (24, 56, 56), (40, 28, 28), (12, 28, 28), (5, 8, 6), (3, 12, 8), (4, 16, 20),
               (8, 4, 12), (4, 20, 4), (6, 33, 16), (4, 5, 8)}


@pytest.mark.parametrize("shape", PLANAR_SHAPES, ids=lambda s: "x".join(map(str, s[:4])) + f"_r{s[4]}")
@pytest.mark.parametrize("mode", ["reflect", "zeros", "replicate"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("similarity", [True, False], ids=["sim", "dist"])
def test_planar_cosine_vs_oracle(shape, mode, dtype, similarity, cuda_device):
    """Maps the streaming kernels do not cover (multi-stage heads, texture_pooling.py:211-268: 16x112x112 ...;
    odd sizes / channel counts) take the planar kernels: same closed forms, no atomics."""
    B, C, H, W, R = shape
    if mode == "reflect" and R >= min(H, W):
        pytest.skip("reflect padding needs pad < dim")
    K = (2 * R + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(B * 1000 + C + H + R)
    x = torch.randn(B, C, H, W, generator=gen)
    if C % 3 == 0:
        x = x.relu()
    x[0, :, 0, 0] = 0.0
    x[-1, :, H - 1, W - 1] *= 1e-9
    g = torch.randn(B, K, H, W, generator=gen)
    if dtype == torch.bfloat16:
        x, g = x.bfloat16().float(), g.bfloat16().float()
    kw = dict(R=R, measure="cosine", padding=R, padding_mode=mode, similarity=similarity)
    cfg = NFPPooling(C, **kw).config
    # TMA-staged row bands where planes and row groups are 16-byte aligned, plain coalesced loads otherwise
    want = "planar/band" if (C, H, W) in PLANAR_BAND else "planar/table"
    if R > 2:
        want = "generic/pairs"   # 7x7 windows and wider: generic kernels
    assert NF.describe(shape[:4], dtype, cfg) == want
    assert NF.describe(shape[:4], dtype, cfg, op=1) == want
    y_ref, gx_ref = O.nfp_forward_backward(x.double(), g.double(), **kw)
    y, gx = _run(x, g, kw, cuda_device, dtype=dtype)
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    assert rel_err(y, y_ref) < tol
    errs = grad_errs(gx, gx_ref, x)
    assert max(errs.values()) < tol, worst(errs)
    if R <= 2:  # bit-reproducible (gather form, no atomics)
        y2, gx2 = _run(x, g, kw, cuda_device, dtype=dtype)
        assert torch.equal(y, y2) and torch.equal(gx, gx2)


@pytest.mark.parametrize("shape", FUSED_SHAPES, ids=lambda s: "x".join(map(str, s[:4])) + f"_r{s[4]}")
@pytest.mark.parametrize("mode", ["reflect", "zeros", "replicate"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_fused_cosine_vs_oracle(shape, mode, dtype, cuda_device):
    B, C, H, W, R = shape
    K = (2 * R + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(B * 1000 + C + H + R)
    x = torch.randn(B, C, H, W, generator=gen)
    if C % 3 == 0:
        x = x.relu()
    x[0, :, 0, 0] = 0.0              # exact zero vector: gradient must follow ATen's clamp semantics
    x[-1, :, H - 1, W - 1] *= 1e-9   # ||x|| < eps
    if dtype == torch.bfloat16:
        x = x.bfloat16().float()
    kw = dict(R=R, measure="cosine", padding=R, padding_mode=mode)
    cfg = NFPPooling(C, **kw).config
    assert NF.describe(shape[:4], dtype, cfg).startswith(("fused/split", "fused/stream")), "shape expected on the streaming fused path"
    g = torch.randn(B, K, H, W, generator=gen)
    if dtype == torch.bfloat16:
        g = g.bfloat16().float()
    # more images than resident CTAs exercises the persistent image loop: oracle on a slice
    sl = slice(B - 4, B) if B > 32 else slice(0, B)
    y_ref, gx_ref = O.nfp_forward_backward(x[sl].double(), g[sl].double(), **kw)
    y, gx = _run(x, g, kw, cuda_device, dtype=dtype)
    y, gx = y[sl], gx[sl]
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    assert rel_err(y, y_ref) < tol
    errs = grad_errs(gx, gx_ref, x[sl])
    assert max(errs.values()) < tol, worst(errs)
    if dtype == torch.float32 and B <= 32:
        # and the CUDA paths agree with each other
        y2, gx2 = _run(x, g, kw, cuda_device, path="generic")
        assert rel_err(y, y2) < FP32_TOL and grad_err(gx, gx2, x) < FP32_TOL
    # the cluster-split kernels (NFPB200_PATH_SPLIT: the measured experiment of DESIGN.md 4.2) on the same problem
    cfg_split = NF.replace(cfg, path="split")
    assert NF.describe(shape[:4], dtype, cfg_split).startswith("fused/split")
    y3, gx3 = _run(x, g, kw, cuda_device, dtype=dtype, path="split")
    y3, gx3 = y3[sl], gx3[sl]
    assert rel_err(y3, y_ref) < tol
    errs = grad_errs(gx3, gx_ref, x[sl])
    assert max(errs.values()) < tol, worst(errs)


@pytest.mark.parametrize("shape", [(40, 8, 7, 7, 1), (40, 16, 7, 7, 2), (24, 2, 14, 14, 1), (24, 4, 14, 14, 2),
                                   (64, 32, 2, 2, 1), (48, 16, 4, 4, 1), (600, 8, 7, 7, 1)],
                         ids=lambda s: "x".join(map(str, s[:4])) + f"_r{s[4]}")
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_fused_stress_repeatable(shape, dtype, cuda_device):
    """compute-sanitizer is closed on this GPU pool, so shared-memory races are hunted the hard way: the smallest
    channel counts (every pipeline phase is as short as it gets, warps drift apart the most), many more images than
    resident CTAs, map and pooled modes, repeated -- results must be bit-identical run to run and match the oracle."""
    B, C, H, W, R = shape
    K = (2 * R + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(sum(shape))
    x = torch.randn(B, C, H, W, generator=gen)
    g = torch.randn(B, K, H, W, generator=gen)
    if dtype == torch.bfloat16:
        x, g = x.bfloat16().float(), g.bfloat16().float()
    kw = dict(R=R, measure="cosine", padding=R)
    cfg = NFPPooling(C, **kw).config
    assert NF.describe(shape[:4], dtype, cfg).startswith(("fused/split", "fused/stream"))
    sl = slice(B - 3, B)
    y_ref, gx_ref = O.nfp_forward_backward(x[sl].double(), g[sl].double(), **kw)
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    first = None
    wa = torch.randn(B, C, generator=gen).to(cuda_device)
    wn = torch.randn(B, K, generator=gen).to(cuda_device)
    for rep in range(6):
        y, gx = _run(x, g, kw, cuda_device, dtype=dtype)
        xp = x.to(cuda_device, dtype).requires_grad_(True)
        ga, gn = NF.nfp_gap_pair(xp, cfg)
        ((ga.float() * wa).sum() + (gn.float() * wn).sum()).backward()
        cur = (y, gx, ga.detach().float().cpu(), gn.detach().float().cpu(), xp.grad.float().cpu())
        if first is None:
            first = cur
            assert rel_err(y[sl], y_ref) < tol and rel_err(gx[sl], gx_ref) < tol
            assert rel_err(cur[3], y.mean((2, 3))) < (1e-5 if dtype == torch.float32 else 2e-2)
        else:
            assert all(torch.equal(a, b) for a, b in zip(first, cur)), f"run {rep} differs from run 0"


def test_fused_is_deterministic(cuda_device):
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(64, 256, 7, 7, generator=gen)
    g = torch.randn(64, 8, 7, 7, generator=gen)
    kw = dict(R=1, measure="cosine", padding=1)
    y1, gx1 = _run(x, g, kw, cuda_device)
    y2, gx2 = _run(x, g, kw, cuda_device)
    assert torch.equal(y1, y2) and torch.equal(gx1, gx2)


def test_wrapper_golden(cuda_device):
    index, arr = load_wrapper_cases()
    for c in index:
        k = c["key"]
        Params = {"num_ftrs": {"m": c["C"]}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 5}}
        pool = nfp_pooling(Params=Params)
        with torch.no_grad():
            pool.nfp_proj.weight.copy_(torch.from_numpy(arr[k + "_w"]))
            pool.nfp_proj.bias.copy_(torch.from_numpy(arr[k + "_b"]))
        pool = pool.to(cuda_device)
        x = torch.from_numpy(arr[k + "_x"]).to(cuda_device).requires_grad_(True)
        out = pool(x)
        out.backward(torch.from_numpy(arr[k + "_g"]).to(cuda_device))
        assert rel_err(out.detach().cpu(), arr[k + "_out"]) < FP32_TOL
        assert grad_err(x.grad.cpu(), arr[k + "_gx"], arr[k + "_x"]) < FP32_TOL
        assert rel_err(pool.nfp_proj.weight.grad.cpu(), arr[k + "_gw"]) < FP32_TOL
        assert rel_err(pool.nfp_proj.bias.grad.cpu(), arr[k + "_gb"]) < FP32_TOL


@pytest.mark.parametrize("shape", [(3, 64, 7, 7), (2, 24, 9, 6)], ids=["fused", "generic"])
def test_pooled_head_equals_map_then_gap(shape, cuda_device):
    B, C, H, W = shape
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(B, C, H, W, generator=gen).to(cuda_device)
    cfg = NFPPooling(C, R=1, measure="cosine", padding=1).config
    xa = x.clone().requires_grad_(True)
    ga, gn = NF.nfp_gap_pair(xa, cfg)
    wa = torch.randn(B, C, generator=gen).to(cuda_device)
    wn = torch.randn(B, 8, generator=gen).to(cuda_device)
    ((ga * wa).sum() + (gn * wn).sum()).backward()
    xb = x.clone().requires_grad_(True)
    yb = NF.nfp_similarity(xb, cfg)
    ((xb.mean((2, 3)) * wa).sum() + (yb.mean((2, 3)) * wn).sum()).backward()
    assert rel_err(ga.detach().cpu(), xb.detach().mean((2, 3)).cpu()) < FP32_TOL
    assert rel_err(gn.detach().cpu(), yb.detach().mean((2, 3)).cpu()) < FP32_TOL
    assert rel_err(xa.grad.cpu(), xb.grad.cpu()) < FP32_TOL


@pytest.mark.parametrize("shape", [(256, 512, 7, 7, 1), (700, 64, 7, 7, 1), (64, 256, 14, 14, 1), (40, 128, 7, 7, 2),
                                   (96, 24, 7, 7, 1)], ids=lambda s: "x".join(map(str, s[:4])) + f"_r{s[4]}")
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_backward_x_stable_hint_same_bits(shape, dtype, cuda_device):
    """NFPB200_HINT_X_STABLE lets the fused backward stream x while the preceding NFP launch drains (PDL) and moves
    the gy-only stencil part behind pass A; in chains of NFP launches the results are bit-identical to the
    conservative order, for every launch of the chain."""
    import ctypes
    from neighbour_feature_pooling_b200 import _capi
    B, C, H, W, R = shape
    K = (2 * R + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(17)
    kd = _capi.F32 if dtype == torch.float32 else _capi.BF16
    xs = [torch.randn(B, C, H, W, generator=gen).to(cuda_device, dtype) for _ in range(3)]
    gys = [torch.randn(B, K, H, W, generator=gen).to(cuda_device, dtype) for _ in range(3)]
    lib = _capi.load()
    st = torch.cuda.current_stream().cuda_stream
    res = {}
    for hint in (0, _capi.HINT_X_STABLE):
        desc = _capi.make_desc(kd, B, C, H, W, R, 1, R, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6, "auto")
        fdesc = _capi.make_desc(kd, B, C, H, W, R, 1, R, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6, "auto")
        desc.path |= hint
        ys = [torch.empty_like(g) for g in gys]
        gxs = [torch.empty_like(x) for x in xs]
        for rep in range(2):
            for i in range(3):   # forward, backward, backward of the next buffer ... back to back on one stream
                _capi.check(lib.nfpb200_forward(ctypes.byref(fdesc), xs[i].data_ptr(), ys[i].data_ptr(), None, 0, st), "fwd")
                _capi.check(lib.nfpb200_backward(ctypes.byref(desc), xs[i].data_ptr(), gys[i].data_ptr(),
                                                 gxs[i].data_ptr(), None, 0, st), "bwd")
                j = (i + 1) % 3
                _capi.check(lib.nfpb200_backward(ctypes.byref(desc), xs[j].data_ptr(), gys[j].data_ptr(),
                                                 gxs[j].data_ptr(), None, 0, st), "bwd")
        torch.cuda.synchronize()
        res[hint] = [t.float().cpu() for t in ys + gxs]
    assert all(torch.equal(a, b) for a, b in zip(res[0], res[_capi.HINT_X_STABLE]))
    y_ref, gx_ref = O.nfp_forward_backward(xs[0][-2:].double().cpu(), gys[0][-2:].double().cpu(), R=R, measure="cosine",
                                           padding=R)
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    assert rel_err(res[_capi.HINT_X_STABLE][0][-2:], y_ref) < tol
    assert rel_err(res[_capi.HINT_X_STABLE][3][-2:], gx_ref) < tol


@pytest.mark.parametrize("shape", [(5, 64, 7, 7), (300, 16, 7, 7), (3, 6, 14, 14)], ids=lambda s: "x".join(map(str, s)))
def test_pool_backward_gradient_row_alignment(shape, cuda_device):
    """nfpb200_pool_backward stages d out / d GAP(x) with one TMA bulk copy per image when its rows are 16-byte
    aligned and sized, with plain loads otherwise (C % 4 != 0, or a gradient view at an odd offset): same bits."""
    import ctypes
    from neighbour_feature_pooling_b200 import _capi
    B, C, H, W = shape
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(B, C, H, W, generator=gen).to(cuda_device)
    ggn = torch.randn(B, 8, generator=gen).to(cuda_device)
    vals = torch.randn(B, C, generator=gen).to(cuda_device)
    buf = torch.empty(B * C + 4, device=cuda_device)
    desc = _capi.make_desc(_capi.F32, B, C, H, W, 1, 1, 1, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6, "auto")
    assert _capi.describe_path(desc, _capi.OP_POOL_BACKWARD).startswith(("fused/split", "fused/stream"))
    lib = _capi.load()
    outs = []
    for off in (0, 1):   # 0: aligned rows, 1: the same values 4 bytes further (misaligned)
        ggx = buf[off:off + B * C].view(B, C)
        ggx.copy_(vals)
        assert (ggx.data_ptr() % 16 == 0) == (off == 0)
        gx = torch.empty_like(x)
        rc = lib.nfpb200_pool_backward(ctypes.byref(desc), x.data_ptr(), ggx.data_ptr(), ggn.data_ptr(), gx.data_ptr(),
                                       None, 0, torch.cuda.current_stream().cuda_stream)
        _capi.check(rc, "nfpb200_pool_backward")
        torch.cuda.synchronize()
        outs.append(gx.cpu())
    assert torch.equal(outs[0], outs[1])
    # and against autograd through the map-mode kernels
    cfg = NFPPooling(C, R=1, measure="cosine", padding=1).config
    xb = x.clone().requires_grad_(True)
    yb = NF.nfp_similarity(xb, cfg)
    ((xb.mean((2, 3)) * vals).sum() + (yb.mean((2, 3)) * ggn).sum()).backward()
    assert rel_err(outs[0], xb.grad.cpu()) < FP32_TOL


@pytest.mark.parametrize("C,H,W", [(512, 7, 7), (256, 14, 14)], ids=["layer4", "layer3"])
@pytest.mark.parametrize("R", [1, 2], ids=["3x3", "5x5"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_full_size_properties(C, H, W, R, dtype, cuda_device):
    """BASELINE.json config 2 at full size (B=256): properties that need no CPU reference."""
    B, K = 256, (2 * R + 1) ** 2 - 1
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(B, C, H, W, generator=gen, device=cuda_device).to(dtype)
    layer = NFPPooling(C, R=R, measure="cosine", padding=R).to(cuda_device)
    xr = x.clone().requires_grad_(True)
    y = layer(xr)
    assert y.shape == (B, K, H, W) and y.dtype == dtype
    yf = y.detach().float()
    assert torch.isfinite(yf).all() and yf.abs().max() <= 1.0 + (1e-5 if dtype == torch.float32 else 1e-2)
    tol = 2e-6 if dtype == torch.float32 else 1e-2
    # symmetry: tap n at pixel p is the same pair as tap K-1-n at the neighbour (interior pixels)
    k = 2 * R + 1
    taps = [(a, b) for a in range(k) for b in range(k) if (a, b) != (R, R)]
    for n, (a, b) in enumerate(taps):
        dy, dx = a - R, b - R
        lhs = yf[:, n, max(0, -dy):H - max(0, dy), max(0, -dx):W - max(0, dx)]
        rhs = yf[:, K - 1 - n, max(0, dy):H - max(0, -dy), max(0, dx):W - max(0, -dx)]
        assert (lhs - rhs).abs().max() <= tol
    # scale invariance of cosine: y(2x) == y(x) exactly (power-of-two scaling is exact in fp)
    y2 = layer(2 * x)
    assert torch.equal(y2, y.detach())
    # per-pixel orthogonality: cosine is invariant to scaling one pixel's vector, so <gx_p, x_p> == 0
    g = torch.randn(y.shape, generator=gen, device=cuda_device).to(dtype)
    y.backward(g)
    gx = xr.grad.float()
    inner = (gx * x.float()).sum(1)
    scale = (gx.norm(dim=1) * x.float().norm(dim=1)).clamp_min(1e-20)
    assert (inner / scale).abs().max() < (1e-4 if dtype == torch.float32 else 3e-2)
    # linearity of backward in the upstream gradient
    xr2 = x.clone().requires_grad_(True)
    layer(xr2).backward(2 * g)
    assert rel_err(xr2.grad.float().cpu(), (2 * gx).cpu()) < (1e-6 if dtype == torch.float32 else 1e-2)
    # a slice of the big batch against the oracle
    y_ref, gx_ref = O.nfp_forward_backward(x[:2].double().cpu(), g[:2].double().cpu(), R=R, measure="cosine", padding=R)
    ptol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    assert rel_err(yf[:2].cpu(), y_ref) < ptol
    assert rel_err(gx[:2].cpu(), gx_ref) < ptol


def test_autocast_and_no_grad(cuda_device):
    import torch.nn.functional as F
    layer = NFPPooling(64, R=1, measure="cosine", padding=1).to(cuda_device)
    x = torch.randn(2, 64, 7, 7, device=cuda_device)
    xb = x.bfloat16()
    y_ref = O.nfp_forward(xb.double().cpu(), R=1, measure="cosine", padding=1)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        # torch's own rule, which the reference inherits (nfp.py:156): cosine_similarity autocasts to fp32
        assert F.cosine_similarity(xb, xb, dim=1).dtype == torch.float32
        y = layer(x)
        yb = layer(xb)          # what a backbone under autocast hands over: bf16 in, fp32 similarity map out
        xg = xb.clone().requires_grad_(True)
        layer(xg).sum().backward()
        head = nfp_pooling(layer).to(cuda_device)
        h_avg, h_nfp = NF.nfp_gap_pair(x, layer.config)
        hb_avg, hb_nfp = NF.nfp_gap_pair(xb, layer.config)
    assert y.dtype == torch.float32 and yb.dtype == torch.float32
    assert rel_err(yb.cpu(), y_ref) < 1e-5          # fp32 map of the bf16 input: no bf16 rounding of y
    assert rel_err(y.cpu(), O.nfp_forward(x.double().cpu(), R=1, measure="cosine", padding=1)) < FP32_TOL
    assert xg.grad.dtype == torch.bfloat16
    # NFP_Pooling.py:27: avgpool(x) keeps x's dtype under autocast; :31 the pooled similarity is fp32
    assert h_avg.dtype == torch.float32 and h_nfp.dtype == torch.float32
    assert hb_avg.dtype == torch.bfloat16 and hb_nfp.dtype == torch.float32
    with torch.no_grad():
        y = layer(x)
    assert y.dtype == torch.float32 and not y.requires_grad
    xh = x.half().requires_grad_(True)
    layer(xh).sum().backward()
    assert xh.grad.dtype == torch.float16
    with pytest.raises(RuntimeError, match="float64"):
        layer(x.double())
    # a view at an odd storage offset (data pointer not 16-byte aligned) is accepted
    big = torch.randn(2 * 64 * 49 + 1, device=cuda_device)
    xo = big[1:].view(2, 64, 7, 7)
    assert xo.data_ptr() % 16 != 0
    assert rel_err(layer(xo).cpu(), layer(xo.clone()).cpu()) == 0.0
    # non-contiguous (channels_last) input is accepted
    xc = x.to(memory_format=torch.channels_last)
    assert rel_err(layer(xc).cpu(), layer(x).cpu()) == 0.0


def test_scs_batch_coupling_matches_reference_quirk(cuda_device):
    """nfp.py:363-374 broadcasts (B,K,H,W)/(B,1,K,H,W): outputs depend on the other batch elements."""
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(4, 6, 5, 5, generator=gen)
    kw = dict(R=1, measure="scs", p=2, padding=1)
    y_ref = O.nfp_forward(x.double(), **kw)
    y, _ = _run(x, torch.zeros_like(y_ref, dtype=torch.float32), kw, cuda_device)
    assert rel_err(y, y_ref) < 1e-4
    y_single = O.nfp_forward(x[:1].double(), **kw)
    assert rel_err(y[:1], y_single) > 1e-3   # genuinely batch-coupled


def test_resnet18_nfp_training_step_runs(cuda_device):
    """bench_train: the reference's model composition on the drop-in trains (loss finite, parameters move)."""
    import bench_train
    out = bench_train.run_gpu("eurosat", batch=16, steps=3, warmup=1)
    assert out["images_per_s"] > 0 and np.isfinite(out["final_loss"])
    out32 = bench_train.run_gpu("ucmerced", batch=4, steps=2, warmup=1, amp=False)
    assert np.isfinite(out32["final_loss"])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_x_stable_hint_in_stacked_chain(dtype, cuda_device):
    """A.fwd -> B.fwd -> B.bwd(hint) with x_B = y_A (stacked NFP layers, or a recomputation that ends in an NFP
    forward): the hinted backward may start streaming x_B early, but never before A.fwd -- the launch that wrote it --
    has completed, because every fused kernel releases its dependents only after its own dependency wait.  Checked
    against the conservative order (same bits) and the oracle, B = 256, 60 repeats, rotating buffers."""
    import ctypes
    from neighbour_feature_pooling_b200 import _capi
    B, CA, H, W = 256, 512, 7, 7
    CB = 8                                   # layer B consumes A's (B, 8, 7, 7) similarity map
    kd = _capi.F32 if dtype == torch.float32 else _capi.BF16
    gen = torch.Generator().manual_seed(23)
    nbuf = 3
    xa = [torch.randn(B, CA, H, W, generator=gen).to(cuda_device, dtype) for _ in range(nbuf)]
    gyb = [torch.randn(B, 8, H, W, generator=gen).to(cuda_device, dtype) for _ in range(nbuf)]
    dA = _capi.make_desc(kd, B, CA, H, W, 1, 1, 1, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6, "auto")
    dB = _capi.make_desc(kd, B, CB, H, W, 1, 1, 1, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6, "auto")
    assert _capi.describe_path(dA, _capi.OP_FORWARD).startswith("fused/")
    assert _capi.describe_path(dB, _capi.OP_BACKWARD).startswith("fused/")
    lib = _capi.load()
    st = torch.cuda.current_stream().cuda_stream
    res = {}
    for hint in (0, _capi.HINT_X_STABLE):
        dBb = _capi.make_desc(kd, B, CB, H, W, 1, 1, 1, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6, "auto")
        dBb.path |= hint
        ya = [torch.zeros(B, 8, H, W, device=cuda_device, dtype=dtype) for _ in range(nbuf)]
        yb = [torch.zeros(B, 8, H, W, device=cuda_device, dtype=dtype) for _ in range(nbuf)]
        gxb = [torch.zeros(B, CB, H, W, device=cuda_device, dtype=dtype) for _ in range(nbuf)]
        outs = []
        for rep in range(60):
            i = rep % nbuf
            ya[i].fill_(float("nan"))       # a too-early read of x_B would see NaNs
            _capi.check(lib.nfpb200_forward(ctypes.byref(dA), xa[i].data_ptr(), ya[i].data_ptr(), None, 0, st), "A.fwd")
            _capi.check(lib.nfpb200_forward(ctypes.byref(dB), ya[i].data_ptr(), yb[i].data_ptr(), None, 0, st), "B.fwd")
            _capi.check(lib.nfpb200_backward(ctypes.byref(dBb), ya[i].data_ptr(), gyb[i].data_ptr(), gxb[i].data_ptr(),
                                             None, 0, st), "B.bwd")
            if rep >= 60 - nbuf:
                outs.append(gxb[i].clone())
        torch.cuda.synchronize()
        res[hint] = [t.float().cpu() for t in outs] + [t.float().cpu() for t in ya]
    assert all(torch.isfinite(t).all() for t in res[_capi.HINT_X_STABLE])
    assert all(torch.equal(a, b) for a, b in zip(res[0], res[_capi.HINT_X_STABLE]))
    i = (60 - 1) % nbuf
    y_a = res[0][nbuf + i][-2:]
    _, gx_ref = O.nfp_forward_backward(y_a.double(), gyb[i][-2:].double().cpu(), R=1, measure="cosine", padding=1)
    assert rel_err(res[_capi.HINT_X_STABLE][nbuf - 1][-2:], gx_ref) < (FP32_TOL if dtype == torch.float32 else BF16_TOL)


POOL_CASES = [  # (B, C, H, W, R, mode, similarity)
    (5, 64, 7, 7, 1, "zeros", True), (5, 64, 7, 7, 1, "replicate", True), (5, 64, 7, 7, 1, "reflect", False),
    (3, 128, 7, 7, 2, "reflect", True), (3, 128, 7, 7, 2, "zeros", False), (2, 64, 14, 14, 1, "replicate", False),
    (2, 64, 14, 14, 2, "reflect", True), (6, 512, 2, 2, 1, "reflect", True), (4, 32, 4, 4, 1, "zeros", False),
    (2, 960, 7, 7, 1, "reflect", True), (3, 20, 9, 6, 1, "reflect", True), (2, 16, 28, 28, 1, "zeros", True),
]


@pytest.mark.parametrize("case", POOL_CASES, ids=lambda c: "x".join(map(str, c[:4])) + f"_r{c[4]}_{c[5]}_{'sim' if c[6] else 'dist'}")
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_pooled_vs_oracle(case, dtype, cuda_device):
    """nfpb200_pool_forward / nfpb200_pool_backward (the nfp_pooling head, NFP_Pooling.py:27-31) directly against the
    oracle: GAP(x), GAP(NFP(x)) and the input gradient of <g1, GAP(x)> + <g2, GAP(NFP(x))>, for every padding mode,
    similarity flag, window and dtype the fused kernels cover, plus shapes that fall to the other paths."""
    B, C, H, W, R, mode, sim = case
    K = (2 * R + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(B * 131 + C + 7 * H + R)
    x = torch.randn(B, C, H, W, generator=gen)
    x[0, :, 0, 0] = 0.0
    g1 = torch.randn(B, C, generator=gen)
    g2 = torch.randn(B, K, generator=gen)
    if dtype == torch.bfloat16:
        x = x.bfloat16().float()
    kw = dict(R=R, measure="cosine", padding=R, padding_mode=mode, similarity=sim)
    # oracle autograd: the upstream gradient of the map is g2 / (H*W), the same value over a tap plane
    gy = (g2.double() / (H * W))[:, :, None, None].expand(B, K, H, W).contiguous()
    y_map, gx_map = O.nfp_forward_backward(x.double(), gy, **kw)
    y_map, gx_map = torch.as_tensor(np.asarray(y_map)), torch.as_tensor(np.asarray(gx_map))
    gap_nfp_ref = y_map.mean((2, 3))
    gx_ref = gx_map + (g1.double() / (H * W))[:, :, None, None]
    gap_x_ref = x.double().mean((2, 3))
    cfg = NFPPooling(C, **kw).config
    xd = x.to(cuda_device, dtype).requires_grad_(True)
    a, n = NF.nfp_gap_pair(xd, cfg)
    ((a.float() * g1.to(cuda_device)).sum() + (n.float() * g2.to(cuda_device)).sum()).backward()
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    assert rel_err(a.detach().float().cpu(), gap_x_ref) < tol
    assert rel_err(n.detach().float().cpu(), gap_nfp_ref) < tol
    assert grad_err(xd.grad.float().cpu(), gx_ref, x) < tol, worst(grad_errs(xd.grad.float().cpu(), gx_ref, x))
    if NF.describe((B, C, H, W), dtype, cfg, op=2).startswith("fused/"):   # the cluster-split pooled kernels as well
        cfg_s = NF.replace(cfg, path="split")
        xs_ = x.to(cuda_device, dtype).requires_grad_(True)
        a2, n2 = NF.nfp_gap_pair(xs_, cfg_s)
        ((a2.float() * g1.to(cuda_device)).sum() + (n2.float() * g2.to(cuda_device)).sum()).backward()
        assert rel_err(a2.detach().float().cpu(), gap_x_ref) < tol
        assert rel_err(n2.detach().float().cpu(), gap_nfp_ref) < tol
        assert grad_err(xs_.grad.float().cpu(), gx_ref, x) < tol, worst(grad_errs(xs_.grad.float().cpu(), gx_ref, x))


def test_nfp_pooling_respects_customised_layers(cuda_device):
    """The one-pass head replaces nfp_layer(x) only for the stock operator (NFP_Pooling.py:29 always calls the layer):
    forward hooks, a re-bound similarity_measure and subclasses overriding forward must see the call."""
    x = torch.randn(3, 64, 7, 7, device=cuda_device)
    params = {"num_ftrs": {"m": 64}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 5}}
    head = nfp_pooling(Params=params).to(cuda_device)
    assert head._fusable()
    base = head(x)
    calls = []
    h = head.nfp_layer.register_forward_hook(lambda m, i, o: calls.append(o.shape))
    assert not head._fusable()
    hooked = head(x)
    h.remove()
    assert calls == [(3, 8, 7, 7)] and rel_err(hooked.detach().cpu(), base.detach().cpu()) < 1e-6
    head.nfp_layer.similarity_measure = lambda t: torch.ones(t.shape[0], 8, 7, 7, device=t.device)
    assert not head._fusable()
    ones = head(x)
    want = x.mean((2, 3)) * head.nfp_proj(torch.ones(3, 8, device=cuda_device))
    assert rel_err(ones.detach().cpu(), want.detach().cpu()) < 1e-6

    class Doubled(NFPPooling):
        def forward(self, t):
            return 2 * super().forward(t)
    head2 = nfp_pooling(nfp_layer=Doubled(64, R=1, measure="cosine", padding=1), Params=params).to(cuda_device)
    head2.nfp_proj.load_state_dict(head.nfp_proj.state_dict())
    assert not head2._fusable()
    want2 = x.mean((2, 3)) * head.nfp_proj(2 * NFPPooling(64, R=1, measure="cosine", padding=1)(x).mean((2, 3)))
    assert rel_err(head2(x).detach().cpu(), want2.detach().cpu()) < 1e-6


TOKEN_SHAPES = [(5, 64, 7, 7, 1), (3, 512, 7, 7, 1), (2, 960, 7, 7, 1), (3, 192, 14, 14, 1), (2, 256, 14, 14, 1),
                (6, 512, 2, 2, 1), (4, 64, 4, 4, 1), (3, 128, 7, 7, 2), (2, 64, 14, 14, 2), (300, 64, 7, 7, 1)]


@pytest.mark.parametrize("shape", TOKEN_SHAPES, ids=lambda s: "x".join(map(str, s[:4])) + f"_r{s[4]}")
@pytest.mark.parametrize("mode,similarity", [("reflect", True), ("zeros", True), ("replicate", False)],
                         ids=["reflect", "zeros", "replicate_dist"])
def test_channels_last_bf16_without_repack(shape, mode, similarity, cuda_device):
    """SURVEY 8 f2: a channels_last bf16 map is consumed where it lies (no .contiguous() repack): the tensor-core
    fused/token kernels (Gram band and gx = M X on mma.sync, bf16 products exact, fp32 accumulate).  Map and pooled
    modes against the oracle on the bf16-rounded input, gradient returned channels_last, bit-repeatable."""
    B, C, H, W, R = shape
    K = (2 * R + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(B * 77 + C + H + R)
    x = torch.randn(B, C, H, W, generator=gen).bfloat16().float()
    if C % 128 == 0:
        x = x.relu()
    x[0, :, 0, 0] = 0.0
    g = torch.randn(B, K, H, W, generator=gen).bfloat16().float()
    kw = dict(R=R, measure="cosine", padding=R, padding_mode=mode, similarity=similarity)
    layer = NFPPooling(C, **kw).to(cuda_device)
    cfg = layer.config
    assert NF.describe(shape[:4], torch.bfloat16, cfg, layout=1).startswith("fused/token")
    y_ref, gx_ref = O.nfp_forward_backward(x.double(), g.double(), **kw)
    xd = x.to(cuda_device, torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    assert NF._channels_last_ok(xd.detach(), cfg), "expected to be consumed in place"
    y = layer(xd)
    y.backward(g.to(cuda_device, torch.bfloat16))
    assert y.is_contiguous() and y.shape == (B, K, H, W)
    assert xd.grad.stride() == xd.stride() or H * W == 1, "gradient comes back channels_last"
    assert rel_err(y.detach().float().cpu(), y_ref) < BF16_TOL
    assert grad_err(xd.grad.float().cpu(), gx_ref, x) < BF16_TOL, worst(grad_errs(xd.grad.float().cpu(), gx_ref, x))
    # the NCHW kernels on the same values agree to bf16 rounding, and the token path repeats bit for bit
    xn = x.to(cuda_device, torch.bfloat16).requires_grad_(True)
    yn = layer(xn)
    yn.backward(g.to(cuda_device, torch.bfloat16))
    assert rel_err(y.detach().float().cpu(), yn.detach().float().cpu()) < 1e-2
    x2 = xd.detach().clone(memory_format=torch.preserve_format).requires_grad_(True)
    y2 = layer(x2)
    y2.backward(g.to(cuda_device, torch.bfloat16))
    assert torch.equal(y2, y) and torch.equal(x2.grad, xd.grad)
    # pooled head on the same layout
    g1 = torch.randn(B, C, generator=gen)
    g2 = torch.randn(B, K, generator=gen)
    gy = (g2.double() / (H * W))[:, :, None, None].expand(B, K, H, W).contiguous()
    y_map, gx_map = O.nfp_forward_backward(x.double(), gy, **kw)
    y_map, gx_map = torch.as_tensor(np.asarray(y_map)), torch.as_tensor(np.asarray(gx_map))
    x3 = xd.detach().clone(memory_format=torch.preserve_format).requires_grad_(True)
    a, n = NF.nfp_gap_pair(x3, cfg)
    ((a.float() * g1.to(cuda_device)).sum() + (n.float() * g2.to(cuda_device)).sum()).backward()
    assert rel_err(a.detach().float().cpu(), x.double().mean((2, 3))) < BF16_TOL
    assert rel_err(n.detach().float().cpu(), y_map.mean((2, 3))) < BF16_TOL
    assert grad_err(x3.grad.float().cpu(), gx_map + (g1.double() / (H * W))[:, :, None, None], x) < BF16_TOL


def test_vit_token_view_without_transpose_copy(cuda_device):
    """The reference's ViT head (texture_pooling.py:181-188) hands NFP `feats[:, 1:].transpose(1, 2).reshape(B, C, H, W)`:
    a VIEW of the (B, 197, 192) token tensor with strides (197*C, 1, W*C, C).  It is consumed in place (batch stride
    197*C, data pointer one token in), forward and backward, and the gradient reaches the token tensor."""
    B, N, C, H, W = 6, 196, 192, 14, 14
    gen = torch.Generator().manual_seed(5)
    feats = torch.randn(B, N + 1, C, generator=gen).bfloat16()
    g = torch.randn(B, 8, H, W, generator=gen).bfloat16()
    layer = NFPPooling(C, R=1, measure="cosine", padding=1).to(cuda_device)
    fd = feats.to(cuda_device).requires_grad_(True)
    fmap = fd[:, 1:].transpose(1, 2).reshape(B, C, H, W)
    assert fmap.data_ptr() == fd.data_ptr() + C * 2 and fmap.stride() == ((N + 1) * C, 1, W * C, C)   # a view, no copy
    assert NF._channels_last_ok(fmap.detach(), layer.config)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y = layer(fmap)
    assert y.dtype == torch.float32          # autocast: fp32 similarity map from bf16 tokens
    y.backward(g.to(cuda_device).float())
    x_ref = feats[:, 1:].transpose(1, 2).reshape(B, C, H, W).double()
    y_ref, gx_ref = O.nfp_forward_backward(x_ref, g.double(), R=1, measure="cosine", padding=1)
    gx_ref = torch.as_tensor(np.asarray(gx_ref))
    assert rel_err(y.detach().cpu(), y_ref) < 1e-5           # fp32 map of bf16 tokens: only accumulation order differs
    gtok = fd.grad.float().cpu()
    assert torch.count_nonzero(gtok[:, 0]) == 0              # the cls token is not part of the map
    assert rel_err(gtok[:, 1:].transpose(1, 2).reshape(B, C, H, W), gx_ref) < BF16_TOL


def test_fp32_tokens_under_autocast_take_the_token_kernels(cuda_device):
    """A ViT's final LayerNorm emits fp32 tokens under bf16 autocast; the reference's extraction convs round them to
    bf16 (nfp.py:152-153).  The drop-in does the same (one cast instead of an NCHW repack) and stays on the
    channels-last tensor-core path; the map comes back fp32, the gradient fp32."""
    B, N, C, H, W = 3, 196, 192, 14, 14
    gen = torch.Generator().manual_seed(9)
    feats = torch.randn(B, N + 1, C, generator=gen)
    g = torch.randn(B, 8, H, W, generator=gen)
    layer = NFPPooling(C, R=1, measure="cosine", padding=1).to(cuda_device)
    fd = feats.to(cuda_device).requires_grad_(True)
    fmap = fd[:, 1:].transpose(1, 2).reshape(B, C, H, W)
    NF.PATH_TRACE = set()
    try:
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = layer(fmap)
    finally:
        paths, NF.PATH_TRACE = NF.PATH_TRACE, None
    assert paths == {"fused/token_14x14_r1 bf16 channels-last map"}
    assert y.dtype == torch.float32
    y.backward(g.to(cuda_device))
    assert fd.grad.dtype == torch.float32
    xq = feats[:, 1:].transpose(1, 2).reshape(B, C, H, W).bfloat16().double()     # what the reference's convs see
    y_ref, gx_ref = O.nfp_forward_backward(xq, g.double(), R=1, measure="cosine", padding=1)
    assert rel_err(y.detach().cpu(), y_ref) < 1e-5
    assert rel_err(fd.grad[:, 1:].transpose(1, 2).reshape(B, C, H, W).cpu(), gx_ref) < BF16_TOL


@pytest.mark.parametrize("shape", [(5, 64, 7, 7, 1), (3, 512, 7, 7, 1), (2, 960, 7, 7, 1), (3, 256, 14, 14, 1),
                                   (6, 512, 2, 2, 1), (3, 128, 7, 7, 2), (300, 16, 7, 7, 1),
                                   (300, 512, 7, 7, 1)],   # full width, more images than resident CTAs (resident-image backward)
                         ids=lambda s: "x".join(map(str, s[:4])) + f"_r{s[4]}")
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_fused_head_matches_composition_and_oracle(shape, dtype, cuda_device):
    """SURVEY 8 f1: the whole nfp_pooling head (NFP_Pooling.py:25-36) -- GAP(x), GAP(NFP(x)), the K -> C projection and
    the product -- is one launch each way (nfpb200_head_forward / _backward).  Output and all three gradients (x,
    nfp_proj.weight, nfp_proj.bias) against the oracle and against the unfused composition."""
    B, C, H, W, R = shape
    K = (2 * R + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(B + 3 * C + H)
    x = torch.randn(B, C, H, W, generator=gen)
    if dtype == torch.bfloat16:
        x = x.bfloat16().float()
    g = torch.randn(B, C, generator=gen)
    params = {"num_ftrs": {"m": C}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 3}}
    layer = NFPPooling(C, R=R, measure="cosine", padding=R)
    torch.manual_seed(7)
    head = nfp_pooling(nfp_layer=layer, Params=params).to(cuda_device)
    Wp, bp = head.nfp_proj.weight.detach().cpu().double(), head.nfp_proj.bias.detach().cpu().double()
    # oracle: fp64 autograd through the gather-form similarity map
    xr = x.double()
    gy_unit = torch.zeros(B, K, H, W, dtype=torch.float64)
    y_map = torch.as_tensor(np.asarray(O.nfp_forward(xr, R=R, measure="cosine", padding=R)))
    gap_n = y_map.mean((2, 3))
    gap_x = xr.mean((2, 3))
    proj = gap_n @ Wp.t() + bp
    out_ref = gap_x * proj
    t = g.double() * gap_x
    gW_ref, gb_ref = t.t() @ gap_n, t.sum(0)
    g_gap_n = t @ Wp
    gy = (g_gap_n / (H * W))[:, :, None, None].expand(B, K, H, W).contiguous()
    _, gx_map = O.nfp_forward_backward(xr, gy, R=R, measure="cosine", padding=R)
    gx_ref = torch.as_tensor(np.asarray(gx_map)) + ((g.double() * proj) / (H * W))[:, :, None, None]
    xd = x.to(cuda_device, dtype).requires_grad_(True)
    NF.PATH_TRACE = set()
    try:
        out = head(xd)
    finally:
        paths, NF.PATH_TRACE = NF.PATH_TRACE, None
    assert any("fused head" in p for p in paths), paths
    out.backward(g.to(cuda_device, out.dtype))
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    assert rel_err(out.detach().float().cpu(), out_ref) < tol
    assert rel_err(xd.grad.float().cpu(), gx_ref) < tol
    assert rel_err(head.nfp_proj.weight.grad.cpu(), gW_ref) < tol
    assert rel_err(head.nfp_proj.bias.grad.cpu(), gb_ref) < tol
    if dtype != torch.float32:
        return   # (bf16 x with fp32 projection parameters is a dtype error in the unfused composition, as in the reference)
    # the unfused composition (forward hook on the projection switches the fused head off) agrees
    head.zero_grad()
    h = head.nfp_proj.register_forward_hook(lambda m, i, o: None)
    x2 = x.to(cuda_device, dtype).requires_grad_(True)
    out2 = head(x2)
    h.remove()
    out2.backward(g.to(cuda_device, out2.dtype))
    assert rel_err(out2.detach().float().cpu(), out.detach().float().cpu()) < (1e-5 if dtype == torch.float32 else 2e-2)
    assert rel_err(x2.grad.float().cpu(), xd.grad.float().cpu()) < (1e-5 if dtype == torch.float32 else 2e-2)


@pytest.mark.parametrize("shape", [(5, 64, 7, 7, 1), (3, 512, 7, 7, 1), (2, 960, 7, 7, 1), (3, 192, 14, 14, 1),
                                   (6, 512, 2, 2, 1), (3, 128, 7, 7, 2)],
                         ids=lambda s: "x".join(map(str, s[:4])) + f"_r{s[4]}")
def test_fused_head_channels_last(shape, cuda_device):
    """The fused nfp_pooling head on the channels-last tensor-core kernels (what the training steps of bench_train.py
    run): output and the gradients of x, nfp_proj.weight and nfp_proj.bias against the oracle."""
    B, C, H, W, R = shape
    K = (2 * R + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(2 * B + C + H)
    x = torch.randn(B, C, H, W, generator=gen).bfloat16().float()
    g = torch.randn(B, C, generator=gen)
    params = {"num_ftrs": {"m": C}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 3}}
    torch.manual_seed(11)
    head = nfp_pooling(nfp_layer=NFPPooling(C, R=R, measure="cosine", padding=R), Params=params).to(cuda_device)
    Wp, bp = head.nfp_proj.weight.detach().cpu().double(), head.nfp_proj.bias.detach().cpu().double()
    xr = x.double()
    y_map = torch.as_tensor(np.asarray(O.nfp_forward(xr, R=R, measure="cosine", padding=R)))
    gap_n, gap_x = y_map.mean((2, 3)), xr.mean((2, 3))
    proj = gap_n @ Wp.t() + bp
    out_ref = gap_x * proj
    t = g.double() * gap_x
    gy = ((t @ Wp) / (H * W))[:, :, None, None].expand(B, K, H, W).contiguous()
    _, gx_map = O.nfp_forward_backward(xr, gy, R=R, measure="cosine", padding=R)
    gx_ref = torch.as_tensor(np.asarray(gx_map)) + ((g.double() * proj) / (H * W))[:, :, None, None]
    xd = x.to(cuda_device, torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    NF.PATH_TRACE = set()
    try:
        out = head(xd)
    finally:
        paths, NF.PATH_TRACE = NF.PATH_TRACE, None
    assert any("fused/token" in p and "channels-last fused head" in p for p in paths), paths
    out.backward(g.to(cuda_device, out.dtype))
    assert rel_err(out.detach().float().cpu(), out_ref) < BF16_TOL
    assert rel_err(xd.grad.float().cpu(), gx_ref) < BF16_TOL
    assert rel_err(head.nfp_proj.weight.grad.cpu(), t.t() @ gap_n) < BF16_TOL
    assert rel_err(head.nfp_proj.bias.grad.cpu(), t.sum(0)) < BF16_TOL


# ---- SURVEY 8 f3: several radii on the same map in one launch (MultiRadiusNFPHead, models/nfp_heads.py:80-118) ---------
MULTI_SHAPES = [(5, 64, 7, 7), (3, 512, 7, 7), (2, 64, 14, 14), (2, 256, 14, 14), (300, 16, 7, 7)]


def _multi_ref(x, g, mode, similarity):
    """cat([NFP_1(x), NFP_2(x)], dim=1) and its input gradient from the oracle, layer by layer as the reference does."""
    kw1 = dict(R=1, measure="cosine", padding=1, padding_mode=mode, similarity=similarity)
    kw2 = dict(R=2, measure="cosine", padding=2, padding_mode=mode, similarity=similarity)
    y1, gx1 = O.nfp_forward_backward(x.double(), g[:, :8].double().contiguous(), **kw1)
    y2, gx2 = O.nfp_forward_backward(x.double(), g[:, 8:].double().contiguous(), **kw2)
    y1, y2, gx1, gx2 = (torch.as_tensor(np.asarray(t)) for t in (y1, y2, gx1, gx2))
    return torch.cat([y1, y2], dim=1), gx1 + gx2


@pytest.mark.parametrize("shape", MULTI_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("mode,similarity", [("reflect", True), ("zeros", False), ("replicate", True)],
                         ids=["reflect", "zeros_dist", "replicate"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_multi_radius_one_launch_vs_oracle(shape, mode, similarity, dtype, cuda_device):
    """R = 1 and R = 2 on the same map from ONE forward and ONE backward launch (desc.inner_R): the 3x3 window is the
    inner part of the 5x5 window under every padding rule, so the result must equal the reference's block-by-block
    evaluation + torch.cat, and the gradient the sum of the two layers' gradients."""
    B, C, H, W = shape
    gen = torch.Generator().manual_seed(B * 31 + C + H)
    x = torch.randn(B, C, H, W, generator=gen)
    if C % 128 == 0:
        x = x.relu()
    x[0, :, 0, 0] = 0.0
    x[-1, :, H - 1, W - 1] *= 1e-9
    g = torch.randn(B, 32, H, W, generator=gen)
    if dtype == torch.bfloat16:
        x, g = x.bfloat16().float(), g.bfloat16().float()
    blocks = nfpb.MultiRadiusNFP(C, padding_mode=mode, similarity=similarity).to(cuda_device)
    cfgs = [b.config for b in blocks.nfp_blocks]
    assert NF.multi_radius_fusable(cfgs)
    sl = slice(B - 4, B) if B > 32 else slice(0, B)
    y_ref, gx_ref = _multi_ref(x[sl], g[sl], mode, similarity)
    NF.PATH_TRACE = set()
    try:
        xd = x.to(cuda_device, dtype).requires_grad_(True)
        y = blocks(xd)
        y.backward(g.to(cuda_device, dtype))
        trace = set(NF.PATH_TRACE)
    finally:
        NF.PATH_TRACE = None
    assert any("radii 1+2 in one launch" in t and "fused/stream" in t for t in trace), trace
    assert y.shape == (B, 32, H, W)
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    assert rel_err(y.detach().float().cpu()[sl], y_ref) < tol
    errs = grad_errs(xd.grad.float().cpu()[sl], gx_ref, x[sl])
    assert max(errs.values()) < tol, worst(errs)
    # against the same kernels launched once per radius (+ cat): the forward values are the same table entries
    x2 = x.to(cuda_device, dtype).requires_grad_(True)
    y2 = torch.cat([b(x2) for b in blocks.nfp_blocks], dim=1)
    y2.backward(g.to(cuda_device, dtype))
    assert rel_err(y.detach().float().cpu(), y2.detach().float().cpu()) < (2e-6 if dtype == torch.float32 else 1e-2)
    assert grad_err(xd.grad.float().cpu(), x2.grad.float().cpu(), x) < (1e-5 if dtype == torch.float32 else 2e-2)
    # bit-repeatable
    x3 = x.to(cuda_device, dtype).requires_grad_(True)
    y3 = blocks(x3)
    y3.backward(g.to(cuda_device, dtype))
    assert torch.equal(y3, y) and torch.equal(x3.grad, xd.grad)


def test_multi_radius_golden(cuda_device):
    """The one-launch multi-radius path against vectors generated by executing the reference itself (two NFPPooling
    layers + torch.cat, tests/golden/nfp_multi_radius.*), fp32 <= 1e-5; the channels-last bf16 path <= 2e-2."""
    index, arr = load_multi_radius_cases()
    for c in index:
        x = torch.from_numpy(arr[c["key"] + "_x"])
        g = torch.from_numpy(arr[c["key"] + "_g"])
        mr = nfpb.MultiRadiusNFP(c["C"], padding_mode=c["padding_mode"], similarity=c["similarity"]).to(cuda_device)
        NF.PATH_TRACE = set()
        try:
            xd = x.to(cuda_device).requires_grad_(True)
            y = mr(xd)
            y.backward(g.to(cuda_device))
            trace = set(NF.PATH_TRACE)
        finally:
            NF.PATH_TRACE = None
        assert any("radii 1+2 in one launch" in t for t in trace), (c, trace)
        assert rel_err(y.detach().cpu(), arr[c["key"] + "_y"]) < FP32_TOL, c
        assert rel_err(xd.grad.cpu(), arr[c["key"] + "_gx"]) < FP32_TOL, c
        if c["C"] % 64 == 0:   # channels-last bf16: tensor-core token kernels, against the fp64 reference on the fp32 values
            xb = x.to(cuda_device, torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
            yb = mr(xb)
            yb.backward(g.to(cuda_device, torch.bfloat16))
            assert rel_err(yb.detach().float().cpu(), arr[c["key"] + "_y"]) < BF16_TOL, c
            assert rel_err(xb.grad.float().cpu(), arr[c["key"] + "_gx"]) < 3e-2, c   # + the rounding of x and g to bf16


@pytest.mark.parametrize("shape", [(5, 64, 7, 7), (3, 512, 7, 7), (2, 64, 14, 14), (200, 64, 7, 7)],
                         ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("autocast", [False, True], ids=["plain", "autocast"])
def test_multi_radius_channels_last(shape, autocast, cuda_device):
    """The same on a channels_last bf16 map: the tensor-core token kernels, one launch each way, gradient back in
    channels_last; under autocast the map is fp32 (F.cosine_similarity is on autocast's fp32 list)."""
    B, C, H, W = shape
    gen = torch.Generator().manual_seed(B * 13 + C + H)
    x = torch.randn(B, C, H, W, generator=gen).bfloat16().float()
    g = torch.randn(B, 32, H, W, generator=gen).bfloat16().float()
    sl = slice(B - 4, B) if B > 32 else slice(0, B)
    y_ref, gx_ref = _multi_ref(x[sl], g[sl], "reflect", True)
    blocks = nfpb.MultiRadiusNFP(C).to(cuda_device)
    xd = x.to(cuda_device, torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    NF.PATH_TRACE = set()
    try:
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            y = blocks(xd)
        y.backward(g.to(cuda_device, y.dtype))
        trace = set(NF.PATH_TRACE)
    finally:
        NF.PATH_TRACE = None
    assert any("radii 1+2 in one launch" in t and "fused/token" in t and "channels-last" in t for t in trace), trace
    assert y.dtype == (torch.float32 if autocast else torch.bfloat16) and y.shape == (B, 32, H, W)
    assert xd.grad.stride() == xd.stride(), "gradient comes back channels_last"
    assert rel_err(y.detach().float().cpu()[sl], y_ref) < BF16_TOL
    assert rel_err(xd.grad.float().cpu()[sl], gx_ref) < BF16_TOL


@pytest.mark.parametrize("shape", [(2, 16, 28, 28), (3, 12, 12, 8), (2, 8, 5, 8)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("mode,similarity", [("reflect", True), ("zeros", False), ("replicate", True)],
                         ids=["reflect", "zeros_dist", "replicate"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_multi_radius_other_map_sizes(shape, mode, similarity, dtype, cuda_device):
    """Maps outside the fused kernels' shape list with 16-byte aligned planes: the planar row-band kernels take the
    multi-radius launch too (one launch each way, both gradient blocks folded into one stencil)."""
    B, C, H, W = shape
    gen = torch.Generator().manual_seed(B * 17 + C + H)
    x = torch.randn(B, C, H, W, generator=gen)
    x[0, :, 0, 0] = 0.0
    g = torch.randn(B, 32, H, W, generator=gen)
    if dtype == torch.bfloat16:
        x, g = x.bfloat16().float(), g.bfloat16().float()
    y_ref, gx_ref = _multi_ref(x, g, mode, similarity)
    mr = nfpb.MultiRadiusNFP(C, padding_mode=mode, similarity=similarity).to(cuda_device)
    NF.PATH_TRACE = set()
    try:
        xd = x.to(cuda_device, dtype).requires_grad_(True)
        y = mr(xd)
        y.backward(g.to(cuda_device, dtype))
        trace = set(NF.PATH_TRACE)
    finally:
        NF.PATH_TRACE = None
    assert any("radii 1+2 in one launch" in t and "planar/band" in t for t in trace), trace
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    assert rel_err(y.detach().float().cpu(), y_ref) < tol
    errs = grad_errs(xd.grad.float().cpu(), gx_ref, x)
    assert max(errs.values()) < tol, worst(errs)
    x2 = x.to(cuda_device, dtype).requires_grad_(True)   # bit-repeatable
    y2 = mr(x2)
    y2.backward(g.to(cuda_device, dtype))
    assert torch.equal(y2, y) and torch.equal(x2.grad, xd.grad)
    if dtype == torch.bfloat16:   # under autocast the map is fp32 (the band kernels' bf16 result is widened)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            assert mr(x2.detach()).dtype == torch.float32


def test_multi_radius_fallbacks_and_head_fusion(cuda_device):
    """(a) configurations the one-launch form does not cover are computed layer by layer + cat (same values);
    (b) fuse_multi_radius() on a ModuleList built exactly like MultiRadiusNFPHead.nfp_blocks (nfp_heads.py:86-93): the
    head's own `torch.cat([blk(fmap) for blk in self.nfp_blocks], dim=1)` then runs one launch each way."""
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(3, 24, 9, 11, generator=gen)          # a map no fused kernel covers
    g = torch.randn(3, 32, 9, 11, generator=gen)
    y_ref, gx_ref = _multi_ref(x, g, "reflect", True)
    mr = nfpb.MultiRadiusNFP(24).to(cuda_device)
    xd = x.to(cuda_device).requires_grad_(True)
    y = mr(xd)
    y.backward(g.to(cuda_device))
    assert rel_err(y.detach().cpu(), y_ref) < FP32_TOL and rel_err(xd.grad.cpu(), gx_ref) < FP32_TOL
    # a non-nested / non-cosine list is never fused
    assert not NF.multi_radius_fusable([nfpb.NFPPooling(8, R=2, measure="cosine", padding=2).config,
                                        nfpb.NFPPooling(8, R=1, measure="cosine", padding=1).config])
    assert not NF.multi_radius_fusable([nfpb.NFPPooling(8, R=1, measure="dot", padding=1).config,
                                        nfpb.NFPPooling(8, R=2, measure="dot", padding=2).config])
    # (b)
    x = torch.randn(4, 64, 7, 7, generator=gen)
    g = torch.randn(4, 32, 7, 7, generator=gen)
    y_ref, gx_ref = _multi_ref(x, g, "reflect", True)
    blocks = torch.nn.ModuleList([nfpb.EnhancedNFPPooling(in_channels=64, R=R, measure="cosine", padding=R)
                                  for R in (1, 2)]).to(cuda_device)
    keys = list(blocks.state_dict().keys())

    def head_cat(fmap):   # the two lines of MultiRadiusNFPHead.forward that touch the blocks (nfp_heads.py:111-112)
        nfp_maps = [blk(fmap) for blk in blocks]
        return torch.cat(nfp_maps, dim=1)

    assert nfpb.fuse_multi_radius(blocks)
    assert list(blocks.state_dict().keys()) == keys
    NF.PATH_TRACE = set()
    try:
        xd = x.to(cuda_device).requires_grad_(True)
        y = head_cat(xd)
        y.backward(g.to(cuda_device))
        trace = set(NF.PATH_TRACE)
    finally:
        NF.PATH_TRACE = None
    assert len(trace) == 1 and "radii 1+2 in one launch" in next(iter(trace)), trace
    assert rel_err(y.detach().cpu(), y_ref) < FP32_TOL and rel_err(xd.grad.cpu(), gx_ref) < FP32_TOL
    nfpb.unfuse_multi_radius(blocks)
    assert blocks[1](x.to(cuda_device)).shape == (4, 24, 7, 7)
    # a customised block (hook) is left alone
    h = blocks[0].register_forward_hook(lambda m, i, o: o)
    assert not nfpb.fuse_multi_radius(blocks)
    h.remove()
