"""GPU (B200): second order of the cosine operator -- the nfpb200_jvp / nfpb200_backward_backward kernels against the
fp64 oracle, and double backward / forward-mode AD through every autograd entry point.

The oracle is ATen in fp64 on the gather form (oracle/nfp_oracle.py, F.cosine_similarity), whose second derivatives
tests/test_second_order_oracle.py pins to the closed forms of tests/second_order_ref.py.
"""
import ctypes

import pytest
import torch
import torch.autograd.forward_ad as fwAD

import neighbour_feature_pooling_b200 as nfpb
from neighbour_feature_pooling_b200 import _capi
from neighbour_feature_pooling_b200 import functional as NF
from oracle import nfp_oracle as O

from _util import Guarded, bits, grad_errs, image_groups, region_groups, rel_err, rounding_errs, worst
from test_parity_gpu import GEOMS

pytestmark = pytest.mark.gpu

EPS = 1e-6
# (B, C, H, W, R, stride, padding, dilation, mode): the parity grid without its 112x112 map (covered below by the
# autograd tests on the row-band kernels), plus edge geometries: 3 channels, a 1-pixel-high output, pad > R.  (With one
# channel the cosine is +-1 and its derivatives are 0 up to rounding: a relative error measures only noise there.)
KERNEL_GEOMS = [g for g in GEOMS if g[2] < 100] + [
    (2, 3, 6, 6, 1, 1, 1, 1, "reflect"),
    (2, 8, 3, 9, 1, 1, 0, 1, "zeros"),
    (2, 8, 5, 5, 1, 1, 3, 1, "zeros"),
    (3, 64, 7, 7, 2, 1, 2, 1, "replicate"),
]
DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
CDT = {torch.float32: _capi.F32, torch.bfloat16: _capi.BF16, torch.float16: _capi.F16}
TAU = 1e-4          # bf16 / fp16: one rounding of an fp32 evaluation within TAU x the group's largest value
FP32_FLOOR, FP32_CAP, FP32_MULT = 1e-5, 1e-4, 8


def gid(g):
    B, C, H, W, R, s, p, d, m = g
    return f"{B}x{C}x{H}x{W}-R{R}-s{s}-p{p}-d{d}-{m}"


def kw_of(g, sim=True):
    B, C, H, W, R, s, p, d, m = g
    return dict(R=R, stride=s, padding=p, dilation=d, padding_mode=m, similarity=sim, eps=EPS)


def make_input(g, degenerate, seed=0):
    B, C, H, W = g[:4]
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, H, W, generator=gen, dtype=torch.float64)
    if degenerate:
        for b in range(B):
            x[b, :, b % H, (1 + b) % W] = 0.0
            x[b, :, (2 + b) % H, 0] *= 1e-8 / x[b, :, (2 + b) % H, 0].norm()
            x[b, :, H - 1, W - 1] *= 1.5 * EPS / x[b, :, H - 1, W - 1].norm()
    return x


def oracle(x, gy, v, kw):
    """ATen in the dtype of x: (gx2, d<v,gx>/dgy, forward-AD tangent) of the gather-form oracle."""
    f = lambda t: O.nfp_forward(t, measure="cosine", **kw)
    xr, gyr = x.clone().requires_grad_(True), gy.clone().requires_grad_(True)
    (gx,) = torch.autograd.grad(f(xr), xr, gyr, create_graph=True)
    gx2, ggy = torch.autograd.grad(gx, (xr, gyr), v)
    with fwAD.dual_level():
        jf = fwAD.unpack_dual(f(fwAD.make_dual(x, v))).tangent
    return gx2.detach(), ggy.detach(), jf.detach()


def desc_of(x, kw, y_f32=False):
    B, C, H, W = x.shape
    d = _capi.make_desc(CDT[x.dtype], B, C, H, W, kw["R"], kw["stride"], kw["padding"], kw["dilation"],
                        kw["padding_mode"], "cosine", kw["similarity"], False, kw["eps"], 1, 1e-6)
    if y_f32:
        d.path |= _capi.FLAG_Y_F32
    return d


def run_kernels(x, gy, v, kw, ws_fill=None):
    """(gx2, ydot by the reverse rule, ydot by the forward-AD rule) from the C ABI directly."""
    d = desc_of(x, kw)
    lib = _capi.load()
    stream = torch.cuda.current_stream().cuda_stream
    gx2 = torch.empty_like(x)
    ws = torch.empty(_capi.workspace_bytes(d, _capi.OP_BACKWARD_BACKWARD), dtype=torch.uint8, device=x.device)
    if ws_fill is not None:
        ws.fill_(ws_fill)
    assert lib.nfpb200_backward_backward(ctypes.byref(d), x.data_ptr(), gy.data_ptr(), v.data_ptr(), gx2.data_ptr(),
                                         ws.data_ptr(), ws.numel(), stream) == 0
    out = []
    for rule in (_capi.JVP_REVERSE, _capi.JVP_FORWARD_AD):
        yd = torch.empty(gy.shape, dtype=x.dtype, device=x.device)
        assert lib.nfpb200_jvp(ctypes.byref(d), x.data_ptr(), v.data_ptr(), yd.data_ptr(), rule, None, 0, stream) == 0
        out.append(yd)
    torch.cuda.synchronize()
    return gx2, out[0], out[1]


def nan_mask_same(got, want):
    return torch.equal(torch.isnan(got.double().cpu()), torch.isnan(want.double().cpu()))


def finite_mask_same(got, want):
    return torch.equal(torch.isfinite(got.double().cpu()), torch.isfinite(want.double().cpu()))


def _map_errs(got, want):
    return {b: rel_err(got.double().cpu()[m.expand_as(got)], want.cpu()[m.expand_as(want)])
            for b, m in image_groups(want.shape).items()}


@pytest.mark.parametrize("degenerate", [False, True], ids=["clean", "degenerate"])
@pytest.mark.parametrize("sim", [True, False], ids=["sim", "dist"])
@pytest.mark.parametrize("g", KERNEL_GEOMS, ids=gid)
def test_kernels_fp32_vs_oracle(g, sim, degenerate, cuda_device):
    kw = kw_of(g, sim)
    x64 = make_input(g, degenerate).to(cuda_device)
    x32 = x64.float().double()      # the oracle sees the fp32 input
    Ho, Wo = O.geometry(g[2], g[3], g[4], g[5], g[6], g[7], g[8]).Ho, O.geometry(g[2], g[3], g[4], g[5], g[6], g[7], g[8]).Wo
    gen = torch.Generator().manual_seed(5)
    gy = torch.randn(g[0], (2 * g[4] + 1) ** 2 - 1, Ho, Wo, generator=gen).to(cuda_device)
    v = torch.randn(x64.shape, generator=gen).to(cuda_device)
    want = oracle(x32, gy.double(), v.double(), kw)
    aten = oracle(x32.float(), gy, v, kw)    # ATen's own fp32 evaluation
    got = run_kernels(x32.float().contiguous(), gy, v, kw)
    xc = x32.cpu()
    for name, gk, wk, ak in zip(("gx2", "jvp_reverse", "jvp_forward_ad"), got, want, aten):
        assert finite_mask_same(gk, wk), name
        if name == "gx2":
            e, ea = grad_errs(gk.cpu(), wk.cpu(), xc, EPS), grad_errs(ak.cpu(), wk.cpu(), xc, EPS)
        else:
            e, ea = _map_errs(gk, wk), _map_errs(ak, wk)
        for key, err in e.items():
            bound = min(FP32_CAP, max(FP32_FLOOR, FP32_MULT * ea.get(key, 0.0)))
            assert err <= bound, (name, key, err, bound, worst(e))
    again = run_kernels(x32.float().contiguous(), gy, v, kw, ws_fill=0xA5)
    for a, b in zip(got, again):
        assert torch.equal(bits(a), bits(b))


@pytest.mark.parametrize("dt", ["bf16", "f16"])
@pytest.mark.parametrize("degenerate", [False, True], ids=["clean", "degenerate"])
@pytest.mark.parametrize("g", KERNEL_GEOMS[:7] + KERNEL_GEOMS[-1:], ids=gid)
def test_kernels_16bit_round_once(g, degenerate, dt, cuda_device):
    dtype = DT[dt]
    kw = kw_of(g)
    xk = make_input(g, degenerate).to(cuda_device).to(dtype)
    geo = O.geometry(g[2], g[3], g[4], g[5], g[6], g[7], g[8])
    gen = torch.Generator().manual_seed(6)
    gyk = torch.randn(g[0], (2 * g[4] + 1) ** 2 - 1, geo.Ho, geo.Wo, generator=gen).to(cuda_device).to(dtype)
    vk = torch.randn(xk.shape, generator=gen).to(cuda_device).to(dtype)
    want = oracle(xk.double(), gyk.double(), vk.double(), kw)
    got = run_kernels(xk, gyk, vk, kw)
    for name, gk, wk in zip(("gx2", "jvp_reverse", "jvp_forward_ad"), got, want):
        assert nan_mask_same(gk, wk), name
        groups = region_groups(xk.double().cpu(), EPS) if name == "gx2" else None
        e = rounding_errs(gk.cpu(), wk.cpu(), dtype, TAU, groups)
        assert max(e.values()) <= 1.0, (name, worst(e))
    # fp32 tangent for 16-bit x (NFPB200_FLAG_Y_F32)
    d = desc_of(xk, kw, y_f32=True)
    yd = torch.empty(gyk.shape, dtype=torch.float32, device=cuda_device)
    assert _capi.load().nfpb200_jvp(ctypes.byref(d), xk.data_ptr(), vk.data_ptr(), yd.data_ptr(), _capi.JVP_FORWARD_AD,
                                    None, 0, torch.cuda.current_stream().cuda_stream) == 0
    e = _map_errs(yd, want[2])
    assert max(e.values()) <= FP32_CAP, worst(e)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("g", [KERNEL_GEOMS[0], KERNEL_GEOMS[5]], ids=gid)
def test_kernels_guarded(g, dtype, cuda_device):
    """No byte outside the outputs is written, the inputs are untouched, and a poisoned workspace changes nothing."""
    kw = kw_of(g)
    x = make_input(g, True).to(dtype)
    geo = O.geometry(g[2], g[3], g[4], g[5], g[6], g[7], g[8])
    gen = torch.Generator().manual_seed(7)
    gy = torch.randn(g[0], (2 * g[4] + 1) ** 2 - 1, geo.Ho, geo.Wo, generator=gen).to(dtype)
    v = torch.randn(x.shape, generator=gen).to(dtype)
    ref = run_kernels(x.to(cuda_device), gy.to(cuda_device), v.to(cuda_device), kw)
    d = desc_of(x, kw)
    lib = _capi.load()
    stream = torch.cuda.current_stream().cuda_stream
    n_ws = _capi.workspace_bytes(d, _capi.OP_BACKWARD_BACKWARD)
    bx = Guarded(x.numel(), dtype, cuda_device, "input", data=x)
    bgy = Guarded(gy.numel(), dtype, cuda_device, "input", data=gy)
    bv = Guarded(v.numel(), dtype, cuda_device, "input", data=v)
    bo = Guarded(x.numel(), dtype, cuda_device, "output")
    bw = Guarded(n_ws, torch.uint8, cuda_device, "workspace")
    assert lib.nfpb200_backward_backward(ctypes.byref(d), bx.ptr(), bgy.ptr(), bv.ptr(), bo.ptr(), bw.ptr(), n_ws,
                                         stream) == 0
    yo = Guarded(gy.numel(), dtype, cuda_device, "output")
    assert lib.nfpb200_jvp(ctypes.byref(d), bx.ptr(), bv.ptr(), yo.ptr(), _capi.JVP_REVERSE, None, 0, stream) == 0
    torch.cuda.synchronize()
    bufs = {"x": bx, "gy": bgy, "v": bv, "gx2": bo, "ydot": yo}
    probs = [m for n, gb in bufs.items() for m in gb.problems(n)]
    probs += [m for m in bw.problems("workspace") if "guard" in m]
    assert not probs, probs
    assert torch.equal(bits(bo.body.view(x.shape)), bits(ref[0])) and torch.equal(bits(yo.body.view(gy.shape)), bits(ref[1]))


# ---- autograd through every entry point --------------------------------------------------------------------------------
def double_backward(f, x, g, v):
    """(d<v, d<g, f(x)>/dx>/dx, d<g, f>/dx) for any f: the second derivative as a gradient penalty takes it."""
    xr = x.detach().clone().requires_grad_(True)
    out = f(xr)
    outs = out if isinstance(out, tuple) else (out,)
    gs = g if isinstance(g, tuple) else (g,)
    (gx,) = torch.autograd.grad(outs, xr, [gi.to(o.dtype) for gi, o in zip(gs, outs)], create_graph=True)
    (gx2,) = torch.autograd.grad(gx, xr, v.to(gx.dtype))
    return gx2.detach(), gx.detach()


def tangent(f, x, v):
    with fwAD.dual_level():
        out = f(fwAD.make_dual(x.detach(), v.to(x.dtype)))
        outs = out if isinstance(out, tuple) else (out,)
        return tuple(fwAD.unpack_dual(o).tangent.detach() for o in outs)


def ref_fn(name, cfgs, w=None, b=None):
    """The oracle composition of entry point `name` (fp64 on the gather form)."""
    def nfp(t, c):
        return O.nfp_forward(t, R=c.R, measure="cosine", stride=c.stride, padding=c.padding, dilation=c.dilation,
                             padding_mode=c.padding_mode, similarity=c.similarity, eps=c.eps)
    c = cfgs[-1]
    if name == "map":
        return lambda t: nfp(t, c)
    if name == "multi":
        return lambda t: torch.cat([nfp(t, k) for k in cfgs], 1)
    if name == "pooled":
        return lambda t: nfp(t, c).mean((2, 3))
    if name == "gap_pair":
        return lambda t: (t.mean((2, 3)), nfp(t, c).mean((2, 3)))
    return lambda t: t.mean((2, 3)) * (nfp(t, c).mean((2, 3)) @ w.t() + b)


def fn(name, cfgs, w=None, b=None, autocast=False):
    c = cfgs[-1]
    def wrap(f):
        if not autocast:
            return f
        def g(t):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return f(t)
        return g
    if name == "map":
        return wrap(lambda t: NF.nfp_similarity(t, c))
    if name == "multi":
        return wrap(lambda t: NF.nfp_multi_radius(t, cfgs))
    if name == "pooled":
        return wrap(lambda t: NF.nfp_pooled_similarity(t, c))
    if name == "gap_pair":
        return wrap(lambda t: NF.nfp_gap_pair(t, c))
    return wrap(lambda t: NF.nfp_head(t, w, b, c))


def cfg(R=1, padding=None, **kw):
    return NF.NFPConfig(R=R, measure="cosine", padding=R if padding is None else padding, **kw)


# (id, entry point, configs, shape, dtype, channels_last + bf16 autocast, expected kernel path of the map forward)
AUTOGRAD = [
    ("ring-f32", "map", [cfg()], (4, 64, 7, 7), torch.float32, False, "fused/stream"),
    ("ring-bf16", "map", [cfg()], (4, 64, 7, 7), torch.bfloat16, False, "fused/stream"),
    ("ring-f16", "map", [cfg()], (4, 64, 7, 7), torch.float16, False, "fused/stream"),
    ("token-bf16-autocast", "map", [cfg()], (3, 64, 14, 14), torch.bfloat16, True, "fused/token"),
    ("band-f32", "map", [cfg()], (2, 16, 112, 112), torch.float32, False, "planar/band"),
    ("generic-stride2", "map", [cfg(stride=2)], (2, 8, 9, 9), torch.float32, False, "generic/pairs"),
    ("multi-ring-f32", "multi", [cfg(1), cfg(2)], (3, 64, 7, 7), torch.float32, False, None),
    ("multi-band-f32", "multi", [cfg(1), cfg(2)], (2, 16, 20, 20), torch.float32, False, None),
    ("pooled-ring-f32", "pooled", [cfg()], (4, 64, 7, 7), torch.float32, False, None),
    ("pooled-band-f32", "pooled", [cfg()], (2, 16, 28, 28), torch.float32, False, None),
    ("pooled-ring-bf16", "pooled", [cfg()], (4, 64, 7, 7), torch.bfloat16, False, None),
    ("gap-ring-f32", "gap_pair", [cfg()], (4, 64, 7, 7), torch.float32, False, None),
    ("gap-generic-f32", "gap_pair", [cfg(stride=2)], (2, 8, 9, 9), torch.float32, False, None),
    ("head-ring-f32", "head", [cfg()], (4, 64, 7, 7), torch.float32, False, None),
    ("head-ring-bf16", "head", [cfg()], (4, 64, 7, 7), torch.bfloat16, False, None),
    ("head-token-bf16", "head", [cfg()], (3, 64, 14, 14), torch.bfloat16, True, None),
]
# the composition's relative error per image / pixel region: fp32 kernels; 16-bit inputs round gy and the results
AUTOGRAD_TOL = {torch.float32: 1e-4, torch.bfloat16: 3e-2, torch.float16: 1e-2}


@pytest.mark.parametrize("case", AUTOGRAD, ids=[c[0] for c in AUTOGRAD])
def test_autograd_double_backward_and_forward_ad(case, cuda_device):
    name, entry, cfgs, shape, dtype, cl, want_path = case
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(shape, generator=gen).to(dtype)
    B, C = shape[:2]
    w = b = None
    if entry == "head":
        K = cfgs[-1].out_channels
        w = (torch.randn(C, K, generator=gen) * 0.1).to(cuda_device)
        b = torch.randn(C, generator=gen).to(cuda_device)
    xd = x.to(cuda_device)
    if cl:
        xd = xd.contiguous(memory_format=torch.channels_last)
    f = fn(entry, cfgs, w, b, autocast=cl)
    if want_path is not None:
        NF.PATH_TRACE = set()
        try:
            f(xd)
        finally:
            trace, NF.PATH_TRACE = NF.PATH_TRACE, None
        assert any(t.startswith(want_path) for t in trace), trace
    with torch.no_grad():
        out = f(xd)
    outs = out if isinstance(out, tuple) else (out,)
    g = tuple(torch.randn(o.shape, generator=gen).to(cuda_device) for o in outs)
    v = torch.randn(shape, generator=gen).to(cuda_device)
    gx2, gx = double_backward(f, xd, g if len(g) > 1 else g[0], v)
    x64 = x.double().to(cuda_device)
    rf = ref_fn(entry, cfgs, w.double() if w is not None else None, b.double() if b is not None else None)
    gx2_ref, gx_ref = double_backward(rf, x64, tuple(t.double() for t in g) if len(g) > 1 else g[0].double(),
                                      v.double())
    tol = AUTOGRAD_TOL[dtype]
    for got, want, what in ((gx, gx_ref, "gx"), (gx2, gx2_ref, "gx2")):
        assert torch.isfinite(got).all(), what
        e = grad_errs(got.double().cpu(), want.cpu(), x64.cpu(), EPS)
        assert max(e.values()) <= tol, (what, worst(e))
    for got, want in zip(tangent(f, xd, v), tangent(rf, x64, v.double())):
        assert rel_err(got.double().cpu(), want.cpu()) <= tol


def test_head_forward_ad_with_dual_weight_and_bias(cuda_device):
    gen = torch.Generator().manual_seed(12)
    c = cfg()
    x = torch.randn(4, 64, 7, 7, generator=gen).to(cuda_device)
    w, b = (torch.randn(64, 8, generator=gen) * 0.1).to(cuda_device), torch.randn(64, generator=gen).to(cuda_device)
    vx, vw, vb = (torch.randn(t.shape, generator=gen).to(cuda_device) for t in (x, w, b))
    with fwAD.dual_level():
        out = NF.nfp_head(fwAD.make_dual(x, vx), fwAD.make_dual(w, vw), fwAD.make_dual(b, vb), c)
        got = fwAD.unpack_dual(out).tangent
    rf = lambda xx, ww, bb: ref_fn("head", [c], ww, bb)(xx)
    with fwAD.dual_level():
        want = fwAD.unpack_dual(rf(fwAD.make_dual(x.double(), vx.double()), fwAD.make_dual(w.double(), vw.double()),
                                   fwAD.make_dual(b.double(), vb.double()))).tangent
    assert rel_err(got.double().cpu(), want.cpu()) <= 1e-4


def test_r1_penalty_training_step_matches_the_oracle(cuda_device):
    """One step of loss = sum(head(x) * t) + gamma ||d sum(head(x))/dx||^2 on the nfp_pooling head (fused kernels)."""
    Params = {"num_ftrs": {"m": 64}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 3}}
    torch.manual_seed(0)
    pool = nfpb.nfp_pooling(Params=Params).to(cuda_device)
    gen = torch.Generator().manual_seed(13)
    x = torch.randn(4, 64, 7, 7, generator=gen)
    tgt = torch.randn(4, 64, generator=gen)

    def step(model_fn, params, xx, tt):
        xr = xx.clone().requires_grad_(True)
        out = model_fn(xr)
        (gx,) = torch.autograd.grad(out.sum(), xr, create_graph=True)
        loss = (out * tt).sum() + 10.0 * gx.pow(2).sum()
        return [t.detach() for t in torch.autograd.grad(loss, params)]

    got = step(pool, [pool.nfp_proj.weight, pool.nfp_proj.bias], x.to(cuda_device), tgt.to(cuda_device))
    w = pool.nfp_proj.weight.detach().double().clone().requires_grad_(True)
    b = pool.nfp_proj.bias.detach().double().clone().requires_grad_(True)
    want = step(lambda t: O.nfp_pooling_forward(t, w, b), [w, b], x.double().to(cuda_device), tgt.double().to(cuda_device))
    for gg, ww in zip(got, want):
        assert rel_err(gg.double().cpu(), ww.cpu()) <= 1e-4


# ---- first order unchanged -------------------------------------------------------------------------------------------
def test_first_order_bits_and_trace_unchanged(cuda_device):
    gen = torch.Generator().manual_seed(14)
    c = cfg()
    x = torch.randn(4, 64, 7, 7, generator=gen).to(cuda_device)
    g = torch.randn(4, 8, 7, 7, generator=gen).to(cuda_device)
    NF.PATH_TRACE = set()
    try:
        xr = x.clone().requires_grad_(True)
        (gx,) = torch.autograd.grad(NF.nfp_similarity(xr, c), xr, g)
        trace, NF.PATH_TRACE = NF.PATH_TRACE, None
    finally:
        NF.PATH_TRACE = None
    assert len(trace) == 1 and all(t.endswith(" map") for t in trace), trace
    d = NF._desc_for(x, c)
    direct = torch.empty_like(x)
    ws, ws_ptr, ws_n = NF._workspace(d, _capi.OP_BACKWARD, x.device)
    assert _capi.load().nfpb200_backward(ctypes.byref(d), x.data_ptr(), g.data_ptr(), direct.data_ptr(), ws_ptr, ws_n,
                                         torch.cuda.current_stream().cuda_stream) == 0
    assert torch.equal(bits(gx), bits(direct))
    # pooled head: one fused head backward call
    w, b = torch.randn(64, 8, generator=gen).to(cuda_device), torch.randn(64, generator=gen).to(cuda_device)
    go = torch.randn(4, 64, generator=gen).to(cuda_device)
    xr = x.clone().requires_grad_(True)
    (gxh,) = torch.autograd.grad(NF.nfp_head(xr, w, b, c), xr, go)
    out, gap_x, gap_nfp = (torch.empty(4, 64, device=cuda_device), torch.empty(4, 64, device=cuda_device),
                           torch.empty(4, 8, device=cuda_device))
    lib, s = _capi.load(), torch.cuda.current_stream().cuda_stream
    assert lib.nfpb200_head_forward(ctypes.byref(d), x.data_ptr(), w.data_ptr(), b.data_ptr(), out.data_ptr(),
                                    gap_x.data_ptr(), gap_nfp.data_ptr(), s) == 0
    direct = torch.empty_like(x)
    assert lib.nfpb200_head_backward(ctypes.byref(d), x.data_ptr(), w.data_ptr(), b.data_ptr(), gap_x.data_ptr(),
                                     gap_nfp.data_ptr(), go.data_ptr(), direct.data_ptr(), s) == 0
    assert torch.equal(bits(gxh), bits(direct))


def test_non_cosine_double_backward_still_raises(cuda_device):
    layer = nfpb.NFPPooling(8, R=1, measure="norm", padding=1).to(cuda_device)
    x = torch.randn(2, 8, 7, 7, device=cuda_device, requires_grad=True)
    (gx,) = torch.autograd.grad(layer(x).sum(), x, create_graph=True)
    with pytest.raises(RuntimeError):
        torch.autograd.grad(gx.sum(), x)
