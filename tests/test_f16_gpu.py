"""GPU: native fp16 (NFPB200_F16) on the NCHW ring kernels and the channels-last token kernels.

* every ring / token cell (all entry points, all ring shapes, the ViT token view and padded gx strides, three padding
  modes, similarity on and off, multi-radius, fp32 maps) against the fp64 oracle on the fp16-rounded input: fp32
  results <= 1e-5, fp16 maps <= 1e-3, input gradients grad_err <= 2e-3 (each image and pixel region on its own scale);
  on the same call: bit-identical reruns, the C ABI's memory contract on guarded buffers at the weakest alignment, and
  a captured CUDA graph with exactly nfpb200_launch_count nodes that replays to the same bits;
* degenerate pixels (norm ~eps) whose gradient overflows fp16: gx is +-inf exactly where the fp16 rounding of the
  oracle's gradient is, and the finite elements are scored per region;
* the ring kernels against what fp16 inputs took before (the fp32 kernels on x.float(), narrowed): within 1 fp16 ulp;
* the module level: autocast, .half() layers, the ViT token view, the fused nfp_pooling head.
"""
import numpy as np
import pytest
import torch

import _util
import test_abi_contract_gpu as AC
from _util import fill_bits, grad_errs, guard_problems, rel_err, worst
from neighbour_feature_pooling_b200 import NFPPooling, _capi, nfp_pooling
from neighbour_feature_pooling_b200 import functional as NF
from oracle import nfp_oracle as O

pytestmark = pytest.mark.gpu

F16 = torch.float16
# guarded-buffer fill patterns for fp16 (quiet NaN, and a NaN with a recognisable payload)
_util.QNAN.setdefault(F16, 0x7E00)
_util.SENTINEL.setdefault(F16, 0x7DA5)
_util._BITS.setdefault(F16, torch.int16)

# bounds, with the worst case test_f16_cell measured over its grid on one B200 (1000 W power limit)
TOL_F32 = 1e-5       # fp32 maps, GAP vectors, head outputs; measured 6.9e-7 (token forward, fp32 map of the ViT view)
TOL_F16_MAP = 1e-3   # fp16 maps; measured 3.9e-4 (one fp16 rounding: 2^-11 = 4.9e-4)
TOL_GRAD = 2e-3      # grad_err of gx; measured 4.8e-4 (token pooled backward)
EPS = 1e-6


def _cell(family, entry, shape, **opts):
    return AC._cell(family, entry, shape, F16, **opts)


class F16Problem(AC.Problem):
    """A grid cell of the C-ABI contract suite with an fp16 descriptor (and optionally similarity off)."""

    def __init__(self, c):
        self.sim = bool(dict(c.opts).get("sim", 1))
        super().__init__(c)
        self.desc.dtype = _capi.F16
        self.desc.similarity = int(self.sim)

    def _kw(self, R=None, padding=None):
        kw = super()._kw(R, padding)
        kw["similarity"] = self.sim
        return kw


def _grid():
    g = []
    for s in AC.STREAM_INST:
        g += [_cell("stream", e, s) for e in AC.ENTRIES]
    for s in [(3, 64, 7, 7, 1), (2, 64, 14, 14, 1)]:
        for mode in ("reflect", "zeros", "replicate"):
            for sim in (1, 0):
                if (mode, sim) != ("reflect", 1):
                    g += [_cell("stream", e, s, mode=mode, sim=sim) for e in ("forward", "backward", "pool_backward")]
    g += [_cell("stream", "forward", s, yf32=1) for s in [(3, 64, 7, 7, 1), (2, 32, 14, 14, 2)]]
    g += [_cell("stream", "backward", (3, 40, 7, 7, 1))]                                  # strip form (C % 64 != 0)
    g += [_cell("stream", e, (3, 512, 7, 7, 1)) for e in ("forward", "backward")]
    for s in [(3, 64, 7, 7, 2), (2, 32, 14, 14, 2)]:
        g += [_cell("stream", e, s, inner=1) for e in ("forward", "backward")]
    vit = (3, 64, 14, 14, 1)
    for e in AC.ENTRIES:
        bwd = e.endswith("backward")
        for i, xbs in enumerate(("dense", "pad8", "vit")):
            g.append(_cell("token", e, vit, xbs=xbs, gxbs=("0", "pad8", "pad64")[i] if bwd else "0"))
    g += [_cell("token", e, (2, 192, 7, 7, 1), xbs="pad8", gxbs="pad64") for e in AC.ENTRIES]
    g += [_cell("token", e, (2, 512, 7, 7, 1)) for e in ("forward", "backward")]
    g += [_cell("token", e, (2, 64, 4, 4, 1)) for e in ("forward", "backward")]
    g += [_cell("token", e, (3, 64, 7, 7, 2), inner=1, xbs="pad8", gxbs="pad8") for e in ("forward", "backward")]
    for mode in ("reflect", "zeros", "replicate"):
        for sim in (1, 0):
            if (mode, sim) != ("reflect", 1):
                g += [_cell("token", e, (2, 64, 7, 7, 1), mode=mode, sim=sim) for e in ("forward", "backward")]
    g += [_cell("token", "forward", (2, 192, 14, 14, 1), yf32=1, xbs="vit")]
    return g


GRID = _grid()


def cell_id(c):
    return AC.cell_id(c).replace("-bf16", "-f16")


def _tol(prob, name):
    if name == "gx":
        return TOL_GRAD
    if name == "y" and not prob.yf32:
        return TOL_F16_MAP
    return TOL_F32


@pytest.mark.parametrize("c", [pytest.param(c, id=cell_id(c)) for c in GRID])
def test_f16_cell(c, cuda_device):
    prob = F16Problem(c)
    assert prob.path().startswith(AC.FAMILIES[c.family][0]), prob.path()
    pb, pws = prob.plain(cuda_device)
    AC._run(prob, pb, pws)
    torch.cuda.synchronize()
    want = AC._out_bits(prob, pb)
    # against the fp64 oracle on the fp16-rounded input
    exp, rows = prob.expected()
    for n, ref in exp.items():
        got = prob.logical(n, pb[n])[rows]
        if n == "gx":
            errs = grad_errs(got, ref, prob.x[rows], EPS)
            assert max(errs.values()) <= TOL_GRAD, worst(errs)
        else:
            e = max(rel_err(got[i], ref[i]) for i in range(len(rows)))
            assert e <= _tol(prob, n), (n, e)
    # reruns: identical bits
    AC._run(prob, pb, pws)
    torch.cuda.synchronize()
    assert all(AC._same_bits(AC._out_bits(prob, pb), want).values()), "rerun"
    # guarded buffers at the weakest alignment (sentinel, then zero workspace)
    for zero_ws in (False, True):
        gb, gws = prob.guarded(cuda_device, zero_ws)
        AC._run(prob, gb, gws)
        torch.cuda.synchronize()
        problems = guard_problems({**gb, "workspace": gws})
        assert not problems, problems
        same = AC._same_bits(AC._out_bits(prob, gb), want)
        assert all(same.values()), ("zero workspace" if zero_ws else "sentinel workspace", same)
    # one call captured alone: nfpb200_launch_count nodes, replaying to the same bits
    for n in prob.outputs:
        fill_bits(pb[n], _util.SENTINEL[pb[n].dtype])
    graph = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.graph(graph):
        AC._run(prob, pb, pws, torch.cuda.current_stream().cuda_stream)
    counts = AC.graph_node_counts(graph)
    launches = counts.get(AC.CU_GRAPH_NODE_TYPE_KERNEL, 0) + counts.get(AC.CU_GRAPH_NODE_TYPE_MEMSET, 0)
    assert launches == prob.launch_count() and sum(counts.values()) == launches, (counts, prob.launch_count())
    graph.instantiate()
    graph.replay()
    torch.cuda.synchronize()
    assert all(AC._same_bits(AC._out_bits(prob, pb), want).values()), "graph replay"


# ---- degenerate pixels: fp16 overflow of the gradient ------------------------------------------------------------------
def _degenerate(B, C, H, W, seed):
    """Positive activations with three pixels per image of norm 0.9 eps.  The map gradient of those pixels is
    >= 1e5 in every channel (far above fp16's 65504), every other gradient element is below 1: no element sits near
    the overflow boundary."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, H, W, generator=g).abs() + 0.5
    for b in range(B):
        for h, w in ((1, 1), (H - 2, W // 2), (H // 2, 0)):
            x[b, :, h, w] = 0.0
            x[b, 0, h, w] = 0.9 * EPS
    gy = torch.rand(B, 8, H, W, generator=g) + 0.5
    return x.half(), gy.half()


@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("hw", [7, 14])
@pytest.mark.parametrize("mode", ["reflect", "zeros", "replicate"])
def test_f16_gradient_overflow(layout, hw, mode, cuda_device):
    x, gy = _degenerate(2, 64, hw, hw, hw)
    _, want = O.nfp_forward_backward(x.double(), gy.double(), R=1, measure="cosine", padding=1, padding_mode=mode,
                                     similarity=True, eps=EPS)
    want = torch.as_tensor(np.asarray(want))
    a = want.abs()
    assert not ((a > 0.9 * 65520) & (a < 1.1 * 65520)).any()    # the planted data keeps away from the boundary
    want16 = want.half()
    cfg = NF.NFPConfig(R=1, measure="cosine", padding=1, padding_mode=mode, eps=EPS)
    xd = x.to(cuda_device)
    if layout == "channels_last":
        xd = xd.contiguous(memory_format=torch.channels_last)
    xd.requires_grad_(True)
    NF.PATH_TRACE = set()
    try:
        y = NF.nfp_similarity(xd, cfg)
        trace = set(NF.PATH_TRACE)
    finally:
        NF.PATH_TRACE = None
    fam = "fused/token_" if layout == "channels_last" else "fused/stream_"
    assert all(t.startswith(fam) and " f16 " in t for t in trace), trace
    y.backward(gy.to(cuda_device))
    got = xd.grad.detach().cpu()
    assert got.dtype == F16
    inf_g, inf_w = torch.isinf(got), torch.isinf(want16)
    assert inf_w.sum() == 2 * 3 * 64
    assert torch.equal(inf_g, inf_w) and torch.equal(torch.sign(got[inf_g]), torch.sign(want16[inf_w]))
    fin = ~inf_w
    errs = grad_errs(torch.where(fin, got.double(), 0.0), torch.where(fin, want, 0.0), x.double(), EPS)
    assert max(errs.values()) <= TOL_GRAD, worst(errs)


# ---- the ring kernels against the widened route -------------------------------------------------------------------
def _ulp16(v):
    """fp16 ulp at |v| (float64 tensor)."""
    e = torch.floor(torch.log2(v.abs().clamp_min(2.0 ** -14)))
    return torch.exp2(e - 10)


def _within_one_ulp(a, b):
    a, b = a.double(), b.double()
    inf = torch.isinf(a) | torch.isinf(b)
    if not torch.equal(a[inf], b[inf]):
        return False
    d = (a - b).abs()[~inf]
    return bool((d <= _ulp16(torch.maximum(a.abs(), b.abs())[~inf])).all())


@pytest.mark.parametrize("shape", AC.STREAM_INST)
def test_f16_ring_matches_widened_route(shape, cuda_device):
    B, C, H, W, R = shape
    g = torch.Generator().manual_seed(B * 1000 + C + H + R)
    x = torch.randn(B, C, H, W, generator=g).half().to(cuda_device)
    cfg = NF.NFPConfig(R=R, measure="cosine", padding=R)
    assert NF.describe(x.shape, F16, cfg).startswith("fused/stream_")
    K = (2 * R + 1) ** 2 - 1
    gy = torch.randn(B, K, H, W, generator=g).half().to(cuda_device)
    # upstream gradients of the fp16 outputs: fp16 values, so that both routes see the same ones
    gg = (torch.randn(B, C, generator=g).half().float().to(cuda_device),
          torch.randn(B, K, generator=g).half().float().to(cuda_device))

    def run(xin, narrow):
        xin = xin.detach().requires_grad_(True)
        y = NF.nfp_similarity(xin, cfg)
        y.backward(gy.to(y.dtype))
        outs = [y.detach(), xin.grad]
        xin2 = xin.detach().requires_grad_(True)
        a, n = NF.nfp_gap_pair(xin2, cfg)
        torch.autograd.backward([a, n], [gg[0].to(a.dtype), gg[1].to(n.dtype)])
        outs += [a.detach(), n.detach(), xin2.grad]
        xin3 = xin.detach().requires_grad_(True)
        p = NF.nfp_pooled_similarity(xin3, cfg)
        p.backward(gg[1].to(p.dtype))
        outs += [p.detach(), xin3.grad]
        return [o.half() if narrow else o for o in outs]
    native = run(x, False)
    widened = run(x.float(), True)
    names = ("y", "gx", "gap_x", "gap_nfp", "gx_pool", "pooled_map", "gx_pooled_map")
    for n, a, b in zip(names, native, widened):
        assert a.dtype == F16, n
        assert _within_one_ulp(a.cpu(), b.cpu()), (n, (a.double() - b.double()).abs().max().item())


# ---- module level ---------------------------------------------------------------------------------------------------
def _traced(fn):
    NF.PATH_TRACE = set()
    try:
        out = fn()
        return out, set(NF.PATH_TRACE)
    finally:
        NF.PATH_TRACE = None


def test_module_channels_last_fp16_under_autocast(cuda_device):
    layer = NFPPooling(64, R=1, measure="cosine", padding=1).to(cuda_device)
    x = torch.randn(2, 64, 7, 7, device=cuda_device).half().contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    with torch.autocast("cuda"):          # fp16 by default
        y, trace = _traced(lambda: layer(x))
    assert trace and all(t.startswith("fused/token_7x7_r1 f16 channels-last") for t in trace), trace
    assert y.dtype == torch.float32
    assert rel_err(y.detach().cpu(), O.nfp_forward(x.detach().double().cpu(), R=1, measure="cosine", padding=1)) <= TOL_F32
    y.sum().backward()
    assert x.grad.dtype == F16 and x.grad.is_contiguous(memory_format=torch.channels_last)


def test_module_half_layer_nchw(cuda_device):
    layer = NFPPooling(64, R=1, measure="cosine", padding=1).to(cuda_device).half()
    x = torch.randn(2, 64, 7, 7, device=cuda_device).half().requires_grad_(True)
    y, trace = _traced(lambda: layer(x))
    assert trace and all(t.startswith("fused/stream_7x7_r1 f16 nchw") for t in trace), trace
    assert y.dtype == F16
    gy = torch.randn_like(y)
    y.backward(gy)
    assert x.grad.dtype == F16
    yr, gr = O.nfp_forward_backward(x.detach().double().cpu(), gy.double().cpu(), R=1, measure="cosine", padding=1)
    assert rel_err(y.detach().cpu(), yr) <= TOL_F16_MAP
    errs = grad_errs(x.grad.cpu(), gr, x.detach().double().cpu(), EPS)
    assert max(errs.values()) <= TOL_GRAD, worst(errs)


def test_module_vit_tokens_under_fp16_autocast(cuda_device):
    """fp32 LayerNorm tokens under fp16 autocast: rounded to fp16 (as the reference's extraction convs do) and taken
    by the token kernels in place of an NCHW repack."""
    B, C, H, W = 2, 192, 14, 14
    feats = torch.randn(B, H * W + 1, C, device=cuda_device, requires_grad=True)
    cfg = NF.NFPConfig(R=1, measure="cosine", padding=1)
    with torch.autocast("cuda", dtype=torch.float16):
        view = feats[:, 1:].transpose(1, 2).reshape(B, C, H, W)
        y, trace = _traced(lambda: NF.nfp_similarity(view, cfg))
    assert trace and all(t.startswith("fused/token_14x14_r1 f16 channels-last") for t in trace), trace
    assert y.dtype == torch.float32
    xq = feats.detach()[:, 1:].transpose(1, 2).reshape(B, C, H, W).half().double().cpu()
    gy = torch.randn_like(y)
    yr, gr = O.nfp_forward_backward(xq, gy.half().double().cpu(), R=1, measure="cosine", padding=1)
    assert rel_err(y.detach().cpu(), yr) <= TOL_F32
    y.backward(gy)
    assert feats.grad.dtype == torch.float32
    got = feats.grad[:, 1:].transpose(1, 2).reshape(B, C, H, W).cpu()
    errs = grad_errs(got, gr, xq, EPS)
    assert max(errs.values()) <= TOL_GRAD, worst(errs)
    assert bool((feats.grad[:, 0] == 0).all())


def test_module_nfp_pooling_fused_head_under_fp16_autocast(cuda_device):
    Params = {"num_ftrs": {"m": 64}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 3}}
    torch.manual_seed(0)
    pool = nfp_pooling(Params=Params).to(cuda_device)
    x = torch.randn(2, 64, 7, 7, device=cuda_device).half().requires_grad_(True)
    with torch.autocast("cuda"):
        out, trace = _traced(lambda: pool(x))
    assert len(trace) == 1 and "fused head" in next(iter(trace)) and " f16 nchw " in next(iter(trace)), trace
    ref = O.nfp_pooling_forward(x.detach().double().cpu(), pool.nfp_proj.weight.detach().cpu().double(),
                                pool.nfp_proj.bias.detach().cpu().double())
    assert rel_err(out.detach().float().cpu(), ref) <= TOL_F16_MAP
    out.float().sum().backward()
    assert x.grad.dtype == F16 and torch.isfinite(x.grad).all()
