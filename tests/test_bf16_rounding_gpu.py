"""GPU: every bf16 kernel path held to one rounding of an fp32 evaluation, and its fp32 outputs to fp32 accuracy.

The kernels read bf16 exactly and compute in fp32; the only error a bf16 result may carry beyond fp32 evaluation is
the final rounding to bf16.  So each cell of the C-ABI grid (tests/test_abi_contract_gpu.py, Problem) is run with a
bf16 descriptor and compared with the fp64 oracle on the bf16-rounded inputs:

* bf16 outputs (y, gx): rounding_errs (tests/_util.py) <= 1, i.e. |got - want| <= 1/2 ulp(want) (1 + 2^-7) + tau S,
  S the largest |want| of the image (y) or of the image's pixel-norm region (gx, as grad_errs groups it);
* fp32 outputs (gap_x, gap_nfp, the head's out, the FLAG_Y_F32 map): rel_err <= tau, each image on its own scale;
* tau is the fp32 budget each family meets in fp32: 1e-5 for cosine, fp32_bound(measure) for the generic measures.

Every (family, entry point) that accepts a bf16 descriptor, with reflect / zeros / replicate padding, similarity on
and off, and clean and degenerate inputs (test_grad_parity_gpu.make_inputs: pixel norms down to 0 and around eps).  The
worst ratio of each cell is recorded as a property.  The module level is checked under torch.autocast(bfloat16): the
fp32 results against the oracle on the bf16-rounded input, the head's bf16 output (the reference's dtype there) within
one rounding, and the paths that return a bf16 map widened to fp32 (planar and generic) against round-to-nearest of
the oracle.  tests/test_bf16_rounding_metric.py shows on the CPU that the
metric passes an honest evaluation, flags the precision bugs this file is meant to catch, and that this grid reaches
every bf16 cell.
"""
import numpy as np
import pytest
import torch

import test_abi_contract_gpu as AC
import test_grad_parity_gpu as GP
from _util import region_groups, rel_err, rn_mismatches, rounding_errs, worst
from neighbour_feature_pooling_b200 import MultiRadiusNFP, NFPPooling, _capi, fuse_pooled_nfp, nfp_pooling
from neighbour_feature_pooling_b200 import functional as NF
from oracle import nfp_oracle as O
from test_generic_parity_gpu import fp32_bound

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
EPS = AC.EPS
TAU = 1e-5   # the fp32 budget of the cosine kernels (the fp32 suites' bound)
# Measured on one B200 (1000 W power limit), worst over the grid: y and gx ratios 0.982-0.989 in every family (the
# token backward's 16-bit M included, so it needs no bound of its own); fp32 outputs <= 6.7e-7 (token gap_nfp).  The
# generic pooled forward, when it pooled a bf16 map, failed every pool_forward / pooled_map_forward cell at up to 358 tau.


def tau_of(measure):
    return TAU if measure == "cosine" else fp32_bound(measure)


def _cell(family, entry, shape, **opts):
    return AC._cell(family, entry, shape, BF16, **opts)


class BF16Problem(AC.Problem):
    """A cell of the C-ABI grid with a bf16 descriptor, similarity on or off, the norm measure's p, and clean or
    degenerate input (kind "deg": test_grad_parity_gpu.make_inputs)."""

    def __init__(self, c):
        o = dict(c.opts)
        self.sim = bool(o.get("sim", 1))
        self.kind = o.get("kind", "clean")
        self.p = o.get("p", 1)
        super().__init__(c)
        self.desc.similarity = int(self.sim)
        self.desc.p = float(self.p)
        self.desc.difference_taps = int(O.uses_difference_taps(self.measure))   # as the oracle reads the spelling
        if c.family == "generic":   # also where a planar kernel would take the map (cosine at stride 1)
            self.desc.path = _capi.PATHS["generic"]

    def _kw(self, R=None, padding=None):
        kw = super()._kw(R, padding)
        kw["similarity"] = self.sim
        kw["p"] = self.p
        return kw

    def _make_data(self):
        super()._make_data()
        if self.kind != "deg":
            return
        seed = 7919 * self.B + 131 * self.C + 17 * self.H + self.W
        x, _ = GP.make_inputs("degenerate", (self.B, self.C, self.H, self.W, self.R), BF16, seed)
        self.x = x.double()
        self.inputs["x"] = (self._x_flat(), BF16)
        if self.c.entry == "head_backward":   # the forward's results, as fp32
            self.gap_x_in = self.x.mean((2, 3)).float().double()
            self.gap_nfp_in = self._map(self.x).mean((2, 3)).float().double()
            self.inputs["gap_x"] = (self.gap_x_in.reshape(-1), torch.float32)
            self.inputs["gap_nfp"] = (self.gap_nfp_in.reshape(-1), torch.float32)

    def expected(self):
        if self.inner and not self.sim:
            raise AssertionError("multi-radius cells: similarity on (the oracle composition below assumes it)")
        return super().expected()


KINDS = ("clean", "deg")
MODE_SIMS = [(m, s) for m in ("reflect", "zeros", "replicate") for s in (1, 0) if (m, s) != ("reflect", 1)]
GENERIC_MEASURES = [dict(measure="cosine"), dict(measure="dot"), dict(measure="norm", p=1), dict(measure="norm", p=2)]


def _grid():
    g = []
    for s in AC.STREAM_INST:   # the six NFP_STREAM_SHAPES instantiations, every entry point
        g += [_cell("stream", e, s, kind=k) for e in AC.ENTRIES for k in KINDS]
    for s in [(3, 64, 7, 7, 1), (2, 64, 14, 14, 1)]:
        for mode, sim in MODE_SIMS:
            g += [_cell("stream", e, s, mode=mode, sim=sim, kind=k) for e in ("forward", "backward", "pool_backward")
                  for k in KINDS]
    g += [_cell("stream", "backward", (3, 40, 7, 7, 1), kind=k) for k in KINDS]          # strip form (C % 64 != 0)
    # more images than resident CTAs at full width: the persistent plan and the two-buffer gradient path
    g += [_cell("stream", e, (300, 512, 7, 7, 1), kind=k) for e in ("forward", "backward") for k in KINDS]
    g += [_cell("stream", "forward", s, yf32=1, kind=k) for s in [(3, 64, 7, 7, 1), (2, 32, 14, 14, 2)] for k in KINDS]
    for s in [(3, 64, 7, 7, 2), (2, 32, 14, 14, 2)]:
        g += [_cell("stream", e, s, inner=1, kind=k) for e in ("forward", "backward") for k in KINDS]
    for s in [(3, 64, 7, 7, 1), (2, 64, 14, 14, 1)]:
        g += [_cell("split", e, s, kind=k) for e in AC.ENTRIES[:6] for k in KINDS]
    band_ops = ("forward", "backward", "pooled_map_forward", "pooled_map_backward")
    for s in [(2, 8, 21, 16, 1), (2, 16, 112, 112, 1)]:
        g += [_cell("band", e, s, kind=k) for e in band_ops for k in KINDS]
    for mode, sim in MODE_SIMS:
        g += [_cell("band", e, (2, 8, 21, 16, 1), mode=mode, sim=sim, kind="deg") for e in band_ops]
    g += [_cell("band", e, (2, 16, 28, 28, 2), inner=1, kind=k) for e in ("forward", "backward") for k in KINDS]
    for s in [(2, 5, 3, 3, 1), (2, 10, 5, 9, 2)]:
        g += [_cell("table", e, s, kind=k) for e in ("forward", "backward") for k in KINDS]
    for mode, sim in MODE_SIMS:
        g += [_cell("table", e, (2, 10, 5, 9, 2), mode=mode, sim=sim, kind="deg") for e in ("forward", "backward")]
    # channels-last token kernels: dense, pad8 and ViT x batch strides; padded gx strides on the backward entries
    vit = (3, 64, 14, 14, 1)
    for e in AC.ENTRIES:
        bwd = e.endswith("backward")
        for i, xbs in enumerate(("dense", "pad8", "vit")):
            g.append(_cell("token", e, vit, xbs=xbs, gxbs=("0", "pad8", "pad64")[i] if bwd else "0"))
        g.append(_cell("token", e, vit, xbs="dense", kind="deg"))
    g += [_cell("token", e, (2, 192, 7, 7, 1), xbs="pad8", gxbs="pad64") for e in AC.ENTRIES]
    g += [_cell("token", e, (2, 512, 7, 7, 1), kind=k) for e in ("forward", "backward") for k in KINDS]
    g += [_cell("token", e, (3, 64, 7, 7, 2), inner=1, xbs="pad8", gxbs="pad8", kind=k) for e in ("forward", "backward")
          for k in KINDS]
    for mode, sim in MODE_SIMS:
        g += [_cell("token", e, (2, 64, 7, 7, 1), mode=mode, sim=sim, kind=k) for e in ("forward", "backward")
              for k in KINDS]
    g += [_cell("token", "forward", (2, 192, 14, 14, 1), yf32=1, xbs="vit", kind=k) for k in KINDS]
    for o in GENERIC_MEASURES:
        g += [_cell("generic", e, (3, 5, 9, 11, 1), kind=k, **o) for e in AC.ENTRIES[:6] for k in KINDS]
    g += [_cell("generic", e, (3, 5, 9, 11, 1), measure="cosine", stride=2, dilation=2, padding=2, mode="circular",
                sim=0) for e in AC.ENTRIES[:6]]
    return g


GRID = _grid()


def cell_id(c):
    return AC.cell_id(c)


def check_cell(prob, got_of):
    """{output: worst ratio to its bound} of one run; got_of(name) -> the output as float64 in its logical shape."""
    exp, rows = prob.expected()
    tau = tau_of(O.canonical_measure(prob.measure))
    out = {}
    for n, ref in exp.items():
        got = got_of(n)[rows]
        if n == "gx":
            errs = rounding_errs(got, ref, BF16, tau, region_groups(prob.x[rows], EPS))
        elif n == "y" and not prob.yf32:
            errs = rounding_errs(got, ref, BF16, tau)
        else:   # fp32 outputs: fp32 accuracy, each image on its own scale
            errs = {i: rel_err(got[i], ref[i]) / tau for i in range(len(rows))}
        out[n] = (max(errs.values()), worst(errs, 3))
    return out


@pytest.mark.parametrize("c", [pytest.param(c, id=cell_id(c)) for c in GRID])
def test_bf16_cell(c, cuda_device, record_property):
    prob = BF16Problem(c)
    assert prob.path().startswith(AC.FAMILIES[c.family][0]), prob.path()
    pb, pws = prob.plain(cuda_device)
    AC._run(prob, pb, pws)
    torch.cuda.synchronize()
    res = check_cell(prob, lambda n: prob.logical(n, pb[n]))
    for n, (r, _) in res.items():
        record_property(f"ratio_{n}", f"{r:.3f}")
    bad = {n: w for n, (r, w) in res.items() if not r <= 1.0}
    assert not bad, bad


# ---- module level, under torch.autocast(bfloat16) -----------------------------------------------------------------
def _traced(fn):
    NF.PATH_TRACE = set()
    try:
        out = fn()
        return out, set(NF.PATH_TRACE)
    finally:
        NF.PATH_TRACE = None


def _x(shape, dev, seed, channels_last=False):
    x = torch.randn(*shape, generator=torch.Generator().manual_seed(seed)).to(BF16)
    x = x.to(dev)
    return x.contiguous(memory_format=torch.channels_last) if channels_last else x


def _per_image(got, want):
    return max(rel_err(got[i], want[i]) for i in range(want.shape[0]))


def _map_ref(xq, R=1, measure="cosine", **kw):
    return torch.as_tensor(np.asarray(O.nfp_forward(xq, R=R, measure=measure, padding=R, **kw)))


@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
def test_autocast_nfp_pooling_layer(layout, cuda_device, record_property):
    """NFPPooling on bf16 activations: the fp32 map within tau of the oracle (the fused kernels write fp32), the input
    gradient (bf16) within one rounding."""
    cl = layout == "channels_last"
    layer = NFPPooling(64, R=1, measure="cosine", padding=1).to(cuda_device)
    x = _x((3, 64, 7, 7), cuda_device, 1, cl).requires_grad_(True)
    with torch.autocast("cuda", dtype=BF16):
        y, trace = _traced(lambda: layer(x))
    assert trace and all(t.startswith("fused/token_" if cl else "fused/stream_") for t in trace), trace
    assert y.dtype == torch.float32
    xq = x.detach().double().cpu()
    gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(2))
    y_ref, gx_ref = O.nfp_forward_backward(xq, gy.to(BF16).double(), R=1, measure="cosine", padding=1)
    e = _per_image(y.detach().cpu(), y_ref)
    y.backward(gy.to(cuda_device))
    r = max(rounding_errs(x.grad.cpu(), gx_ref, BF16, TAU, region_groups(xq, EPS)).values())
    record_property("y_err", f"{e:.2e}")
    record_property("ratio_gx", f"{r:.3f}")
    assert e <= TAU and r <= 1.0, (e, r)


@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
def test_autocast_nfp_pooling_head(layout, cuda_device, record_property):
    """The fused nfp_pooling head on bf16 activations: out has the reference's dtype, bf16 (GAP(x) of bf16 x times the
    autocast Linear), and is the kernel's fp32 result rounded once: within one rounding of the oracle."""
    Params = {"num_ftrs": {"m": 64}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 3}}
    torch.manual_seed(0)
    pool = nfp_pooling(Params=Params).to(cuda_device)
    x = _x((3, 64, 7, 7), cuda_device, 3, layout == "channels_last")
    with torch.autocast("cuda", dtype=BF16):
        out, trace = _traced(lambda: pool(x))
    assert len(trace) == 1 and "fused head" in next(iter(trace)), trace
    assert out.dtype == BF16
    ref = O.nfp_pooling_forward(x.double().cpu(), pool.nfp_proj.weight.detach().cpu().double(),
                                pool.nfp_proj.bias.detach().cpu().double())
    r = max(rounding_errs(out.detach(), ref, BF16, TAU).values())
    record_property("ratio_out", f"{r:.3f}")
    assert r <= 1.0, r


@pytest.mark.parametrize("case", ["stream", "band", "token"])
def test_autocast_multi_radius(case, cuda_device, record_property):
    """MultiRadiusNFP on bf16 activations: the ring and token kernels write the fp32 map (within tau); the planar band
    kernels write bf16, widened: exactly round-to-nearest of the oracle, except within tau S of a tie."""
    C, H = {"stream": (64, 7), "band": (16, 28), "token": (64, 7)}[case]
    blocks = MultiRadiusNFP(C).to(cuda_device)
    x = _x((2, C, H, H), cuda_device, 4, case == "token")
    with torch.autocast("cuda", dtype=BF16):
        y, trace = _traced(lambda: blocks(x))
    assert trace and all("radii 1+2 in one launch" in t for t in trace), trace
    assert y.dtype == torch.float32
    xq = x.double().cpu()
    ref = torch.cat([_map_ref(xq, 1), _map_ref(xq, 2)], 1)
    got = y.detach().cpu()
    if case == "band":
        assert all(t.startswith("planar/band") for t in trace), trace
        bad = rn_mismatches(got, ref, BF16, TAU)
        record_property("rn_mismatches", bad)
        assert bad == 0, bad
    else:
        e = _per_image(got, ref)
        record_property("y_err", f"{e:.2e}")
        assert e <= TAU, e


@pytest.mark.parametrize("case", ["stream", "band", "token", "generic-dot", "generic-norm"])
def test_autocast_pooled_similarity(case, cuda_device, record_property):
    """nfp_pooled_similarity (and fuse_pooled_nfp on a stock layer) on bf16 activations: GAP(NFP(x)), fp32, within tau
    of the oracle on every path, the generic one included (its map stays fp32 before the pooling)."""
    C, H, W, measure, p = {"stream": (64, 7, 7, "cosine", 1), "band": (16, 28, 30, "cosine", 1),
                           "token": (64, 7, 7, "cosine", 1), "generic-dot": (5, 9, 11, "dot", 1),
                           "generic-norm": (5, 9, 11, "norm", 2)}[case]
    layer = NFPPooling(C, R=1, measure=measure, p=p, padding=1).to(cuda_device)
    x = _x((3, C, H, W), cuda_device, 5, case == "token")
    with torch.autocast("cuda", dtype=BF16):
        y, trace = _traced(lambda: NF.nfp_pooled_similarity(x, layer.config))
    prefix = {"stream": "fused/stream_", "band": "planar/band", "token": "fused/token_"}.get(case, "generic/pairs")
    assert trace and all(t.startswith(prefix) for t in trace), trace
    assert y.dtype == torch.float32
    ref = _map_ref(x.double().cpu(), 1, measure, p=p).mean((2, 3))
    e = _per_image(y.cpu(), ref)
    record_property("gap_nfp_err", f"{e:.2e}")
    assert e <= tau_of(measure), e
    if measure == "cosine":
        assert fuse_pooled_nfp(layer)
        with torch.autocast("cuda", dtype=BF16):
            yf = layer(x)
        assert yf.shape == (3, 8, 1, 1) and torch.equal(yf.flatten(1), y)


def test_autocast_vit_tokens(cuda_device, record_property):
    """fp32 LayerNorm tokens under bf16 autocast, as a (B, C, H, W) view: rounded to bf16 (as the reference's
    extraction convs do), fp32 map within tau, fp32 token gradient within one bf16 rounding (the kernels' gx)."""
    B, C, H, W = 2, 192, 14, 14
    feats = torch.randn(B, H * W + 1, C, generator=torch.Generator().manual_seed(6)).to(cuda_device)
    feats.requires_grad_(True)
    cfg = NF.NFPConfig(R=1, measure="cosine", padding=1)
    with torch.autocast("cuda", dtype=BF16):
        view = feats[:, 1:].transpose(1, 2).reshape(B, C, H, W)
        y, trace = _traced(lambda: NF.nfp_similarity(view, cfg))
    assert trace and all(t.startswith("fused/token_14x14_r1 bf16 channels-last") for t in trace), trace
    assert y.dtype == torch.float32
    xq = feats.detach()[:, 1:].transpose(1, 2).reshape(B, C, H, W).to(BF16).double().cpu()
    gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(7))
    y_ref, gx_ref = O.nfp_forward_backward(xq, gy.to(BF16).double(), R=1, measure="cosine", padding=1)
    e = _per_image(y.detach().cpu(), y_ref)
    y.backward(gy.to(cuda_device))
    got = feats.grad[:, 1:].transpose(1, 2).reshape(B, C, H, W).cpu()
    r = max(rounding_errs(got, gx_ref, BF16, TAU, region_groups(xq, EPS)).values())
    record_property("y_err", f"{e:.2e}")
    record_property("ratio_gx", f"{r:.3f}")
    assert e <= TAU and r <= 1.0, (e, r)
    assert bool((feats.grad[:, 0] == 0).all())


@pytest.mark.parametrize("case", ["band", "table", "generic-cosine", "generic-dot"])
def test_autocast_widened_bf16_map(case, cuda_device, record_property):
    """The planar and generic map paths have no fp32 map output: under autocast their bf16 map is widened to fp32.
    Pinned exactly: every element is round-to-nearest of the oracle, except within tau S of a tie."""
    C, H, W, measure = {"band": (16, 28, 28, "cosine"), "table": (5, 3, 3, "cosine"),
                        "generic-cosine": (5, 9, 11, "cosine"), "generic-dot": (5, 9, 11, "dot")}[case]
    cfg = NFPPooling(C, R=1, measure=measure, padding=1).config
    if case.startswith("generic"):
        cfg = NF.replace(cfg, path="generic")
    x = _x((3, C, H, W), cuda_device, 8)
    with torch.autocast("cuda", dtype=BF16):
        y, trace = _traced(lambda: NF.nfp_similarity(x, cfg))
    prefix = {"band": "planar/band", "table": "planar/table"}.get(case, "generic/pairs")
    assert trace and all(t.startswith(prefix) for t in trace), trace
    assert y.dtype == torch.float32
    bad = rn_mismatches(y.cpu(), _map_ref(x.double().cpu(), 1, measure), BF16, tau_of(measure))
    record_property("rn_mismatches", bad)
    assert bad == 0, bad
