"""CPU: the input-gradient metric of tests/test_generic_parity_gpu.py (elem_grad_errs, tests/_util.py) and its bounds.

* the fp32 bounds come from ATen's own fp32 error over the GPU grid (measured again here and printed beside them);
  ATen's fp32 evaluation passes every cell; the cells where that evaluation is ill-conditioned are listed;
* the metric flags, under every measure's bound, the kernel bugs the GPU file is meant to catch;
* every cell of the GPU grid takes generic/pairs with the expected launch count (host-only path query, no GPU);
* the oracle's index tables equal the reference's one-hot Conv2d extraction at every new edge geometry.
"""
import collections
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from neighbour_feature_pooling_b200 import _capi
from oracle import nfp_oracle as O
from oracle.ref_loader import reference_available

import test_generic_parity_gpu as G
from _util import elem_grad_err, elem_grad_errs, reached_pixels, rel_err
from test_parity_gpu import LOOSE

F32 = torch.float32


def _cells():
    for m, g in G.GRID:
        for op, dt, kind in G.runs(m, g):
            if dt == F32:
                yield m, g, op, kind


def _cell(m, g, op, kind):
    x = G.make_inputs(kind, g, F32, G.seed(m, g, kind), m)
    return x, G.grads(op, g, m, kind, F32)


@pytest.fixture(scope="module")
def aten():
    """{(spelling, geom, op, kind): aten_fp32} over the fp32 cells of the GPU grid."""
    return {(m, g, op, k): G.aten_fp32(op, *_cell(m, g, op, k), G.case_kw(m, g)) for m, g, op, k in _cells()}


def test_bounds_from_aten_fp32(aten):
    """ATEN_FP32 is ATen's largest fp32 error in the cells where it stays below LOOSE / FP32_MULT (within a factor 2:
    other CPUs round other sums); every bound is FP32_MULT x that, at least 1e-5 and at most LOOSE; the other cells
    are printed with ATen's error."""
    worst = collections.defaultdict(float)
    ill = collections.defaultdict(list)
    for (m, g, op, kind), (outs, gx) in aten.items():
        cm = O.canonical_measure(m)
        cap = LOOSE.get(cm, 1e-5) / G.FP32_MULT
        for key, e in [(("out", i), e) for i, e in enumerate(outs)] + list(gx.items()):
            if e < cap:
                worst[cm] = max(worst[cm], e)
            else:
                ill[cm].append((e, m, G.geom_id(g), op, kind, key))
    print(f"\n{'measure':13s} {'fp32 bound':>10s} {'ATen fp32':>10s} {'re-measured':>11s} {'LOOSE':>7s}  ill-conditioned cells")
    for m in O.MEASURES:
        print(f"{m:13s} {G.fp32_bound(m):10.1e} {G.ATEN_FP32[m]:10.1e} {worst[m]:11.1e} {LOOSE.get(m, 1e-5):7.0e}  "
              f"{len(ill[m])}" + (f" (worst {max(ill[m])[0]:.1e} at {max(ill[m])[1:]})" if ill[m] else ""))
    for m in O.MEASURES:
        assert G.ATEN_FP32[m] / 2 <= worst[m] <= 2 * G.ATEN_FP32[m], (m, worst[m], G.ATEN_FP32[m])
        assert 1e-5 <= G.fp32_bound(m) <= LOOSE.get(m, 1e-5), m
        assert G.fp32_bound(m) == min(LOOSE.get(m, 1e-5), max(1e-5, G.FP32_MULT * G.ATEN_FP32[m])), m


def test_aten_fp32_passes_every_cell(aten):
    """Specificity: ATen's own fp32 evaluation passes every cell under allowed(), except geman's input gradient
    (NO_CELL_ALLOWANCE), which ATen gets wrong by construction (the number is printed)."""
    failed = []
    geman = 0.0
    for (m, g, op, kind), (outs, gx) in aten.items():
        t_out, t_gx = G.allowed(m, F32, (outs, gx))
        if not all(e < t_out for e in outs):
            failed.append((m, G.geom_id(g), op, kind, outs))
        over = {k: e for k, e in gx.items() if not e < t_gx[k]}
        if O.canonical_measure(m) in G.NO_CELL_ALLOWANCE:
            geman = max([geman] + list(over.values()))
        elif over:
            failed.append((m, G.geom_id(g), op, kind, over))
    print(f"\ngeman: ATen's fp32 input gradient is up to {geman:.1e} off in a bucket (bound {G.fp32_bound('geman'):.1e})")
    assert not failed, failed[:5]


# ---- the metric flags each bug -----------------------------------------------------------------------------------
MUTATION_GEOMS = [(3, 20, 7, 7, 1, 1, 1, 1, "reflect"), (2, 8, 9, 8, 1, 2, 1, 1, "replicate"),
                  (2, 6, 5, 6, 1, 1, 5, 1, "circular"), (2, 6, 3, 4, 1, 1, 6, 1, "replicate"),
                  (2, 6, 5, 7, 1, 1, 4, 1, "reflect")]


def _gx(x, gs, kw, op="map", gap_div=None):
    if op == "map":
        return G.oracle_map(x, gs[0], kw)[1]
    return G.oracle_pooled(x, gs[0], gs[1], kw, gap_div)[2]


def _fold_dropped(x, g, kw):
    """The map-mode gradient with the part that the padding rule folds back onto one border pixel left out (the pixel
    with the largest such part): a gather backward that misses one branch of its padding rule."""
    pad, mode = kw["padding"], kw["padding_mode"]
    xr = x.double().requires_grad_(True)
    xp = F.pad(xr, (pad,) * 4, mode=mode)
    xp.retain_grad()
    y = O.nfp_forward(xp, **{**kw, "padding": 0, "padding_mode": "zeros"})
    y.backward(g.double())
    H, W = x.shape[2:]
    direct = xp.grad[:, :, pad:pad + H, pad:pad + W]
    fold = (xr.grad - direct).abs().sum((0, 1)).nan_to_num(nan=0.0)   # not a pixel of the NaN footprint
    h, w = np.unravel_index(int(fold.argmax()), fold.shape)
    if not fold[h, w] > 0:
        return None   # every folded pixel is in the NaN footprint (rmse / hellinger at a zero difference)
    out = xr.grad.clone()
    out[:, :, h, w] = direct[:, :, h, w]
    return out


def _flagged(got, want, geo, bounds):
    errs = elem_grad_errs(got, want, geo)
    return any(not e < bounds.get(k, 0.0) for k, e in errs.items())


@pytest.mark.parametrize("measure", G.SPELLINGS)
@pytest.mark.parametrize("geom", MUTATION_GEOMS, ids=G.geom_id)
def test_metric_flags_each_mutation(measure, geom):
    """Every mutation of the fp64 input gradient is flagged under the cell's bounds (allowed()), on both inputs and in
    both ops."""
    kw = G.case_kw(measure, geom)
    geo = G.case_geo(geom)
    m = O.canonical_measure(measure)
    missed = {}
    for kind in G.KINDS:
        for op in G.OPS:
            x, gs = _cell(measure, geom, op, kind)
            want = _gx(x, gs, kw, op)
            _, bounds = G.allowed(measure, F32, G.aten_fp32(op, x, gs, kw))
            assert not _flagged(want, want, geo, bounds)
            errs = elem_grad_errs(want, want, geo)
            assert errs, "nothing to score"
            mut = {}
            # every bulk element zeroed, and the largest bulk element off by 1e-4 (relative)
            mag = want.abs()
            struct = ~reached_pixels(geo)
            med = torch.stack([mag[b][:, ~struct][mag[b][:, ~struct] > 0].median() for b in range(x.shape[0])])
            bulk = (mag <= 10 * med[:, None, None, None]) & ~struct
            mut["bulk zeroed"] = torch.where(bulk, torch.zeros_like(want), want)
            i = int(torch.where(bulk, mag, torch.zeros_like(mag)).flatten().argmax())
            one = want.clone().flatten()
            one[i] *= 1 + 1e-4
            mut["one bulk element x (1 + 1e-4)"] = one.view_as(want)
            for other in ("reflect", "replicate", "circular", "zeros"):
                if other != kw["padding_mode"]:
                    try:
                        mut[f"{other} padding rule"] = _gx(x, gs, {**kw, "padding_mode": other}, op)
                    except RuntimeError:   # not a valid padding for this map (reflect / circular limits)
                        pass
            mut["similarity sign flipped"] = _gx(x, gs, {**kw, "similarity": not kw["similarity"]}, op)
            if m == "scs":
                mut["scs per image"] = torch.cat([_gx(x[b:b + 1], [t[b:b + 1] for t in gs], kw, op)
                                                  for b in range(x.shape[0])])
            if m == "attention":
                mut["attention without its softmax pass"] = _gx(x, gs, {**kw, "measure": "dot"}, op)
            if op == "map" and kw["padding_mode"] != "zeros":
                mut["one border pixel's fold dropped"] = _fold_dropped(x, gs[0], kw)
            if op == "pooled" and geo.Ho * geo.Wo != geom[2] * geom[3]:
                mut["GAP(NFP) gradient divided by H*W"] = _gx(x, gs, kw, op, gap_div=geom[2] * geom[3])
            for name, got in mut.items():
                fin = torch.isfinite(want)
                if got is None or torch.equal(got[fin], want[fin]):
                    continue   # changes nothing outside the NaN footprint (rmse / hellinger at a zero difference)
                # a 1e-4 error is below the allowance of the cells where ATen's own fp32 error is larger: held to the
                # measure's bound; every other mutation to the cell's bounds
                b = {k: G.fp32_bound(measure) for k in errs} if name.startswith("one bulk") else bounds
                if not _flagged(got, want, geo, b):
                    missed[(kind, op, name)] = sorted(elem_grad_errs(got, want, geo).items(), key=lambda kv: -kv[1])[:2]
    assert not missed, missed


ISSUE_TABLE = [((3, 20, 7, 7, 1, 1, 1, 1, "reflect"), ("geman", "chisquared2", "jeffrey", "canberra")),
               ((2, 8, 9, 8, 1, 2, 1, 1, "replicate"),
                ("geman", "chisquared2", "hellinger", "canberra"))]
# rmse and smith are in that table too, but on this draw what the recipe zeroes there is the NaN footprint of
# replicate's zero differences (rmse) and elements below 1e-7 of their bucket (smith): nothing to flag


@pytest.mark.parametrize("geom,measures", ISSUE_TABLE, ids=lambda v: G.geom_id(v) if isinstance(v[0], int) else "")
def test_whole_tensor_scale_misses_zeroed_elements(geom, measures):
    """Why the generic tests score gx with elem_grad_err: on the randn recipe of test_random_vs_oracle_generic,
    zeroing every gradient element below LOOSE x the largest passes the old whole-tensor rel_err bound; elem_grad_err
    flags the same tensor."""
    B, C, H, W, R, s, pad, d, mode = geom
    geo = G.case_geo(geom)
    zeroed = {}
    for measure in measures:
        gen = torch.Generator().manual_seed(G.seed(measure, geom))
        x = torch.randn(B, C, H, W, generator=gen)
        kw = dict(R=R, measure=measure, p=1, stride=s, padding=pad, dilation=d, padding_mode=mode)
        g = torch.randn(B, (2 * R + 1) ** 2 - 1, geo.Ho, geo.Wo, generator=gen)
        _, want = G.oracle_map(x, g, kw)
        tol = max(LOOSE.get(measure, 1e-5), 2e-5)
        keep = want.abs() >= 0.999 * tol * want[torch.isfinite(want)].abs().max()
        got = torch.where(keep, want, torch.zeros_like(want))
        zeroed[measure] = f"{1 - keep.double().mean().item():.0%}"
        assert rel_err(got, want) < tol, measure
        zeroed[measure] += f", elem_grad_err {elem_grad_err(got, want, geo):.2f}"
        assert elem_grad_err(got, want, geo) >= G.fp32_bound(measure), measure
    print("\nelements zeroed:", zeroed)


# ---- grid reach ---------------------------------------------------------------------------------------------------
def _expected_launches(measure, op):
    m = O.canonical_measure(measure)
    fwd = 1 + (m in ("attention", "scs"))
    bwd = 2 + {"attention": 1, "scs": 2}.get(m, 0)
    return {_capi.OP_FORWARD: fwd, _capi.OP_BACKWARD: bwd, _capi.OP_POOL_FORWARD: fwd + 2,
            _capi.OP_POOL_BACKWARD: bwd + 1}[op]


def test_grid_reaches_generic_pairs():
    """Every (measure, geometry, op, dtype) cell of the GPU grid takes generic/pairs, with the expected launch count
    and a workspace that holds the 5 pair coefficients (backward) and the map (pooled)."""
    wrong = []
    ops = (_capi.OP_FORWARD, _capi.OP_BACKWARD, _capi.OP_POOL_FORWARD, _capi.OP_POOL_BACKWARD)
    for m, g in G.GRID:
        cfg = G.config(m, g)
        geo = G.case_geo(g)
        B, C, H, W = g[:4]
        npairs = B * cfg.out_channels * geo.Ho * geo.Wo
        for dt in G.DTYPES:
            desc = _capi.make_desc(_capi.F32 if dt == F32 else _capi.BF16, B, C, H, W, cfg.R, cfg.stride, cfg.padding,
                                   cfg.dilation, cfg.padding_mode, cfg.measure, cfg.similarity, cfg.difference_taps,
                                   cfg.eps, cfg.p, cfg.q_scs, cfg.path)
            assert _capi.output_shape(desc) == (geo.Ho, geo.Wo)
            for op in ops:
                if op >= _capi.OP_POOL_FORWARD and not any(o == "pooled" for o, _, _ in G.runs(m, g)):
                    continue
                esz = 4 if dt == F32 else 2
                need = {_capi.OP_FORWARD: 0, _capi.OP_BACKWARD: 20 * npairs, _capi.OP_POOL_FORWARD: esz * npairs,
                        _capi.OP_POOL_BACKWARD: 4 * npairs + 20 * npairs}[op]   # fp32 map gradient
                got = (_capi.describe_path(desc, op), _capi.launch_count(desc, op), _capi.workspace_bytes(desc, op))
                if got[0] != "generic/pairs" or got[1] != _expected_launches(m, op) or got[2] < need:
                    wrong.append((m, G.geom_id(g), op, dt, got))
    assert not wrong, wrong[:5]
    # the grid holds every measure spelling, both similarity values per measure, both ops and dtypes per geometry
    sims = {(O.canonical_measure(m), G.case_sim(m, g)) for m, g in G.GRID}
    assert sims == {(m, s) for m in O.MEASURES for s in (True, False)}
    assert {m for m, _ in G.GRID} == set(G.SPELLINGS)
    for geom in G.ALL_GEOMS:
        assert {G.case_sim(m, g) for m, g in G.GRID if g == geom} == {True, False}, geom


# ---- oracle pin ---------------------------------------------------------------------------------------------------
def _one_hot_extraction(x, geom):
    """The reference's extraction: depthwise Conv2d with frozen one-hot weights (nfp.py:42-82), pure-neighbour taps."""
    B, C, H, W, R, s, pad, d, mode = geom
    k = 2 * R + 1
    taps = O.tap_offsets(R)
    conv = nn.Conv2d(C, len(taps) * C, k, stride=s, padding=pad, dilation=d, groups=C, bias=False,
                     padding_mode=mode).double()
    centre = nn.Conv2d(C, C, k, stride=s, padding=pad, dilation=d, groups=C, bias=False, padding_mode=mode).double()
    with torch.no_grad():
        conv.weight.zero_()
        centre.weight.zero_()
        for ch in range(C):
            for t, (a, b) in enumerate(taps):
                conv.weight[ch * len(taps) + t, 0, a, b] = 1.0
            centre.weight[ch, 0, R, R] = 1.0
        n = conv(x)
        c = centre(x)
    Ho, Wo = n.shape[2:]
    return c.unsqueeze(2), n.view(B, C, len(taps), Ho, Wo)


@pytest.mark.parametrize("geom", G.EDGE_GEOMS, ids=G.geom_id)
def test_oracle_gather_equals_one_hot_conv(geom):
    x = torch.randn(*geom[:4], dtype=torch.float64, generator=torch.Generator().manual_seed(G.seed(geom)))
    c, n = O.gather_centre_neighbours(x, G.case_geo(geom))
    c_ref, n_ref = _one_hot_extraction(x, geom)
    assert torch.equal(c, c_ref) and torch.equal(n, n_ref)


@pytest.mark.skipif(not reference_available(), reason="needs the original project: NFP_REFERENCE_ROOT or a copy staged under oracle/_ref")
@pytest.mark.parametrize("geom", G.EDGE_GEOMS, ids=G.geom_id)
def test_oracle_matches_reference_at_edge_geometries(geom):
    """The oracle's forward and backward equal the reference NFPPooling's own, in fp64, for every measure spelling."""
    from oracle.ref_loader import load_reference
    RefNFP, _ = load_reference()
    B, C, H, W = geom[:4]
    for measure in G.SPELLINGS:
        kw = G.case_kw(measure, geom)
        x = G.make_inputs("conditioned", geom, F32, G.seed(measure, geom, "ref"), measure).double()
        layer = RefNFP(C, **{k: v for k, v in kw.items()}).double()
        xr = x.clone().requires_grad_(True)
        y = layer(xr)
        g = torch.randn(y.shape, dtype=torch.float64, generator=torch.Generator().manual_seed(G.seed(measure, geom)))
        (gx,) = torch.autograd.grad(y, xr, g)
        y_o, gx_o = G.oracle_map(x, g, kw)
        assert rel_err(y_o, y.detach()) < 1e-12, measure
        assert rel_err(gx_o, gx) < 1e-10, measure


@pytest.mark.parametrize("measure,geom", [("cosine", (3, 20, 7, 7, 1, 1, 1, 1, "reflect")),
                                          ("chisquared2", (3, 20, 7, 7, 1, 1, 1, 1, "reflect")),
                                          ("scs", (2, 6, 6, 6, 1, 1, 4, 1, "zeros"))],
                         ids=lambda v: v if isinstance(v, str) else G.geom_id(v))
def test_flags_pooled_map_gradient_rounded_to_bf16(measure, geom):
    """The generic pooled backward once stored the map gradient g_gap_nfp / (Ho*Wo) in the dtype of x.  For bf16 its
    2^-9 rounding is multiplied by per-tap derivatives that cancel to far smaller sums at pixels near a clamp, and
    the GPU grid failed there.  The same rounding, applied to the fp64 oracle on the conditioned bf16 input, is flagged
    at the bf16 bound; kept in fp32 (what the kernel does now) it passes."""
    kw = G.case_kw(measure, geom)
    geo = G.case_geo(geom)
    x = G.make_inputs("conditioned", geom, torch.bfloat16, G.seed(measure, geom, "conditioned"), measure)
    g1, g2 = G.grads("pooled", geom, measure, "conditioned", torch.bfloat16)
    want = G.oracle_pooled(x, g1, g2, kw)[2]
    B, C, H, W = x.shape

    def with_map_gradient(cast):
        gy = cast(g2.double() / (geo.Ho * geo.Wo))[:, :, None, None].expand(B, g2.shape[1], geo.Ho, geo.Wo)
        return G.oracle_map(x, gy.double().contiguous(), kw)[1] + (g1.double() / (H * W))[:, :, None, None]
    rounded = with_map_gradient(lambda t: t.bfloat16())
    kept = with_map_gradient(lambda t: t.float())
    assert elem_grad_err(rounded, want, geo, torch.bfloat16) >= G.BF16_TOL
    assert elem_grad_err(kept, want, geo, torch.bfloat16) < G.BF16_TOL / 100
