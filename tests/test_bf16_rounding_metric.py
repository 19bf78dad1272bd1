"""CPU: the one-rounding metric of tests/test_bf16_rounding_gpu.py (rounding_errs, tests/_util.py) and its grid.

* ulp and round_nearest agree with the formats bit for bit, subnormals and overflow included;
* an honest kernel passes: the oracle evaluated in fp32 and rounded once to nearest scores <= 1 on every op (map,
  backward, pooled, pooled map, head, multi-radius), clean and degenerate input, bf16 and fp16, and its fp32 outputs
  are within tau;
* each bf16-only precision bug the GPU file is meant to catch scores > 1 (or > tau for fp32 outputs), and the table
  printed beside it shows which of them the flat 2e-2 relative bound of the other suites lets through;
* the GPU grid reaches every (family, entry point) that accepts a bf16 descriptor (host-only path queries).
"""
import ctypes

import numpy as np
import pytest
import torch

from neighbour_feature_pooling_b200 import _capi
from oracle import nfp_oracle as O

import test_abi_contract_gpu as AC
import test_abi_contract_host as ACH
import test_bf16_rounding_gpu as B
import test_grad_parity_gpu as G
from _util import grad_err, region_groups, rel_err, rn_mismatches, round_nearest, rounding_err, ulp

BF16, F16 = torch.bfloat16, torch.float16
TAU = 1e-5
OLD_TOL = 2e-2   # the flat bf16 bound of the other suites
EPS = 1e-6
OPS = ("map", "backward", "pooled", "pooled_map", "head", "multi")


# ---- ulp and rounding -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [BF16, F16], ids=["bf16", "f16"])
def test_ulp_and_round_nearest_match_the_format(dtype):
    g = torch.Generator().manual_seed(0)
    tiny = torch.finfo(dtype).tiny
    v = torch.cat([torch.randn(4000, generator=g, dtype=torch.float64) * 10.0 ** torch.randint(-6, 5, (4000,),
                                                                                               generator=g),
                   torch.rand(2000, generator=g, dtype=torch.float64) * 4 * tiny,    # subnormals
                   torch.tensor([0.0, tiny, -tiny, 1.0, -2.0, torch.finfo(dtype).max], dtype=torch.float64)])
    v = v[v.abs() < torch.finfo(dtype).max]
    qd = v.to(dtype).double()
    # ulp(v) is the spacing of the format around v: the gap above a representable value that is not a power of two
    exact = qd[(qd != 0) & (torch.frexp(qd.abs())[0] != 0.5)]
    up_e = torch.nextafter(exact.to(dtype), torch.tensor(float("inf"), dtype=dtype)).double()
    assert torch.equal(ulp(dtype, exact), (up_e - exact).abs())
    assert float(ulp(dtype, torch.tensor([0.0]))) == float(torch.nextafter(torch.tensor(0.0, dtype=dtype),
                                                                           torch.tensor(1.0, dtype=dtype)))
    r = round_nearest(dtype, v)
    assert torch.equal(r.to(dtype).double(), r)   # representable
    # nearest: no representable neighbour of r is closer to v
    for n in (torch.nextafter(r.to(dtype), torch.tensor(float("inf"), dtype=dtype)).double(),
              torch.nextafter(r.to(dtype), torch.tensor(-float("inf"), dtype=dtype)).double()):
        assert bool(((n - v).abs() >= (r - v).abs()).all())
    # fp32 -> 16-bit is a single rounding in torch: round_nearest agrees with it on fp32 values
    v32 = v.float().double()
    assert torch.equal(round_nearest(dtype, v32), v32.float().to(dtype).double())
    ovf = {BF16: (2 - 2.0 ** -8) * 2.0 ** 127, F16: 65520.0}[dtype]   # half-way past the largest finite value
    below = torch.nextafter(torch.tensor(ovf, dtype=torch.float64), torch.tensor(0.0, dtype=torch.float64))
    assert float(round_nearest(dtype, below.view(1))) == torch.finfo(dtype).max
    assert torch.equal(round_nearest(dtype, torch.tensor([ovf, -ovf], dtype=torch.float64)),
                       torch.tensor([float("inf"), -float("inf")], dtype=torch.float64))


def test_rounding_errs_overflow_and_nan():
    want = torch.tensor([[1.0, 70000.0, -1e6, float("nan")]], dtype=torch.float64)
    got = torch.tensor([[1.0, float("inf"), -float("inf"), 5.0]], dtype=torch.float64)
    assert rounding_err(got, want, F16, TAU) == 0.0
    assert rounding_err(torch.tensor([[1.0, 65504.0, -float("inf"), 5.0]]), want, F16, TAU) == float("inf")
    assert rounding_err(torch.tensor([[float("inf"), float("inf"), -float("inf"), 5.0]]), want, F16, TAU) == float("inf")


# ---- one op: fp64 oracle and its fp32 evaluation ----------------------------------------------------------------
def _shape(op):
    return (3, 64, 7, 7, 2) if op == "multi" else (3, 64, 7, 7, 1)


def _problem(op, kind, dtype, mode="reflect", sim=True, shape=None):
    """(x rounded to dtype, the op's other inputs): gy in dtype for map gradients, fp32 vectors for the pooled ones."""
    B, C, H, W, R = shape or _shape(op)
    seed = 7 * OPS.index(op) + 3 * G.KINDS.index(kind) + G.MODES.index(mode) + 31 * sim
    x, _ = G.make_inputs(kind, (B, C, H, W, R), torch.float32, seed)
    x = round_nearest(dtype, x)
    gen = torch.Generator().manual_seed(seed + 1)
    K = (2 * R + 1) ** 2 - 1
    ins = dict(R=R, mode=mode, sim=sim)
    if op in ("backward", "multi"):
        ins["gy"] = round_nearest(dtype, torch.randn(B, K + (8 if op == "multi" else 0), H, W, generator=gen))
    if op in ("pooled", "pooled_map"):
        ins["g1"] = torch.randn(B, C, generator=gen).float().double() if op == "pooled" else torch.zeros(B, C,
                                                                                                        dtype=torch.float64)
        ins["g2"] = torch.randn(B, K, generator=gen).float().double()
    if op == "head":
        ins["w"] = (0.1 * torch.randn(C, K, generator=gen)).float().double()
        ins["b"] = torch.randn(C, generator=gen).float().double()
        ins["g"] = torch.randn(B, C, generator=gen).float().double()
    return x, ins


def _np(t):
    return torch.as_tensor(np.asarray(t))


def evaluate(op, x, ins, prec):
    """{output name: (value as float64, "T" or "f32")} of the op, every step of the oracle in `prec`."""
    R, kw = ins["R"], dict(measure="cosine", padding_mode=ins["mode"], similarity=ins["sim"])
    xp = x.to(prec)
    B, C, H, W = x.shape
    if op == "map":
        return {"y": (_np(O.nfp_forward(xp, R=R, padding=R, **kw)).double(), "T")}
    if op == "backward":
        y, gx = O.nfp_forward_backward(xp, ins["gy"].to(prec), R=R, padding=R, **kw)
        return {"gx": (_np(gx).double(), "T")}
    if op == "multi":
        gy = ins["gy"].to(prec)
        y1, g1 = O.nfp_forward_backward(xp, gy[:, :8].contiguous(), R=1, padding=1, **kw)
        y2, g2 = O.nfp_forward_backward(xp, gy[:, 8:].contiguous(), R=2, padding=2, **kw)
        return {"y": (torch.cat([_np(y1), _np(y2)], 1).double(), "T"), "gx": ((_np(g1) + _np(g2)).double(), "T")}
    if op in ("pooled", "pooled_map"):
        g1, g2 = ins["g1"].to(prec), ins["g2"].to(prec)
        gy = (g2 / (H * W))[:, :, None, None].expand(B, g2.shape[1], H, W).contiguous()
        y, gx = O.nfp_forward_backward(xp, gy, R=R, padding=R, **kw)
        out = {"gap_nfp": (_np(y).mean((2, 3)).double(), "f32"),
               "gx": ((_np(gx) + (g1 / (H * W))[:, :, None, None]).double(), "T")}
        if op == "pooled":
            out["gap_x"] = (xp.mean((2, 3)).double(), "f32")
        return out
    # head: out = GAP(x) * (W GAP(NFP(x)) + b); backward of <g, out> with the forward's fp32 vectors
    w, b, g = ins["w"].to(prec), ins["b"].to(prec), ins["g"].to(prec)
    y = _np(O.nfp_forward(xp, R=R, padding=R, **kw))
    gap_x, gap_n = xp.mean((2, 3)), y.mean((2, 3))
    proj = gap_n @ w.t() + b
    gy = (((g * gap_x) @ w) / (H * W))[:, :, None, None].expand(B, w.shape[1], H, W).contiguous()
    _, gx = O.nfp_forward_backward(xp, gy, R=R, padding=R, **kw)
    gx = _np(gx) + ((g * proj) / (H * W))[:, :, None, None]
    return {"out": ((gap_x * proj).double(), "f32"), "gx": (gx.double(), "T")}


def score(name, got, want, x, dtype, tau=TAU):
    """The GPU file's check: ratio to the bound (<= 1 passes) for 16-bit outputs, rel_err / tau per image for fp32."""
    if name == "gx":
        return rounding_err(got, want, dtype, tau, region_groups(x, EPS))
    if name == "y":
        return rounding_err(got, want, dtype, tau)
    return max(rel_err(got[i], want[i]) for i in range(want.shape[0])) / tau


def old_score(name, got, want, x):
    """What the other suites assert for bf16 (pass < 2e-2): rel_err of maps and vectors, grad_err of gradients."""
    return grad_err(got, want, x) if name == "gx" else rel_err(got, want)


@pytest.mark.parametrize("dtype", [BF16, F16], ids=["bf16", "f16"])
@pytest.mark.parametrize("kind", G.KINDS)
@pytest.mark.parametrize("op", OPS)
def test_honest_evaluation_passes(op, kind, dtype):
    """Specificity: fp32 evaluation rounded once to nearest (fp32 outputs left fp32) passes, in every padding mode and
    for both similarity flags."""
    worst = {}
    for mode in G.MODES:
        for sim in (True, False):
            x, ins = _problem(op, kind, dtype, mode, sim)
            want = evaluate(op, x, ins, torch.float64)
            got = evaluate(op, x, ins, torch.float32)
            for n, (w, kind_of) in want.items():
                g = round_nearest(dtype, got[n][0]) if kind_of == "T" else got[n][0]
                worst[(mode, sim, n)] = score(n, g, w, x, dtype)
    bad = {k: v for k, v in worst.items() if not v <= 1.0}
    assert not bad, bad
    print(f"\n{op} {kind} {dtype}: worst ratio {max(worst.values()):.3f} at {max(worst, key=worst.get)}")


# ---- mutations: bf16-only precision bugs ------------------------------------------------------------------------
def _rz_bf16(v):
    """fp32 -> bf16 rounded toward zero (the low 16 bits dropped)."""
    b = v.float().contiguous().view(torch.int32) & -65536
    return b.view(torch.float32).double()


def _rn(v):
    return round_nearest(BF16, v)


def _parts(x32, R, mode, round_gram=False):
    """The cosine kernels' forward intermediates in fp32: centre / neighbours, dot, inverse norms, y."""
    geo = O.geometry(x32.shape[2], x32.shape[3], R, 1, R, 1, mode)
    c, n = O.gather_centre_neighbours(x32, geo)
    dot, cc, nn = (c * n).sum(1), (c * c).sum(1), (n * n).sum(1)
    if round_gram:   # Gram entries (dot products and squared norms) kept in bf16
        dot, cc, nn = dot.bfloat16().float(), cc.bfloat16().float(), nn.bfloat16().float()
    inc = 1.0 / cc.sqrt().clamp_min(EPS)
    inn = 1.0 / nn.sqrt().clamp_min(EPS)
    return c, n, dot, inc, inn


def _map_variant(x, R, mode, how):
    x32 = x.float()
    c, n, dot, inc, inn = _parts(x32, R, mode, round_gram=(how == "gram"))
    if how == "inv_norms":
        inc, inn = inc.bfloat16().float(), inn.bfloat16().float()
    y = dot * inc * inn
    return _rz_bf16(y) if how == "rz" else _rn(y)


def _grad_variant(x, gy, R, mode, how):
    """The cosine map's input gradient as a kernel contracts it: per pair, dy/dc = a n - bc c and dy/dn = a c - bn n
    with a = g / (|c| |n|), bc = g y / |c|^2, bn = g y / |n|^2 (fp32), scattered onto the input pixels; then one
    rounding to bf16.  how: "ok", "coef" (a, bc, bn rounded to bf16 before the contraction), "taps" (each tap's
    contribution added to a bf16 accumulator)."""
    x32 = x.float().clone().requires_grad_(True)
    c, n, dot, inc, inn = _parts(x32, R, mode)
    g = gy.float()
    with torch.no_grad():
        y = dot * inc * inn
        a, bc, bn = g * inc * inn, g * y * inc * inc, g * y * inn * inn
        if how == "coef":
            a, bc, bn = a.bfloat16().float(), bc.bfloat16().float(), bn.bfloat16().float()
    cc, nn = (c * c).sum(1), (n * n).sum(1)

    def contraction(t):
        s = slice(None) if t is None else slice(t, t + 1)
        L = (a[:, s] * dot[:, s]).sum() - 0.5 * (bc[:, s] * cc).sum() - 0.5 * (bn[:, s] * nn[:, s]).sum()
        return torch.autograd.grad(L, x32, retain_graph=True)[0]
    if how != "taps":
        return _rn(contraction(None))
    acc = torch.zeros_like(x32)
    for t in range(g.shape[1]):
        acc = (acc + contraction(t)).bfloat16().float()
    return acc.double()


def _mutations():
    """{name: (output, got, want, x)} on the clean input, reflect padding, similarity on (bf16)."""
    out = {}
    x, ins = _problem("map", "clean", BF16)
    y_ref = evaluate("map", x, ins, torch.float64)["y"][0]
    for how, name in (("inv_norms", "inverse norms rounded to bf16"), ("gram", "Gram / dot entries rounded to bf16"),
                      ("rz", "y rounded toward zero")):
        out[name] = ("y", _map_variant(x, 1, "reflect", how), y_ref, x)
    out["control: map, fp32 then one rounding"] = ("y", _map_variant(x, 1, "reflect", "ok"), y_ref, x)
    # the generic pooled forward as it was: GAP of a map already rounded to bf16
    xp, insp = _problem("pooled", "clean", BF16)
    gap_ref = evaluate("pooled", xp, insp, torch.float64)["gap_nfp"][0]
    y32 = _np(O.nfp_forward(xp.float(), R=1, padding=1, measure="cosine")).double()
    out["GAP of a bf16-rounded map"] = ("gap_nfp", _rn(y32).mean((2, 3)), gap_ref, xp)
    out["control: GAP of the fp32 map"] = ("gap_nfp", y32.mean((2, 3)), gap_ref, xp)
    # backward
    xb, insb = _problem("backward", "clean", BF16)
    gx_ref = evaluate("backward", xb, insb, torch.float64)["gx"][0]
    for how, name in (("coef", "backward coefficients rounded to bf16 (token M without lo)"),
                      ("taps", "per-tap partial gradients accumulated in bf16"),
                      ("ok", "control: backward, fp32 contraction then one rounding")):
        out[name] = ("gx", _grad_variant(xb, insb["gy"], 1, "reflect", how), gx_ref, xb)
    # the pooled upstream gradient g_gap_nfp / (HW), rounded to bf16 before the map backward
    B, C, H, W = xp.shape
    want = evaluate("pooled", xp, insp, torch.float64)["gx"][0]
    gy = _rn((insp["g2"] / (H * W)).float().double())[:, :, None, None].expand(B, 8, H, W).contiguous()
    _, gx = O.nfp_forward_backward(xp.float(), gy.float(), R=1, measure="cosine", padding=1)
    got = _rn(_np(gx).double() + (insp["g1"] / (H * W))[:, :, None, None])
    out["pooled upstream gradient g_gap_nfp / HW rounded to bf16"] = ("gx", got, want, xp)
    return out


MUTATIONS = _mutations()


def test_each_mutation_is_flagged():
    """Sensitivity: every mutation scores > 1 (its controls <= 1).  The printed table is the gap the flat 2e-2 bound
    leaves; the two mutations checked when the bound was questioned (inverse norms in bf16, GAP of a bf16 map) pass it."""
    rows, missed_new, old_misses = [], [], set()
    for name, (out, got, want, x) in MUTATIONS.items():
        new, old = score(out, got, want, x, BF16), old_score(out, got, want, x)
        verdict = "" if name.startswith("control") else ("passes (missed)" if old < OLD_TOL else "fails")
        rows.append(f"{name:62s} {out:8s} ratio {new:10.3g}   2e-2 metric {old:9.2e} {verdict}")
        if name.startswith("control"):
            assert new <= 1.0, (name, new)
            continue
        if not new > 1.0:
            missed_new.append((name, new))
        if old < OLD_TOL:
            old_misses.add(name)
    print("\n" + "\n".join(rows))
    assert not missed_new, missed_new
    assert {"inverse norms rounded to bf16", "GAP of a bf16-rounded map"} <= old_misses, old_misses


# ---- the GPU grid reaches every bf16 cell -------------------------------------------------------------------------
def test_grid_reaches_every_bf16_cell():
    """Every cell of the GPU grid takes the family it is filed under; together they cover every (family, entry point)
    that accepts a bf16 descriptor, all six ring instantiations on every entry point, the options named for each family,
    the three padding modes and both similarity flags on every map family, and clean and degenerate inputs."""
    lib = _capi.load()
    seen, wrong = {}, []
    for c in B.GRID:
        p = B.BF16Problem(c)
        assert p.desc.dtype == _capi.BF16
        path = p.path()
        if not path.startswith(AC.FAMILIES[c.family][0]) or p.launch_count() < 1:
            wrong.append((B.cell_id(c), path))
        if p.head:
            assert lib.nfpb200_head_supported(ctypes.byref(p.desc)) == 0, B.cell_id(c)
        seen.setdefault(c.family, set()).add(c.entry)
    assert not wrong, wrong[:5]
    # every entry point a bf16 descriptor of the family is accepted on (host-only query) is in the grid
    accepted = {}
    for fam, shape, opts in [("stream", (3, 64, 7, 7, 1), {}), ("split", (3, 64, 7, 7, 1), {}),
                             ("band", (2, 8, 21, 16, 1), {}), ("table", (2, 10, 5, 9, 2), {}),
                             ("token", (3, 64, 14, 14, 1), {}), ("generic", (3, 5, 9, 11, 1), {"measure": "dot"})]:
        for e in AC.ENTRIES:
            p = B.BF16Problem(B._cell(fam, e, shape, **opts))
            try:
                ok = p.path().startswith(AC.FAMILIES[fam][0])
            except RuntimeError:
                ok = False
            if ok and p.head:
                ok = lib.nfpb200_head_supported(ctypes.byref(p.desc)) == 0
            if ok:
                accepted.setdefault(fam, set()).add(e)
    assert accepted == ACH.EXPECTED_ENTRIES, accepted
    assert seen == accepted, {f: accepted[f] - seen.get(f, set()) for f in accepted}
    ids = [B.cell_id(c) for c in B.GRID]
    assert len(ids) == len(set(ids))
    # the six ring instantiations on every entry point
    inst = {(B.BF16Problem(c).path(), c.entry) for c in B.GRID if c.family == "stream"}
    for n in ("7x7_r1", "7x7_r2", "14x14_r1", "14x14_r2", "2x2_r1", "4x4_r1"):
        assert {e for m, e in inst if m.endswith(n)} == set(AC.ENTRIES), n
    opts = {(c.family, k, v) for c in B.GRID for k, v in c.opts}
    for want in [("stream", "yf32", 1), ("stream", "inner", 1), ("band", "inner", 1), ("token", "inner", 1),
                 ("token", "yf32", 1), ("token", "xbs", "vit"), ("token", "xbs", "pad8"), ("token", "gxbs", "pad64"),
                 ("token", "gxbs", "pad8"), ("generic", "measure", "cosine"), ("generic", "measure", "dot"),
                 ("generic", "p", 2), ("generic", "measure", "norm")]:
        assert want in opts, want
    assert any(c.shape == (3, 40, 7, 7, 1) and c.entry == "backward" for c in B.GRID)            # strip form
    assert {c.entry for c in B.GRID if c.shape == (300, 512, 7, 7, 1)} == {"forward", "backward"}
    assert any(c.family == "token" and c.shape[1] == 512 for c in B.GRID)
    for fam in ("stream", "band", "table", "token"):
        ms = {(dict(c.opts).get("mode", "reflect"), dict(c.opts).get("sim", 1)) for c in B.GRID if c.family == fam}
        assert ms == {(m, s) for m in G.MODES for s in (1, 0)}, (fam, ms)
        for e in ("forward", "backward"):
            assert {dict(c.opts).get("kind", "clean") for c in B.GRID if c.family == fam and c.entry == e} == \
                {"clean", "deg"}, (fam, e)
    for fam, es in accepted.items():   # degenerate input on every entry point
        for e in es:
            assert "deg" in {dict(c.opts).get("kind") for c in B.GRID if c.family == fam and c.entry == e}, (fam, e)


def test_gpu_check_passes_the_honest_evaluation():
    """The GPU file's own check_cell, handed fp32 evaluations rounded once instead of kernel results, passes a sample
    of its cells (every family, entry point and input kind): the bound is met by what a correct kernel computes."""
    seen, bad = set(), []
    for c in B.GRID:
        key = (c.family, c.entry, dict(c.opts).get("kind", "clean"))
        if key in seen or dict(c.opts).get("inner") or c.shape[0] > 8:
            continue
        seen.add(key)
        p = B.BF16Problem(c)
        exp64, rows = p.expected()
        x32 = p.x.float().double()
        q = B.BF16Problem(c)
        q.x = x32.float()   # the same evaluation in fp32
        for attr in ("gy", "g_gap_x", "g_gap_nfp", "proj_w", "proj_b", "g_out", "gap_x_in", "gap_nfp_in"):
            if hasattr(q, attr):
                setattr(q, attr, getattr(q, attr).float())
        exp32, _ = q.expected()

        def got_of(n):
            v = torch.zeros((p.B,) + tuple(exp32[n].shape[1:]), dtype=torch.float64)
            v[rows] = exp32[n].double()
            return v if (n not in ("y", "gx") or (n == "y" and p.yf32)) else round_nearest(BF16, v)
        res = B.check_cell(p, got_of)
        if not all(r <= 1.0 for r, _ in res.values()):
            bad.append((B.cell_id(c), res))
    assert not bad, bad[:3]


def test_rn_mismatches():
    """The widened-map pin: an fp32 evaluation rounded once to nearest has no mismatch (ties within tau S excused);
    rounding toward zero, or one element off by an ulp, is counted."""
    x, ins = _problem("map", "clean", BF16)
    want = evaluate("map", x, ins, torch.float64)["y"][0]
    y32 = evaluate("map", x, ins, torch.float32)["y"][0]
    assert rn_mismatches(round_nearest(BF16, y32), want, BF16, TAU) == 0
    assert rn_mismatches(_rz_bf16(y32), want, BF16, TAU) > want.numel() // 10
    off = round_nearest(BF16, want).clone()
    i = int(off.abs().flatten().argmax())
    off.view(-1)[i] += ulp(BF16, off.view(-1)[i:i + 1])[0]
    assert rn_mismatches(off, want, BF16, TAU) == 1
