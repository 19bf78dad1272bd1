"""GPU: the persistent fused kernels past their first wave, checked image by image.

The ring (fused/stream_*), cluster-split (fused/split_*) and token (fused/token_*) kernels are persistent: the grid is
the resident CTAs (ring, token: min(B, resident CTAs); split: every resident cluster), and CTA i takes images i,
i + grid, i + 2 grid, ...  More images than resident CTAs changes more than the loop count: the ring backward switches
to a double-buffered upstream gradient without per-lane partial tables (and re-plans its stages), the token kernels
prefetch a CTA's next image into their second buffer, the split kernels' image ring wraps.  The other suites run
almost everything at B <= 8, inside one wave.

Every cell here measures its resident grid g once (nfpb200_debug_phase_timing at a large B: the CTAs that stamped),
then runs at B = g (one full wave), g + 1 (one CTA takes a second image; the ring backward's two-buffer plan) and
2g + 3 (three rounds on some CTAs: an odd round count for the barrier phase bits, a wrap of the split image ring):

1. the fp64 oracle on images 0, g-1, g, min(2g, B-1) and B-1 (the first and last image of round one, the first of
   round two, the last), with each suite's bounds: fp32 1e-5 (grad_errs for gx), bf16 rounding_errs <= 1 with its fp32
   outputs at 1e-5, fp16 the TOL_* bounds of test_f16_gpu;
2. every image against the same entry point called on slices of at most 8 images (device views at the image offsets,
   batch strides kept): the forward entries bit-identical, the backward entries (a different plan) within fp32
   grad_errs 1e-5, or one 16-bit ulp + tau S (S the image's largest |gx|);
3. outputs pre-filled with a NaN sentinel: no element of any image still holds it after the big call or the slices;
4. a rerun of the big call: identical bits.

The grid (GRID) holds a multi-round cell for every (family, instantiation, dtype, entry point) the library serves
(tests/test_batch_waves_host.py checks that on the CPU) and the channel counts that reach each planner configuration.
The measured g of each cell is recorded as the property "grid".

Also here: the planar row-band kernels put B in gridDim.y and hand B > 65535 to the generic kernels; both sides of
that boundary against each other and the oracle.
"""
import copy
import ctypes
from collections import namedtuple

import numpy as np
import pytest
import torch

import _util
import test_abi_contract_gpu as AC
import test_bf16_rounding_gpu as BR
import test_f16_gpu as F16T
from _util import SENTINEL, bits, fill_bits, grad_errs, rel_err, worst
from neighbour_feature_pooling_b200 import _capi
from oracle import nfp_oracle as O

pytestmark = pytest.mark.gpu

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
ENTRIES = AC.ENTRIES
FWD_ENTRIES = ("forward", "pool_forward", "pooled_map_forward", "head_forward")
FB = ("forward", "backward")
TAU = 1e-5            # the fp32 budget of the cosine kernels (every fp32 bound below, and tau of the 16-bit ones)
SLICE = 8             # images per single-wave call
STAMPS_PER_CTA = {"stream": 8, "split": 16, "token": 16}   # include/nfp_b200.h, nfpb200_debug_phase_timing
PROBLEM = {F32: AC.Problem, BF16: BR.BF16Problem, F16: F16T.F16Problem}
DTYPE_NAME = {F32: "fp32", BF16: "bf16", F16: "f16"}

# a cell without its batch size: shape = (C, H, W, R)
WCell = namedtuple("WCell", "family entry shape dtype opts")


def _cells(family, entries, shape, dtypes, **opts):
    out = []
    for e in entries:
        o = dict(opts)
        if family == "token" and not e.endswith("backward"):
            o.pop("gxbs", None)   # gx batch strides only where there is a gx
        out += [WCell(family, e, shape, dt, tuple(sorted(o.items()))) for dt in dtypes]
    return out


def _grid():
    g = []
    # ring: every entry point at one channel count per instantiation (the bench workloads' where there is one)
    for s in [(512, 7, 7, 1), (512, 7, 7, 2), (256, 14, 14, 1), (256, 14, 14, 2), (512, 2, 2, 1), (64, 4, 4, 1)]:
        g += _cells("stream", ENTRIES, s, (F32, BF16, F16))
    # the other ring plans: lane-per-channel NCH = 1 (64), streamed NCH = 15 (960), the strip form (40 = C % 64 != 0),
    # small-C R = 2, bf16 resident image at 14x14 (112)
    for s in [(64, 7, 7, 1), (960, 7, 7, 1), (40, 7, 7, 1), (32, 7, 7, 2), (112, 14, 14, 1), (32, 14, 14, 2)]:
        g += _cells("stream", FB, s, (F32, BF16))
    # the two multi-radius bench workloads (R = 2 with the inner radius-1 map), the x-stable hint, fp32 maps
    for s in [(512, 7, 7, 2), (256, 14, 14, 2)]:
        g += _cells("stream", FB, s, (F32, BF16, F16), inner=1)
        g += _cells("stream", ("backward",), s, (F32, BF16), hint=1)
        g += _cells("stream", ("forward",), s, (BF16,), yf32=1)
    # token (channels-last): every entry point per instantiation; the ViT-Tiny view (class token in front, padded gx)
    tok = (BF16, F16)
    g += _cells("token", ENTRIES, (64, 7, 7, 1), tok)                          # two 8-warp CTAs per SM
    g += _cells("token", ENTRIES, (512, 7, 7, 2), tok)                         # 16 warps, two image buffers
    g += _cells("token", ENTRIES, (192, 14, 14, 1), tok, xbs="vit", gxbs="pad64")   # 16 warps, one buffer
    for s in [(64, 14, 14, 2), (64, 2, 2, 1), (64, 4, 4, 1)]:
        g += _cells("token", ENTRIES, s, tok)
    g += _cells("token", FB, (512, 7, 7, 1), tok)
    g += _cells("token", FB, (960, 7, 7, 1), tok)                              # 16 warps, one buffer
    g += _cells("token", ("backward",), (64, 14, 14, 1), tok)                  # 16 warps, two image buffers
    g += _cells("token", FB, (512, 7, 7, 2), tok, inner=1, xbs="pad8", gxbs="pad8")
    # cluster-split (NFPB200_PATH_SPLIT), every instantiation
    for s in [(64, 7, 7, 1), (64, 14, 14, 1), (64, 2, 2, 1), (64, 4, 4, 1), (64, 7, 7, 2), (64, 14, 14, 2)]:
        g += _cells("split", ENTRIES[:6], s, (F32, BF16))
    return g


GRID = _grid()


def wave_id(w):
    C, H, W, R = w.shape
    extra = "".join(f"-{k}{v}" for k, v in w.opts)
    return f"{w.family}-{w.entry}-{C}x{H}x{W}_r{R}-{DTYPE_NAME[w.dtype]}{extra}"


def batch_sizes(g):
    """One full wave, one CTA with a second image, three rounds on some CTAs."""
    return (g, g + 1, 2 * g + 3)


def scored_rows(g, B):
    """The images the oracle scores: first / last of round one, first of round two, the last image."""
    return sorted({r for r in (0, g - 1, g, min(2 * g, B - 1), B - 1) if 0 <= r < B})


def problem(w, B):
    return PROBLEM[w.dtype](AC._cell(w.family, w.entry, (B,) + tuple(w.shape), w.dtype, **dict(w.opts)))


# ---- buffers by image ----------------------------------------------------------------------------------------------
def image_elems(prob, name):
    """Elements from one image of a buffer to the next (0: the buffer is shared by every image)."""
    dense = prob.C * prob.H * prob.W
    if name == "x":
        return (prob.xbs or dense) if prob.nhwc else dense
    if name == "gx":
        return (prob.gxbs or dense) if prob.nhwc else dense
    if name in ("y", "gy"):
        return prob.Ky * prob.Ho * prob.Wo
    if name in ("gap_x", "g_gap_x", "out", "g_out"):
        return prob.C
    if name in ("gap_nfp", "g_gap_nfp"):
        return prob.K
    return 0   # proj_w, proj_b


def _ptrs_at(prob, bufs, lo):
    """Pointers of every buffer at image `lo` (x one class token further in for the ViT view)."""
    p = {}
    for n, t in bufs.items():
        lead = prob.lead if n == "x" else 0
        p[n] = t.data_ptr() + (lead + lo * image_elems(prob, n)) * t.element_size()
    return p


def _resized(prob, B):
    """A shallow copy of `prob` whose descriptor says B images (its buffers are the caller's)."""
    sub = copy.copy(prob)
    sub.desc = type(prob.desc).from_buffer_copy(prob.desc)
    sub.desc.B = B
    sub.B = B
    return sub


def _call(prob, bufs, lo=0, ws=None):
    wn = prob.workspace_bytes()
    if wn and ws is None:
        ws = torch.empty(wn, dtype=torch.uint8, device=next(iter(bufs.values())).device)
    rc = prob.call(_ptrs_at(prob, bufs, lo), ws.data_ptr() if wn else None, wn,
                   torch.cuda.current_stream().cuda_stream)
    assert rc == 0, _capi.status_string(rc)


def _sentinel_outputs(prob, dev):
    outs = {}
    for n, (sz, dt, _) in prob.outputs.items():
        outs[n] = torch.empty(sz, dtype=dt, device=dev)
        fill_bits(outs[n], SENTINEL[dt])
    return outs


def _unwritten(prob, outs):
    """{output: elements (inside its images) still holding the sentinel}."""
    left = {}
    for n, (_, dt, mask) in prob.outputs.items():
        want = torch.empty(1, dtype=dt)
        fill_bits(want, SENTINEL[dt])
        hit = (bits(outs[n]).cpu() == bits(want))
        if mask is not None:
            hit &= mask
        if hit.any():
            left[n] = int(hit.sum())
    return left


# ---- the resident grid ----------------------------------------------------------------------------------------------
_GRIDS = {}


def resident_grid(w, dev):
    """CTAs of the call's grid at a batch past one wave: the CTAs that wrote a phase stamp, at the first of 4, 16, 64
    images per SM where fewer CTAs than images stamped."""
    if w in _GRIDS:
        return _GRIDS[w]
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    for per_sm in (4, 16, 64):
        g = _stamped_ctas(w, dev, per_sm * sms)
        if g < per_sm * sms:
            break
    assert 0 < g < per_sm * sms, (g, per_sm * sms)   # the grid is the resident CTAs, not the batch
    _GRIDS[w] = g
    return g


def _stamped_ctas(w, dev, Bbig):
    small = problem(w, 2)
    big = _resized(small, Bbig)
    bufs = {}
    for n, (d, dt) in small.inputs.items():
        e = image_elems(small, n)
        numel = d.numel() + (Bbig - 2) * e   # the same tail and lead, more images
        bufs[n] = torch.randn(numel, device=dev).to(dt)
    for n, (sz, dt, _) in small.outputs.items():
        bufs[n] = torch.empty(sz + (Bbig - 2) * image_elems(small, n), dtype=dt, device=dev)
    stamps = torch.zeros(16 * Bbig, dtype=torch.int64, device=dev)
    lib = _capi.load()
    torch.cuda.synchronize()
    lib.nfpb200_debug_phase_timing(ctypes.c_void_p(stamps.data_ptr()))
    try:
        _call(big, bufs)
        torch.cuda.synchronize()
    finally:
        lib.nfpb200_debug_phase_timing(None)
    return int((stamps.view(-1, STAMPS_PER_CTA[w.family])[:, 0] != 0).sum())


# ---- checks ---------------------------------------------------------------------------------------------------------
def check_oracle(prob, outs):
    """Failures of the scored images against the fp64 oracle, with the suite's bounds of the dtype."""
    dt = prob.c.dtype
    got_of = lambda n: prob.logical(n, outs[n])   # noqa: E731
    bad = {}
    if dt == BF16:
        for n, (r, w) in BR.check_cell(prob, got_of).items():
            if not r <= 1.0:
                bad[n] = w
        return bad
    exp, rows = prob.expected()
    for n, ref in exp.items():
        got = got_of(n)[rows]
        if n == "gx":
            errs = {(rows[i], k): v for (i, k), v in grad_errs(got, ref, prob.x[rows], AC.EPS).items()}
            tol = TAU if dt == F32 else F16T.TOL_GRAD
        else:
            errs = {rows[i]: rel_err(got[i], ref[i]) for i in range(len(rows))}
            tol = TAU if dt == F32 else F16T._tol(prob, n)
        if not max(errs.values()) <= tol:
            bad[n] = (tol, worst(errs, 3))
    return bad


def gx_mismatch(prob, a, b):
    """Images whose gx differs between two runs by more than the backward's tolerance: fp32 grad_errs <= tau per
    image and pixel region; 16-bit one ulp + tau S, S the image's largest |gx|.  {image: error} of the failures."""
    bad = {}
    if prob.c.dtype == F32:
        for lo in range(0, prob.B, SLICE):
            hi = min(lo + SLICE, prob.B)
            errs = grad_errs(a[lo:hi], b[lo:hi], prob.x[lo:hi], AC.EPS)
            for (i, k), v in errs.items():
                if not v <= TAU:
                    bad[(lo + i, k)] = v
        return bad
    m = torch.maximum(a.abs(), b.abs())
    S = m.flatten(1).amax(1).view(-1, 1, 1, 1)
    ratio = ((a - b).abs() / (_util.ulp(prob.c.dtype, m) + TAU * S)).flatten(1).amax(1)
    for i in (~(ratio <= 1.0)).nonzero().flatten().tolist():
        bad[i] = ratio[i].item()
    return bad


@pytest.mark.parametrize("w", [pytest.param(w, id=wave_id(w)) for w in GRID])
def test_batch_waves(w, cuda_device, record_property):
    g = resident_grid(w, cuda_device)
    record_property("grid", g)
    prefix = AC.FAMILIES[w.family][0]
    for B in batch_sizes(g):
        assert B == g or g < B
        prob = problem(w, B)
        prob.rows = scored_rows(g, B)
        path = prob.path()
        assert path.startswith(prefix), path
        where = f"B={B} g={g}"
        ins = {n: d.to(cuda_device, dt) for n, (d, dt) in prob.inputs.items()}
        big = _sentinel_outputs(prob, cuda_device)
        _call(prob, {**ins, **big})
        torch.cuda.synchronize()
        left = _unwritten(prob, big)
        assert not left, (where, "never written", left)
        want = AC._out_bits(prob, big)
        bad = check_oracle(prob, big)
        assert not bad, (where, "oracle", bad)
        # the big call again: the same bits
        _call(prob, {**ins, **big})
        torch.cuda.synchronize()
        same = AC._same_bits(AC._out_bits(prob, big), want)
        assert all(same.values()), (where, "rerun", same)
        # every image from single-wave calls on slices of at most SLICE images
        sl = _sentinel_outputs(prob, cuda_device)
        sub = _resized(prob, SLICE)
        assert sub.path() == path and sub.launch_count() == prob.launch_count(), (sub.path(), path)
        ws = torch.empty(max(sub.workspace_bytes(), 1), dtype=torch.uint8, device=cuda_device)
        for lo in range(0, B, SLICE):
            part = sub if B - lo >= SLICE else _resized(prob, B - lo)
            _call(part, {**ins, **sl}, lo, ws)
        torch.cuda.synchronize()
        left = _unwritten(prob, sl)
        assert not left, (where, "never written by the slices", left)
        if w.entry in FWD_ENTRIES:
            same = AC._same_bits(AC._out_bits(prob, sl), want)
            assert all(same.values()), (where, "single-wave slices differ", same)
        else:
            bad = gx_mismatch(prob, prob.logical("gx", big["gx"]), prob.logical("gx", sl["gx"]))
            assert not bad, (where, "single-wave slices differ", len(bad), sorted(bad.items())[:6])
        del ins, big, sl, ws


# ---- the planar kernels' batch limit ------------------------------------------------------------------------------
PLANAR_LIMIT = 65535   # gridDim.y


def _band_desc(B):
    return _capi.make_desc(_capi.F32, B, 8, 21, 16, 1, 1, 1, 1, "reflect", "cosine", True, False, AC.EPS, 1, 1e-6)


def test_planar_batch_limit(cuda_device):
    """B = 65535 takes the row-band kernels (B in gridDim.y), B = 65536 the generic kernels: the two agree on the
    images they share, and both match the fp64 oracle on a few of them."""
    B, C, H, W = PLANAR_LIMIT + 1, 8, 21, 16
    lib = _capi.load()
    gen = torch.Generator(device=cuda_device).manual_seed(65536)
    x = torch.randn(B, C, H, W, device=cuda_device, generator=gen)
    gy = torch.randn(B, 8, H, W, device=cuda_device, generator=gen)
    paths = {}
    res = {}
    for n in (PLANAR_LIMIT, PLANAR_LIMIT + 1):
        d = _band_desc(n)
        paths[n] = tuple(_capi.describe_path(d, op) for op in (_capi.OP_FORWARD, _capi.OP_BACKWARD))
        y = torch.empty(n, 8, H, W, device=cuda_device)
        gx = torch.empty(n, C, H, W, device=cuda_device)
        s = torch.cuda.current_stream().cuda_stream
        for op, call in ((_capi.OP_FORWARD, lambda p, k: lib.nfpb200_forward(ctypes.byref(d), x.data_ptr(),
                                                                              y.data_ptr(), p, k, s)),
                         (_capi.OP_BACKWARD, lambda p, k: lib.nfpb200_backward(ctypes.byref(d), x.data_ptr(),
                                                                               gy.data_ptr(), gx.data_ptr(), p, k, s))):
            k = _capi.workspace_bytes(d, op)
            ws = torch.empty(max(k, 1), dtype=torch.uint8, device=cuda_device)
            rc = call(ws.data_ptr() if k else None, k)
            assert rc == 0, _capi.status_string(rc)
        torch.cuda.synchronize()
        res[n] = (y, gx)
    assert all(p.startswith("planar/band") for p in paths[PLANAR_LIMIT]), paths
    assert all(p.startswith("generic/pairs") for p in paths[PLANAR_LIMIT + 1]), paths
    rows = [0, 1, 32767, PLANAR_LIMIT - 2, PLANAR_LIMIT - 1]
    xr = x[rows].double().cpu()
    y_ref, gx_ref = O.nfp_forward_backward(xr, gy[rows].double().cpu(), R=1, measure="cosine", padding=1,
                                           padding_mode="reflect", similarity=True, eps=AC.EPS)
    y_ref, gx_ref = torch.as_tensor(np.asarray(y_ref)), torch.as_tensor(np.asarray(gx_ref))
    for n, (y, gx) in res.items():
        yr, gr = y[rows].double().cpu(), gx[rows].double().cpu()
        e = max(rel_err(yr[i], y_ref[i]) for i in range(len(rows)))
        errs = grad_errs(gr, gx_ref, xr, AC.EPS)
        assert e <= TAU and max(errs.values()) <= TAU, (n, e, worst(errs))
    # every shared image: the two paths within fp32 accuracy of each other, image by image
    (ya, ga), (yb, gb) = res[PLANAR_LIMIT], res[PLANAR_LIMIT + 1]
    yb, gb = yb[:PLANAR_LIMIT], gb[:PLANAR_LIMIT]
    for a, b in ((ya, yb), (ga, gb)):
        err = ((a - b).abs().flatten(1).amax(1) / b.abs().flatten(1).amax(1).clamp_min(1e-30))
        assert bool((err <= TAU).all()), (int((err > TAU).sum()), err.max().item())
