"""Shared helpers of the test-suite (golden fixtures, error norms)."""
import json
import math
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_measure_cases():
    with open(os.path.join(GOLDEN, "nfp_measures.json")) as f:
        index = json.load(f)["cases"]
    arrays = {}
    for part in (1, 2):   # stored in two halves by case (oracle/make_golden.py) to keep each file under 1 MB
        arrays.update(np.load(os.path.join(GOLDEN, f"nfp_measures_{part}.npz")))
    return index, arrays


def load_wrapper_cases():
    with open(os.path.join(GOLDEN, "nfp_pooling_wrapper.json")) as f:
        index = json.load(f)["cases"]
    arrays = np.load(os.path.join(GOLDEN, "nfp_pooling_wrapper.npz"))
    return index, arrays


def load_multi_radius_cases():
    with open(os.path.join(GOLDEN, "nfp_multi_radius.json")) as f:
        index = json.load(f)["cases"]
    arrays = np.load(os.path.join(GOLDEN, "nfp_multi_radius.npz"))
    return index, arrays


def case_kwargs(c):
    return dict(R=c["R"], measure=c["measure"], p=c["p"], stride=c["stride"], padding=c["padding"],
                dilation=c["dilation"], padding_mode=c["padding_mode"], similarity=c["similarity"])


def case_id(c):
    return f'{c["key"]}-{c["measure"]}-{c["geom"]}-sim{int(c["similarity"])}-p{c["p"]}'


def rel_err(got, want):
    """max |got - want| over the finite entries of `want`, relative to max(1e-30, max |want|)."""
    got = torch.as_tensor(np.asarray(got), dtype=torch.float64)
    want = torch.as_tensor(np.asarray(want), dtype=torch.float64)
    fin = torch.isfinite(want)
    if not fin.any():
        return 0.0
    if not torch.isfinite(got[fin]).all():
        return float("inf")
    scale = max(want[fin].abs().max().item(), 1e-30)
    return ((got - want)[fin].abs().max() / scale).item()


SMALL_NORM = 1e-3   # well below any ordinary activation's norm, far above eps


def pixel_regions(x, eps=1e-6):
    """(B, H, W) region label of every pixel of the (B, C, H, W) input `x`, by its norm over channels.

    The cosine gradient at a pixel scales like |gy| / max(||x_pixel||, eps): pixels with ||x|| <= 2 eps ("deg") get
    gradients near 1 / eps = 1e6, pixels a little above that ("small", up to SMALL_NORM) up to 5e5, ordinary pixels
    about |gy| / ||x||.  Scored on a common scale, the first two hide every error in the third."""
    n = torch.linalg.vector_norm(torch.as_tensor(np.asarray(x), dtype=torch.float64), dim=1)
    lab = torch.full(n.shape, 2, dtype=torch.int64)
    lab[n < SMALL_NORM] = 1
    lab[n <= 2 * eps] = 0
    return lab


REGION_NAMES = ("deg", "small", "ordinary")


def grad_errs(got, want, x, eps=1e-6, per_image=True):
    """{(image, region): rel_err of the input gradient over that image's pixels of that region} (pixel_regions);
    image None when per_image=False (each region over the whole batch)."""
    got = torch.as_tensor(np.asarray(got), dtype=torch.float64)
    want = torch.as_tensor(np.asarray(want), dtype=torch.float64)
    lab = pixel_regions(x, eps)
    assert got.shape == want.shape and lab.shape == (want.shape[0],) + tuple(want.shape[2:]), (got.shape, lab.shape)
    # (C, B, H, W): a boolean (B, H, W) mask then selects whole pixels
    got, want = got.transpose(0, 1), want.transpose(0, 1)
    out = {}
    for b in (range(want.shape[1]) if per_image else [None]):
        for r, name in enumerate(REGION_NAMES):
            m = lab == r
            if b is not None:
                m = m & (torch.arange(m.shape[0]) == b)[:, None, None]
            if m.any():
                out[(b, name)] = rel_err(got[:, m], want[:, m])
    return out


def grad_err(got, want, x, eps=1e-6, per_image=True):
    """Max-norm relative error of an input gradient with each image and each pixel region (pixel_regions) on its
    own scale.  Use it instead of rel_err for input gradients: with a whole-tensor scale the 1e6-sized gradients of
    pixels with ||x|| <= 2 eps hide every error elsewhere, and one image's large gradients hide another's.
    `x` is the input the reference saw."""
    return max(grad_errs(got, want, x, eps, per_image).values())


def reached_pixels(geo):
    """(H, W) bool: the input pixels that some output reads, as its centre or as one of its taps, under the oracle's
    index tables (oracle.nfp_oracle.geometry).  Every other pixel gets no gradient from the map in any measure."""
    from oracle import nfp_oracle as O
    ids = torch.arange(1, geo.H * geo.W + 1, dtype=torch.float64).view(1, 1, geo.H, geo.W)
    c, n = O.gather_centre_neighbours(ids, geo)   # an implicit zero of 'zeros' padding reads id 0
    seen = torch.cat([c.flatten(), n.flatten()]).long()
    hit = torch.zeros(geo.H * geo.W + 1, dtype=torch.bool)
    hit[seen] = True
    return hit[1:].view(geo.H, geo.W)


# |want| relative to the median nonzero |want| of its image.  Up to 10x ("bulk") is the ordinary gradient of randn
# inputs; between 10x and 1000x ("high") sit the pixels next to a 1e3-scaled pixel and the moderately small
# denominators; above 1000x ("spike") the denominators within a few eps of 0 (|c| + |n| + eps, ||c|| ~ eps), whose
# gradients reach 1e5-1e7 x the median and would otherwise set the scale of the whole image.
ELEM_BUCKETS = ((10.0, "bulk"), (1000.0, "high"), (math.inf, "spike"))
_MANTISSA_BITS = {torch.float32: 23, torch.bfloat16: 7}


def elem_grad_errs(got, want, geo, dtype=torch.float32):
    """{(image, bucket): error} of an input gradient, for any measure (the companion of grad_errs, which is built for
    the cosine measure's pixel-norm regions).

    * "struct": elements of pixels no output reaches (reached_pixels).  Their gradient is exact by construction: 0.0 in
      map mode, g_gap_x / (H*W) in pooled mode (already in `want`).  The entry is 0.0 when every such element of the
      image is within one ulp of `dtype` of `want` (so exactly 0.0 where want is 0), else inf.
    * "bulk", "high", "spike": the other elements, by |want| over the image's median nonzero |want| (ELEM_BUCKETS),
      each scored with rel_err on its own scale.  A few elements whose denominator is near 0 carry gradients 1e6 x
      the rest; on a common scale they would hide any error in the others.
    """
    got = torch.as_tensor(np.asarray(got), dtype=torch.float64)
    want = torch.as_tensor(np.asarray(want), dtype=torch.float64)
    assert got.shape == want.shape and tuple(want.shape[2:]) == (geo.H, geo.W), (got.shape, want.shape)
    struct = ~reached_pixels(geo)
    out = {}
    for b in range(want.shape[0]):
        gb, wb = got[b], want[b]
        if struct.any():
            gs, ws = gb[:, struct], wb[:, struct]
            e = torch.floor(torch.log2(ws.abs().clamp_min(1e-300)))
            ulp = torch.where(ws == 0, torch.zeros_like(ws), torch.exp2(e - _MANTISSA_BITS[dtype]))
            out[(b, "struct")] = 0.0 if bool(((gs - ws).abs() <= ulp).all()) else math.inf
        gr, wr = gb[:, ~struct], wb[:, ~struct]
        mag = wr.abs()
        nz = mag[(mag > 0) & torch.isfinite(mag)]
        med = nz.median().item() if nz.numel() else 1.0
        lo = -1.0   # the bulk bucket starts below 0: it holds the zero elements too
        for hi, name in ELEM_BUCKETS:
            m = (mag > lo * med) & (mag <= hi * med)
            if m.any():
                out[(b, name)] = rel_err(gr[m], wr[m])
            lo = hi
    return out


def elem_grad_err(got, want, geo, dtype=torch.float32):
    """max of elem_grad_errs: the input-gradient error of the generic kernels' tests (0.0 when `want` has no finite
    element: the NaN footprint of a zero difference in rmse / hellinger is not compared)."""
    return max(elem_grad_errs(got, want, geo, dtype).values(), default=0.0)


def worst(errs, k=4):
    """The k largest entries of a grad_errs() table, for assertion messages."""
    return sorted(errs.items(), key=lambda kv: -kv[1])[:k]


# ---- guarded buffers (tests/test_abi_contract_*.py) ------------------------------------------------------------------
# A typed body inside one larger uint8 allocation, with a lead and a tail guard.  Inputs: body = data, guards = quiet
# NaN, so a read past either end that feeds a result turns it into NaN.  Outputs and the workspace: body and guards
# hold a NaN with a recognisable payload (SENTINEL), so a write outside the body, and an element never written, show.
GUARD_BYTES = 256 * 1024   # larger than any single transfer of any path (a ring chunk, a band slab)
QNAN = {torch.float32: 0x7FC00000, torch.bfloat16: 0x7FC0, torch.uint8: 0x7F}
SENTINEL = {torch.float32: 0x7FA5A5A5, torch.bfloat16: 0x7FA5, torch.uint8: 0xA5}
_BITS = {torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.uint8: torch.uint8}


def bits(t):
    """The raw bit patterns of a float tensor (for exact, NaN-aware comparison)."""
    return t.contiguous().view(_BITS[t.dtype])


def fill_bits(t, pattern):
    """Fill a float tensor with one bit pattern (e.g. a NaN with a payload, which a float fill cannot express)."""
    esz = t.element_size()
    if _BITS[t.dtype] is not torch.uint8 and pattern >= 2 ** (8 * esz - 1):
        pattern -= 2 ** (8 * esz)   # the same bits as a signed integer
    t.view(_BITS[t.dtype]).fill_(pattern)


class Guarded:
    """`numel` elements of `dtype` at byte address % 512 == `place`, GUARD_BYTES of guard on each side.

    kind "input": body = `data` (flat, NaN where `data` is NaN), guards quiet NaN; the whole allocation must stay
    bit-unchanged.  kind "output" / "workspace": body and guards SENTINEL; the guards must stay unchanged, and so must
    every body element outside `written` (a flat bool mask, default all), while no element inside it may still hold
    SENTINEL after the call."""

    def __init__(self, numel, dtype, device, kind, data=None, place=16, written=None, guard=GUARD_BYTES):
        esz = torch.empty(0, dtype=dtype).element_size()
        assert place % esz == 0 and kind in ("input", "output", "workspace")
        self.dtype, self.kind, self.numel = dtype, kind, numel
        self.raw = torch.empty(2 * guard + numel * esz + 512 + 16, dtype=torch.uint8, device=device)
        lead = guard + (place - (self.raw.data_ptr() + guard)) % 512
        self.lo, self.hi = lead, lead + numel * esz
        fill = QNAN[dtype] if kind == "input" else SENTINEL[dtype]
        n_el = self.raw.numel() // esz
        fill_bits(self.raw[:n_el * esz].view(dtype), fill)
        self.raw[n_el * esz:].fill_(0xFF)
        if data is not None:
            self.body.copy_(data.reshape(-1).to(device, dtype))
        self.written = written
        self.snapshot = self.raw.clone()

    @property
    def body(self):
        return self.raw[self.lo:self.hi].view(self.dtype)

    def ptr(self):
        return self.raw.data_ptr() + self.lo

    def problems(self, name):
        """What the last call did wrong to this buffer (empty list: nothing)."""
        out = []
        raw, ref = self.raw, self.snapshot
        for side, a, b in (("lead guard", 0, self.lo), ("tail guard", self.hi, raw.numel())):
            bad = (raw[a:b] != ref[a:b]).nonzero()
            if bad.numel():
                out.append(f"{name}: {side} changed at {bad.numel()} bytes, first at {int(bad[0]) - (self.lo if a else a)}"
                           f" bytes from the body")
        if self.kind == "input":
            bad = (raw[self.lo:self.hi] != ref[self.lo:self.hi]).nonzero()
            if bad.numel():
                out.append(f"{name}: input body written at {bad.numel()} bytes, first at byte {int(bad[0])}")
            return out
        got = bits(self.body)
        want = bits(ref[self.lo:self.hi].view(self.dtype))
        wr = self.written if self.written is not None else torch.ones(self.numel, dtype=torch.bool)
        wr = wr.to(got.device)
        if self.kind == "output":
            left = ((got == want) & wr).nonzero()
            if left.numel():
                out.append(f"{name}: {left.numel()} elements never written, first at {int(left[0])}")
        gap = ((got != want) & ~wr).nonzero()
        if gap.numel():
            out.append(f"{name}: {gap.numel()} elements written outside the output, first at {int(gap[0])}")
        return out


def guard_problems(bufs):
    """Every problem of every buffer of a call: {name: Guarded} -> list of messages."""
    return [m for name, g in bufs.items() if g is not None for m in g.problems(name)]
