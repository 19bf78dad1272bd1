"""TEST INFRASTRUCTURE ONLY -- CPU restatement of Neighbourhood Feature Pooling.

This is the parity oracle for the CUDA path.  It restates the algorithm of the
reference operator in *gather form*: instead of the reference's two frozen
one-hot depthwise convolutions (reference ``models/pooling/nfp.py:42-82``) it
indexes the centre pixel and the ``k*k-1`` neighbour pixels directly, which is
the same arithmetic (multiplying by a one-hot kernel is a copy) and lets the
oracle run in fp64.  The floating-point semantics that live in ATen
(``cosine_similarity``, ``linalg.norm``, ``softmax``) are kept by calling the
same ATen ops the reference calls.

Pinned against the reference itself by ``oracle/check_against_reference.py``
(run where a reference checkout is named by ``NFP_REFERENCE_ROOT``) and by the
fixtures in ``tests/golden/`` (``oracle/make_golden.py``).

Citations are ``file:line`` relative to the reference checkout.

Never import this module from the product package.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F

# nfp.py:85-118 -- the 18 accepted (lower-cased) spellings -> 17 distinct measures
MEASURES = (
    "norm", "cosine", "dot", "rmse", "geman", "attention", "emd", "canberra",
    "hellinger", "chisquared1", "chisquared2", "gfc", "pearson", "jeffrey",
    "squaredchord", "smith", "scs",
)
_ALIASES = {"sharpened_cosine": "scs"}  # nfp.py:117
PADDING_MODES = ("zeros", "reflect", "replicate", "circular")  # torch.nn.Conv2d


def canonical_measure(measure: str) -> str:
    """nfp.py:21 lower-cases; nfp.py:119-120 raises RuntimeError when unknown."""
    m = _ALIASES.get(measure.lower(), measure.lower())
    if m not in MEASURES:
        raise RuntimeError(f"Similarity measure {measure.lower()} not implemented")
    return m


def uses_difference_taps(measure_as_given: str) -> bool:
    """nfp.py:74 tests the *raw* constructor string (case-sensitive quirk).

    When true the neighbour conv emits ``centre - neighbour``; otherwise it
    emits the pure neighbour (nfp.py:78-80).  Only Norm and RMSE read that
    tensor without a separate centre (nfp.py:143, 174).
    """
    return measure_as_given in ("norm", "rmse", "mahalanobis")


def tap_offsets(R: int):
    """Row-major k x k window with the centre removed (nfp.py:64-67)."""
    k = 2 * R + 1
    return [(a, b) for a in range(k) for b in range(k) if not (a == R and b == R)]


def _map_index(i: int, n: int, mode: str) -> int:
    """Source index for padded coordinate ``i`` (already shifted by -pad), or -1
    for an implicit zero.  Semantics of F.pad / Conv2d padding_mode."""
    if 0 <= i < n:
        return i
    if mode == "zeros":
        return -1
    if mode == "reflect":
        return -i if i < 0 else 2 * (n - 1) - i
    if mode == "replicate":
        return 0 if i < 0 else n - 1
    if mode == "circular":
        return i % n
    raise ValueError(f"padding_mode {mode!r}")


@dataclass
class Geometry:
    H: int
    W: int
    R: int
    stride: int
    padding: int
    dilation: int
    padding_mode: str
    Ho: int
    Wo: int
    row_c: np.ndarray  # (Ho,)   source row of the centre, -1 = zero
    row_n: np.ndarray  # (Ho,k)  source row of window row a
    col_c: np.ndarray  # (Wo,)
    col_n: np.ndarray  # (Wo,k)


def geometry(H, W, R=1, stride=1, padding=0, dilation=1, padding_mode="reflect") -> Geometry:
    """Index tables of the stencil.  Output size as Conv2d computes it
    (nfp.py:42-47; the formula the reference restates at nfp.py:128-129)."""
    k = 2 * R + 1
    if padding_mode not in PADDING_MODES:
        raise ValueError(f"padding_mode {padding_mode!r}")
    if padding_mode == "reflect" and padding > 0 and (padding >= H or padding >= W):
        # ATen reflection_pad2d's own check, reached through Conv2d._conv_forward
        raise RuntimeError(
            "Padding size should be less than the corresponding input dimension, "
            f"but got: padding ({padding}, {padding}) at dimension 3 of input {[H, W]}")
    if padding_mode == "circular" and (padding > H or padding > W):
        raise RuntimeError("Padding value causes wrapping around more than once.")
    Ho = (H + 2 * padding - dilation * (k - 1) - 1) // stride + 1
    Wo = (W + 2 * padding - dilation * (k - 1) - 1) // stride + 1
    if Ho <= 0 or Wo <= 0:
        raise RuntimeError(
            f"Calculated padded input size per channel: ({H + 2 * padding} x {W + 2 * padding}). "
            f"Kernel size: ({dilation * (k - 1) + 1} x {dilation * (k - 1) + 1}). "
            "Kernel size can't be greater than actual input size")
    row_c = np.array([_map_index(i * stride + R * dilation - padding, H, padding_mode)
                      for i in range(Ho)], dtype=np.int64)
    col_c = np.array([_map_index(j * stride + R * dilation - padding, W, padding_mode)
                      for j in range(Wo)], dtype=np.int64)
    row_n = np.array([[_map_index(i * stride + a * dilation - padding, H, padding_mode)
                       for a in range(k)] for i in range(Ho)], dtype=np.int64)
    col_n = np.array([[_map_index(j * stride + b * dilation - padding, W, padding_mode)
                       for b in range(k)] for j in range(Wo)], dtype=np.int64)
    return Geometry(H, W, R, stride, padding, dilation, padding_mode, Ho, Wo,
                    row_c, row_n, col_c, col_n)


def gather_centre_neighbours(x: torch.Tensor, g: Geometry):
    """``(B,C,H,W) -> centre (B,C,1,Ho,Wo), neighbours (B,C,K,Ho,Wo)``.

    Equivalent of ``center_value(x).unsqueeze(2)`` and
    ``reshape_tensor(comp_neighbors(x))`` with pure-neighbour taps
    (nfp.py:152-155, 136-139)."""
    B, C, H, W = x.shape
    assert (H, W) == (g.H, g.W)
    xz = F.pad(x, (0, 1, 0, 1))  # index H / W = the implicit zero of 'zeros' padding
    def fix(a, n):
        t = torch.as_tensor(a)
        return torch.where(t < 0, torch.full_like(t, n), t)
    rc, cc = fix(g.row_c, H), fix(g.col_c, W)
    rn, cn = fix(g.row_n, H), fix(g.col_n, W)
    centre = xz[:, :, rc[:, None], cc[None, :]].unsqueeze(2)
    taps = [xz[:, :, rn[:, a][:, None], cn[:, b][None, :]] for (a, b) in tap_offsets(g.R)]
    return centre, torch.stack(taps, dim=2)


def nfp_forward(x: torch.Tensor, R=1, measure="norm", p=1, stride=1, padding=0,
                dilation=1, padding_mode="reflect", similarity=True, eps=1e-6,
                q_scs=1e-6, difference_taps=None) -> torch.Tensor:
    """Restatement of ``NFPPooling.forward`` (nfp.py:132-134) for every measure.

    ``difference_taps`` reproduces the case-sensitivity quirk of nfp.py:74; by
    default it is derived from ``measure`` as given."""
    if difference_taps is None:
        difference_taps = uses_difference_taps(measure)
    m = canonical_measure(measure)
    g = geometry(x.shape[2], x.shape[3], R, stride, padding, dilation, padding_mode)
    c, n = gather_centre_neighbours(x, g)

    if m == "norm":  # nfp.py:141-148
        v = (c - n) if difference_taps else n
        y = torch.linalg.norm(v, ord=p, dim=1)
        return -y if similarity else y
    if m == "rmse":  # nfp.py:172-179
        v = (c - n) if difference_taps else n
        y = torch.sqrt(torch.mean(v ** 2, dim=1))
        return -y if similarity else y
    if m == "cosine":  # nfp.py:150-159
        y = F.cosine_similarity(c, n, dim=1, eps=eps)
        return y if similarity else 1 - y
    if m == "dot":  # nfp.py:161-170
        y = torch.sum(c * n, dim=1)
        return y if similarity else -y
    if m == "geman":  # nfp.py:181-193
        d = (c - n) ** 2
        y = (d / (d + eps)).mean(dim=1)
        return y if similarity else 1 - y
    if m == "attention":  # nfp.py:195-205
        y = F.softmax(torch.sum(c * n, dim=1), dim=1)
        return y if similarity else -y
    if m == "emd":  # nfp.py:207-216
        y = torch.sum(torch.abs(c - n), dim=1)
        return -y if similarity else y
    if m == "canberra":  # nfp.py:218-227
        y = torch.sum(torch.abs(c - n) / (torch.abs(c) + torch.abs(n) + eps), dim=1)
        return -y if similarity else y
    if m == "hellinger":  # nfp.py:229-241
        ca, na = torch.abs(c) + eps, torch.abs(n) + eps
        y = torch.sqrt(0.5 * torch.sum((torch.sqrt(ca) - torch.sqrt(na)) ** 2, dim=1))
        return -y if similarity else y
    if m == "chisquared1":  # nfp.py:243-252
        y = torch.sum((c - n) ** 2 / (torch.abs(c) + torch.abs(n) + eps), dim=1)
        return -y if similarity else y
    if m == "chisquared2":  # nfp.py:254-263
        y = torch.sum((c - n) ** 2 / (torch.abs(c) + eps), dim=1)
        return -y if similarity else y
    if m == "gfc":  # nfp.py:265-276
        num = torch.sum(c * n, dim=1)
        den = torch.norm(c, dim=1) * torch.norm(n, dim=1) + eps
        y = num / den
        return y if similarity else -y
    if m == "pearson":  # nfp.py:278-293
        cc = c - c.mean(dim=1, keepdim=True)
        nc = n - n.mean(dim=1, keepdim=True)
        num = torch.sum(cc * nc, dim=1)
        den = torch.sqrt(torch.sum(cc ** 2, dim=1) * torch.sum(nc ** 2, dim=1) + eps)
        y = num / den
        return y if similarity else -y
    if m == "jeffrey":  # nfp.py:295-308
        ca, na = torch.abs(c) + eps, torch.abs(n) + eps
        y = torch.sum(ca * torch.log(ca / na) + na * torch.log(na / ca), dim=1)
        return -y if similarity else y
    if m == "squaredchord":  # nfp.py:310-324
        ca, na = torch.abs(c) + eps, torch.abs(n) + eps
        y = torch.sum(torch.square(torch.sqrt(ca) - torch.sqrt(na)), dim=1)
        return -y if similarity else y
    if m == "smith":  # nfp.py:326-342
        ca, na = torch.abs(c), torch.abs(n)
        mins = torch.sum(torch.minimum(ca, na), dim=1)
        y = 1 - mins / (torch.minimum(ca.sum(dim=1), na.sum(dim=1)) + eps)
        return y if similarity else -y
    if m == "scs":  # nfp.py:344-374, including its cross-batch broadcast
        dot = torch.sum(c * n, dim=1)                                   # (B,K,Ho,Wo)
        den = (torch.norm(c, dim=1) + q_scs) * (torch.norm(n, dim=1) + q_scs)  # (B,K,Ho,Wo)
        # reference: (B,K,Ho,Wo) / (B,1,K,Ho,Wo) -> (B,B,K,Ho,Wo): [b, b'] = dot[b'] / den[b]
        t = dot.unsqueeze(0) / den.unsqueeze(1)
        s = torch.sign(t) * (torch.abs(t) ** p)
        s = torch.nan_to_num(s, nan=0.0, posinf=0.0, neginf=0.0)
        if not similarity:
            s = 1 - s
        return s.mean(dim=1)
    raise AssertionError(m)


def nfp_forward_backward(x: torch.Tensor, gy: torch.Tensor, **kw):
    """Forward and the gradient w.r.t. ``x`` for upstream gradient ``gy`` --
    what autograd computes through the reference module."""
    xr = x.detach().clone().requires_grad_(True)
    y = nfp_forward(xr, **kw)
    (gx,) = torch.autograd.grad(y, xr, gy)
    return y.detach(), gx


# --------------------------------------------------------------------------- #
# Closed forms for the cosine measure (what the CUDA kernels implement).
# --------------------------------------------------------------------------- #

def cosine_forward_np(x: np.ndarray, R=1, stride=1, padding=0, dilation=1,
                      padding_mode="reflect", similarity=True, eps=1e-6) -> np.ndarray:
    """fp64 closed form of nfp.py:150-159 with the installed ATen semantics of
    ``cosine_similarity``: each norm is clamped separately at ``eps``."""
    x = np.asarray(x, dtype=np.float64)
    B, C, H, W = x.shape
    g = geometry(H, W, R, stride, padding, dilation, padding_mode)
    taps = tap_offsets(R)
    y = np.zeros((B, len(taps), g.Ho, g.Wo))
    zero = np.zeros((B, C))
    def px(r, c):
        return zero if (r < 0 or c < 0) else x[:, :, r, c]
    for i in range(g.Ho):
        for j in range(g.Wo):
            cv = px(g.row_c[i], g.col_c[j])
            Nc = np.maximum(np.sqrt((cv * cv).sum(1)), eps)
            for t, (a, b) in enumerate(taps):
                nv = px(g.row_n[i, a], g.col_n[j, b])
                Nn = np.maximum(np.sqrt((nv * nv).sum(1)), eps)
                y[:, t, i, j] = (cv * nv).sum(1) / (Nc * Nn)
    return y if similarity else 1 - y


def cosine_backward_np(x: np.ndarray, gy: np.ndarray, R=1, stride=1, padding=0,
                       dilation=1, padding_mode="reflect", similarity=True,
                       eps=1e-6) -> np.ndarray:
    """fp64 closed-form gradient of the cosine measure.

    For one (centre c, neighbour n) pair with ``N = max(||.||, eps)`` and
    ``y = <c,n>/(Nc Nn)``, ATen's backward gives
    ``dy/dc = n/(Nc Nn) - y c/(Nc ||c||)`` (second term 0 when ``c == 0``) and
    symmetrically for n -- the value is clamped, the gradient still carries the
    norm term (probed on torch 2.11; SURVEY.md section 8 row a3)."""
    x = np.asarray(x, dtype=np.float64)
    gy = np.asarray(gy, dtype=np.float64)
    B, C, H, W = x.shape
    g = geometry(H, W, R, stride, padding, dilation, padding_mode)
    taps = tap_offsets(R)
    gx = np.zeros_like(x)
    sign = 1.0 if similarity else -1.0
    for i in range(g.Ho):
        for j in range(g.Wo):
            rc, cc = g.row_c[i], g.col_c[j]
            if rc < 0 or cc < 0:
                continue  # centre is an implicit zero: y == 0 and no gradient path
            cv = x[:, :, rc, cc]
            nc = np.sqrt((cv * cv).sum(1))
            Nc = np.maximum(nc, eps)
            for t, (a, b) in enumerate(taps):
                rn, cn = g.row_n[i, a], g.col_n[j, b]
                if rn < 0 or cn < 0:
                    # neighbour is an implicit zero: y = 0; dy/dc = 0/(..) - 0 = 0
                    continue
                nv = x[:, :, rn, cn]
                nn = np.sqrt((nv * nv).sum(1))
                Nn = np.maximum(nn, eps)
                yv = (cv * nv).sum(1) / (Nc * Nn)
                gg = sign * gy[:, t, i, j]
                w = gg / (Nc * Nn)
                with np.errstate(divide="ignore", invalid="ignore"):
                    dc = np.where(nc > 0, gg * yv / (Nc * nc), 0.0)
                    dn = np.where(nn > 0, gg * yv / (Nn * nn), 0.0)
                gx[:, :, rc, cc] += w[:, None] * nv - dc[:, None] * cv
                gx[:, :, rn, cn] += w[:, None] * cv - dn[:, None] * nv
    return gx


# --------------------------------------------------------------------------- #
# The pooling wrapper (reference models/NFP_Pooling.py:25-36).
# --------------------------------------------------------------------------- #

def nfp_pooling_forward(x: torch.Tensor, proj_weight=None, proj_bias=None, **kw) -> torch.Tensor:
    """``GAP(x) * nfp_proj(GAP(NFP(x)))`` -> (B, C)  (NFP_Pooling.py:27-35).
    ``kw`` defaults follow NFP_Pooling.py:10-16 (R=1, cosine, padding=1)."""
    kw = {"R": 1, "measure": "cosine", "padding": 1, **kw}
    x_avg = x.mean(dim=(2, 3))
    x_nfp = nfp_forward(x, **kw).mean(dim=(2, 3))
    if proj_weight is not None:
        x_nfp = F.linear(x_nfp, proj_weight, proj_bias)
    return x_avg * x_nfp


def algorithmic_bytes_per_map(C, H, W, R, elem_bytes, Ho=None, Wo=None, pooled=False):
    """SURVEY.md section 8(d3): read x (fwd) + write y + read x (bwd) + read gy
    + write gx = 3*C*H*W*e + 2*K*Ho*Wo*e ; pooled mode replaces the maps by
    O(C+K) vectors."""
    K = (2 * R + 1) ** 2 - 1
    Ho = H if Ho is None else Ho
    Wo = W if Wo is None else Wo
    if pooled:
        return 3 * C * H * W * elem_bytes + 2 * (C + K) * elem_bytes
    return 3 * C * H * W * elem_bytes + 2 * K * Ho * Wo * elem_bytes
