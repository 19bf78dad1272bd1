"""fp64 closed forms of the cosine NFP operator's second-order derivatives (test reference; never imported by the package).

Per (centre a, neighbour b) pair, with ``n = ||.||``, ``N = max(n, eps)``, ``P = N_a N_b``, ``y = a.b / P`` and a
direction ``v`` on the input (``v_a`` at the centre pixel, ``v_b`` at the neighbour pixel):

* JVP:  ``y' = (v_a.b + a.v_b) / P - y (t_a a.v_a + t_b b.v_b)``.  Reverse mode (what ATen's backward differentiates)
  uses ``t = 1 / (N n)``, 0 at ``n = 0``: each ``N`` takes the clamped value but differentiates as ``n``.  Forward AD
  (``torch.autograd.forward_ad``) gives a norm clamped at eps a zero tangent: ``t = 1 / (N n)`` where ``n >= eps``, else 0.
  The reverse-rule JVP is also the part of the double backward that flows to ``gy``.
* backward of the backward: ``gx2 = d<v, gx(x, gy)>/dx`` with ``G = +-gy`` (``-`` for ``similarity=False``) is, per pair,
      centre    += G (k_aa a + k_ab b + k_ava v_a + k_avb v_b)
      neighbour += G (k_bb b + k_ab a + k_avb v_a... )   (see pair_coefs)
  with ``S = t_a a.v_a + t_b b.v_b``, ``u = t (1/N + 1/n) / n`` (the derivative of ``t``: ``dt/dx = -u x``):
      k_aa = -t_a p / P + y t_a S + y u_a a.v_a      k_bb = -t_b p / P + y t_b S + y u_b b.v_b
      k_ab = -S / P   (on b at the centre, on a at the neighbour)
      k_ava = -y t_a  (on v_a at the centre)         k_bvb = -y t_b  (on v_b at the neighbour)
      k_v = 1 / P     (on v_b at the centre, on v_a at the neighbour)
  ``p = v_a.b + a.v_b``.  At an all-zero pixel ``u (a.v_a)`` is inf * 0: NaN in every channel of that pixel, which is
  what ATen's norm double backward gives there.
"""
from __future__ import annotations

import numpy as np

from oracle.nfp_oracle import geometry, tap_offsets

RULE_FORWARD_AD, RULE_REVERSE = 0, 1


def _pairs(g, R):
    """(i, j, t, centre (r, c), neighbour (r, c)) of every output element; -1 = an implicit zero."""
    for i in range(g.Ho):
        for j in range(g.Wo):
            for t, (a, b) in enumerate(tap_offsets(R)):
                yield i, j, t, (g.row_c[i], g.col_c[j]), (g.row_n[i, a], g.col_n[j, b])


def _px(x, rc):
    r, c = rc
    return np.zeros(x.shape[:2]) if (r < 0 or c < 0) else x[:, :, r, c]


def _t(n, N, rule, eps):
    with np.errstate(divide="ignore", invalid="ignore"):
        t = 1.0 / (N * n)
    keep = (n >= eps) if rule == RULE_FORWARD_AD else (n > 0)
    return np.where(keep, t, 0.0)


def _dots(x, v, cp, npx):
    a, b, va, vb = _px(x, cp), _px(x, npx), _px(v, cp), _px(v, npx)
    return a, b, va, vb, (a * a).sum(1), (b * b).sum(1), (a * b).sum(1), (a * va).sum(1), (b * vb).sum(1), \
        (va * b).sum(1) + (a * vb).sum(1)


def cosine_jvp_np(x, v, rule, R=1, stride=1, padding=0, dilation=1, padding_mode="reflect", similarity=True,
                  eps=1e-6) -> np.ndarray:
    """fp64 ``y'`` (B, K, H', W') of the cosine map at ``x`` in direction ``v`` by the given rule."""
    x, v = np.asarray(x, np.float64), np.asarray(v, np.float64)
    B, C, H, W = x.shape
    g = geometry(H, W, R, stride, padding, dilation, padding_mode)
    out = np.zeros((B, len(tap_offsets(R)), g.Ho, g.Wo))
    for i, j, t, cp, npx in _pairs(g, R):
        a, b, va, vb, aa, bb, ab, qa, qb, p = _dots(x, v, cp, npx)
        na, nb = np.sqrt(aa), np.sqrt(bb)
        Na, Nb = np.maximum(na, eps), np.maximum(nb, eps)
        P = Na * Nb
        y = ab / P
        out[:, t, i, j] = p / P - y * (_t(na, Na, rule, eps) * qa + _t(nb, Nb, rule, eps) * qb)
    return out if similarity else -out


def pair_coefs(aa, bb, ab, qa, qb, p, eps):
    """(k_aa, k_bb, k_ab, k_ava, k_bvb, k_v) of one pair (arrays over the batch), without the factor G."""
    na, nb = np.sqrt(aa), np.sqrt(bb)
    Na, Nb = np.maximum(na, eps), np.maximum(nb, eps)
    P = Na * Nb
    y = ab / P
    ta, tb = _t(na, Na, RULE_REVERSE, eps), _t(nb, Nb, RULE_REVERSE, eps)
    S = ta * qa + tb * qb
    with np.errstate(divide="ignore", invalid="ignore"):
        # u x.v = t (1/N + 1/n) (x.v / n): x.v / n is 0/0 = NaN at an all-zero pixel
        wa = ta * (1.0 / Na + 1.0 / na) * (qa / na)
        wb = tb * (1.0 / Nb + 1.0 / nb) * (qb / nb)
        wa = np.where(na > 0, wa, np.nan)
        wb = np.where(nb > 0, wb, np.nan)
    k_aa = -ta * p / P + y * ta * S + y * wa
    k_bb = -tb * p / P + y * tb * S + y * wb
    return k_aa, k_bb, -S / P, -y * ta, -y * tb, 1.0 / P


def cosine_backward_backward_np(x, gy, v, R=1, stride=1, padding=0, dilation=1, padding_mode="reflect",
                                similarity=True, eps=1e-6) -> np.ndarray:
    """fp64 ``gx2 = d<v, gx(x, gy)>/dx`` (B, C, H, W), gx the cosine map's input gradient (cosine_backward_np)."""
    x, gy, v = np.asarray(x, np.float64), np.asarray(gy, np.float64), np.asarray(v, np.float64)
    B, C, H, W = x.shape
    g = geometry(H, W, R, stride, padding, dilation, padding_mode)
    sign = 1.0 if similarity else -1.0
    out = np.zeros_like(x)
    for i, j, t, cp, npx in _pairs(g, R):
        a, b, va, vb, aa, bb, ab, qa, qb, p = _dots(x, v, cp, npx)
        k_aa, k_bb, k_ab, k_ava, k_bvb, k_v = pair_coefs(aa, bb, ab, qa, qb, p, eps)
        G = (sign * gy[:, t, i, j])[:, None]
        if cp[0] >= 0 and cp[1] >= 0:
            out[:, :, cp[0], cp[1]] += G * (k_aa[:, None] * a + k_ab[:, None] * b + k_ava[:, None] * va
                                            + k_v[:, None] * vb)
        if npx[0] >= 0 and npx[1] >= 0:
            out[:, :, npx[0], npx[1]] += G * (k_bb[:, None] * b + k_ab[:, None] * a + k_bvb[:, None] * vb
                                              + k_v[:, None] * va)
    return out
