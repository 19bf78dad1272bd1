"""CPU: the fp64 closed forms of the cosine operator's second order (tests/second_order_ref.py) against ATen.

The double backward (``torch.autograd.grad(..., create_graph=True)`` differentiated again, both halves: to x and to
gy) and forward-mode AD (``torch.autograd.forward_ad``) are taken through ATen on two restatements of the reference:
the gather-form oracle (``oracle/nfp_oracle.py``, which calls ``F.cosine_similarity``) and the conv form
(``oracle/nfp_convform.py``, the reference's exact op sequence).  Inputs include all-zero pixels, pixels below eps and
pixels just above it.  Pass: <= 1e-12 relative on the finite elements of each image and pixel-norm region, and the same
non-finite mask (the conv form: a larger one, see test_closed_forms_match_aten).
"""
import numpy as np
import pytest
import torch
import torch.autograd.forward_ad as fwAD

from oracle import nfp_oracle as O
from oracle.nfp_convform import ConvFormCosineNFP

import second_order_ref as S
from _util import grad_errs, image_groups, rel_err

TOL = 1e-12
EPS = 1e-6

# (B, C, H, W, R, stride, padding, dilation, padding_mode, similarity)
CASES = [
    (2, 5, 6, 7, 1, 1, 1, 1, "reflect", True),
    (2, 4, 7, 6, 2, 1, 2, 1, "reflect", True),
    (2, 3, 8, 8, 3, 1, 3, 1, "replicate", True),
    (2, 5, 9, 8, 1, 2, 1, 1, "zeros", True),
    (2, 4, 9, 9, 1, 1, 2, 2, "circular", True),
    (2, 5, 7, 7, 1, 1, 2, 1, "zeros", False),       # pad != R: implicit-zero centres
    (2, 5, 7, 8, 1, 1, 0, 1, "reflect", True),      # no padding
    (2, 4, 9, 10, 2, 2, 1, 2, "replicate", False),
    (2, 3, 7, 7, 1, 1, 1, 1, "circular", False),
]


def case_id(c):
    B, C, H, W, R, s, p, d, mode, sim = c
    return f"{B}x{C}x{H}x{W}-R{R}-s{s}-p{p}-d{d}-{mode}-sim{int(sim)}"


def degenerate_input(B, C, H, W, seed=0):
    """randn with an all-zero pixel, a pixel of norm ~1e-8 (below eps) and one at 1.5 eps in every image."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, H, W, generator=g, dtype=torch.float64)
    for b in range(B):
        x[b, :, (1 + b) % H, 2 % W] = 0.0
        x[b, :, 3 % H, (1 + b) % W] *= 1e-8 / x[b, :, 3 % H, (1 + b) % W].norm()
        x[b, :, H - 1, W - 2] *= 1.5 * EPS / x[b, :, H - 1, W - 2].norm()
    return x


def kwargs(c):
    B, C, H, W, R, s, p, d, mode, sim = c
    return dict(R=R, stride=s, padding=p, dilation=d, padding_mode=mode, similarity=sim, eps=EPS)


def _aten_gather(c):
    kw = kwargs(c)
    return lambda x: O.nfp_forward(x, measure="cosine", **kw)


def _aten_conv(c):
    B, C, H, W, R, s, p, d, mode, sim = c
    layer = ConvFormCosineNFP(C, R=R, stride=s, padding=p, dilation=d, padding_mode=mode, similarity=sim,
                              eps=EPS).double()
    return layer


def _same_mask(got, want):
    return torch.equal(torch.isfinite(torch.as_tensor(np.asarray(got))), torch.isfinite(torch.as_tensor(np.asarray(want))))


def _aten_second_order(f, x, gy, v):
    xr = x.clone().requires_grad_(True)
    gyr = gy.clone().requires_grad_(True)
    (gx,) = torch.autograd.grad(f(xr), xr, gyr, create_graph=True)
    gx2, ggy = torch.autograd.grad(gx, (xr, gyr), v)
    with fwAD.dual_level():
        jf = fwAD.unpack_dual(f(fwAD.make_dual(x, v))).tangent
    return gx2, ggy, jf


@pytest.mark.parametrize("form", ["gather", "conv"])
@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_closed_forms_match_aten(c, form):
    B, C, H, W = c[:4]
    x = degenerate_input(B, C, H, W)
    f = _aten_gather(c) if form == "gather" else _aten_conv(c)
    g = torch.Generator().manual_seed(1)
    gy = torch.randn(f(x).shape, generator=g, dtype=torch.float64)
    v = torch.randn(x.shape, generator=g, dtype=torch.float64)
    gx2, ggy, jf = _aten_second_order(f, x, gy, v)
    kw = kwargs(c)
    want_gx2 = S.cosine_backward_backward_np(x.numpy(), gy.numpy(), v.numpy(), **kw)
    want_rev = S.cosine_jvp_np(x.numpy(), v.numpy(), S.RULE_REVERSE, **kw)
    want_fwd = S.cosine_jvp_np(x.numpy(), v.numpy(), S.RULE_FORWARD_AD, **kw)
    assert _same_mask(ggy, want_rev) and _same_mask(jf, want_fwd)
    if form == "gather":
        assert _same_mask(gx2, want_gx2)
    else:
        # the conv form's one-hot conv backward multiplies the zero pixel's NaN by the kernel's zeros (0 * NaN = NaN):
        # its NaN reaches every pixel whose window holds an all-zero pixel.  It keeps the closed form's NaN, and
        # elsewhere its finite values are the closed form's
        want_nan = ~np.isfinite(want_gx2)
        got_nan = ~torch.isfinite(gx2).numpy()
        assert (got_nan | ~want_nan).all()
        want_gx2 = np.where(got_nan, np.nan, want_gx2)
    e2 = grad_errs(gx2, want_gx2, x.numpy(), EPS)
    assert max(e2.values()) <= TOL, sorted(e2.items(), key=lambda kv: -kv[1])[:4]
    for got, want in ((ggy, want_rev), (jf, want_fwd)):
        for b, m in image_groups(got.shape).items():
            wb = torch.as_tensor(want)[m.expand_as(got)]
            assert rel_err(got[m.expand_as(got)], wb) <= TOL, b


def test_non_finite_footprint_is_the_zero_pixels():
    """The double backward is NaN in exactly the channels of all-zero pixels and reaches ~1e12 below eps."""
    c = CASES[0]
    B, C, H, W = c[:4]
    x = degenerate_input(B, C, H, W)
    g = torch.Generator().manual_seed(2)
    gy = torch.randn(B, 8, H, W, generator=g, dtype=torch.float64)
    v = torch.randn(x.shape, generator=g, dtype=torch.float64)
    gx2 = torch.as_tensor(S.cosine_backward_backward_np(x.numpy(), gy.numpy(), v.numpy(), **kwargs(c)))
    zero_px = (x == 0).all(1, keepdim=True).expand_as(x)
    assert torch.equal(~torch.isfinite(gx2), zero_px)
    small = (x.norm(dim=1, keepdim=True) < EPS).expand_as(x) & ~zero_px
    assert gx2[small].abs().max() > 1e9


def test_rules_differ_only_below_eps():
    """Forward AD and the reverse-mode JVP agree wherever no pair touches a pixel whose norm is below eps."""
    c = CASES[0]
    B, C, H, W = c[:4]
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, C, H, W, generator=g, dtype=torch.float64)
    v = torch.randn(x.shape, generator=g, dtype=torch.float64)
    a = S.cosine_jvp_np(x.numpy(), v.numpy(), S.RULE_FORWARD_AD, **kwargs(c))
    b = S.cosine_jvp_np(x.numpy(), v.numpy(), S.RULE_REVERSE, **kwargs(c))
    assert np.array_equal(a, b)
    x = degenerate_input(B, C, H, W)
    a = S.cosine_jvp_np(x.numpy(), v.numpy(), S.RULE_FORWARD_AD, **kwargs(c))
    b = S.cosine_jvp_np(x.numpy(), v.numpy(), S.RULE_REVERSE, **kwargs(c))
    assert np.abs(a - b).max() > 1e3
