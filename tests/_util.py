"""Shared helpers of the test-suite (golden fixtures, error norms)."""
import json
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


def worst(errs, k=4):
    """The k largest entries of a grad_errs() table, for assertion messages."""
    return sorted(errs.items(), key=lambda kv: -kv[1])[:k]
