"""TEST INFRASTRUCTURE ONLY -- pin the oracle against the reference itself.

Needs a checkout of the original project:

    NFP_REFERENCE_ROOT=/path/to/Neighbour_Feature_Pooling python -m oracle.check_against_reference

For every measure x geometry case it executes the unmodified reference module
(forward and autograd backward, fp64) and the oracle restatement on the same
seeded input and reports the max abs difference.  Exit code 1 on any mismatch.
"""
from __future__ import annotations

import itertools
import sys

import numpy as np
import torch

from . import nfp_oracle as O
from .ref_loader import load_reference

# (C, H, W, R, stride, padding, dilation, padding_mode)
GEOMETRIES = [
    (6, 7, 7, 1, 1, 1, 1, "reflect"),     # the live path: pad = R (NFP_Pooling.py:10-16)
    (5, 6, 9, 2, 1, 2, 1, "reflect"),     # 5x5, non-square
    (4, 5, 5, 1, 1, 0, 1, "reflect"),     # module default padding=0 (nfp.py:16)
    (4, 6, 6, 1, 1, 2, 1, "reflect"),     # pad > R: centre itself lands in the halo
    (4, 8, 7, 1, 2, 1, 1, "reflect"),     # stride 2
    (4, 9, 9, 1, 1, 2, 2, "reflect"),     # dilation 2
    (3, 2, 2, 1, 1, 1, 1, "reflect"),     # EuroSAT-shaped 2x2 map
    (4, 6, 5, 1, 1, 1, 1, "zeros"),
    (4, 6, 5, 2, 1, 2, 1, "replicate"),
    (4, 6, 5, 1, 1, 1, 1, "circular"),
    (4, 7, 7, 1, 2, 3, 2, "zeros"),
]


def run_case(NFPPooling, measure, geom, similarity, p, B=3, seed=0, dtype=torch.float64):
    C, H, W, R, s, pad, d, mode = geom
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, H, W, generator=gen, dtype=dtype)
    if seed % 2:  # post-ReLU style maps with exact zeros
        x = x.relu()
    ref = NFPPooling(C, R=R, measure=measure, p=p, stride=s, padding=pad, dilation=d,
                     padding_mode=mode, similarity=similarity).to(dtype)
    xr = x.clone().requires_grad_(True)
    y_ref = ref(xr)
    g = torch.randn(y_ref.shape, generator=gen, dtype=dtype)
    (gx_ref,) = torch.autograd.grad(y_ref, xr, g)
    y, gx = O.nfp_forward_backward(x, g, R=R, measure=measure, p=p, stride=s, padding=pad,
                                   dilation=d, padding_mode=mode, similarity=similarity)
    ey = (y - y_ref.detach()).abs().max().item()
    fin = torch.isfinite(gx_ref) & torch.isfinite(gx)
    # Degenerate inputs (sqrt'(0) in rmse/hellinger/norm on an all-zero difference, e.g. two
    # zero-padded taps or post-ReLU zeros) give NaN gradients in the reference.  Its conv
    # backward multiplies that NaN by the zero taps of the one-hot kernel, so the NaN spreads
    # over the whole k x k window of real pixels; the gather form only poisons the elements it
    # actually touches (or none, for implicit zeros).  The NaN footprint is therefore not part
    # of the contract.  Require: wherever the reference gradient is finite the oracle is finite
    # and agrees.
    same_nan = bool((torch.isfinite(gx) | ~torch.isfinite(gx_ref)).all())
    eg = (gx - gx_ref)[fin].abs().max().item() if fin.any() else 0.0
    scale = max(1.0, y_ref.abs().max().item())
    gscale = max(1.0, gx_ref[fin].abs().max().item()) if fin.any() else 1.0
    return ey / scale, eg / gscale, same_nan


def main():
    NFPPooling, nfp_pooling = load_reference()
    worst = 0.0
    bad = 0
    n = 0
    spellings = list(O.MEASURES) + ["sharpened_cosine", "Norm", "RMSE", "Cosine"]
    for measure, geom, sim in itertools.product(spellings, GEOMETRIES, (True, False)):
        for p in ((1, 2, 3.0) if measure.lower() in ("norm", "scs", "sharpened_cosine") else (1,)):
            for seed in (0, 1):
                ey, eg, same_nan = run_case(NFPPooling, measure, geom, sim, p, seed=seed)
                n += 1
                worst = max(worst, ey, eg)
                if ey > 1e-12 or eg > 1e-10 or not same_nan:
                    bad += 1
                    print(f"MISMATCH measure={measure} geom={geom} sim={sim} p={p} seed={seed} "
                          f"ey={ey:.3e} eg={eg:.3e} same_nan={same_nan}")
    # closed-form cosine (numpy fp64) vs the reference, including degenerate vectors
    for geom in GEOMETRIES:
        C, H, W, R, s, pad, d, mode = geom
        gen = torch.Generator().manual_seed(7)
        x = torch.randn(2, C, H, W, generator=gen, dtype=torch.float64)
        x[0, :, 0, 0] = 0.0                 # exact zero vector
        x[1, :, H // 2, W // 2] *= 1e-9     # ||x|| < eps
        ref = NFPPooling(C, R=R, measure="cosine", stride=s, padding=pad, dilation=d,
                         padding_mode=mode).double()
        xr = x.clone().requires_grad_(True)
        y_ref = ref(xr)
        g = torch.randn(y_ref.shape, generator=gen, dtype=torch.float64)
        (gx_ref,) = torch.autograd.grad(y_ref, xr, g)
        kw = dict(R=R, stride=s, padding=pad, dilation=d, padding_mode=mode)
        y = O.cosine_forward_np(x.numpy(), **kw)
        gx = O.cosine_backward_np(x.numpy(), g.numpy(), **kw)
        ey = np.abs(y - y_ref.detach().numpy()).max()
        eg = np.abs(gx - gx_ref.numpy()).max() / max(1.0, np.abs(gx_ref.numpy()).max())
        n += 1
        worst = max(worst, ey, eg)
        if ey > 1e-12 or eg > 1e-12:
            bad += 1
            print(f"MISMATCH closed-form cosine geom={geom} ey={ey:.3e} eg={eg:.3e}")
    # the pooling wrapper (NFP_Pooling.py:25-36)
    Params = {"num_ftrs": {"m": 6}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 3}}
    pool = nfp_pooling(Params=Params).double()
    x = torch.randn(3, 6, 7, 7, dtype=torch.float64, generator=torch.Generator().manual_seed(3))
    out_ref = pool(x)
    out = O.nfp_pooling_forward(x, pool.nfp_proj.weight, pool.nfp_proj.bias)
    e = (out - out_ref).abs().max().item()
    n += 1
    worst = max(worst, e)
    if e > 1e-12:
        bad += 1
        print(f"MISMATCH nfp_pooling wrapper e={e:.3e}")
    print(f"{n} cases, {bad} mismatches, worst scaled error {worst:.3e}")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
