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
