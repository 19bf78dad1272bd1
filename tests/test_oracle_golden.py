"""CPU: the oracle restatement against the golden vectors generated from the unmodified reference
(oracle/make_golden.py), and -- where the reference checkout exists -- against the reference itself."""
import numpy as np
import pytest
import torch

from oracle import nfp_oracle as O
from oracle.ref_loader import reference_available

from _util import case_id, case_kwargs, load_measure_cases, load_multi_radius_cases, load_wrapper_cases, rel_err

INDEX, ARR = load_measure_cases()


@pytest.mark.parametrize("c", INDEX, ids=case_id)
def test_oracle_matches_reference_golden(c):
    x = torch.from_numpy(ARR[c["key"] + "_x"]).double()
    g = torch.from_numpy(ARR[c["key"] + "_g"]).double()
    y, gx = O.nfp_forward_backward(x, g, **case_kwargs(c))
    assert rel_err(y, ARR[c["key"] + "_y_f64"]) < 1e-12
    # NaN footprint of degenerate gradients is not part of the contract (see oracle/check_against_reference.py)
    assert rel_err(gx, ARR[c["key"] + "_gx_f64"]) < 1e-10


@pytest.mark.parametrize("c", [c for c in INDEX if c["measure"] == "cosine"], ids=case_id)
def test_closed_form_cosine_matches_golden(c):
    kw = case_kwargs(c)
    kw.pop("measure"); kw.pop("p")
    y = O.cosine_forward_np(ARR[c["key"] + "_x"], **kw)
    gx = O.cosine_backward_np(ARR[c["key"] + "_x"], ARR[c["key"] + "_g"], **kw)
    assert rel_err(y, ARR[c["key"] + "_y_f64"]) < 1e-12
    assert rel_err(gx, ARR[c["key"] + "_gx_f64"]) < 1e-12
    # the reference's own fp32 rounding noise is far below the 1e-5 parity bar of the CUDA path
    assert rel_err(ARR[c["key"] + "_y_f32"], ARR[c["key"] + "_y_f64"]) < 2e-6
    assert rel_err(ARR[c["key"] + "_gx_f32"], ARR[c["key"] + "_gx_f64"]) < 2e-6


def test_multi_radius_golden_and_nesting():
    """The reference's multi-radius composition (two NFPPooling layers, R = 1, 2, padding = R, torch.cat -- as
    models/nfp_heads.py:86-93,111-112 builds it): the oracle reproduces it layer by layer, and the radius-1 map is exactly the
    inner taps of the radius-2 map (what lets the CUDA path produce both from one pass, include/nfp_b200.h inner_R)."""
    index, arr = load_multi_radius_cases()
    inner = [6, 7, 8, 11, 12, 15, 16, 17]   # taps of the 5x5 window (centre removed) with |dy|, |dx| <= 1, row-major
    for c in index:
        x = torch.from_numpy(arr[c["key"] + "_x"]).double()
        g = torch.from_numpy(arr[c["key"] + "_g"]).double()
        ys, gxs = [], []
        for R, sl in ((1, slice(0, 8)), (2, slice(8, 32))):
            y, gx = O.nfp_forward_backward(x, g[:, sl].contiguous(), R=R, measure="cosine", padding=R,
                                           padding_mode=c["padding_mode"], similarity=c["similarity"])
            ys.append(torch.as_tensor(np.asarray(y)))
            gxs.append(torch.as_tensor(np.asarray(gx)))
        assert rel_err(torch.cat(ys, 1), arr[c["key"] + "_y"]) < 1e-12
        assert rel_err(gxs[0] + gxs[1], arr[c["key"] + "_gx"]) < 1e-10
        y_ref = torch.from_numpy(arr[c["key"] + "_y"])
        # radius-1 map = inner taps of the radius-2 map (the reference's two convs sum in different orders: 1e-16 apart)
        assert rel_err(y_ref[:, :8], y_ref[:, 8:][:, inner]) < 1e-13


def test_wrapper_golden():
    index, arr = load_wrapper_cases()
    for c in index:
        k = c["key"]
        x = torch.from_numpy(arr[k + "_x"]).double().requires_grad_(True)
        w = torch.from_numpy(arr[k + "_w"]).double().requires_grad_(True)
        b = torch.from_numpy(arr[k + "_b"]).double().requires_grad_(True)
        out = O.nfp_pooling_forward(x, w, b)
        gx, gw, gb = torch.autograd.grad(out, (x, w, b), torch.from_numpy(arr[k + "_g"]).double())
        assert rel_err(out.detach(), arr[k + "_out"]) < 1e-12
        assert rel_err(gx, arr[k + "_gx"]) < 1e-12
        assert rel_err(gw, arr[k + "_gw"]) < 1e-12
        assert rel_err(gb, arr[k + "_gb"]) < 1e-12


def test_tap_order_and_geometry():
    assert O.tap_offsets(1) == [(0, 0), (0, 1), (0, 2), (1, 0), (1, 2), (2, 0), (2, 1), (2, 2)]
    g = O.geometry(7, 7, R=1, padding=1)
    assert (g.Ho, g.Wo) == (7, 7)
    assert list(g.row_n[0]) == [1, 0, 1] and list(g.row_n[6]) == [5, 6, 5]   # reflect, edge not repeated
    with pytest.raises(RuntimeError, match="Padding size should be less"):
        O.geometry(2, 2, R=1, padding=2)
    with pytest.raises(RuntimeError, match="Kernel size can't be greater"):
        O.geometry(2, 2, R=1, padding=0)
    with pytest.raises(RuntimeError, match="not implemented"):
        O.canonical_measure("mahalanobis")


def test_algorithmic_bytes_table():
    # SURVEY.md 8(d3) / BASELINE.md section 3
    assert O.algorithmic_bytes_per_map(512, 7, 7, 1, 4) == 304192
    assert O.algorithmic_bytes_per_map(256, 14, 14, 1, 4) == 614656
    assert O.algorithmic_bytes_per_map(512, 7, 7, 2, 4) == 310464
    assert O.algorithmic_bytes_per_map(256, 14, 14, 2, 2) == 319872


@pytest.mark.skipif(not reference_available(), reason="needs the original project: NFP_REFERENCE_ROOT or a copy staged under oracle/_ref")
def test_oracle_against_live_reference_subset():
    from oracle import check_against_reference as chk
    from oracle.ref_loader import load_reference
    NFPPooling, _ = load_reference()
    for measure in ("cosine", "norm", "Norm", "pearson", "scs", "attention", "smith"):
        for geom in chk.GEOMETRIES[:7]:
            ey, eg, same_nan = chk.run_case(NFPPooling, measure, geom, True, 1, seed=0)
            assert ey < 1e-12 and eg < 1e-10 and same_nan, (measure, geom, ey, eg)


def test_conv_form_port_equals_gather_form():
    """bench.py's CPU baseline (the reference's operator sequence, oracle/nfp_convform.py) computes the
    same function as the gather-form oracle."""
    from oracle.nfp_convform import ConvFormCosineNFP, forward_backward
    for (C, H, W, R, s, pad, d, mode) in [(6, 7, 7, 1, 1, 1, 1, "reflect"), (5, 6, 9, 2, 1, 2, 1, "reflect"),
                                          (4, 8, 7, 1, 2, 1, 1, "zeros"), (4, 9, 9, 1, 1, 2, 2, "replicate")]:
        gen = torch.Generator().manual_seed(C * H)
        x = torch.randn(3, C, H, W, generator=gen, dtype=torch.float64)
        kw = dict(R=R, stride=s, padding=pad, dilation=d, padding_mode=mode)
        layer = ConvFormCosineNFP(C, **kw).double()
        y_ref = O.nfp_forward(x, measure="cosine", **kw)
        g = torch.randn(y_ref.shape, generator=gen, dtype=torch.float64)
        y_ref, gx_ref = O.nfp_forward_backward(x, g, measure="cosine", **kw)
        y, gx = forward_backward(layer, x, g)
        assert rel_err(y, y_ref) < 1e-12 and rel_err(gx, gx_ref) < 1e-12
