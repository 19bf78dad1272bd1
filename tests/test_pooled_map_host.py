"""CPU: the pooled-map ops of the C ABI (GAP(NFP(x)) alone, NFPB200_OP_POOLED_MAP_*) -- path, workspace and launch-count
queries, no compute -- and fuse_pooled_nfp on the CPU (pickle / deepcopy, state_dict, refusals, shape probes)."""
import copy
import ctypes
import io
import math
import os
import pickle

import pytest
import torch
import torch.nn.functional as F

import neighbour_feature_pooling_b200 as nfpb
from neighbour_feature_pooling_b200 import EnhancedNFPPooling, NFPPooling, _capi, modules

FWD, BWD = _capi.OP_POOLED_MAP_FORWARD, _capi.OP_POOLED_MAP_BACKWARD
MAPS = [(16, 112, 112), (24, 56, 56), (40, 28, 28), (112, 14, 14), (960, 7, 7)]   # the multi-stage head's maps


def _desc(**kw):
    base = dict(dtype=_capi.F32, B=64, C=8, H=7, W=7, R=1, stride=1, padding=1, dilation=1,
                padding_mode="reflect", measure="cosine", similarity=True, difference_taps=False,
                eps=1e-6, p=1, q_scs=1e-6, path="auto")
    layout = kw.pop("layout", _capi.LAYOUT_NCHW)
    inner = kw.pop("inner_R", 0)
    base.update(kw)
    d = _capi.make_desc(**base)
    d.layout, d.inner_R = layout, inner
    return d


def _rc(d, op):
    n = ctypes.c_size_t()
    return _capi.load().nfpb200_workspace_bytes(ctypes.byref(d), op, ctypes.byref(n))


def _partials_floor(d):
    """B * n_bands * K * 4 bytes: the band partials.  A band has at most round_up(cap, g) rows, cap = NFPB200_PLANAR_TH
    (default 8) and g the row granule that keeps each bulk copy 16-byte aligned (fused_plan), so
    n_bands >= ceil(H / round_up(cap, g))."""
    K = (2 * d.R + 1) ** 2 - 1
    g = 16 // math.gcd(16, d.W * (2 if d.dtype == _capi.BF16 else 4))
    th_max = max(-(-int(os.environ.get("NFPB200_PLANAR_TH", "8")) // g) * g, g)
    return d.B * -(-d.H // th_max) * K * 4


@pytest.mark.parametrize("dtype", [_capi.F32, _capi.BF16])
@pytest.mark.parametrize("chw", MAPS[:3], ids=lambda s: "x".join(map(str, s)))
def test_band_shapes(chw, dtype):
    C, H, W = chw
    d = _desc(C=C, H=H, W=W, dtype=dtype)
    assert _capi.describe_path(d, FWD) == "planar/band" and _capi.describe_path(d, BWD) == "planar/band"
    assert _capi.launch_count(d, FWD) == 2 and _capi.launch_count(d, BWD) == 1
    assert _capi.workspace_bytes(d, FWD) >= _partials_floor(d)
    assert _capi.workspace_bytes(d, BWD) == 0
    # the existing pooled head ops keep their dispatch
    assert _capi.describe_path(d, _capi.OP_POOL_FORWARD) == "generic/pairs"
    assert _capi.describe_path(d, _capi.OP_POOL_BACKWARD) == "generic/pairs"


def test_ring_and_token_shapes():
    for (C, H, W), name in ((MAPS[3], "fused/stream_14x14_r1"), (MAPS[4], "fused/stream_7x7_r1")):
        d = _desc(C=C, H=H, W=W)
        for op in (FWD, BWD):
            assert _capi.describe_path(d, op) == name
            assert _capi.workspace_bytes(d, op) >= 64 * C * 4   # GAP(x) out / zero g_gap_x in
        assert _capi.launch_count(d, FWD) == 1 and _capi.launch_count(d, BWD) == 2   # + the memset
        assert _capi.describe_path(d, _capi.OP_POOL_FORWARD) == name
    tok = _desc(C=960, dtype=_capi.BF16, layout=_capi.LAYOUT_NHWC)
    assert _capi.describe_path(tok, FWD) == "fused/token_7x7_r1" == _capi.describe_path(tok, BWD)
    assert _capi.workspace_bytes(tok, BWD) >= 64 * 960 * 4
    assert _capi.launch_count(tok, FWD) == 1 and _capi.launch_count(tok, BWD) == 2


def test_generic_fallbacks():
    for d in (_desc(B=3, C=20, H=9, W=6),                 # unaligned planes (the map takes planar/table)
              _desc(C=512, H=56, W=56),                   # too wide for one band slab
              _desc(C=16, H=112, W=112, path="generic"),
              _desc(C=16, H=28, W=28, measure="dot"),
              _desc(C=16, H=28, W=28, stride=2),
              _desc(C=16, H=28, W=28, padding_mode="circular")):
        for op in (FWD, BWD):
            assert _capi.describe_path(d, op) == "generic/pairs", d
        assert _capi.launch_count(d, FWD) == _capi.launch_count(d, _capi.OP_POOL_FORWARD) - 1   # no GAP(x) pass
        assert _capi.launch_count(d, BWD) == _capi.launch_count(d, _capi.OP_POOL_BACKWARD)
    assert _capi.describe_path(_desc(B=3, C=20, H=9, W=6), _capi.OP_BACKWARD) == "planar/table"


def test_refusals():
    assert _rc(_desc(C=16, H=112, W=112, path="fused"), FWD) == -5
    assert _rc(_desc(C=16, H=112, W=112, path="fused"), BWD) == -5
    inner = _desc(C=16, H=28, W=28, R=2, padding=2, inner_R=1)
    assert _capi.describe_path(inner, _capi.OP_FORWARD) == "planar/band"   # the map mode carries it
    assert _rc(inner, FWD) == -5 and _rc(inner, BWD) == -5
    inner7 = _desc(C=64, R=2, padding=2, inner_R=1)
    assert _rc(inner7, FWD) == -5
    for op in (6, -1):
        assert _rc(_desc(), op) == -1
        buf = ctypes.create_string_buffer(64)
        assert _capi.load().nfpb200_describe_path(ctypes.byref(_desc()), op, buf, 64) == -1
        n = ctypes.c_int32()
        assert _capi.load().nfpb200_launch_count(ctypes.byref(_desc()), op, ctypes.byref(n)) == -1
    # null pointers are refused before anything touches the device
    lib = _capi.load()
    assert lib.nfpb200_pooled_map_forward(ctypes.byref(_desc()), None, None, None, 0, None) == -1
    assert lib.nfpb200_pooled_map_backward(ctypes.byref(_desc()), None, None, None, None, 0, None) == -1
    assert lib.nfpb200_pooled_map_forward(ctypes.byref(_desc()), 0x1004, 0x2000, None, 0, None) == -7


def test_existing_pool_ops_unchanged():
    """The pooled-map ops add paths; the answers of the four existing ops stay what they were."""
    for (C, H, W) in MAPS:
        for dt in (_capi.F32, _capi.BF16):
            d = _desc(C=C, H=H, W=W, dtype=dt)
            want = "generic/pairs" if H > 14 else f"fused/stream_{H}x{W}_r1"
            assert _capi.describe_path(d, _capi.OP_POOL_FORWARD) == want
            assert _capi.describe_path(d, _capi.OP_POOL_BACKWARD) == want
            assert _capi.describe_path(d, _capi.OP_FORWARD) == ("planar/band" if H > 14 else want)
    assert _capi.describe_path(_desc(C=16, H=112, W=112), _capi.OP_POOL_FORWARD) == "generic/pairs"
    assert _capi.launch_count(_desc(C=16, H=112, W=112), _capi.OP_POOL_FORWARD) == 3


# ---- fuse_pooled_nfp on the CPU ---------------------------------------------------------------------------------------

def _layer(cls=NFPPooling, **kw):
    return cls(16, R=1, measure=kw.pop("measure", "cosine"), padding=1, **kw)


def test_fuse_keeps_state_dict_and_tree():
    layer = _layer()
    keys = list(layer.state_dict().keys())
    children = [n for n, _ in layer.named_modules()]
    assert nfpb.fuse_pooled_nfp(layer)
    assert isinstance(layer.__dict__["forward"], modules._PooledForward)
    assert list(layer.state_dict().keys()) == keys
    assert [n for n, _ in layer.named_modules()] == children
    assert not nfpb.fuse_pooled_nfp(layer)   # already fused: a re-bound forward is not stock
    nfpb.unfuse_pooled_nfp(layer)
    assert "forward" not in layer.__dict__ and modules._stock(layer)


def test_fuse_round_trips_pickle_and_deepcopy():
    layer = _layer(EnhancedNFPPooling)
    assert nfpb.fuse_pooled_nfp(layer)
    for clone in (pickle.loads(pickle.dumps(layer)), copy.deepcopy(layer)):
        fwd = clone.__dict__["forward"]
        assert isinstance(fwd, modules._PooledForward) and fwd.layer is clone and clone is not layer
        assert clone.state_dict().keys() == layer.state_dict().keys()
    buf = io.BytesIO()
    torch.save(layer, buf)
    buf.seek(0)
    loaded = torch.load(buf, weights_only=False)
    assert loaded.__dict__["forward"].layer is loaded


def test_fuse_refuses_non_stock_layers():
    class Sub(NFPPooling):
        pass

    hooked = _layer()
    hooked.register_forward_hook(lambda m, i, o: None)
    rebound = _layer()
    rebound.similarity_measure = lambda x: x
    for layer in (_layer(Sub), hooked, rebound, _layer(measure="norm"), _layer(measure="dot"), torch.nn.Identity()):
        before = dict(layer.__dict__)
        assert not nfpb.fuse_pooled_nfp(layer)
        assert "forward" not in layer.__dict__ or layer.__dict__["forward"] is before.get("forward")


def test_fused_cpu_probe_is_the_stock_answer():
    layer = _layer()
    assert nfpb.fuse_pooled_nfp(layer)
    x = torch.randn(2, 16, 9, 11)
    with torch.no_grad():
        y = layer(x)
    assert y.shape == (2, 8, 9, 11) and not y.any()   # the stock shape probe: zeros of the map's shape
    with pytest.raises(RuntimeError, match="only on CUDA"):
        layer(x)                                       # autograd enabled: CPU compute is refused as before


def test_fused_output_is_identity_under_the_heads_pool():
    """The head pools the (B, K, 1, 1) output again and views it as (B, K): both are exact identities."""
    t = torch.randn(4, 8, 1, 1)
    assert torch.equal(F.adaptive_avg_pool2d(t, (1, 1)).view(4, -1), t.flatten(1))


def test_functional_rejects_cpu_tensors():
    cfg = _layer().config
    with pytest.raises(RuntimeError, match="only on CUDA"):
        nfpb.nfp_pooled_similarity(torch.randn(1, 16, 8, 8), cfg)
    with torch.no_grad(), pytest.raises(RuntimeError, match="only on CUDA"):
        nfpb.nfp_pooled_similarity(torch.randn(1, 16, 8, 8), cfg)
