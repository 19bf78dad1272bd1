"""CPU: the drop-in nn.Module surface (SURVEY.md section 8 row b1): constructor arguments, attributes,
state_dict compatibility with the reference, shape probes, error behaviour, import-path shims."""
import os
import sys

import numpy as np
import pytest
import torch

import neighbour_feature_pooling_b200 as nfpb
from neighbour_feature_pooling_b200 import NFPPooling, EnhancedNFPPooling, nfp_pooling
from oracle.ref_loader import REFERENCE_ROOT, reference_available

from _util import GOLDEN


def test_constructor_defaults_and_attributes():
    m = NFPPooling(6)
    assert (m.R, m.measure, m.p, m.stride, m.padding, m.dilation, m.bias, m.padding_mode, m.similarity,
            m.eps, m.in_size, m.q_scs) == (1, "norm", 1, 1, 0, 1, False, "reflect", True, 1e-6, 224, 1e-6)
    assert m.kernel_size == 3 and m.out_channels == 8 and m.in_channels == 6
    assert m.output_size == 222            # nfp.py:125-130 with input_size=224, padding=0
    m.in_channels = 99                     # reference callers assign it after construction (resnet18.py:166)
    assert m.in_channels == 99
    m2 = NFPPooling(4, R=2, measure="Cosine", padding=2, input_size=14)
    assert m2.measure == "cosine" and m2.kernel_size == 5 and m2.out_channels == 24 and m2.output_size == 14
    assert callable(m2.similarity_measure)


def test_unknown_measure_and_rejections():
    with pytest.raises(RuntimeError, match="Similarity measure mahalanobis not implemented"):
        NFPPooling(4, measure="mahalanobis")
    with pytest.raises(RuntimeError, match="Similarity measure foo not implemented"):
        NFPPooling(4, measure="Foo")
    with pytest.raises(NotImplementedError):
        NFPPooling(4, bias=True)
    with pytest.raises(TypeError):
        NFPPooling(None)                   # the reference crashes in nn.Conv2d the same way


def test_state_dict_matches_reference_layout():
    ref = np.load(os.path.join(GOLDEN, "nfp_state_dict.npz"))
    for measure in ("cosine", "norm"):
        m = NFPPooling(3, R=1, measure=measure, padding=1)
        sd = m.state_dict()
        assert list(sd.keys()) == ["comp_neighbors.weight", "center_value.weight"]
        for k, v in sd.items():
            np.testing.assert_array_equal(v.numpy(), ref[f"{measure}_{k}"])
        # strict load of the reference's tensors
        m.load_state_dict({k: torch.from_numpy(ref[f"{measure}_{k}"]) for k in sd}, strict=True)
    params = dict(NFPPooling(3, measure="cosine").named_parameters())
    assert set(params) == {"comp_neighbors.weight", "center_value.weight"}
    assert all(not p.requires_grad for p in params.values())
    # a checkpoint whose frozen taps were trained/edited would be a different operator: refuse it
    bad = {k: v.clone() for k, v in NFPPooling(3, measure="cosine").state_dict().items()}
    bad["comp_neighbors.weight"][0, 0, 0, 0] = 0.5
    with pytest.raises(RuntimeError, match="not the frozen one-hot taps"):
        NFPPooling(3, measure="cosine").load_state_dict(bad)
    # case quirk of nfp.py:74: 'Norm' builds similarity-style taps, 'norm' difference taps
    assert NFPPooling(2, measure="Norm").comp_neighbors.weight.min() == 0
    assert NFPPooling(2, measure="norm").comp_neighbors.weight.min() == -1


def test_cpu_shape_probe_and_cpu_rejection():
    m = NFPPooling(8, R=1, measure="cosine", padding=1)
    with torch.no_grad():
        out = m(torch.randn(1, 8, 7, 7))
    assert out.shape == (1, 8, 7, 7) and torch.isfinite(out).all()   # finite: probes may feed train-mode BatchNorm
    with torch.no_grad():
        assert NFPPooling(8, R=2, measure="cosine", padding=0, stride=2)(torch.randn(2, 8, 9, 11)).shape == (2, 24, 3, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 8, 7, 7))          # grad mode on: a real CPU computation is being asked for
    with torch.no_grad(), pytest.raises(RuntimeError, match="Padding size should be less"):
        NFPPooling(8, measure="cosine", padding=2)(torch.randn(1, 8, 2, 2))
    with torch.no_grad(), pytest.raises(RuntimeError, match="Kernel size can't be greater"):
        NFPPooling(8, measure="cosine", padding=0)(torch.randn(1, 8, 2, 2))


def test_shape_probe_keeps_batchnorm_buffers_finite():
    """The reference's MOBILENETV3_NFP_INSERT.__init__ (mobilenetv3.py:337-353) pipes its CPU dummy through NFP and on
    through train-mode Conv+BatchNorm blocks under no_grad: BatchNorm updates its running statistics there, so the
    probe's values must be finite or every later eval() / checkpoint carries NaNs."""
    import torch.nn as nn
    nfp = NFPPooling(16, R=1, measure="cosine", padding=1)
    tail = nn.Sequential(nn.Conv2d(nfp.out_channels, 16, 1, bias=False), nn.BatchNorm2d(16), nn.ReLU(),
                         nn.Conv2d(16, 4, 3, padding=1), nn.BatchNorm2d(4))
    tail.train()
    with torch.no_grad():
        out = tail(nfp(torch.randn(2, 16, 14, 14)))
    assert out.shape == (2, 4, 14, 14)
    for name, buf in tail.named_buffers():
        assert torch.isfinite(buf).all(), name


def test_wrapper_contract():
    Params = {"num_ftrs": {"resnet18": 16}, "Model_name": "resnet18", "Dataset": "UCMerced",
              "num_classes": {"UCMerced": 21}, "feature_extraction": False}
    w = nfp_pooling(Params=Params)
    assert isinstance(w.nfp_layer, NFPPooling)
    assert (w.nfp_layer.in_channels, w.nfp_layer.R, w.nfp_layer.measure, w.nfp_layer.padding, w.nfp_layer.in_size) == \
        (16, 1, "cosine", 1, 7)
    assert (w.model_name, w.dataset, w.num_classes, w.feature_extraction) == ("resnet18", "UCMerced", 21, False)
    assert w.nfp_proj.in_features == 8 and w.nfp_proj.out_features == 16
    assert sorted(w.state_dict().keys()) == sorted(
        ["nfp_layer.comp_neighbors.weight", "nfp_layer.center_value.weight", "nfp_proj.weight", "nfp_proj.bias"])
    assert [n for n, p in w.named_parameters() if p.requires_grad] == ["nfp_proj.weight", "nfp_proj.bias"]
    with torch.no_grad():
        assert w(torch.randn(2, 16, 7, 7)).shape == (2, 16)   # CPU shape probe
    bare = nfp_pooling()
    assert bare.nfp_proj is None and bare.nfp_layer.in_channels == 2048 and bare.model_name is None
    custom = nfp_pooling(nfp_layer=NFPPooling(4, R=2, measure="dot", padding=2), Params=None)
    assert custom.nfp_layer.out_channels == 24


def test_enhanced_symbol():
    e = EnhancedNFPPooling(in_channels=8, R=2, measure="cosine", padding=2)
    assert isinstance(e, NFPPooling) and e.out_channels == 24


def test_install_dropin_import_paths():
    nfpb.install_dropin()
    try:
        from models.pooling.nfp import NFPPooling as A
        from models.NFP_Pooling import nfp_pooling as B
        from models.pooling.enhanced_nfp import EnhancedNFPPooling as C
        assert A is NFPPooling and B is nfp_pooling and C is EnhancedNFPPooling
    finally:
        nfpb.uninstall_dropin()
    assert "models.pooling.nfp" not in sys.modules


@pytest.mark.skipif(not reference_available(), reason="needs the original project: NFP_REFERENCE_ROOT or a copy staged under oracle/_ref")
def test_reference_heads_run_unchanged_on_the_dropin():
    """models/nfp_heads.py is un-importable upstream (missing EnhancedNFPPooling); with the drop-in
    installed it imports, and its constructors' CPU dummy probes (nfp_heads.py:24-27,95-97) work."""
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "models" or k.startswith("models.")}
    nfpb.install_dropin()
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        import models.nfp_heads as heads
        h = heads.NFPHead(in_c=32, bottleneck_dim=16)
        assert isinstance(h.nfp, NFPPooling) and h.nfp_out_channels == 8
        mr = heads.MultiRadiusNFPHead(in_c=32, bottleneck_dim=16)
        assert mr.compress[0].in_channels == 8 + 24
        # SURVEY 8 f3: the head's two radii in one launch -- only the blocks' forward attributes are bound, the module
        # tree / state_dict are untouched, and CPU shape probes still answer block by block
        keys = list(mr.state_dict().keys())
        assert nfpb.fuse_multi_radius(mr.nfp_blocks)
        assert list(mr.state_dict().keys()) == keys
        with torch.no_grad():
            assert [b(torch.randn(1, 32, 7, 7)).shape[1] for b in mr.nfp_blocks] == [8, 24]
        nfpb.unfuse_multi_radius(mr.nfp_blocks)
        assert not any("forward" in b.__dict__ for b in mr.nfp_blocks)
    finally:
        sys.path.remove(REFERENCE_ROOT)
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
            sys.modules.pop(k)
        sys.modules.update(saved)
