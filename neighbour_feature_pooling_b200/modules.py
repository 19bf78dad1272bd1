"""Drop-in ``nn.Module`` surface of the NFP hot path.

Mirrors, name for name, the classes the reference's callers construct:

* ``NFPPooling``          <- reference ``models/pooling/nfp.py:15-134``
* ``nfp_pooling``         <- reference ``models/NFP_Pooling.py:5-36``
* ``EnhancedNFPPooling``  <- the class ``models/nfp_heads.py:6`` imports from the
  module ``models.pooling.enhanced_nfp`` that the reference does not ship

Same constructor arguments and defaults, same attributes, same ``state_dict``
keys, same output layout -- but ``forward`` launches the hand-written sm_100a
kernels of ``libnfp_b200.so`` instead of composing ATen ops, and the
``(B, C*(k*k-1), H', W')`` neighbour tensor is never materialised.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import functional as NF
from ._capi import MEASURES as _MEASURE_IDS


class _FrozenTaps(nn.Module):
    """Holds the frozen one-hot ``weight`` the reference keeps in its two
    depthwise ``nn.Conv2d`` layers (nfp.py:42-82), so that checkpoints written by
    the reference load strictly and ours carry the same keys.  It is never used
    in the computation: the kernels index the taps directly."""

    def __init__(self, weight: torch.Tensor):
        super().__init__()
        self.weight = nn.Parameter(weight, requires_grad=False)

    def forward(self, x):  # pragma: no cover - not a compute path
        raise RuntimeError("the one-hot tap tensors are checkpoint ballast; call the NFPPooling module instead")


def _tap_weights(in_channels: int, R: int, difference_taps: bool):
    """One-hot tensors with the contents of nfp.py:53-82.

    ``comp`` is ``(K*C, 1, k, k)``: output channel ``g*K + n`` has +1 at tap ``n``
    (row-major window, centre removed), or centre=+1 / tap=-1 for the distance
    family.  ``centre`` is ``(C, 1, k, k)`` with +1 in the middle."""
    k = 2 * R + 1
    K = k * k - 1
    taps = [(a, b) for a in range(k) for b in range(k) if (a, b) != (R, R)]
    one = torch.zeros(K, 1, k, k)
    for n, (a, b) in enumerate(taps):
        if difference_taps:
            one[n, 0, R, R] = 1.0
            one[n, 0, a, b] = -1.0
        else:
            one[n, 0, a, b] = 1.0
    comp = one.repeat(in_channels, 1, 1, 1)
    centre = torch.zeros(in_channels, 1, k, k)
    centre[:, 0, R, R] = 1.0
    return comp, centre


class NFPPooling(nn.Module):
    """``(B, C, H, W) -> (B, (2R+1)^2 - 1, H', W')`` similarity of every pixel's
    channel vector with each of its window neighbours.

    Constructor signature and defaults are those of the reference
    (nfp.py:16-18).  Deviations, all loud:

    * ``bias=True`` (a random *trainable* bias added to the extracted taps,
      nfp.py:46,57) is rejected with ``NotImplementedError``;
    * float64 inputs are rejected (the kernels accumulate in fp32);
    * CPU inputs are rejected, except shape probes under ``torch.no_grad()``
      (see ``functional.shape_probe``).
    """

    def __init__(self, in_channels, R=1, measure='norm', p=1, stride=1, padding=0,
                 dilation=1, bias=False, padding_mode='reflect', similarity=True,
                 eps=1e-6, input_size=224, q_scs=1e-6):
        super().__init__()
        self.in_size = input_size
        self.measure = measure.lower()
        self.in_channels = in_channels
        self.R = R
        self.stride = stride
        self.padding = padding
        self.padding_mode = padding_mode
        self.similarity = similarity
        self.p = p
        self.dilation = dilation
        self.bias = bias
        self.eps = eps
        self.q_scs = q_scs
        self.kernel_size = int(2 * self.R + 1)
        self.out_channels = int(self.kernel_size ** 2 - 1)
        if bias:
            raise NotImplementedError(
                "NFPPooling(bias=True) adds a randomly initialised trainable bias to the extracted "
                "neighbours (reference nfp.py:46,57); the B200 kernels do not implement it")
        if padding_mode not in ("zeros", "reflect", "replicate", "circular"):
            raise ValueError("padding_mode must be one of 'zeros', 'reflect', 'replicate' or 'circular', "
                             f"but got padding_mode='{padding_mode}'")
        # nfp.py:74 tests the constructor string as given (case-sensitive), nfp.py:21 lower-cases
        difference_taps = measure in ('norm', 'rmse', 'mahalanobis')
        comp, centre = _tap_weights(in_channels, int(R), difference_taps)
        self.comp_neighbors = _FrozenTaps(comp)
        self.center_value = _FrozenTaps(centre)
        if self.measure not in _MEASURE_IDS:
            raise RuntimeError(f'Similarity measure {self.measure} not implemented')  # nfp.py:119-120
        self._cfg = NF.NFPConfig(R=int(R), measure=self.measure, p=p, stride=int(stride), padding=int(padding),
                                 dilation=int(dilation), padding_mode=padding_mode, similarity=bool(similarity),
                                 eps=float(eps), q_scs=float(q_scs), difference_taps=difference_taps)
        self.similarity_measure = self._measure
        self.register_load_state_dict_post_hook(NFPPooling._verify_taps)

    @property
    def config(self) -> NF.NFPConfig:
        return self._cfg

    @property
    def output_size(self):
        """nfp.py:125-130 -- computed from ``in_size``, not from the input."""
        return (self.in_size + 2 * self.padding - self.dilation * (self.kernel_size - 1) - 1) // self.stride + 1

    @staticmethod
    def _verify_taps(module, incompatible_keys):
        # A checkpoint whose frozen taps differ from the one-hot pattern would mean a different
        # operator than the one the kernels compute; refuse it instead of silently ignoring it.
        comp, centre = _tap_weights(module.center_value.weight.shape[0], module._cfg.R, module._cfg.difference_taps)
        for name, got, want in (("comp_neighbors.weight", module.comp_neighbors.weight, comp),
                                ("center_value.weight", module.center_value.weight, centre)):
            if got.shape != want.shape or not torch.equal(got.detach().float().cpu(), want):
                incompatible_keys.unexpected_keys.append(
                    f"{name} (loaded values are not the frozen one-hot taps of NFPPooling)")

    def _measure(self, x):
        return NF.nfp_similarity(x, self._cfg)

    def forward(self, x):
        return self.similarity_measure(x)

    def extra_repr(self):
        c = self._cfg
        return (f"in_channels={self.in_channels}, R={c.R}, measure={c.measure!r}, stride={c.stride}, "
                f"padding={c.padding}, dilation={c.dilation}, padding_mode={c.padding_mode!r}, "
                f"similarity={c.similarity}")


class EnhancedNFPPooling(NFPPooling):
    """The symbol ``models/nfp_heads.py:6`` imports.  The reference does not ship
    its source, so its semantics are **parity-unpinned**; the heads call it as
    ``EnhancedNFPPooling(in_channels=, R=, measure=, padding=)``
    (nfp_heads.py:18-23,58-63,88-93) exactly like ``resnet18.py:16-21`` calls
    ``NFPPooling``, which is what this is."""

    def __init__(self, in_channels, R=1, measure='cosine', padding=0, **kwargs):
        super().__init__(in_channels, R=R, measure=measure, padding=padding, **kwargs)


class nfp_pooling(nn.Module):
    """``GAP(x) * nfp_proj(GAP(NFP(x)))`` -> ``(B, C)`` (NFP_Pooling.py:25-36).

    With the stock ``NFPPooling`` layer both global-average-pools and the NFP map
    come out of ONE pass over ``x`` (``nfpb200_pool_forward``): the similarity
    map is reduced on chip and never written to HBM."""

    def __init__(self, nfp_layer=None, Params=None):
        super().__init__()
        if nfp_layer is None:
            dense_feature_dim = Params["num_ftrs"][Params["Model_name"]] if Params else 2048
            nfp_layer = NFPPooling(in_channels=dense_feature_dim, R=1, measure='cosine', padding=1,
                                   input_size=Params.get('input_size', 7) if Params else 7)
        self.nfp_layer = nfp_layer
        self.model_name = Params["Model_name"] if Params is not None else None
        self.dataset = Params["Dataset"] if Params is not None else None
        self.num_classes = Params["num_classes"][self.dataset] if Params is not None else None
        self.feature_extraction = (Params['feature_extraction']
                                   if Params is not None and 'feature_extraction' in Params else None)
        self.avgpool = nn.AdaptiveAvgPool2d(1)
        # as in the reference, a user-supplied nfp_layer together with Params=None leaves
        # dense_feature_dim undefined only when Params is given; nfp_proj exists iff Params does
        self.nfp_proj = (nn.Linear(self.nfp_layer.out_channels, Params["num_ftrs"][Params["Model_name"]])
                         if Params else None)

    def _fusable(self):
        """The one-pass head (nfp_gap_pair) stands in for ``self.nfp_layer(x)`` only when that call would run the
        stock operator: a subclass overriding ``forward``, a re-bound ``similarity_measure`` or forward hooks on the
        layer must see the call, as in the reference (NFP_Pooling.py:29)."""
        return _stock(self.nfp_layer)

    def forward(self, x):
        layer = self.nfp_layer
        if x.device.type == "cuda" and self._fusable():
            if (type(self.nfp_proj) is nn.Linear and not self.nfp_proj._forward_hooks
                    and not self.nfp_proj._forward_pre_hooks):
                # the whole head in one launch each way: GAP(x), GAP(NFP(x)), the K -> C projection and the product
                out = NF.nfp_head(x, self.nfp_proj.weight, self.nfp_proj.bias, layer.config)
                if out is not None:
                    return out
            x_avg, x_nfp = NF.nfp_gap_pair(x, layer.config)
        else:
            # foreign / customised nfp_layer module, or a CPU shape probe (NFPPooling answers those itself)
            x_avg = self.avgpool(x).view(x.size(0), -1)
            x_nfp = layer(x)
            x_nfp = nn.functional.adaptive_avg_pool2d(x_nfp, (1, 1)).view(x_nfp.size(0), -1)
        if self.nfp_proj is not None:
            x_nfp = self.nfp_proj(x_nfp)
        return x_avg * x_nfp


def _stock(layer) -> bool:
    """True when calling ``layer(x)`` runs the stock operator (no subclass ``forward``, no re-bound
    ``similarity_measure`` or ``forward``, no hooks): only then may a fused kernel stand in for the call."""
    return (type(layer) in (NFPPooling, EnhancedNFPPooling)
            and "forward" not in layer.__dict__
            and getattr(layer.similarity_measure, "__func__", None) is NFPPooling._measure
            and getattr(layer.similarity_measure, "__self__", None) is layer
            and not layer._forward_hooks and not layer._forward_pre_hooks
            and not layer._backward_hooks and not layer._backward_pre_hooks)


class MultiRadiusNFP(nn.Module):
    """``torch.cat([NFP_R(x) for R in R_list], dim=1)`` -- the operator inside the reference's
    ``MultiRadiusNFPHead`` (models/nfp_heads.py:86-93,111-112) -- as one module.  With ``R_list = (1, 2)`` (the
    reference's default), cosine and ``padding = R`` both maps come out of ONE launch each way (SURVEY 8 f3): the 3x3
    window is the inner part of the 5x5 window, so the radius-1 map and the concatenation are free."""

    def __init__(self, in_channels, R_list=(1, 2), measure="cosine", **kwargs):
        super().__init__()
        self.nfp_blocks = nn.ModuleList([
            EnhancedNFPPooling(in_channels=in_channels, R=R, measure=measure, padding=R, **kwargs) for R in R_list])
        self.out_channels = sum(b.out_channels for b in self.nfp_blocks)

    def forward(self, x):
        if x.device.type == "cuda" and all(_stock(b) for b in self.nfp_blocks):
            return NF.nfp_multi_radius(x, [b.config for b in self.nfp_blocks])
        return torch.cat([b(x) for b in self.nfp_blocks], dim=1)


def fuse_multi_radius(blocks) -> bool:
    """Make the UNMODIFIED reference ``MultiRadiusNFPHead`` (models/nfp_heads.py:80-118) run its two radii in one
    launch: ``fuse_multi_radius(head.nfp_blocks)``.  The head evaluates ``[blk(fmap) for blk in self.nfp_blocks]`` and
    concatenates; after this call the first block returns the complete concatenated map and the second an empty
    ``(B, 0, H, W)`` tensor, so the head's own ``torch.cat`` reproduces the same result.  Module structure, parameters
    and ``state_dict`` keys are untouched (only the two instances' ``forward`` attributes are bound);
    ``unfuse_multi_radius`` restores them.  Returns False (and changes nothing) when the blocks are not two stock
    cosine layers with nested windows (``functional.multi_radius_fusable``)."""
    blocks = list(blocks)
    if len(blocks) != 2 or not all(_stock(b) for b in blocks):
        return False
    first, second = blocks
    cfgs = (first.config, second.config)
    if not NF.multi_radius_fusable(cfgs):
        return False

    def fused_forward(x):
        if x.device.type != "cuda":
            return type(first).forward(first, x)
        return NF.nfp_multi_radius(x, cfgs)

    def empty_forward(x):
        if x.device.type != "cuda":
            return type(second).forward(second, x)
        return x.new_empty((x.shape[0], 0, x.shape[2], x.shape[3]),
                           dtype=torch.float32 if torch.is_autocast_enabled("cuda") else x.dtype)

    first.forward = fused_forward
    second.forward = empty_forward
    return True


def unfuse_multi_radius(blocks):
    for b in blocks:
        b.__dict__.pop("forward", None)


class _PooledForward:
    """``forward`` of a layer fused by ``fuse_pooled_nfp``: ``GAP(NFP(x))`` as a ``(B, K, 1, 1)`` tensor on CUDA, the
    stock forward for every other input.  A module-level class holding the layer (not a closure), so that ``pickle`` /
    ``torch.save`` and ``copy.deepcopy`` round-trip a fused layer, and a copy's forward runs on the copy."""

    def __init__(self, layer):
        self.layer = layer

    def __call__(self, x):
        layer = self.layer
        if x.device.type != "cuda":   # CPU shape probes and CPU errors: exactly as the stock layer answers them
            return type(layer).forward(layer, x)
        return NF.nfp_pooled_similarity(x, layer.config)[:, :, None, None]


def fuse_pooled_nfp(layer) -> bool:
    """Make a stock ``NFPPooling`` / ``EnhancedNFPPooling`` layer return ``adaptive_avg_pool2d(NFP(x), 1)``, shape
    ``(B, K, 1, 1)``, computed without writing the similarity map (``functional.nfp_pooled_similarity``).

    For callers that global-pool the layer's output right away, as every stage of the reference's
    ``MobileNetV3_MultiStageNFP`` does (models/texture_pooling.py:249-256: ``adaptive_avg_pool2d(nfp(x), (1, 1))`` then
    ``.view(B, -1)``): their own pool and view are then exact identities, so the unmodified head gets the same values.
    It is valid ONLY for such callers: anything else that reads the layer's output sees a 1 x 1 map.  Forward hooks
    registered on the layer after this call see the ``(B, K, 1, 1)`` tensor.  CPU inputs (constructor shape probes
    included) take the stock forward.

    Only the instance's ``forward`` attribute is set; parameters, ``state_dict`` keys and the module tree are unchanged,
    and ``unfuse_pooled_nfp`` restores the stock forward.  Returns False and changes nothing when the layer is not a
    stock cosine layer (a subclass, a re-bound ``forward`` / ``similarity_measure``, hooks, another measure)."""
    if not _stock(layer) or layer.config.measure != "cosine":
        return False
    layer.forward = _PooledForward(layer)
    return True


def unfuse_pooled_nfp(layer):
    if isinstance(layer.__dict__.get("forward"), _PooledForward):
        del layer.__dict__["forward"]


__all__ = ["NFPPooling", "EnhancedNFPPooling", "nfp_pooling", "MultiRadiusNFP", "fuse_multi_radius",
           "unfuse_multi_radius", "fuse_pooled_nfp", "unfuse_pooled_nfp"]
