"""Autograd bindings of the NFP C ABI.

``nfp_similarity``  -- the operator behind ``NFPPooling.forward``
                       (reference models/pooling/nfp.py:132-134): (B,C,H,W) -> (B,K,H',W')
``nfp_gap_pair``    -- the fused head of ``nfp_pooling.forward``
                       (reference models/NFP_Pooling.py:27-31): (GAP(x), GAP(NFP(x)))
``nfp_pooled_similarity`` -- what every stage of the multi-stage head keeps of its map
                       (reference models/texture_pooling.py:249-256): GAP(NFP(x)) -> (B, K)

Both launch the hand-written sm_100a kernels of libnfp_b200.so on the current
CUDA stream.  Backward recomputes the similarities from ``x``; nothing but ``x``
is saved.  There is no CPU or PyTorch implementation behind these functions:
CPU tensors are rejected (except the constructor-time shape probes described in
``shape_probe``).
"""
from __future__ import annotations

import ctypes
import os
import math
from dataclasses import dataclass, replace

import torch

from . import _capi


@dataclass(frozen=True)
class NFPConfig:
    """Constructor arguments of the reference NFPPooling (nfp.py:16-18) that shape the math."""
    R: int = 1
    measure: str = "norm"          # lower-cased spelling, nfp.py:21
    p: float = 1
    stride: int = 1
    padding: int = 0
    dilation: int = 1
    padding_mode: str = "reflect"
    similarity: bool = True
    eps: float = 1e-6
    q_scs: float = 1e-6
    difference_taps: bool = False  # nfp.py:74: raw measure string in ('norm','rmse','mahalanobis')
    path: str = "auto"             # 'auto' | 'generic' | 'fused'

    @property
    def kernel_size(self) -> int:
        return 2 * self.R + 1

    @property
    def out_channels(self) -> int:
        return self.kernel_size ** 2 - 1


def conv_output_size(n: int, cfg: NFPConfig) -> int:
    """Conv2d output-size rule (what nfp.py:128-129 restates)."""
    return (n + 2 * cfg.padding - cfg.dilation * (cfg.kernel_size - 1) - 1) // cfg.stride + 1


def _check_geometry(H: int, W: int, cfg: NFPConfig):
    # same failure modes as the reference's Conv2d(padding_mode=...) forward
    if cfg.padding_mode == "reflect" and cfg.padding > 0 and (cfg.padding >= H or cfg.padding >= W):
        raise RuntimeError(
            "Padding size should be less than the corresponding input dimension, but got: padding "
            f"({cfg.padding}, {cfg.padding}) at dimension 3 of input {[H, W]}")
    if cfg.padding_mode == "circular" and (cfg.padding > H or cfg.padding > W):
        raise RuntimeError("Padding value causes wrapping around more than once.")
    Ho, Wo = conv_output_size(H, cfg), conv_output_size(W, cfg)
    if Ho <= 0 or Wo <= 0:
        span = cfg.dilation * (cfg.kernel_size - 1) + 1
        raise RuntimeError(
            f"Calculated padded input size per channel: ({H + 2 * cfg.padding} x {W + 2 * cfg.padding}). "
            f"Kernel size: ({span} x {span}). Kernel size can't be greater than actual input size")
    return Ho, Wo


def shape_probe(x: torch.Tensor, cfg: NFPConfig) -> torch.Tensor:
    """Answer a constructor-time shape probe without computing anything.

    The reference heads discover NFP's output width by running a CPU dummy
    through the layer inside ``__init__`` under ``torch.no_grad()``
    (resnet18.py:22-25, nfp_heads.py:24-27, mobilenetv3.py:337-353).  This
    package has no CPU implementation, so a CPU input with autograd disabled is
    answered with a ZERO tensor of the correct shape.  Some of those callers pipe
    the probe through train-mode ``BatchNorm`` layers (mobilenetv3.py:347-353),
    which update their running statistics even under ``no_grad``: the values must
    therefore be finite (a NaN probe would poison the running buffers for good).
    The result carries no information beyond its shape; real CPU inference is
    rejected whenever autograd is enabled, and documented as unsupported otherwise.
    """
    B, C, H, W = x.shape
    Ho, Wo = _check_geometry(H, W, cfg)
    return torch.zeros((B, cfg.out_channels, Ho, Wo), dtype=x.dtype, device=x.device)


def _reject_cpu(x: torch.Tensor):
    raise RuntimeError(
        "neighbour_feature_pooling_b200 runs only on CUDA (sm_100a) tensors; got a "
        f"{x.device.type} tensor.  There is no CPU fallback by design.  (CPU inputs are accepted only "
        "as shape probes under torch.no_grad().)")


_KERNEL_DTYPES = {torch.float32: _capi.F32, torch.bfloat16: _capi.BF16}
# diagnostics: when a set is installed here (bench_train.py does during its eager warm-up), every forward records the
# kernel path it takes ("fused/token_7x7_r1 bf16 pool", ...)
PATH_TRACE = None


def _trace(desc, op, what):
    if PATH_TRACE is not None:
        PATH_TRACE.add(f"{_capi.describe_path(desc, op)} {'bf16' if desc.dtype == _capi.BF16 else 'f32'} "
                       f"{'channels-last' if desc.layout else 'nchw'} {what}")

# NFPB200_HINT_X_STABLE (include/nfp_b200.h) is opt-in: it pays only when the backward directly follows another fused NFP
# launch on the stream (-1.9 us per backward in such chains); after any other kernel -- the normal case inside a network --
# there is nothing to overlap and the reordered prologue costs ~0.9 us.  NFPB200_X_STABLE_HINT=1 switches it on.
_X_STABLE_HINT = os.environ.get("NFPB200_X_STABLE_HINT", "0") == "1"


def _prepare(x: torch.Tensor, cfg: NFPConfig = None):
    """-> (tensor in a kernel dtype, dtype to return results in, memory layout the kernels will read)

    Under ``torch.autocast('cuda')`` the reference extracts the neighbours with convs in the autocast dtype and then
    runs ``F.cosine_similarity`` (``norm``, ``sum``, ``softmax`` ... for the other measures), which is on autocast's
    fp32 list: its similarity map is float32.  A bf16 input therefore gives an fp32 map (the fused forward writes
    fp32 directly, NFPB200_FLAG_Y_F32).  An fp32 input is NOT rounded to the autocast dtype first: the kernels
    accumulate in fp32 anyway, so the result only differs from the reference's by the reference's own input rounding
    (well inside the 2e-2 bf16 tolerance), and the cast kernel is saved."""
    if x.dim() != 4:
        raise RuntimeError(f"NFP expects a 4-D (B, C, H, W) input, got {tuple(x.shape)}")
    if not x.is_floating_point():
        raise RuntimeError(f"NFP expects a floating-point input, got {x.dtype}")
    out_dtype = x.dtype
    if torch.is_autocast_enabled("cuda"):
        out_dtype = torch.float32
    if x.dtype == torch.float64:
        raise RuntimeError("NFP kernels compute in fp32; float64 inputs are not supported")
    if x.dtype not in _KERNEL_DTYPES:  # fp16: widen, the kernels accumulate in fp32 anyway
        x = x.float()
    if cfg is not None and _channels_last_ok(x, cfg):
        return x, out_dtype, _capi.LAYOUT_NHWC     # consumed in place: no repack copy
    if (cfg is not None and x.dtype == torch.float32 and x.dim() == 4 and torch.is_autocast_enabled("cuda")
            and torch.get_autocast_dtype("cuda") == torch.bfloat16 and _is_channels_last_view(x)):
        # fp32 channels-last map under bf16 autocast (a ViT's final LayerNorm emits fp32 tokens): the reference's
        # extraction convs would round it to bf16 (nfp.py:152-153); doing the same costs one cast kernel (4 B in,
        # 2 B out per element) instead of an NCHW repack (4 B in, 4 B out) and keeps the tensor-core path
        xb = x.to(torch.bfloat16)
        if _channels_last_ok(xb, cfg):
            return xb, out_dtype, _capi.LAYOUT_NHWC
    x = x.contiguous()
    if x.data_ptr() % 16:   # a view at an odd storage offset: the kernels move data with 16-byte TMA copies
        x = x.clone()
    return x, out_dtype, _capi.LAYOUT_NCHW


def _is_channels_last_view(x: torch.Tensor) -> bool:
    """x[b, c, h, w] lives at b*sB + (h*W + w)*C + c: a torch channels_last map, or the (B, C, H, W) VIEW the
    reference's ViT head makes of the backbone's (B, 1+N, C) token tensor (texture_pooling.py:181-188)."""
    B, C, H, W = x.shape
    sb, sc, sh, sw = x.stride()
    return C > 1 and sc == 1 and sw == C and sh == W * C and (B == 1 or sb >= H * W * C) and not x.is_contiguous()


def _channels_last_ok(x: torch.Tensor, cfg: NFPConfig) -> bool:
    """True when the tensor-core channels-last kernels (fused/token_*) take x as it lies in memory."""
    if x.dtype != torch.bfloat16 or x.dim() != 4 or not _is_channels_last_view(x):
        return False
    if x.data_ptr() % 16 or (x.shape[0] > 1 and x.stride(0) % 8):
        return False
    if cfg.path == "generic":
        return False
    desc = _desc_for(x, cfg, _capi.LAYOUT_NHWC)
    buf = ctypes.create_string_buffer(64)
    return _capi.load().nfpb200_describe_path(ctypes.byref(desc), _capi.OP_BACKWARD, buf, 64) == 0


def _desc_for(x: torch.Tensor, cfg: NFPConfig, layout: int = 0) -> _capi.Desc:
    B, C, H, W = x.shape
    xbs = x.stride(0) if (layout == _capi.LAYOUT_NHWC and B > 1) else 0
    return _capi.make_desc(_KERNEL_DTYPES[x.dtype], B, C, H, W, cfg.R, cfg.stride, cfg.padding,
                           cfg.dilation, cfg.padding_mode, cfg.measure, cfg.similarity,
                           cfg.difference_taps, cfg.eps, cfg.p, cfg.q_scs, cfg.path, layout=layout,
                           x_batch_stride=xbs, gx_batch_stride=0)


def _empty_like_layout(x: torch.Tensor, layout: int) -> torch.Tensor:
    if layout == _capi.LAYOUT_NHWC:   # dense channels_last: what a cuDNN NHWC backbone wants back
        B, C, H, W = x.shape
        return torch.empty_strided((B, C, H, W), (H * W * C, 1, W * C, C), dtype=x.dtype, device=x.device)
    return torch.empty_like(x)


def _workspace(desc, op, device):
    n = _capi.workspace_bytes(desc, op)
    if n == 0:
        return None, 0, 0
    ws = torch.empty(n, dtype=torch.uint8, device=device)
    return ws, ws.data_ptr(), n


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class _NFPSimilarity(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, cfg, y_f32=False, layout=0):
        desc = _desc_for(x, cfg, layout)
        Ho, Wo = _capi.output_shape(desc)
        # bf16 x, fp32 map (autocast): the fused kernels write fp32 directly; other paths write bf16 (widened by
        # the caller)
        y_f32 = bool(y_f32) and x.dtype == torch.bfloat16 and \
            _capi.describe_path(desc, _capi.OP_FORWARD).startswith("fused/")
        if y_f32:
            desc.path |= _capi.FLAG_Y_F32
        y = torch.empty((x.shape[0], cfg.out_channels, Ho, Wo), dtype=torch.float32 if y_f32 else x.dtype,
                        device=x.device)
        _trace(desc, _capi.OP_FORWARD, "map")
        with torch.cuda.device(x.device):
            ws, ws_ptr, ws_n = _workspace(desc, _capi.OP_FORWARD, x.device)
            rc = _capi.load().nfpb200_forward(ctypes.byref(desc), x.data_ptr(), y.data_ptr(), ws_ptr, ws_n,
                                              _stream(x.device))
        _capi.check(rc, "nfpb200_forward")
        ctx.save_for_backward(x)
        ctx.cfg = cfg
        ctx.layout = layout
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        desc = _desc_for(x, ctx.cfg, ctx.layout)
        # x is a saved forward activation: the launch that precedes this one on the stream did not write it, so the
        # hint would be valid here; see _X_STABLE_HINT for why it is opt-in
        if _X_STABLE_HINT:
            desc.path |= _capi.HINT_X_STABLE
        gy = gy.to(x.dtype).contiguous()
        if gy.data_ptr() % 16:
            gy = gy.clone()
        gx = _empty_like_layout(x, ctx.layout)
        with torch.cuda.device(x.device):
            ws, ws_ptr, ws_n = _workspace(desc, _capi.OP_BACKWARD, x.device)
            rc = _capi.load().nfpb200_backward(ctypes.byref(desc), x.data_ptr(), gy.data_ptr(), gx.data_ptr(),
                                               ws_ptr, ws_n, _stream(x.device))
        _capi.check(rc, "nfpb200_backward")
        return gx, None, None, None


class _NFPGapPair(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, cfg, layout=0):
        desc = _desc_for(x, cfg, layout)
        B, C = x.shape[:2]
        gap_x = torch.empty((B, C), dtype=torch.float32, device=x.device)
        gap_nfp = torch.empty((B, cfg.out_channels), dtype=torch.float32, device=x.device)
        _trace(desc, _capi.OP_POOL_FORWARD, "pooled head")
        with torch.cuda.device(x.device):
            ws, ws_ptr, ws_n = _workspace(desc, _capi.OP_POOL_FORWARD, x.device)
            rc = _capi.load().nfpb200_pool_forward(ctypes.byref(desc), x.data_ptr(), gap_x.data_ptr(),
                                                   gap_nfp.data_ptr(), ws_ptr, ws_n, _stream(x.device))
        _capi.check(rc, "nfpb200_pool_forward")
        ctx.save_for_backward(x)
        ctx.cfg = cfg
        ctx.layout = layout
        return gap_x, gap_nfp

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_gap_x, g_gap_nfp):
        (x,) = ctx.saved_tensors
        desc = _desc_for(x, ctx.cfg, ctx.layout)
        # x is a saved forward activation: the launch that precedes this one on the stream did not write it, so the
        # hint would be valid here; see _X_STABLE_HINT for why it is opt-in
        if _X_STABLE_HINT:
            desc.path |= _capi.HINT_X_STABLE
        g_gap_x = g_gap_x.float().contiguous()
        g_gap_nfp = g_gap_nfp.float().contiguous()
        gx = _empty_like_layout(x, ctx.layout)
        with torch.cuda.device(x.device):
            ws, ws_ptr, ws_n = _workspace(desc, _capi.OP_POOL_BACKWARD, x.device)
            rc = _capi.load().nfpb200_pool_backward(ctypes.byref(desc), x.data_ptr(), g_gap_x.data_ptr(),
                                                    g_gap_nfp.data_ptr(), gx.data_ptr(), ws_ptr, ws_n,
                                                    _stream(x.device))
        _capi.check(rc, "nfpb200_pool_backward")
        return gx, None, None


class _NFPPooledMap(torch.autograd.Function):
    """GAP(NFP(x)) (B, K) fp32 without writing the map (nfpb200_pooled_map_forward / _backward)."""

    @staticmethod
    def forward(ctx, x, cfg, layout=0):
        desc = _desc_for(x, cfg, layout)
        gap_nfp = torch.empty((x.shape[0], cfg.out_channels), dtype=torch.float32, device=x.device)
        _trace(desc, _capi.OP_POOLED_MAP_FORWARD, "pooled map")
        with torch.cuda.device(x.device):
            ws, ws_ptr, ws_n = _workspace(desc, _capi.OP_POOLED_MAP_FORWARD, x.device)
            rc = _capi.load().nfpb200_pooled_map_forward(ctypes.byref(desc), x.data_ptr(), gap_nfp.data_ptr(),
                                                         ws_ptr, ws_n, _stream(x.device))
        _capi.check(rc, "nfpb200_pooled_map_forward")
        ctx.save_for_backward(x)
        ctx.cfg = cfg
        ctx.layout = layout
        return gap_nfp

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_gap_nfp):
        (x,) = ctx.saved_tensors
        desc = _desc_for(x, ctx.cfg, ctx.layout)
        if _X_STABLE_HINT:
            desc.path |= _capi.HINT_X_STABLE
        g_gap_nfp = g_gap_nfp.float().contiguous()   # fp32 whatever the dtype of x
        gx = _empty_like_layout(x, ctx.layout)
        with torch.cuda.device(x.device):
            ws, ws_ptr, ws_n = _workspace(desc, _capi.OP_POOLED_MAP_BACKWARD, x.device)
            rc = _capi.load().nfpb200_pooled_map_backward(ctypes.byref(desc), x.data_ptr(), g_gap_nfp.data_ptr(),
                                                          gx.data_ptr(), ws_ptr, ws_n, _stream(x.device))
        _capi.check(rc, "nfpb200_pooled_map_backward")
        return gx, None, None


class _NFPHead(torch.autograd.Function):
    """out = GAP(x) * (W GAP(NFP(x)) + b) in ONE launch each way (nfpb200_head_forward / _backward); the projection's
    parameter gradients are three tiny PyTorch ops on the (B, C) / (B, K) tensors the forward leaves behind."""

    @staticmethod
    def forward(ctx, x, weight, bias, cfg, layout=0):
        desc = _desc_for(x, cfg, layout)
        B, C = x.shape[:2]
        w = weight.detach().float().contiguous()
        bvec = bias.detach().float().contiguous() if bias is not None else None
        out = torch.empty((B, C), dtype=torch.float32, device=x.device)
        gap_x = torch.empty((B, C), dtype=torch.float32, device=x.device)
        gap_nfp = torch.empty((B, cfg.out_channels), dtype=torch.float32, device=x.device)
        if PATH_TRACE is not None:
            PATH_TRACE.add(f"{_capi.describe_path(desc, _capi.OP_POOL_FORWARD)} "
                           f"{'bf16' if desc.dtype == _capi.BF16 else 'f32'} {'channels-last' if layout else 'nchw'} "
                           "fused head (GAP, GAP(NFP), proj, product)")
        with torch.cuda.device(x.device):
            rc = _capi.load().nfpb200_head_forward(ctypes.byref(desc), x.data_ptr(), w.data_ptr(),
                                                   bvec.data_ptr() if bvec is not None else None, out.data_ptr(),
                                                   gap_x.data_ptr(), gap_nfp.data_ptr(), _stream(x.device))
        _capi.check(rc, "nfpb200_head_forward")
        ctx.save_for_backward(x, w, bvec if bvec is not None else w.new_empty(0), gap_x, gap_nfp)
        ctx.cfg = cfg
        ctx.layout = layout
        ctx.has_bias = bias is not None
        ctx.param_dtypes = (weight.dtype, bias.dtype if bias is not None else None)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_out):
        x, w, bvec, gap_x, gap_nfp = ctx.saved_tensors
        desc = _desc_for(x, ctx.cfg, ctx.layout)
        if _X_STABLE_HINT:
            desc.path |= _capi.HINT_X_STABLE
        g_out = g_out.float().contiguous()
        gx = _empty_like_layout(x, ctx.layout)
        with torch.cuda.device(x.device):
            rc = _capi.load().nfpb200_head_backward(ctypes.byref(desc), x.data_ptr(), w.data_ptr(),
                                                    bvec.data_ptr() if ctx.has_bias else None, gap_x.data_ptr(),
                                                    gap_nfp.data_ptr(), g_out.data_ptr(), gx.data_ptr(),
                                                    _stream(x.device))
        _capi.check(rc, "nfpb200_head_backward")
        t = g_out * gap_x                                   # d loss / d proj  (B, C)
        gw = (t.t() @ gap_nfp).to(ctx.param_dtypes[0]) if ctx.needs_input_grad[1] else None
        gb = t.sum(0).to(ctx.param_dtypes[1]) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return gx, gw, gb, None, None


def nfp_head(x: torch.Tensor, weight: torch.Tensor, bias, cfg: NFPConfig):
    """``GAP(x) * (weight @ GAP(NFP(x)) + bias)`` -> (B, C): the whole nfp_pooling head (NFP_Pooling.py:25-36) fused
    into the pooled kernels.  Returns None when the problem is not covered (the caller composes the pieces)."""
    if x.device.type != "cuda" or x.dim() != 4 or weight.device != x.device:
        return None
    _check_geometry(x.shape[2], x.shape[3], cfg)
    xk, out_dtype, layout = _prepare(x, cfg)
    desc = _desc_for(xk, cfg, layout)
    if _capi.load().nfpb200_head_supported(ctypes.byref(desc)) != 0:
        return None
    out = _NFPHead.apply(xk, weight, bias, cfg, layout)
    # NFP_Pooling.py:35: x_avg (dtype of x) * nfp_proj(...) (autocast dtype under autocast, else the parameter dtype)
    proj_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else weight.dtype
    return out.to(torch.promote_types(x.dtype, proj_dtype))


class _NFPMultiRadius(torch.autograd.Function):
    """[NFP_r(x) | NFP_R(x)] along the channel axis in ONE launch each way (desc.inner_R, include/nfp_b200.h)."""

    @staticmethod
    def forward(ctx, x, cfg, inner_R, y_f32=False, layout=0):
        desc = _desc_for(x, cfg, layout)
        desc.inner_R = inner_R
        Ho, Wo = _capi.output_shape(desc)
        # bf16 x, fp32 map (autocast): the fused kernels write fp32 directly; the planar band kernels write bf16 (widened
        # by the caller)
        y_f32 = bool(y_f32) and x.dtype == torch.bfloat16 and \
            _capi.describe_path(desc, _capi.OP_FORWARD).startswith("fused/")
        if y_f32:
            desc.path |= _capi.FLAG_Y_F32
        k_in = (2 * inner_R + 1) ** 2 - 1
        y = torch.empty((x.shape[0], k_in + cfg.out_channels, Ho, Wo), dtype=torch.float32 if y_f32 else x.dtype,
                        device=x.device)
        _trace(desc, _capi.OP_FORWARD, f"map, radii {inner_R}+{cfg.R} in one launch")
        with torch.cuda.device(x.device):
            rc = _capi.load().nfpb200_forward(ctypes.byref(desc), x.data_ptr(), y.data_ptr(), None, 0,
                                              _stream(x.device))
        _capi.check(rc, "nfpb200_forward (multi-radius)")
        ctx.save_for_backward(x)
        ctx.cfg, ctx.inner_R, ctx.layout = cfg, inner_R, layout
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        desc = _desc_for(x, ctx.cfg, ctx.layout)
        desc.inner_R = ctx.inner_R
        if _X_STABLE_HINT:
            desc.path |= _capi.HINT_X_STABLE
        gy = gy.to(x.dtype).contiguous()
        if gy.data_ptr() % 16:
            gy = gy.clone()
        gx = _empty_like_layout(x, ctx.layout)
        with torch.cuda.device(x.device):
            rc = _capi.load().nfpb200_backward(ctypes.byref(desc), x.data_ptr(), gy.data_ptr(), gx.data_ptr(),
                                               None, 0, _stream(x.device))
        _capi.check(rc, "nfpb200_backward (multi-radius)")
        return gx, None, None, None, None


def multi_radius_fusable(cfgs) -> bool:
    """Two cosine layers whose windows nest -- (inner radius r, outer radius R > r), each with padding = its radius,
    stride 1, dilation 1 and otherwise equal options: the radius-r window is then the inner part of the radius-R
    window (the padding rule maps an index, whatever the pad width), so one pass over x yields both maps."""
    if len(cfgs) != 2:
        return False
    a, b = cfgs
    return (a.measure == "cosine" and b.measure == "cosine" and a.R < b.R and a.padding == a.R and b.padding == b.R
            and a.stride == b.stride == 1 and a.dilation == b.dilation == 1 and a.padding_mode == b.padding_mode
            and a.padding_mode != "circular" and a.similarity == b.similarity and a.eps == b.eps
            and a.path == b.path and a.path != "generic")


def nfp_multi_radius(x: torch.Tensor, cfgs) -> torch.Tensor:
    """``torch.cat([nfp_similarity(x, c) for c in cfgs], dim=1)`` -- what the reference's ``MultiRadiusNFPHead``
    computes block by block (models/nfp_heads.py:80-118: R_list = (1, 2), then ``torch.cat``) -- in ONE launch each
    way when ``multi_radius_fusable(cfgs)`` and the fused kernels cover the map (SURVEY 8 f3): the radius-1 map costs
    nothing beyond the radius-2 launch, and the concatenation copy disappears.  Anything else is computed layer by
    layer and concatenated (same values)."""
    cfgs = tuple(cfgs)
    if x.device.type == "cuda" and x.dim() == 4 and multi_radius_fusable(cfgs):
        inner, outer = cfgs
        _check_geometry(x.shape[2], x.shape[3], outer)
        xk, out_dtype, layout = _prepare(x, outer)
        desc = _desc_for(xk, outer, layout)
        desc.inner_R = inner.R
        buf = ctypes.create_string_buffer(64)
        lib = _capi.load()
        if (lib.nfpb200_describe_path(ctypes.byref(desc), _capi.OP_FORWARD, buf, 64) == 0
                and lib.nfpb200_describe_path(ctypes.byref(desc), _capi.OP_BACKWARD, buf, 64) == 0):
            y = _NFPMultiRadius.apply(xk, outer, inner.R, out_dtype == torch.float32, layout)
            return y if y.dtype == out_dtype else y.to(out_dtype)
    return torch.cat([nfp_similarity(x, c) for c in cfgs], dim=1)


def nfp_similarity(x: torch.Tensor, cfg: NFPConfig) -> torch.Tensor:
    """(B, C, H, W) -> (B, k*k-1, H', W') similarity map; differentiable w.r.t. ``x``."""
    if x.device.type != "cuda":
        if x.device.type == "cpu" and not torch.is_grad_enabled():
            return shape_probe(x, cfg)
        _reject_cpu(x)
    if x.dim() == 4:
        _check_geometry(x.shape[2], x.shape[3], cfg)
    xk, out_dtype, layout = _prepare(x, cfg)
    y = _NFPSimilarity.apply(xk, cfg, out_dtype == torch.float32, layout)
    return y if y.dtype == out_dtype else y.to(out_dtype)


def nfp_gap_pair(x: torch.Tensor, cfg: NFPConfig):
    """``(GAP(x), GAP(NFP(x)))`` -> ((B, C), (B, k*k-1)) in one pass over ``x``."""
    if x.device.type != "cuda":
        _reject_cpu(x)
    if x.dim() == 4:
        _check_geometry(x.shape[2], x.shape[3], cfg)
    xk, out_dtype, layout = _prepare(x, cfg)
    gx, gn = _NFPGapPair.apply(xk, cfg, layout)   # both fp32 (the kernels accumulate in fp32)
    # NFP_Pooling.py:27: avgpool(x) keeps the dtype of x (also under autocast); :31: the similarity map's dtype
    return gx.to(x.dtype), gn.to(out_dtype)


def nfp_pooled_similarity(x: torch.Tensor, cfg: NFPConfig) -> torch.Tensor:
    """``adaptive_avg_pool2d(nfp_similarity(x, cfg), 1).flatten(1)`` -> (B, k*k-1), differentiable w.r.t. ``x``,
    without writing the similarity map: what each stage of the reference's multi-stage head keeps of its map
    (models/texture_pooling.py:249-256).  The result has the map's dtype: float32 under CUDA autocast, else the dtype of
    ``x``; the kernels accumulate in fp32 either way.  Only ``x`` is saved for the backward."""
    if x.device.type != "cuda":
        _reject_cpu(x)
    if x.dim() == 4:
        _check_geometry(x.shape[2], x.shape[3], cfg)
    xk, out_dtype, layout = _prepare(x, cfg)
    gn = _NFPPooledMap.apply(xk, cfg, layout)   # fp32
    return gn if gn.dtype == out_dtype else gn.to(out_dtype)


def describe(x_shape, dtype: torch.dtype, cfg: NFPConfig, op: int = _capi.OP_FORWARD, layout: int = 0) -> str:
    """Name of the kernel path a problem would take (for tests / bench reporting)."""
    B, C, H, W = x_shape
    desc = _capi.make_desc(_KERNEL_DTYPES[dtype], B, C, H, W, cfg.R, cfg.stride, cfg.padding, cfg.dilation,
                           cfg.padding_mode, cfg.measure, cfg.similarity, cfg.difference_taps, cfg.eps,
                           cfg.p, cfg.q_scs, cfg.path, layout=layout)
    return _capi.describe_path(desc, op)


__all__ = ["NFPConfig", "nfp_similarity", "nfp_gap_pair", "nfp_pooled_similarity", "nfp_head", "nfp_multi_radius", "multi_radius_fusable", "shape_probe", "conv_output_size", "describe",
           "replace", "math"]
