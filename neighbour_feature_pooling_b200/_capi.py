"""ctypes binding of libnfp_b200.so (the C ABI in include/nfp_b200.h).

This is the only place the Python host code touches native code.  There is no
CPU or PyTorch fallback: if the library is missing or a call fails, a
RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
import math
import os
import threading

# NFPB200_LIB selects another BUILD of the same native library (kernel A/B experiments: `build.py --variant`)
_LIB_PATH = os.environ.get("NFPB200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib",
                                                          "libnfp_b200.so")

ABI_VERSION = 5

F32, BF16, F16 = 0, 1, 2   # F16 (ABI v5): ring and token kernels only, anything else is NFPB200_EUNSUPPORTED
PAD_MODES = {"zeros": 0, "reflect": 1, "replicate": 2, "circular": 3}
MEASURES = {
    "norm": 0, "cosine": 1, "dot": 2, "rmse": 3, "geman": 4, "attention": 5, "emd": 6,
    "canberra": 7, "hellinger": 8, "chisquared1": 9, "chisquared2": 10, "gfc": 11,
    "pearson": 12, "jeffrey": 13, "squaredchord": 14, "smith": 15, "scs": 16,
    "sharpened_cosine": 16,  # nfp.py:117 accepts both spellings
}
PATHS = {"auto": 0, "generic": 1, "fused": 2, "split": 3}
HINT_X_STABLE = 0x100   # NFPB200_HINT_X_STABLE, OR-ed into Desc.path for the backward entry points
FLAG_Y_F32 = 0x200      # NFPB200_FLAG_Y_F32, OR-ed into Desc.path for nfpb200_forward with bf16 / fp16 x: y is fp32
OP_FORWARD, OP_BACKWARD, OP_POOL_FORWARD, OP_POOL_BACKWARD = 0, 1, 2, 3
OP_POOLED_MAP_FORWARD, OP_POOLED_MAP_BACKWARD = 4, 5   # GAP(NFP(x)) alone (ABI v4)
OP_JVP, OP_BACKWARD_BACKWARD = 7, 8                   # second order of the cosine measure (6 is not an op)
JVP_FORWARD_AD, JVP_REVERSE = 0, 1                    # nfpb200_jvp rule: forward AD / the map nfpb200_backward transposes
LAYOUT_NCHW, LAYOUT_NHWC = 0, 1

EXPORTS = (
    "nfpb200_abi_version", "nfpb200_status_string", "nfpb200_output_shape",
    "nfpb200_workspace_bytes", "nfpb200_describe_path", "nfpb200_launch_count",
    "nfpb200_forward", "nfpb200_backward", "nfpb200_pool_forward", "nfpb200_pool_backward",
    "nfpb200_debug_phase_timing", "nfpb200_head_supported", "nfpb200_head_forward", "nfpb200_head_backward",
    "nfpb200_pooled_map_forward", "nfpb200_pooled_map_backward", "nfpb200_jvp", "nfpb200_backward_backward",
)


class Desc(ctypes.Structure):
    """Mirror of nfpb200_desc_t."""
    _fields_ = [
        ("struct_bytes", ctypes.c_int32), ("dtype", ctypes.c_int32),
        ("B", ctypes.c_int32), ("C", ctypes.c_int32), ("H", ctypes.c_int32), ("W", ctypes.c_int32),
        ("R", ctypes.c_int32), ("stride", ctypes.c_int32), ("padding", ctypes.c_int32),
        ("dilation", ctypes.c_int32), ("padding_mode", ctypes.c_int32), ("measure", ctypes.c_int32),
        ("similarity", ctypes.c_int32), ("difference_taps", ctypes.c_int32),
        ("eps", ctypes.c_float), ("p", ctypes.c_float), ("q_scs", ctypes.c_float),
        ("path", ctypes.c_int32),
        ("layout", ctypes.c_int32), ("inner_R", ctypes.c_int32),
        ("x_batch_stride", ctypes.c_int64), ("gx_batch_stride", ctypes.c_int64),
    ]


_lib = None
_lock = threading.Lock()


def library_path() -> str:
    return _LIB_PATH


def load():
    """Load the shared library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(_LIB_PATH):
            raise RuntimeError(
                f"{_LIB_PATH} is missing: build it with `python -m neighbour_feature_pooling_b200.build` "
                "(or __graft_entry__.build()).  There is no CPU / PyTorch fallback for the NFP operator.")
        lib = ctypes.CDLL(_LIB_PATH)
        vp, i32p, szp = ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_size_t)
        dp = ctypes.POINTER(Desc)
        lib.nfpb200_abi_version.restype = ctypes.c_int
        lib.nfpb200_abi_version.argtypes = []
        lib.nfpb200_status_string.restype = ctypes.c_char_p
        lib.nfpb200_status_string.argtypes = [ctypes.c_int]
        lib.nfpb200_output_shape.restype = ctypes.c_int
        lib.nfpb200_output_shape.argtypes = [dp, i32p, i32p]
        lib.nfpb200_workspace_bytes.restype = ctypes.c_int
        lib.nfpb200_workspace_bytes.argtypes = [dp, ctypes.c_int32, szp]
        lib.nfpb200_describe_path.restype = ctypes.c_int
        lib.nfpb200_describe_path.argtypes = [dp, ctypes.c_int32, ctypes.c_char_p, ctypes.c_size_t]
        lib.nfpb200_launch_count.restype = ctypes.c_int
        lib.nfpb200_launch_count.argtypes = [dp, ctypes.c_int32, i32p]
        lib.nfpb200_forward.restype = ctypes.c_int
        lib.nfpb200_forward.argtypes = [dp, vp, vp, vp, ctypes.c_size_t, vp]
        lib.nfpb200_backward.restype = ctypes.c_int
        lib.nfpb200_backward.argtypes = [dp, vp, vp, vp, vp, ctypes.c_size_t, vp]
        lib.nfpb200_pool_forward.restype = ctypes.c_int
        lib.nfpb200_pool_forward.argtypes = [dp, vp, vp, vp, vp, ctypes.c_size_t, vp]
        lib.nfpb200_pool_backward.restype = ctypes.c_int
        lib.nfpb200_pool_backward.argtypes = [dp, vp, vp, vp, vp, vp, ctypes.c_size_t, vp]
        lib.nfpb200_debug_phase_timing.restype = ctypes.c_int
        lib.nfpb200_debug_phase_timing.argtypes = [vp]
        lib.nfpb200_head_supported.restype = ctypes.c_int
        lib.nfpb200_head_supported.argtypes = [dp]
        lib.nfpb200_head_forward.restype = ctypes.c_int
        lib.nfpb200_head_forward.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp]
        lib.nfpb200_head_backward.restype = ctypes.c_int
        lib.nfpb200_head_backward.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp, vp]
        lib.nfpb200_pooled_map_forward.restype = ctypes.c_int
        lib.nfpb200_pooled_map_forward.argtypes = [dp, vp, vp, vp, ctypes.c_size_t, vp]
        lib.nfpb200_pooled_map_backward.restype = ctypes.c_int
        lib.nfpb200_pooled_map_backward.argtypes = [dp, vp, vp, vp, vp, ctypes.c_size_t, vp]
        lib.nfpb200_jvp.restype = ctypes.c_int
        lib.nfpb200_jvp.argtypes = [dp, vp, vp, vp, ctypes.c_int32, vp, ctypes.c_size_t, vp]
        lib.nfpb200_backward_backward.restype = ctypes.c_int
        lib.nfpb200_backward_backward.argtypes = [dp, vp, vp, vp, vp, vp, ctypes.c_size_t, vp]
        got = lib.nfpb200_abi_version()
        if got != ABI_VERSION:
            raise RuntimeError(f"libnfp_b200.so ABI version {got}, host code expects {ABI_VERSION}; rebuild")
        _lib = lib
    return _lib


def status_string(rc: int) -> str:
    return load().nfpb200_status_string(rc).decode()


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what} failed: {status_string(rc)} (status {rc})")


def make_desc(dtype: int, B: int, C: int, H: int, W: int, R: int, stride: int, padding: int,
              dilation: int, padding_mode: str, measure: str, similarity: bool,
              difference_taps: bool, eps: float, p: float, q_scs: float, path: str = "auto",
              layout: int = 0, x_batch_stride: int = 0, gx_batch_stride: int = 0, inner_R: int = 0) -> Desc:
    d = Desc()
    d.struct_bytes = ctypes.sizeof(Desc)
    d.dtype = dtype
    d.B, d.C, d.H, d.W = B, C, H, W
    d.R, d.stride, d.padding, d.dilation = R, stride, padding, dilation
    d.padding_mode = PAD_MODES[padding_mode]
    d.measure = MEASURES[measure]
    d.similarity = int(bool(similarity))
    d.difference_taps = int(bool(difference_taps))
    d.eps = float(eps)
    d.p = float(p) if not (isinstance(p, str)) else (math.inf if p == "inf" else float(p))
    d.q_scs = float(q_scs)
    d.path = PATHS[path]
    d.layout = layout
    d.inner_R = inner_R   # multi-radius launch: y / gy = [radius inner_R map | radius R map] (0 = off)
    d.x_batch_stride = x_batch_stride
    d.gx_batch_stride = gx_batch_stride
    return d


def output_shape(desc: Desc):
    ho, wo = ctypes.c_int32(), ctypes.c_int32()
    check(load().nfpb200_output_shape(ctypes.byref(desc), ctypes.byref(ho), ctypes.byref(wo)), "nfpb200_output_shape")
    return ho.value, wo.value


def workspace_bytes(desc: Desc, op: int) -> int:
    n = ctypes.c_size_t()
    check(load().nfpb200_workspace_bytes(ctypes.byref(desc), op, ctypes.byref(n)), "nfpb200_workspace_bytes")
    return n.value


def describe_path(desc: Desc, op: int) -> str:
    buf = ctypes.create_string_buffer(128)
    check(load().nfpb200_describe_path(ctypes.byref(desc), op, buf, 128), "nfpb200_describe_path")
    return buf.value.decode()


def launch_count(desc: Desc, op: int) -> int:
    n = ctypes.c_int32()
    check(load().nfpb200_launch_count(ctypes.byref(desc), op, ctypes.byref(n)), "nfpb200_launch_count")
    return n.value
