"""GPU: the ring kernels warm L2 with their inputs before griddepcontrol.wait (cp.async.bulk.prefetch.L2), also while
the preceding grid is still writing those inputs.  The kernels read x and gy only after the wait, through L2, so every
chain below must give the same bits as the same launches with a device synchronize between them, and match the oracle.

Each chain feeds a buffer that the launch immediately before it writes into the next launch; the buffer is filled with
NaN before the chain starts, so a read of stale data would show.  B = 256 (512x7x7: the backward runs one image per
CTA, the forward two CTAs per SM), 60 repeats over rotating buffers, no NFPB200_HINT_X_STABLE."""
import ctypes

import pytest
import torch

from oracle import nfp_oracle as O

from _util import rel_err

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
BF16_TOL = 2e-2
B, C, H, W = 256, 512, 7, 7
K = 8
REPS, NBUF = 60, 3
DTYPES = pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])


def _desc(dtype, c):
    from neighbour_feature_pooling_b200 import _capi
    kd = _capi.F32 if dtype == torch.float32 else _capi.BF16
    d = _capi.make_desc(kd, B, c, H, W, 1, 1, 1, 1, "reflect", "cosine", True, False, 1e-6, 1, 1e-6, "auto")
    assert _capi.describe_path(d, _capi.OP_FORWARD).startswith("fused/stream")
    assert _capi.describe_path(d, _capi.OP_BACKWARD).startswith("fused/stream")
    return d


class _Chain:
    def __init__(self):
        from neighbour_feature_pooling_b200 import _capi
        self.capi, self.lib = _capi, _capi.load()
        self.sync = False

    def _after(self):
        if self.sync:
            torch.cuda.synchronize()

    def fwd(self, d, x, y):
        st = torch.cuda.current_stream().cuda_stream
        self.capi.check(self.lib.nfpb200_forward(ctypes.byref(d), x.data_ptr(), y.data_ptr(), None, 0, st), "forward")
        self._after()

    def bwd(self, d, x, gy, gx):
        st = torch.cuda.current_stream().cuda_stream
        self.capi.check(self.lib.nfpb200_backward(ctypes.byref(d), x.data_ptr(), gy.data_ptr(), gx.data_ptr(), None, 0,
                                                  st), "backward")
        self._after()


def _run_both(step, bufs):
    """step(chain, i) for REPS repeats on buffer set i = rep % NBUF, once chained and once with a synchronize after
    every launch; returns (chained, synchronized) copies of the buffers named in `bufs` at the end."""
    res = []
    for sync in (False, True):
        ch = _Chain()
        ch.sync = sync
        for rep in range(REPS):
            step(ch, rep % NBUF)
        torch.cuda.synchronize()
        res.append({k: [t.float().cpu() for t in bufs[k]] for k in bufs})
    return res


def _randn(gen, dtype, dev, *shape):
    return [torch.randn(*shape, generator=gen).to(dev, dtype) for _ in range(NBUF)]


def _tol(dtype):
    return FP32_TOL if dtype == torch.float32 else BF16_TOL


def _assert_same_finite(chained, synced):
    for k in chained:
        for a, b in zip(chained[k], synced[k]):
            assert torch.isfinite(a).all(), k
            assert torch.equal(a, b), k


@DTYPES
def test_stacked_chain_conservative(dtype, cuda_device):
    """A.fwd -> B.fwd -> B.bwd with x_B = y_A: B's forward and backward prefetch y_A while A (resp. B.fwd) runs."""
    gen = torch.Generator().manual_seed(41)
    dA, dB = _desc(dtype, C), _desc(dtype, K)
    xa = _randn(gen, dtype, cuda_device, B, C, H, W)
    gyb = _randn(gen, dtype, cuda_device, B, K, H, W)
    ya = [torch.zeros(B, K, H, W, device=cuda_device, dtype=dtype) for _ in range(NBUF)]
    yb = [torch.zeros(B, K, H, W, device=cuda_device, dtype=dtype) for _ in range(NBUF)]
    gxb = [torch.zeros(B, K, H, W, device=cuda_device, dtype=dtype) for _ in range(NBUF)]

    def step(ch, i):
        ya[i].fill_(float("nan"))
        ch.fwd(dA, xa[i], ya[i])
        ch.fwd(dB, ya[i], yb[i])
        ch.bwd(dB, ya[i], gyb[i], gxb[i])

    chained, synced = _run_both(step, {"ya": ya, "yb": yb, "gxb": gxb})
    _assert_same_finite(chained, synced)
    i = (REPS - 1) % NBUF
    x_b = chained["ya"][i][-2:].double()
    y_ref, gx_ref = O.nfp_forward_backward(x_b, gyb[i][-2:].double().cpu(), R=1, measure="cosine", padding=1)
    assert rel_err(chained["yb"][i][-2:], y_ref) < _tol(dtype)
    assert rel_err(chained["gxb"][i][-2:], gx_ref) < _tol(dtype)


@DTYPES
def test_backward_of_gradient_just_written(dtype, cuda_device):
    """A.fwd -> bwd with gy = y_A, the (256, 8, 7, 7) map the forward has just written: the backward prefetches it."""
    gen = torch.Generator().manual_seed(43)
    d = _desc(dtype, C)
    xa = _randn(gen, dtype, cuda_device, B, C, H, W)
    xb = _randn(gen, dtype, cuda_device, B, C, H, W)
    ya = [torch.zeros(B, K, H, W, device=cuda_device, dtype=dtype) for _ in range(NBUF)]
    gx = [torch.zeros(B, C, H, W, device=cuda_device, dtype=dtype) for _ in range(NBUF)]

    def step(ch, i):
        ya[i].fill_(float("nan"))
        ch.fwd(d, xa[i], ya[i])
        ch.bwd(d, xb[i], ya[i], gx[i])

    chained, synced = _run_both(step, {"ya": ya, "gx": gx})
    _assert_same_finite(chained, synced)
    i = (REPS - 1) % NBUF
    _, gx_ref = O.nfp_forward_backward(xb[i][-2:].double().cpu(), chained["ya"][i][-2:].double(), R=1,
                                       measure="cosine", padding=1)
    assert rel_err(chained["gx"][i][-2:], gx_ref) < _tol(dtype)


@DTYPES
def test_forward_of_gradient_just_written(dtype, cuda_device):
    """bwd -> fwd with x = gx, the input gradient the backward has just written: the forward prefetches it."""
    gen = torch.Generator().manual_seed(47)
    d = _desc(dtype, C)
    xa = _randn(gen, dtype, cuda_device, B, C, H, W)
    gy = _randn(gen, dtype, cuda_device, B, K, H, W)
    gx = [torch.zeros(B, C, H, W, device=cuda_device, dtype=dtype) for _ in range(NBUF)]
    y = [torch.zeros(B, K, H, W, device=cuda_device, dtype=dtype) for _ in range(NBUF)]

    def step(ch, i):
        gx[i].fill_(float("nan"))
        ch.bwd(d, xa[i], gy[i], gx[i])
        ch.fwd(d, gx[i], y[i])

    chained, synced = _run_both(step, {"gx": gx, "y": y})
    _assert_same_finite(chained, synced)
    i = (REPS - 1) % NBUF
    y_ref = O.nfp_forward(chained["gx"][i][-2:].double(), R=1, measure="cosine", padding=1)
    assert rel_err(chained["y"][i][-2:], y_ref) < _tol(dtype)
