"""GPU: the C ABI's memory and stream contract on every kernel path.

The parity suites check each kernel's arithmetic on buffers from PyTorch's caching allocator (512-byte aligned bases,
sizes rounded up, neighbours full of finite data), on the current stream, eagerly.  Here the test owns every pointer:

* guarded buffers (tests/_util.py, Guarded): every tensor sits at the weakest alignment include/nfp_b200.h allows
  (16 bytes, or 4 for the fp32 vectors) inside 256 KiB guards.  Input guards hold quiet NaN, output bodies and guards
  and the workspace a NaN sentinel.  After each call: every guard and every input byte is unchanged, no output element
  still holds the sentinel, the outputs are bit-identical to the same call on plain torch allocations, and again with
  a zero-filled workspace; the plain call matches the fp64 oracle on its first and last image;
* channels-last batch strides: x with padded and ViT-token strides (gaps NaN), gx with padded strides (gaps must keep
  the sentinel);
* CUDA graphs: each call captured alone has exactly nfpb200_launch_count kernel / memset nodes and replays to the
  eager bits; autograd forward + backward captured in global mode replays to the eager bits;
* streams: a call handed a side stream puts every launch on it (a NaN-then-spin-then-data sequence on that stream
  poisons any launch that runs elsewhere), and the autograd API honours torch.cuda.stream;
* a fresh process whose first launches of each family happen inside a capture, and one whose first launches happen
  on two host threads at once.

tests/test_abi_contract_host.py checks on the CPU that the guard checker flags what it should, that this grid reaches
every (family, entry point) cell, and that every pointer below its documented alignment is refused.
"""
import ctypes
import os
import subprocess
import sys
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch

from neighbour_feature_pooling_b200 import _capi
from oracle import nfp_oracle as O

from _util import SENTINEL, Guarded, bits, fill_bits, guard_problems, rel_err

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 1e-6
ENTRIES = ("forward", "backward", "pool_forward", "pool_backward", "pooled_map_forward", "pooled_map_backward",
           "head_forward", "head_backward")
OP_OF = {"forward": _capi.OP_FORWARD, "backward": _capi.OP_BACKWARD, "pool_forward": _capi.OP_POOL_FORWARD,
         "pool_backward": _capi.OP_POOL_BACKWARD, "pooled_map_forward": _capi.OP_POOLED_MAP_FORWARD,
         "pooled_map_backward": _capi.OP_POOLED_MAP_BACKWARD, "head_forward": _capi.OP_POOL_FORWARD,
         "head_backward": _capi.OP_POOL_BACKWARD}
# family -> (describe_path prefix, cfg.path, layout)
FAMILIES = {
    "stream": ("fused/stream_", "auto", _capi.LAYOUT_NCHW),
    "split": ("fused/split_", "split", _capi.LAYOUT_NCHW),
    "band": ("planar/band", "auto", _capi.LAYOUT_NCHW),
    "table": ("planar/table", "auto", _capi.LAYOUT_NCHW),
    "token": ("fused/token_", "auto", _capi.LAYOUT_NHWC),
    "generic": ("generic/pairs", "auto", _capi.LAYOUT_NCHW),
}
F32, BF16 = torch.float32, torch.bfloat16
# fp32 vectors (4-byte alignment); every other pointer is placed 16 bytes past a 512-byte boundary
F32_VECTORS = ("gap_x", "gap_nfp", "g_gap_x", "g_gap_nfp", "out", "g_out", "proj_b")

Cell = namedtuple("Cell", "family entry shape dtype opts")


def _cell(family, entry, shape, dtype, **opts):
    return Cell(family, entry, shape, dtype, tuple(sorted(opts.items())))


# ---- the grid ------------------------------------------------------------------------------------------------------
STREAM_INST = [(3, 64, 7, 7, 1), (3, 64, 7, 7, 2), (2, 64, 14, 14, 1), (2, 32, 14, 14, 2), (4, 64, 2, 2, 1),
               (3, 64, 4, 4, 1)]   # the six NFP_STREAM_SHAPES instantiations
GENERIC = [dict(measure="cosine", stride=2, dilation=2, padding=2, mode="circular"), dict(measure="attention"),
           dict(measure="scs")]


def _grid():
    g = []
    for s in STREAM_INST:
        for dt in (F32, BF16):
            g += [_cell("stream", e, s, dt) for e in ENTRIES]
    for s in [(3, 64, 7, 7, 1), (2, 64, 14, 14, 1)]:
        for dt in (F32, BF16):
            g += [_cell("stream", "backward", s, dt, hint=1)]
            g += [_cell("split", e, s, dt) for e in ENTRIES[:6]]
    g += [_cell("stream", "forward", s, BF16, yf32=1) for s in [(3, 64, 7, 7, 1), (2, 32, 14, 14, 2)]]
    g += [_cell("stream", "backward", (3, 40, 7, 7, 1), dt) for dt in (F32, BF16)]      # strip form (C % 64 != 0)
    g += [_cell("stream", e, (300, 512, 7, 7, 1), F32) for e in ("forward", "backward")]  # persistent, resident image
    for s in [(3, 64, 7, 7, 2), (2, 32, 14, 14, 2)]:
        g += [_cell("stream", e, s, dt, inner=1) for e in ("forward", "backward") for dt in (F32, BF16)]
    band_ops = ("forward", "backward", "pooled_map_forward", "pooled_map_backward")
    for s in [(2, 8, 21, 16, 1), (2, 16, 112, 112, 1)]:    # H = 21: the last band is partial
        g += [_cell("band", e, s, dt) for e in band_ops for dt in (F32, BF16)]
    g += [_cell("band", e, (2, 16, 28, 28, 2), dt, inner=1) for e in ("forward", "backward") for dt in (F32, BF16)]
    g += [_cell("table", e, s, dt) for e in ("forward", "backward")
          for s, dt in [((2, 5, 3, 3, 1), F32), ((2, 10, 5, 9, 2), BF16)]]
    # channels-last token kernels: every entry with each x batch stride, each gx batch stride on the backward entries
    vit = (3, 64, 14, 14, 1)
    for e in ENTRIES:
        bwd = e.endswith("backward")
        for i, xbs in enumerate(("dense", "pad8", "vit")):
            g.append(_cell("token", e, vit, BF16, xbs=xbs, gxbs=("0", "pad8", "pad64")[i] if bwd else "0"))
    g += [_cell("token", "backward", vit, BF16, xbs=x, gxbs=gx) for x in ("dense", "pad8", "vit")
          for gx in ("0", "pad8", "pad64") if (x, gx) not in (("dense", "0"), ("pad8", "pad8"), ("vit", "pad64"))]
    g += [_cell("token", e, (2, 192, 7, 7, 1), BF16, xbs="pad8", gxbs="pad64") for e in ENTRIES]
    g += [_cell("token", e, (2, 512, 7, 7, 1), BF16) for e in ("forward", "backward")]
    g += [_cell("token", e, (3, 64, 7, 7, 2), BF16, inner=1, xbs="pad8", gxbs="pad8") for e in ("forward", "backward")]
    for o in GENERIC:
        g += [_cell("generic", e, (3, 5, 9, 11, 1), dt, **o) for e in ENTRIES[:6] for dt in (F32, BF16)]
    return g


GRID = _grid()


def cell_id(c):
    o = dict(c.opts)
    extra = "".join(f"-{k}{v}" for k, v in sorted(o.items()))
    return (f'{c.family}-{c.entry}-{"x".join(map(str, c.shape[:4]))}_r{c.shape[4]}-'
            f'{"fp32" if c.dtype == F32 else "bf16"}{extra}')


# ---- one ABI call ---------------------------------------------------------------------------------------------------
class Problem:
    """The buffers and the ABI call of one grid cell.  Flat host data; `run` places them in any allocation."""

    def __init__(self, c):
        self.c = c
        o = dict(c.opts)
        B, C, H, W, R = c.shape
        self.B, self.C, self.H, self.W, self.R = c.shape
        self.measure = o.get("measure", "cosine")
        self.stride, self.dil = o.get("stride", 1), o.get("dilation", 1)
        self.pad, self.mode = o.get("padding", R), o.get("mode", "reflect")
        self.inner = o.get("inner", 0)
        self.nhwc = FAMILIES[c.family][2] == _capi.LAYOUT_NHWC
        dense = H * W * C
        self.lead = C if o.get("xbs") == "vit" else 0   # the ViT token view: x starts one (class) token in
        self.xbs = {None: 0, "dense": 0, "pad8": dense + 8, "vit": 197 * C}[o.get("xbs")]
        self.gxbs = {"0": 0, "pad8": dense + 8, "pad64": dense + 64}[o.get("gxbs", "0")]
        kd = _capi.F32 if c.dtype == F32 else _capi.BF16
        self.desc = _capi.make_desc(kd, B, C, H, W, R, self.stride, self.pad, self.dil, self.mode, self.measure, True,
                                    False, EPS, 1, 1e-6, FAMILIES[c.family][1], layout=FAMILIES[c.family][2],
                                    x_batch_stride=self.xbs, gx_batch_stride=self.gxbs, inner_R=self.inner)
        if o.get("hint"):
            self.desc.path |= _capi.HINT_X_STABLE
        self.yf32 = bool(o.get("yf32"))
        if self.yf32:
            self.desc.path |= _capi.FLAG_Y_F32
        self.Ho, self.Wo = _capi.output_shape(self.desc)
        self.K = (2 * R + 1) ** 2 - 1
        self.Ky = self.K + ((2 * self.inner + 1) ** 2 - 1 if self.inner else 0)
        self.op = OP_OF[c.entry]
        self.head = c.entry.startswith("head")
        self._make_data()

    # -- host data --
    def _make_data(self):
        c, B, C, H, W, K = self.c, self.B, self.C, self.H, self.W, self.K
        gen = torch.Generator().manual_seed(zlib.crc32(cell_id(c).encode()))
        x = torch.randn(B, C, H, W, generator=gen)
        self.x = x.to(c.dtype).double()   # what the kernels see
        e = c.entry
        self.inputs = {"x": (self._x_flat(), c.dtype)}
        self.outputs = {}
        if e == "forward":
            self.outputs["y"] = (B * self.Ky * self.Ho * self.Wo, F32 if self.yf32 else c.dtype, None)
        if e == "backward":
            self.gy = torch.randn(B, self.Ky, self.Ho, self.Wo, generator=gen).to(c.dtype).double()
            self.inputs["gy"] = (self.gy.reshape(-1), c.dtype)
        if e == "pool_backward":
            self.g_gap_x = torch.randn(B, C, generator=gen).double()
            self.inputs["g_gap_x"] = (self.g_gap_x.reshape(-1), F32)
        if e in ("pool_backward", "pooled_map_backward"):
            self.g_gap_nfp = torch.randn(B, K, generator=gen).double()
            self.inputs["g_gap_nfp"] = (self.g_gap_nfp.reshape(-1), F32)
        if e == "pool_forward":
            self.outputs["gap_x"] = (B * C, F32, None)
        if e in ("pool_forward", "pooled_map_forward"):
            self.outputs["gap_nfp"] = (B * K, F32, None)
        if self.head:
            self.proj_w = (0.1 * torch.randn(C, K, generator=gen)).double()
            self.proj_b = torch.randn(C, generator=gen).double()
            self.inputs["proj_w"] = (self.proj_w.reshape(-1), F32)
            self.inputs["proj_b"] = (self.proj_b.reshape(-1), F32)
        if e == "head_forward":
            for n, sz in (("out", B * C), ("gap_x", B * C), ("gap_nfp", B * K)):
                self.outputs[n] = (sz, F32, None)
        if e == "head_backward":   # the forward's results, as fp32
            self.gap_x_in = self.x.mean((2, 3)).float().double()
            self.gap_nfp_in = self._map(self.x).mean((2, 3)).float().double()
            self.g_out = torch.randn(B, C, generator=gen).double()
            self.inputs["gap_x"] = (self.gap_x_in.reshape(-1), F32)
            self.inputs["gap_nfp"] = (self.gap_nfp_in.reshape(-1), F32)
            self.inputs["g_out"] = (self.g_out.reshape(-1), F32)
        if e.endswith("backward"):
            n, mask = self._gx_extent()
            self.outputs["gx"] = (n, c.dtype, mask)

    def _x_flat(self):
        B, C, H, W = self.x.shape
        if not self.nhwc:
            return self.x.reshape(-1)
        dense = H * W * C
        s = self.xbs or dense
        flat = torch.full((self.lead + (B - 1) * s + dense,), float("nan"), dtype=torch.float64)
        img = self.x.permute(0, 2, 3, 1).reshape(B, dense)
        for b in range(B):
            flat[self.lead + b * s:self.lead + b * s + dense] = img[b]
        return flat

    def _gx_extent(self):
        B, C, H, W = self.B, self.C, self.H, self.W
        if not self.nhwc or not self.gxbs:
            return B * C * H * W, None
        dense = H * W * C
        n = (B - 1) * self.gxbs + dense
        mask = torch.zeros(n, dtype=torch.bool)
        for b in range(B):
            mask[b * self.gxbs:b * self.gxbs + dense] = True
        return n, mask

    def logical(self, name, flat):
        """A flat output as float64 in its logical shape ((B, C, H, W) for gx)."""
        t = flat.detach().cpu().double()
        B, C, H, W = self.B, self.C, self.H, self.W
        if name == "y":
            return t.view(B, self.Ky, self.Ho, self.Wo)
        if name == "gx":
            if not self.nhwc:
                return t.view(B, C, H, W)
            s = self.gxbs or H * W * C
            return torch.stack([t[b * s:b * s + H * W * C] for b in range(B)]).view(B, H, W, C).permute(0, 3, 1, 2)
        return t.view(B, -1)

    # -- fp64 oracle --
    def _kw(self, R=None, padding=None):
        return dict(R=R or self.R, measure=self.measure, stride=self.stride, padding=self.pad if padding is None
                    else padding, dilation=self.dil, padding_mode=self.mode, similarity=True, eps=EPS)

    def _map(self, x):
        return torch.as_tensor(np.asarray(O.nfp_forward(x, **self._kw())))

    def _map_grad(self, x, gy):
        y, gx = O.nfp_forward_backward(x, gy, **self._kw())
        return torch.as_tensor(np.asarray(y)), torch.as_tensor(np.asarray(gx))

    def expected(self):
        """{output name: fp64 expectation} of the images the oracle scores, and those images."""
        x, e, B = self.x, self.c.entry, self.B
        rows = list(range(B)) if B <= 8 else [0, B - 1]
        if self.measure == "scs":     # batch-coupled: the oracle needs every image
            rows = list(range(B))
        xr = x[rows]
        HoWo, HW = self.Ho * self.Wo, self.H * self.W
        if self.inner:
            kw = dict(measure="cosine", padding_mode=self.mode, similarity=True)
            gy = self.gy[rows] if e == "backward" else torch.zeros(len(rows), self.Ky, self.H, self.W,
                                                                  dtype=torch.float64)
            ki = self.Ky - self.K
            y1, g1 = O.nfp_forward_backward(xr, gy[:, :ki].contiguous(), R=self.inner, padding=self.inner, **kw)
            y2, g2 = O.nfp_forward_backward(xr, gy[:, ki:].contiguous(), R=self.R, padding=self.R, **kw)
            if e == "forward":
                return {"y": torch.cat([torch.as_tensor(np.asarray(y1)), torch.as_tensor(np.asarray(y2))], 1)}, rows
            return {"gx": torch.as_tensor(np.asarray(g1)) + torch.as_tensor(np.asarray(g2))}, rows
        if e == "forward":
            return {"y": self._map(xr)}, rows
        if e == "backward":
            return {"gx": self._map_grad(xr, self.gy[rows])[1]}, rows
        if e in ("pool_forward", "pooled_map_forward"):
            out = {"gap_nfp": self._map(xr).mean((2, 3))}
            if e == "pool_forward":
                out["gap_x"] = xr.mean((2, 3))
            return out, rows
        if e in ("pool_backward", "pooled_map_backward"):
            gy = (self.g_gap_nfp[rows] / HoWo)[:, :, None, None].expand(len(rows), self.K, self.Ho, self.Wo)
            gx = self._map_grad(xr, gy.contiguous())[1]
            if e == "pool_backward":
                gx = gx + (self.g_gap_x[rows] / HW)[:, :, None, None]
            return {"gx": gx}, rows
        if e == "head_forward":
            gap_x, gap_n = xr.mean((2, 3)), self._map(xr).mean((2, 3))
            return {"gap_x": gap_x, "gap_nfp": gap_n, "out": gap_x * (gap_n @ self.proj_w.t() + self.proj_b)}, rows
        # head backward: d/dx of <g_out, gap_x * (W gap_nfp + b)> with gap_x / gap_nfp read back from the forward
        g, gx_, gn = self.g_out[rows], self.gap_x_in[rows], self.gap_nfp_in[rows]
        g1 = g * (gn @ self.proj_w.t() + self.proj_b)
        g2 = (g * gx_) @ self.proj_w
        gy = (g2 / HoWo)[:, :, None, None].expand(len(rows), self.K, self.Ho, self.Wo)
        return {"gx": self._map_grad(xr, gy.contiguous())[1] + (g1 / HW)[:, :, None, None]}, rows

    # -- the call --
    def call(self, p, ws, ws_n, stream):
        lib, d, e = _capi.load(), ctypes.byref(self.desc), self.c.entry
        if e == "forward":
            return lib.nfpb200_forward(d, p["x"], p["y"], ws, ws_n, stream)
        if e == "backward":
            return lib.nfpb200_backward(d, p["x"], p["gy"], p["gx"], ws, ws_n, stream)
        if e == "pool_forward":
            return lib.nfpb200_pool_forward(d, p["x"], p["gap_x"], p["gap_nfp"], ws, ws_n, stream)
        if e == "pool_backward":
            return lib.nfpb200_pool_backward(d, p["x"], p["g_gap_x"], p["g_gap_nfp"], p["gx"], ws, ws_n, stream)
        if e == "pooled_map_forward":
            return lib.nfpb200_pooled_map_forward(d, p["x"], p["gap_nfp"], ws, ws_n, stream)
        if e == "pooled_map_backward":
            return lib.nfpb200_pooled_map_backward(d, p["x"], p["g_gap_nfp"], p["gx"], ws, ws_n, stream)
        if e == "head_forward":
            return lib.nfpb200_head_forward(d, p["x"], p["proj_w"], p["proj_b"], p["out"], p["gap_x"], p["gap_nfp"],
                                            stream)
        return lib.nfpb200_head_backward(d, p["x"], p["proj_w"], p["proj_b"], p["gap_x"], p["gap_nfp"], p["g_out"],
                                         p["gx"], stream)

    def workspace_bytes(self):
        return 0 if self.head else _capi.workspace_bytes(self.desc, self.op)

    def launch_count(self):
        return 1 if self.head else _capi.launch_count(self.desc, self.op)

    def path(self):
        return _capi.describe_path(self.desc, self.op)

    def plain(self, dev):
        """Inputs on plain torch allocations, outputs torch.empty, a fresh workspace: {name: tensor}, ws tensor."""
        bufs = {n: d.to(dev, dt) for n, (d, dt) in self.inputs.items()}
        bufs.update({n: torch.empty(sz, dtype=dt, device=dev) for n, (sz, dt, _) in self.outputs.items()})
        n = self.workspace_bytes()
        return bufs, (torch.empty(n, dtype=torch.uint8, device=dev) if n else None)

    def guarded(self, dev, zero_ws=False):
        bufs = {n: Guarded(d.numel(), dt, dev, "input", data=d, place=4 if n in F32_VECTORS else 16)
                for n, (d, dt) in self.inputs.items()}
        bufs.update({n: Guarded(sz, dt, dev, "output", place=4 if n in F32_VECTORS else 16, written=m)
                     for n, (sz, dt, m) in self.outputs.items()})
        n = self.workspace_bytes()
        ws = Guarded(n, torch.uint8, dev, "workspace") if n else None
        if ws is not None and zero_ws:
            ws.body.zero_()
            ws.snapshot = ws.raw.clone()
        return bufs, ws


def _ptrs(prob, bufs):
    p = {n: (b.ptr() if isinstance(b, Guarded) else b.data_ptr()) for n, b in bufs.items()}
    # the ViT token view: the buffer starts at the class token (NaN), x one token further in
    p["x"] += prob.lead * torch.empty(0, dtype=prob.c.dtype).element_size()
    return p


def _run(prob, bufs, ws, stream=None):
    s = torch.cuda.current_stream().cuda_stream if stream is None else stream
    wp = None if ws is None else (ws.ptr() if isinstance(ws, Guarded) else ws.data_ptr())
    wn = 0 if ws is None else prob.workspace_bytes()
    rc = prob.call(_ptrs(prob, bufs), wp, wn, s)
    assert rc == 0, _capi.status_string(rc)


def _out_bits(prob, bufs):
    """{output: bits of its written elements} on the host."""
    out = {}
    for n, (_, _, mask) in prob.outputs.items():
        t = bufs[n].body if isinstance(bufs[n], Guarded) else bufs[n]
        t = bits(t).cpu()
        out[n] = t[mask] if mask is not None else t
    return out


def _same_bits(a, b):
    return {n: bool(torch.equal(a[n], b[n])) for n in a}


# ---- libcuda: stream flags and graph nodes --------------------------------------------------------------------------
_cu = None


def libcuda():
    global _cu
    if _cu is None:
        _cu = ctypes.CDLL("libcuda.so.1")
        _cu.cuStreamGetFlags.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint)]
        _cu.cuGraphGetNodes.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t)]
        _cu.cuGraphNodeGetType.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int)]
    return _cu


CU_GRAPH_NODE_TYPE_KERNEL, CU_GRAPH_NODE_TYPE_MEMSET = 0, 2


def graph_node_counts(graph):
    """{node type: count} of a captured torch.cuda.CUDAGraph(keep_graph=True)."""
    cu, g = libcuda(), ctypes.c_void_p(graph.raw_cuda_graph())
    n = ctypes.c_size_t(0)
    assert cu.cuGraphGetNodes(g, None, ctypes.byref(n)) == 0
    nodes = (ctypes.c_void_p * n.value)()
    assert cu.cuGraphGetNodes(g, nodes, ctypes.byref(n)) == 0
    counts = {}
    for i in range(n.value):
        t = ctypes.c_int()
        assert cu.cuGraphNodeGetType(ctypes.c_void_p(nodes[i]), ctypes.byref(t)) == 0
        counts[t.value] = counts.get(t.value, 0) + 1
    return counts


# ---- §1-§3, §5: guard bands, oracle, graph capture of each cell ---------------------------------------------------
TOL = {("cosine", F32): 1e-5, ("cosine", BF16): 2e-2, ("other", F32): 1e-4, ("other", BF16): 5e-2}


@pytest.mark.parametrize("c", [pytest.param(c, id=cell_id(c)) for c in GRID])
def test_guarded_call(c, cuda_device):
    prob = Problem(c)
    assert prob.path().startswith(FAMILIES[c.family][0]), prob.path()
    # plain allocations: the oracle, and the bits every other run must reproduce
    pb, pws = prob.plain(cuda_device)
    _run(prob, pb, pws)
    torch.cuda.synchronize()
    want = _out_bits(prob, pb)
    exp, rows = prob.expected()
    tol = TOL[("cosine" if prob.measure == "cosine" else "other", c.dtype)]
    for n, ref in exp.items():
        got = prob.logical(n, pb[n])[rows]
        for i in dict.fromkeys((0, len(rows) - 1)):   # first and last image, each on its own scale
            assert rel_err(got[i], ref[i]) < tol, (n, rows[i], rel_err(got[i], ref[i]))
    # guarded buffers at the weakest alignment, sentinel workspace, then zero workspace
    for zero_ws in (False, True):
        gb, gws = prob.guarded(cuda_device, zero_ws)
        _run(prob, gb, gws)
        torch.cuda.synchronize()
        problems = guard_problems({**gb, "workspace": gws})
        assert not problems, problems
        same = _same_bits(_out_bits(prob, gb), want)
        assert all(same.values()), ("zero workspace" if zero_ws else "sentinel workspace", same)
    # one call captured alone: exactly nfpb200_launch_count kernel / memset nodes, and the replay reproduces the bits
    for n in prob.outputs:
        fill_bits(pb[n], SENTINEL[pb[n].dtype])
    graph = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.graph(graph):
        _run(prob, pb, pws, torch.cuda.current_stream().cuda_stream)
    counts = graph_node_counts(graph)
    launches = counts.get(CU_GRAPH_NODE_TYPE_KERNEL, 0) + counts.get(CU_GRAPH_NODE_TYPE_MEMSET, 0)
    assert launches == prob.launch_count() and sum(counts.values()) == launches, (counts, prob.launch_count())
    graph.instantiate()
    graph.replay()
    torch.cuda.synchronize()
    same = _same_bits(_out_bits(prob, pb), want)
    assert all(same.values()), ("graph replay", same)


# ---- §4: streams ----------------------------------------------------------------------------------------------------
def _one_per_family_entry():
    seen, out = set(), []
    for c in GRID:
        o = dict(c.opts)
        plain = o.get("gxbs", "0") == "0" and o.get("xbs", "dense") == "dense" and not {"hint", "yf32", "inner"} & set(o)
        if (c.family, c.entry) in seen or not plain:
            continue
        seen.add((c.family, c.entry))
        out.append(c)
    return out


STREAM_CELLS = _one_per_family_entry()
SPIN_CYCLES = 20_000_000   # ~10 ms at B200 clocks: far longer than any of these calls


def _is_nonblocking(stream):
    flags = ctypes.c_uint(0)
    assert libcuda().cuStreamGetFlags(ctypes.c_void_p(stream.cuda_stream), ctypes.byref(flags)) == 0
    return bool(flags.value & 1)   # CU_STREAM_NON_BLOCKING


def _side_stream_bits(prob, dev, s, handle):
    """On side stream s: x := NaN, spin, x := data, poison outputs; the call on `handle`; copy the outputs out on s."""
    bufs, ws = prob.plain(dev)
    real = {n: bufs[n].clone() for n in prob.inputs}
    for n in prob.inputs:
        bufs[n].fill_(float("nan"))
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for n in prob.inputs:
            bufs[n].fill_(float("nan"))
        torch.cuda._sleep(SPIN_CYCLES)
        for n in prob.inputs:
            bufs[n].copy_(real[n])
        for n in prob.outputs:
            bufs[n].fill_(-1.0)
    _run(prob, bufs, ws, handle)
    with torch.cuda.stream(s):
        copies = {n: bufs[n].clone() for n in prob.outputs}
    s.synchronize()
    out = _out_bits(prob, copies)
    torch.cuda.synchronize()   # (the legacy-stream self-test) nothing left running
    return out


@pytest.mark.parametrize("c", [pytest.param(c, id=cell_id(c)) for c in STREAM_CELLS])
def test_side_stream(c, cuda_device):
    prob = Problem(c)
    pb, pws = prob.plain(cuda_device)
    _run(prob, pb, pws)
    torch.cuda.synchronize()
    want = _out_bits(prob, pb)
    s = torch.cuda.Stream()
    assert _is_nonblocking(s)
    same = _same_bits(_side_stream_bits(prob, cuda_device, s, s.cuda_stream), want)
    assert all(same.values()), same


def test_side_stream_check_can_fail(cuda_device):
    """The same sequence handed the legacy default stream instead of s: the launches run during the spin and read NaN."""
    prob = Problem(_cell("stream", "forward", (3, 64, 7, 7, 1), F32))
    pb, pws = prob.plain(cuda_device)
    _run(prob, pb, pws)
    torch.cuda.synchronize()
    want = _out_bits(prob, pb)
    s = torch.cuda.Stream()
    assert _is_nonblocking(s)
    same = _same_bits(_side_stream_bits(prob, cuda_device, s, 0), want)
    assert not all(same.values())


# ---- autograd ops: side stream, warm graph capture, second device ---------------------------------------------------
def _autograd_ops():
    import neighbour_feature_pooling_b200 as nfpb
    from neighbour_feature_pooling_b200 import NFPPooling, functional as NF

    def cfg(C, R=1, path="auto", **kw):
        return NF.replace(NFPPooling(C, R=R, measure=kw.pop("measure", "cosine"), padding=kw.pop("padding", R),
                                     **kw).config, path=path)

    def head(C, R=1):
        gen = torch.Generator().manual_seed(C + R)
        w, b = 0.1 * torch.randn(C, (2 * R + 1) ** 2 - 1, generator=gen), torch.randn(C, generator=gen)
        params = {}   # per device, made on the first (eager) call: nothing is copied from the host under capture

        def f(x):
            if x.device not in params:
                params[x.device] = (w.to(x.device), b.to(x.device))
            return NF.nfp_head(x, *params[x.device], cfg(C, R))
        return f

    def multi(C):
        blocks = {}

        def f(x):
            if x.device not in blocks:
                blocks[x.device] = nfpb.MultiRadiusNFP(C).to(x.device)
            return blocks[x.device](x)
        return f

    cl = torch.channels_last
    return {   # name -> (fn, shape (B, C, H, W), dtype, memory format)
        "map-stream": (lambda x: NF.nfp_similarity(x, cfg(64)), (3, 64, 7, 7), F32, None),
        "map-split": (lambda x: NF.nfp_similarity(x, cfg(64, path="split")), (2, 64, 14, 14), F32, None),
        "map-band": (lambda x: NF.nfp_similarity(x, cfg(8)), (2, 8, 21, 16), BF16, None),
        "map-table": (lambda x: NF.nfp_similarity(x, cfg(5)), (2, 5, 3, 3), F32, None),
        "map-token": (lambda x: NF.nfp_similarity(x, cfg(64)), (3, 64, 14, 14), BF16, cl),
        "map-generic": (lambda x: NF.nfp_similarity(x, cfg(5, measure="attention")), (3, 5, 9, 11), F32, None),
        "pool-stream": (lambda x: NF.nfp_gap_pair(x, cfg(64)), (3, 64, 7, 7), BF16, None),
        "pool-token": (lambda x: NF.nfp_gap_pair(x, cfg(64)), (3, 64, 7, 7), BF16, cl),
        "pool-generic": (lambda x: NF.nfp_gap_pair(x, cfg(5, measure="scs")), (3, 5, 9, 11), F32, None),
        "pooled-stream": (lambda x: NF.nfp_pooled_similarity(x, cfg(64)), (3, 64, 7, 7), F32, None),
        "pooled-band": (lambda x: NF.nfp_pooled_similarity(x, cfg(16)), (2, 16, 28, 28), F32, None),
        "pooled-token": (lambda x: NF.nfp_pooled_similarity(x, cfg(64)), (3, 64, 14, 14), BF16, cl),
        "pooled-generic": (lambda x: NF.nfp_pooled_similarity(x, cfg(5, stride=2, dilation=2, padding=2,
                                                                     padding_mode="circular")),
                           (3, 5, 9, 11), BF16, None),
        "head-stream": (head(64), (3, 64, 7, 7), F32, None),
        "head-token": (head(64), (3, 64, 7, 7), BF16, cl),
        "multi-stream": (multi(64), (3, 64, 7, 7), F32, None),
        "multi-band": (multi(16), (2, 16, 28, 28), BF16, None),
        "multi-token": (multi(64), (3, 64, 7, 7), BF16, cl),
    }


AUTOGRAD_OPS = list(_autograd_ops())


def _ag_input(name, dev, seed):
    fn, shape, dt, fmt = _autograd_ops()[name]
    x = torch.randn(*shape, generator=torch.Generator().manual_seed(seed)).to(dev, dt)
    return x.contiguous(memory_format=fmt) if fmt is not None else x


def _ag_step(fn, x):
    """Forward and backward; the loss weights every output element differently."""
    xl = x.detach().clone().requires_grad_(True)
    out = fn(xl)
    outs = out if isinstance(out, tuple) else (out,)
    loss = sum((o.float() * torch.linspace(-1, 1, o.numel(), device=o.device).view(o.shape)).sum() for o in outs)
    (gx,) = torch.autograd.grad(loss, xl)
    return [o.detach() for o in outs] + [gx]


def _ag_bits(ts):
    return [bits(t).cpu() for t in ts]


def _eq(a, b):
    return all(torch.equal(u, v) for u, v in zip(a, b)) and len(a) == len(b)


@pytest.mark.parametrize("name", AUTOGRAD_OPS)
def test_autograd_side_stream_and_graph(name, cuda_device):
    fn = _autograd_ops()[name][0]
    x1, x2 = _ag_input(name, cuda_device, 1), _ag_input(name, cuda_device, 2)
    eager1, eager2 = _ag_bits(_ag_step(fn, x1)), _ag_bits(_ag_step(fn, x2))
    # under torch.cuda.stream(s)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = _ag_step(fn, x1)
    s.synchronize()
    assert _eq(_ag_bits(got), eager1)
    # warm up on a side stream, capture forward + backward in global capture mode, replay with two inputs
    xs = x1.clone()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            _ag_step(fn, xs)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = _ag_step(fn, xs)
    for x, want in ((x2, eager2), (x1, eager1)):
        xs.copy_(x)
        graph.replay()
        torch.cuda.synchronize()
        assert _eq(_ag_bits(static), want)


def test_second_device(cuda_device, record_property):
    """Autograd ops on cuda:1 while cuda:0 is current: the same bits as on cuda:0 (per-device one-time setup)."""
    if torch.cuda.device_count() < 2:
        record_property("second_device", "skipped: one device visible")
        pytest.skip("one CUDA device visible")
    d1 = torch.device("cuda:1")
    torch.cuda.set_device(0)
    for name in AUTOGRAD_OPS:
        fn = _autograd_ops()[name][0]
        want = _ag_bits(_ag_step(fn, _ag_input(name, cuda_device, 1)))
        got = _ag_step(fn, _ag_input(name, d1, 1))
        torch.cuda.synchronize(d1)
        assert torch.cuda.current_device() == 0
        assert _eq(_ag_bits(got), want), name


# ---- fresh processes: first launches inside a capture, and on two threads ------------------------------------------
FIRST_LAUNCHES = [   # a ring, split, token, band-map and band-pooled call (and their backward) in a fresh process
    _cell("stream", "forward", (3, 64, 7, 7, 1), F32), _cell("stream", "pooled_map_backward", (3, 64, 7, 7, 1), F32),
    _cell("split", "backward", (2, 64, 14, 14, 1), BF16), _cell("token", "forward", (3, 64, 14, 14, 1), BF16),
    _cell("token", "pooled_map_backward", (3, 64, 14, 14, 1), BF16, xbs="vit"),
    _cell("band", "forward", (2, 16, 112, 112, 1), F32), _cell("band", "backward", (2, 16, 112, 112, 1), BF16),
    _cell("band", "pooled_map_forward", (2, 8, 21, 16, 1), F32),
    _cell("band", "pooled_map_backward", (2, 8, 21, 16, 1), BF16),
]

_CHILD = r"""
import sys, threading, torch
sys.path[:0] = [{root!r}, {tests!r}]
import test_abi_contract_gpu as T
mode = sys.argv[1]
dev = torch.device("cuda:0")
probs = [T.Problem(c) for c in T.FIRST_LAUNCHES]
bufs = [p.plain(dev) for p in probs]
torch.cuda.synchronize()
if mode == "capture":   # the library's first launches of every family happen inside this capture
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for p, (b, ws) in zip(probs, bufs):
            T._run(p, b, ws, torch.cuda.current_stream().cuda_stream)
    g.replay()
else:                   # two host threads, each making the first launches of its own families on its own stream
    halves = [[i for i, c in enumerate(T.FIRST_LAUNCHES) if c.family in fams]
              for fams in (("stream", "band"), ("split", "token"))]
    errors = []
    def work(idx):
        try:
            s = torch.cuda.Stream()
            for i in idx:
                T._run(probs[i], bufs[i][0], bufs[i][1], s.cuda_stream)
            s.synchronize()
        except BaseException as e:
            errors.append(repr(e))
    ts = [threading.Thread(target=work, args=(h,)) for h in halves]
    for t in ts: t.start()
    for t in ts: t.join()
    assert not errors, errors
torch.cuda.synchronize()
first = [T._out_bits(p, b) for p, (b, _) in zip(probs, bufs)]
for p, (b, ws) in zip(probs, bufs):   # sequential, eager, on the current stream
    T._run(p, b, ws)
torch.cuda.synchronize()
bad = [T.cell_id(p.c) for p, f, (b, _) in zip(probs, first, bufs) if not all(T._same_bits(f, T._out_bits(p, b)).values())]
assert not bad, bad
print("OK", mode, len(probs))
"""


@pytest.mark.parametrize("mode", ["capture", "threads"])
def test_first_launches_fresh_process(mode, cuda_device):
    code = _CHILD.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    r = subprocess.run([sys.executable, "-c", code, mode], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and f"OK {mode}" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
