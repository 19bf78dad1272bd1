"""CPU: routing of fp16 (NFPB200_F16, ABI v5) through the C ABI and the Python host code.  No compute calls.

fp16 is served by the NCHW streaming-ring kernels ("fused/stream_*") and the channels-last token kernels
("fused/token_*") only, on exactly the problems a bf16 descriptor sends to them; every other fp16 problem is
NFPB200_EUNSUPPORTED (-5) and the Python side widens it to fp32."""
import ctypes
import itertools
import json
import os
import re
import subprocess
import sys

import pytest
import torch

from neighbour_feature_pooling_b200 import _capi
from neighbour_feature_pooling_b200 import functional as NF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EUNSUPPORTED = -5
SERVED_PREFIXES = ("fused/stream_", "fused/token_")
OPS = (_capi.OP_FORWARD, _capi.OP_BACKWARD, _capi.OP_POOL_FORWARD, _capi.OP_POOL_BACKWARD,
       _capi.OP_POOLED_MAP_FORWARD, _capi.OP_POOLED_MAP_BACKWARD)
PATHS = ("auto", "fused", "generic", "split")

# (B, C, H, W, R, padding, stride, measure, padding_mode, layout, inner_R): what each kernel family takes for bf16
SHAPES = {
    "ring": [(4, 64, 7, 7, 1, 1, 1, "cosine", "reflect", 0, 0), (2, 512, 7, 7, 1, 1, 1, "cosine", "zeros", 0, 0),
             (2, 64, 14, 14, 1, 1, 1, "cosine", "replicate", 0, 0), (2, 32, 14, 14, 2, 2, 1, "cosine", "reflect", 0, 0),
             (4, 64, 2, 2, 1, 1, 1, "cosine", "reflect", 0, 0), (3, 64, 4, 4, 1, 1, 1, "cosine", "reflect", 0, 0),
             (3, 64, 7, 7, 2, 2, 1, "cosine", "reflect", 0, 1), (256, 960, 7, 7, 1, 1, 1, "cosine", "reflect", 0, 0),
             (3, 40, 7, 7, 1, 1, 1, "cosine", "reflect", 0, 0)],
    "token": [(3, 64, 14, 14, 1, 1, 1, "cosine", "reflect", 1, 0), (2, 192, 7, 7, 1, 1, 1, "cosine", "zeros", 1, 0),
              (2, 512, 7, 7, 1, 1, 1, "cosine", "replicate", 1, 0), (3, 64, 7, 7, 2, 2, 1, "cosine", "reflect", 1, 1),
              (2, 32, 7, 7, 1, 1, 1, "cosine", "reflect", 1, 0)],   # C % 64 != 0: not a token shape
    "band": [(2, 16, 112, 112, 1, 1, 1, "cosine", "reflect", 0, 0), (2, 8, 21, 16, 1, 1, 1, "cosine", "zeros", 0, 0),
             (2, 16, 28, 28, 2, 2, 1, "cosine", "reflect", 0, 1)],
    "table": [(2, 5, 3, 3, 1, 1, 1, "cosine", "reflect", 0, 0), (2, 10, 5, 9, 2, 2, 1, "cosine", "reflect", 0, 0)],
    "generic": [(3, 5, 9, 11, 1, 2, 2, "cosine", "circular", 0, 0), (2, 64, 7, 7, 1, 1, 1, "attention", "reflect", 0, 0),
                (2, 64, 7, 7, 1, 0, 1, "cosine", "reflect", 0, 0), (2, 64, 7, 7, 1, 1, 1, "attention", "reflect", 1, 0)],
}


def _desc(dtype, shape, path="auto", yf32=False):
    B, C, H, W, R, pad, stride, measure, mode, layout, inner = shape
    d = _capi.make_desc(dtype, B, C, H, W, R, stride, pad, 1, mode, measure, True, False, 1e-6, 1, 1e-6, path,
                        layout=layout, inner_R=inner)
    if yf32:
        d.path |= _capi.FLAG_Y_F32
    return d


def _query(d, op):
    """(describe_path rc, name, workspace bytes, launch count) of one op."""
    lib = _capi.load()
    buf = ctypes.create_string_buffer(128)
    rc = lib.nfpb200_describe_path(ctypes.byref(d), op, buf, 128)
    if rc:
        n = ctypes.c_size_t()
        assert lib.nfpb200_workspace_bytes(ctypes.byref(d), op, ctypes.byref(n)) == rc
        k = ctypes.c_int32()
        assert lib.nfpb200_launch_count(ctypes.byref(d), op, ctypes.byref(k)) == rc
        return rc, None, None, None
    return 0, buf.value.decode(), _capi.workspace_bytes(d, op), _capi.launch_count(d, op)


def routing_table():
    """{(family, shape index, op, path, yf32): (bf16 query, f16 query, bf16 head_supported, f16 head_supported)}."""
    lib = _capi.load()
    out = {}
    for fam, shapes in SHAPES.items():
        for si, s in enumerate(shapes):
            for op, path, yf32 in itertools.product(OPS, PATHS, (False, True)):
                b, h = _desc(_capi.BF16, s, path, yf32), _desc(_capi.F16, s, path, yf32)
                out[(fam, si, op, path, yf32)] = (_query(b, op), _query(h, op),
                                                  lib.nfpb200_head_supported(ctypes.byref(b)),
                                                  lib.nfpb200_head_supported(ctypes.byref(h)))
    return out


def check_routing(table):
    """The fp16 routing rules over a routing_table(); returns how many cells fp16 is served on."""
    served = 0
    for key, (qb, qh, hb, hh) in table.items():
        bf16_on_f16_family = qb[0] == 0 and qb[1].startswith(SERVED_PREFIXES)
        if qh[0] == 0:
            served += 1
            # a ring / token name, and the very path, workspace and launch count of bf16
            assert qh[1].startswith(SERVED_PREFIXES), (key, qh)
            assert qh == qb, (key, qb, qh)
        else:
            assert qh[0] == EUNSUPPORTED or qh[0] == qb[0], (key, qh, qb)
        # coverage: fp16 is served exactly where bf16 takes the ring or token kernels
        assert (qh[0] == 0) == bf16_on_f16_family, (key, qb, qh)
        # the fused head follows the same rule: where bf16 takes it, fp16 does
        assert hh == hb or (hh == EUNSUPPORTED and hb != 0), (key, hb, hh)
    return served


def test_abi_version_is_5_everywhere():
    with open(os.path.join(ROOT, "include", "nfp_b200.h")) as f:
        header = f.read()
    assert int(re.search(r"#define NFPB200_ABI_VERSION (\d+)", header).group(1)) == 5
    assert _capi.ABI_VERSION == 5 and _capi.load().nfpb200_abi_version() == 5
    assert re.search(r"NFPB200_F16 = 2\b", header) and _capi.F16 == 2
    assert ctypes.sizeof(_capi.Desc) == 96   # the descriptor did not change


def test_f16_routing_matches_bf16():
    table = routing_table()
    served = check_routing(table)
    # the grid does reach both families and the unsupported side
    names = {qh[1] for qb, qh, _, _ in table.values() if qh[0] == 0}
    assert any(n.startswith("fused/stream_") for n in names) and any(n.startswith("fused/token_") for n in names)
    assert served < len(table)
    # every family of SHAPES keeps its bf16 meaning (the grid tests what it says it tests)
    prefix = {"ring": "fused/stream_", "token": "fused/token_", "band": "planar/band", "table": "planar/table",
              "generic": "generic/pairs"}
    for fam, shapes in SHAPES.items():
        for si, s in enumerate(shapes):
            if fam in ("ring", "token") and s[1] % 64 and s[9] == 1:
                continue   # the control shapes the token kernels do not take
            if fam == "generic" and s[9] == 1:
                continue   # NHWC outside the token kernels: -5 for both dtypes
            q = table[(fam, si, _capi.OP_FORWARD, "auto", False)][0]
            assert q[0] == 0 and q[1].startswith(prefix[fam]), (fam, s, q)


def test_f16_refusals():
    lib = _capi.load()
    n = ctypes.c_size_t()
    ring = SHAPES["ring"][0]
    for op in OPS:
        # forced generic, and the cluster-split kernels (PATH_SPLIT), carry no fp16
        for path in ("generic", "split"):
            d = _desc(_capi.F16, ring, path)
            assert lib.nfpb200_workspace_bytes(ctypes.byref(d), op, ctypes.byref(n)) == EUNSUPPORTED, (op, path)
        # band / table / generic problems
        for fam in ("band", "table", "generic"):
            for s in SHAPES[fam]:
                d = _desc(_capi.F16, s)
                assert lib.nfpb200_workspace_bytes(ctypes.byref(d), op, ctypes.byref(n)) == EUNSUPPORTED, (op, s)
    # an unknown dtype is still an argument error
    d = _desc(_capi.F16, ring)
    d.dtype = 3
    assert lib.nfpb200_workspace_bytes(ctypes.byref(d), _capi.OP_FORWARD, ctypes.byref(n)) == -1


def test_f16_y_f32_flag_is_accepted_where_bf16_is():
    for s in SHAPES["ring"][:2] + SHAPES["token"][:2]:
        for dt in (_capi.BF16, _capi.F16):
            assert _query(_desc(dt, s, yf32=True), _capi.OP_FORWARD)[0] == 0


_SPLIT_SCRIPT = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import test_f16_host as T
t = T.routing_table()
served = T.check_routing(t)
split = sum(1 for qb, qh, _, _ in t.values() if qb[0] == 0 and qb[1].startswith("fused/split_"))
print(json.dumps({"served": served, "split": split}))
"""


def test_f16_under_split_selection():
    """NFPB200_FUSED_IMPL=split sends bf16 ring problems to the cluster-split kernels: those are -5 for fp16."""
    env = dict(os.environ, NFPB200_FUSED_IMPL="split")
    r = subprocess.run([sys.executable, "-c", _SPLIT_SCRIPT, os.path.dirname(os.path.abspath(__file__))],
                       capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert got["split"] > 0 and got["served"] > 0, got


# ---- _prepare: keep fp16 when the caller's ops take it, widen otherwise ------------------------------------------------
def _cfg(R=1, **kw):
    return NF.NFPConfig(R=R, measure="cosine", padding=R, **kw)


@pytest.mark.parametrize("ops,name", [(NF.MAP_OPS, "map"), (NF.POOL_OPS, "pool"), (NF.POOLED_MAP_OPS, "pooled_map")])
def test_prepare_keeps_or_widens_fp16(ops, name):
    cases = [
        # (x, cfg, kept?, layout when kept)
        (torch.randn(2, 64, 7, 7).half(), _cfg(), True, _capi.LAYOUT_NCHW),                        # ring
        (torch.randn(2, 64, 7, 7).half().contiguous(memory_format=torch.channels_last), _cfg(), True,
         _capi.LAYOUT_NHWC),                                                                         # token
        (torch.randn(2, 32, 7, 7).half().contiguous(memory_format=torch.channels_last), _cfg(), True,
         _capi.LAYOUT_NCHW),                                                                         # token no, ring yes
        (torch.randn(2, 16, 28, 28).half(), _cfg(), False, None),                                   # band: widened
        (torch.randn(2, 5, 3, 3).half(), _cfg(), False, None),                                      # table: widened
        (torch.randn(2, 64, 7, 7).half(), NF.NFPConfig(R=1, measure="attention", padding=1), False, None),
        (torch.randn(2, 64, 7, 7).half(), _cfg(path="generic"), False, None),
    ]
    for x, cfg, kept, layout in cases:
        xk, out_dtype, lay = NF._prepare(x, cfg, ops)
        assert out_dtype == torch.float16
        if kept:
            assert xk.dtype == torch.float16 and lay == layout, (name, tuple(x.shape), lay)
            if lay == _capi.LAYOUT_NHWC:
                assert xk.data_ptr() == x.data_ptr()   # consumed in place
            desc = NF._desc_for(xk, cfg, lay)
            for op in ops:
                assert _capi.describe_path(desc, op).startswith(SERVED_PREFIXES)
        else:
            assert xk.dtype == torch.float32, (name, tuple(x.shape), cfg)


def test_prepare_probes_the_callers_ops(monkeypatch):
    """The keep-or-widen decision asks about the ops the caller will issue (not always the map backward)."""
    seen = []
    served = NF._served

    def spy(x, cfg, layout, ops):
        seen.append((layout, tuple(ops)))
        return served(x, cfg, layout, ops)
    monkeypatch.setattr(NF, "_served", spy)
    cfg = _cfg()
    for ops in (NF.MAP_OPS, NF.POOL_OPS, NF.POOLED_MAP_OPS):
        seen.clear()
        assert NF._prepare(torch.randn(2, 64, 7, 7).half(), cfg, ops)[0].dtype == torch.float16
        assert seen == [(_capi.LAYOUT_NCHW, ops)], seen
        seen.clear()
        xc = torch.randn(2, 64, 7, 7).half().contiguous(memory_format=torch.channels_last)
        assert NF._prepare(xc, cfg, ops)[2] == _capi.LAYOUT_NHWC
        assert seen == [(_capi.LAYOUT_NHWC, ops)], seen
    # fp32 and bf16 inputs are untouched by the fp16 rule
    xf = torch.randn(2, 64, 7, 7)
    assert NF._prepare(xf, cfg, NF.POOL_OPS)[0].dtype == torch.float32
    assert NF._prepare(xf.bfloat16(), cfg, NF.POOL_OPS)[0].dtype == torch.bfloat16


def test_describe_and_trace_name_f16():
    cfg = _cfg()
    assert NF.describe((2, 64, 7, 7), torch.float16, cfg).startswith("fused/stream_7x7_r1")
    assert NF.describe((2, 64, 7, 7), torch.float16, cfg, layout=1).startswith("fused/token_7x7_r1")
    assert NF._DTYPE_NAMES[_capi.F16] == "f16"
