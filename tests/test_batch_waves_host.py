"""CPU: the grid of tests/test_batch_waves_gpu.py keeps up with the library.

* every ring and token instantiation of NFP_STREAM_SHAPES (read from the source), every dtype and entry point the
  library serves there (asked through nfpb200_describe_path / nfpb200_head_supported, which need no GPU), and every
  shape the cluster-split kernels accept under NFPB200_PATH_SPLIT has a cell in the grid, so a new shape, dtype or
  entry point cannot go without a multi-round check;
* each cell takes its family's path at a small and at a large batch;
* the batch sizes and scored images reach the regimes they are named for, for any measured grid;
* the planar row-band kernels' batch limit sits where the GPU test expects it.
"""
import ctypes
import os
import re

import pytest
import torch

from neighbour_feature_pooling_b200 import _capi

import test_abi_contract_gpu as AC
import test_batch_waves_gpu as BW

DTYPES = (torch.float32, torch.bfloat16, torch.float16)
FAMILY_ENTRIES = {"stream": AC.ENTRIES, "token": AC.ENTRIES, "split": AC.ENTRIES[:6]}
PROBE_CHANNELS = (64, 32)   # the channel counts a (shape, dtype, entry) is probed with


def stream_shapes():
    with open(os.path.join(AC.ROOT, "neighbour_feature_pooling_b200", "csrc", "nfp_stream.h")) as f:
        src = f.read()
    block = src[src.index("#define NFP_STREAM_SHAPES(X)"):].split("\n\n", 1)[0]
    shapes = [tuple(int(v) for v in m[:3]) for m in re.findall(r"X\((\d+),\s*(\d+),\s*(\d+),\s*\d+\)", block)]
    assert len(shapes) >= 6, block
    return shapes


def served(family, entry, hwr, dtype):
    """Whether the library sends (family, entry point, H x W radius R, dtype) to that family's fused kernels."""
    H, W, R = hwr
    lib = _capi.load()
    for C in PROBE_CHANNELS:
        try:
            p = BW.PROBLEM[dtype](AC._cell(family, entry, (3, C, H, W, R), dtype))
            path = p.path()
        except RuntimeError:
            continue
        if not path.startswith(AC.FAMILIES[family][0]):
            continue
        if p.head and lib.nfpb200_head_supported(ctypes.byref(p.desc)) != 0:
            continue
        return True
    return False


def test_grid_has_a_cell_for_everything_served():
    have = {(w.family, tuple(w.shape[1:]), w.dtype, w.entry) for w in BW.GRID}
    missing, count = [], 0
    for family, entries in FAMILY_ENTRIES.items():
        for hwr in stream_shapes():
            for dt in DTYPES:
                for e in entries:
                    if served(family, e, hwr, dt):
                        count += 1
                        if (family, hwr, dt, e) not in have:
                            missing.append((family, hwr, BW.DTYPE_NAME[dt], e))
    assert not missing, missing
    # ring: 6 shapes x 3 dtypes x 8 entries at least; token and split serve something too
    assert count >= 144 + 2 * 8 + 2 * 6, count
    ids = [BW.wave_id(w) for w in BW.GRID]
    assert len(ids) == len(set(ids))


@pytest.mark.parametrize("B", [3, 1201])
def test_every_cell_takes_its_family_path(B):
    lib = _capi.load()
    for w in BW.GRID:
        small = BW.problem(w, 3)
        p = BW._resized(small, B)
        assert p.path().startswith(AC.FAMILIES[w.family][0]), (BW.wave_id(w), B, p.path())
        if p.head:
            assert lib.nfpb200_head_supported(ctypes.byref(p.desc)) == 0, BW.wave_id(w)


def test_grid_reaches_the_planner_configurations():
    cells = {(w.family, w.entry, w.shape, w.dtype, w.opts) for w in BW.GRID}
    f32, bf16, f16 = DTYPES
    for want in [("stream", "backward", (960, 7, 7, 1), f32, ()), ("stream", "backward", (40, 7, 7, 1), bf16, ()),
                 ("stream", "backward", (64, 7, 7, 1), f32, ()), ("stream", "backward", (112, 14, 14, 1), bf16, ()),
                 ("stream", "backward", (32, 14, 14, 2), f32, ()),
                 ("stream", "backward", (512, 7, 7, 2), f32, (("inner", 1),)),
                 ("stream", "backward", (256, 14, 14, 2), f16, (("inner", 1),)),
                 ("stream", "backward", (256, 14, 14, 2), bf16, (("hint", 1),)),
                 ("stream", "forward", (512, 7, 7, 2), bf16, (("yf32", 1),)),
                 ("token", "backward", (192, 14, 14, 1), bf16, (("gxbs", "pad64"), ("xbs", "vit"))),
                 ("token", "backward", (960, 7, 7, 1), f16, ()), ("token", "backward", (64, 14, 14, 1), bf16, ()),
                 ("token", "backward", (512, 7, 7, 2), f16, (("gxbs", "pad8"), ("inner", 1), ("xbs", "pad8")))]:
        assert want in cells, want


@pytest.mark.parametrize("g", [1, 2, 148, 296, 444, 1184])
def test_batch_sizes_reach_their_regimes(g):
    one, two, three = BW.batch_sizes(g)
    assert one == g and two == g + 1 and three >= 2 * g + 1
    # B = g + 1: image g is CTA 0's second image; 2g + 3: images 2g .. are third-round images
    assert BW.scored_rows(g, two)[-1] == g
    rows = BW.scored_rows(g, three)
    for r in (0, g - 1, g, 2 * g, three - 1):
        assert r in rows
    assert (three - 1) // g >= 2
    assert BW.scored_rows(g, one) == sorted({0, g - 1})


def test_planar_batch_limit_paths():
    assert BW.PLANAR_LIMIT == 65535
    for B, prefix in ((BW.PLANAR_LIMIT, "planar/band"), (BW.PLANAR_LIMIT + 1, "generic/pairs")):
        d = BW._band_desc(B)
        for op in (_capi.OP_FORWARD, _capi.OP_BACKWARD):
            assert _capi.describe_path(d, op).startswith(prefix), (B, op)
