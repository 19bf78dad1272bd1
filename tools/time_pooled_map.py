#!/usr/bin/env python
"""GAP(NFP(x)) on the five maps of the reference's MobileNetV3_MultiStageNFP (models/texture_pooling.py:211-268), two ways:

    (a) composed: nfp_similarity + adaptive_avg_pool2d (the map is written, re-read by the pool; its gradient is
        expanded to a full map by the pool's backward and read by the NFP backward);
    (b) pooled:   nfp_pooled_similarity (nfpb200_pooled_map_*: the map never exists).

Per map: forward (no_grad) and forward + backward are each captured in a CUDA graph of NBUF iterations that rotate over
NBUF input buffers holding > 2 x the 126 MB L2 in all (so x comes from HBM, not L2), timed with CUDA events over whole
replays after warm-up; the median of WINDOWS windows is reported per iteration.  backward = (forward + backward) -
forward.  Then one graph replay of the whole five-map set, forward + backward, each way.  Algorithmic bytes are from the
shapes: what each way must move through HBM at least (x, the map, its gradient, gx, the pooled vectors).

    python tools/time_pooled_map.py [B] [dtype]      (B = 64; dtype fp32 | bf16, default: both)
"""
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from neighbour_feature_pooling_b200 import NFPPooling, functional as NF  # noqa: E402

MAPS = [(16, 112, 112), (24, 56, 56), (40, 28, 28), (112, 14, 14), (960, 7, 7)]
K = 8
L2_BYTES = 126 * 2 ** 20
WINDOWS = 7


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return f"{name}, power limit {pl or 'unknown'}"


class Map:
    def __init__(self, dev, B, C, H, W, dtype):
        self.shape, self.dtype = (B, C, H, W), dtype
        self.cfg = NFPPooling(C, R=1, measure="cosine", padding=1).config
        xbytes = B * C * H * W * dtype.itemsize
        self.nbuf = max(2, min(64, -(-2 * L2_BYTES // xbytes)))
        gen = torch.Generator(device=dev).manual_seed(C)
        self.xs = [torch.randn(B, C, H, W, device=dev, generator=gen).to(dtype).requires_grad_(True)
                   for _ in range(self.nbuf)]
        self.g = torch.randn(B, K, device=dev, generator=gen)
        esz, P = dtype.itemsize, H * W
        x, y, gap = B * C * P * esz, B * K * P * esz, B * K * 4
        # (a) fwd: read x, write y, pool reads y, writes the pooled vector;  bwd: pool backward writes gy, NFP backward
        #     reads x and gy, writes gx.   (b) fwd: read x, write the pooled vector;  bwd: read x, write gx.
        self.bytes = {"composed": (x + y + y + gap, gap + y + x + y + x), "pooled": (x + gap, gap + x + x)}

    def composed(self, x):
        return F.adaptive_avg_pool2d(NF.nfp_similarity(x, self.cfg), 1).flatten(1)

    def pooled(self, x):
        return NF.nfp_pooled_similarity(x, self.cfg)

    def step(self, way, i, backward):
        x = self.xs[i % self.nbuf]
        if backward:
            y = getattr(self, way)(x)
            torch.autograd.grad(y, x, self.g.to(y.dtype))
        else:
            with torch.no_grad():
                getattr(self, way)(x)


def graph_time(fn, iters):
    """Per-iteration time (s) of fn(i), i in [0, iters), captured as one CUDA graph: median over WINDOWS replays."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(3):
            fn(i)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(iters):
            fn(i)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(WINDOWS):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3 / iters)
    del g
    return statistics.median(ts)


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
    dtypes = {"fp32": torch.float32, "bf16": torch.bfloat16}
    which = [sys.argv[2]] if len(sys.argv) > 2 else ["fp32", "bf16"]
    dev = torch.device("cuda:0")
    print(f"card: {card()}")
    print(f"B = {B}; inputs rotate over buffers holding > 2 x L2 (HBM-cold x); median of {WINDOWS} graph replays; "
          "us per call; MB = algorithmic HBM bytes")
    for dn in which:
        maps = [Map(dev, B, c, h, w, dtypes[dn]) for c, h, w in MAPS]
        print(f"\n{dn}")
        print(f"{'map':>12} {'path (pooled)':>22} | {'composed fwd':>12} {'bwd':>8} {'MB f/b':>13} | "
              f"{'pooled fwd':>10} {'bwd':>8} {'MB f/b':>13} | {'speed-up f+b':>12}")
        for m in maps:
            t = {}
            for way in ("composed", "pooled"):
                f = graph_time(lambda i: m.step(way, i, False), m.nbuf)
                fb = graph_time(lambda i: m.step(way, i, True), m.nbuf)
                t[way] = (f, fb - f, fb)
            path = NF.describe(m.shape, m.dtype, m.cfg, NF._capi.OP_POOLED_MAP_FORWARD)
            bc, bp = m.bytes["composed"], m.bytes["pooled"]
            B_, C, H, W = m.shape
            print(f"{C:>4}x{H}x{W:<4} {path:>22} | {t['composed'][0] * 1e6:12.1f} {t['composed'][1] * 1e6:8.1f} "
                  f"{bc[0] / 1e6:6.1f}/{bc[1] / 1e6:6.1f} | {t['pooled'][0] * 1e6:10.1f} {t['pooled'][1] * 1e6:8.1f} "
                  f"{bp[0] / 1e6:6.1f}/{bp[1] / 1e6:6.1f} | {t['composed'][2] / t['pooled'][2]:11.2f}x")
        n = min(m.nbuf for m in maps)
        for way in ("composed", "pooled"):
            def full_set(i, way=way):
                for m in maps:
                    m.step(way, i, True)
            ts = graph_time(full_set, n)
            mb = sum(sum(m.bytes[way]) for m in maps) / 1e6
            print(f"whole five-map set, forward + backward, {way:>8}: {ts * 1e6:8.1f} us per set ({mb:.1f} MB)")


if __name__ == "__main__":
    main()
