"""Time one second-order training call of the cosine NFP map: forward + create_graph backward + double backward.

    python tools/time_second_order.py [--out FILE]

Per row: this package (nfp_similarity: fused / planar forward and backward, then nfpb200_backward_backward and
nfpb200_jvp) against the reference's conv form (oracle/nfp_convform.py: one-hot convs + F.cosine_similarity) run by
ATen on the same GPU.  One CUDA graph holds one call on each of N inputs, N chosen so that the inputs span more than
twice the 126 MB L2: every call reads its input from HBM.  Median of 7 replays, divided by N.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from neighbour_feature_pooling_b200 import functional as NF  # noqa: E402
from oracle.nfp_convform import ConvFormCosineNFP  # noqa: E402

L2_BYTES = 126 * 2 ** 20
ROWS = [  # (B, C, H, W, dtype)
    (256, 512, 7, 7, torch.float32),
    (256, 512, 7, 7, torch.bfloat16),
    (64, 16, 112, 112, torch.float32),
]


def call(f, x, gy, v):
    y = f(x)
    (gx,) = torch.autograd.grad(y, x, gy.to(y.dtype), create_graph=True)
    (gx2,) = torch.autograd.grad(gx, x, v)
    return gx2


def time_graph(f, xs, gys, vs, reps=7):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            for x, gy, v in zip(xs, gys, vs):
                call(f, x, gy, v)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = [call(f, x, gy, v) for x, gy, v in zip(xs, gys, vs)]
    g.replay()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e3 / len(xs))
    del outs, g
    return sorted(times)[len(times) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the table here (profiles/second_order_b200.txt)")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    lines = [f"# {torch.cuda.get_device_name(dev)}; nvidia-smi: {smi}",
             "# forward + create_graph backward + double backward of the cosine map (R = 1, pad 1, reflect), one call;",
             "# CUDA-graph replays over N inputs spanning > 2x L2, median of 7, microseconds per call",
             f"{'shape':<22}{'dtype':<7}{'N':>4}{'path (forward)':>26}{'package us':>12}{'ATen conv form us':>19}"
             f"{'speed-up':>10}"]
    print("\n".join(lines), flush=True)
    cfg = NF.NFPConfig(R=1, measure="cosine", padding=1)
    for B, C, H, W, dtype in ROWS:
        esz = torch.empty(0, dtype=dtype).element_size()
        n = max(3, -(-2 * L2_BYTES // (B * C * H * W * esz)) + 1)
        gen = torch.Generator().manual_seed(0)
        xs = [torch.randn(B, C, H, W, generator=gen).to(dev, dtype).requires_grad_(True) for _ in range(n)]
        gys = [torch.randn(B, 8, H, W, generator=gen).to(dev, dtype) for _ in range(n)]
        vs = [torch.randn(B, C, H, W, generator=gen).to(dev, dtype) for _ in range(n)]
        ours = time_graph(lambda t: NF.nfp_similarity(t, cfg), xs, gys, vs)
        ref = ConvFormCosineNFP(C, R=1, padding=1).to(dev, dtype)
        aten = time_graph(ref, xs, gys, vs)
        path = NF.describe((B, C, H, W), dtype, cfg)
        lines.append(f"{f'{B}x{C}x{H}x{W}':<22}{str(dtype).split('.')[-1]:<7}{n:>4}{path:>26}{ours:>12.1f}{aten:>19.1f}"
                     f"{aten / ours:>10.2f}")
        print(lines[-1], flush=True)
        del xs, gys, vs, ref
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
