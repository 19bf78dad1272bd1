#!/usr/bin/env python
"""Time the NFP forward and backward each right after a non-NFP torch kernel, on rotating HBM-cold buffers.

    python tools/time_isolated.py [--shape l4] [--R 1] [--dtype fp32|bf16] [--batch 256] [--steps 200]

Inside a network an NFP launch follows some other kernel (the backward follows the gradient kernel of the layer above),
and that kernel does not release its dependents early: nothing of the NFP launch overlaps it, so whatever an NFP kernel
does before its dependency wait (e.g. the L2 prefetch of its inputs) is pure cost there.  Each timed call is one small
elementwise torch kernel followed by one NFP launch; the torch kernel alone is timed the same way and subtracted.
Graph replays, median of --windows windows (bench.LayerBench.timed).
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import SHAPES, LayerBench  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--shape", default="l4", choices=sorted(SHAPES))
ap.add_argument("--R", type=int, default=1)
ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"])
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--steps", type=int, default=200)
ap.add_argument("--windows", type=int, default=11)
args = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("time_isolated.py needs a CUDA device")
C, H, W, _ = SHAPES[args.shape]
dev = torch.device("cuda:0")
lb = LayerBench(dev, args.batch, C, H, W, args.R, args.dtype)
other = [torch.ones(1 << 16, device=dev) for _ in range(lb.nbuf)]   # 256 KB each: a short non-NFP kernel


def torch_only(i):
    other[i].mul_(1.0001)


def then_fwd(i):
    other[i].mul_(1.0001)
    lb.fwd(i)


def then_bwd(i):
    other[i].mul_(1.0001)
    lb.bwd_conservative(i)


n = args.steps
t = {nm: lb.timed(fn, n, 5, windows=args.windows) / n * 1e6
     for nm, fn in (("torch_only", torch_only), ("then_fwd", then_fwd), ("then_bwd", then_bwd))}
print(json.dumps({"workload": f"B={args.batch} {C}x{H}x{W} R={args.R} {args.dtype}",
                  "lib": os.path.basename(os.environ.get("NFPB200_LIB", "") or "libnfp_b200.so"),
                  "us_torch_kernel": round(t["torch_only"], 3),
                  "us_fwd_after_torch_kernel": round(t["then_fwd"] - t["torch_only"], 3),
                  "us_bwd_after_torch_kernel": round(t["then_bwd"] - t["torch_only"], 3)}))
