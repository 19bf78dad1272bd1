#!/usr/bin/env python
"""fp16 NFP, forward + backward, three ways:

    f16      native fp16: the ring (NCHW) or token (channels-last) kernels read and write half;
    widened  what an fp16 input took before the kernels had an fp16 dtype: the same call on x.float() (the fp32 kernels;
             a channels-last map is repacked to NCHW), its result narrowed with .half() -- the cast kernels, the fp32
             traffic and autograd's narrowing of gx included;
    bf16     the same call on a bf16 input, for reference.

Shapes (B = 256): 512x7x7 NCHW and channels-last, 960x7x7 NCHW, the ViT head's 192x14x14 token view of fp32 tokens under
autocast (f16: fp16 autocast, rounded to fp16 and read in place by the token kernels; widened: the fp32 NCHW repack
fp16 autocast took before; bf16: bf16 autocast), and the nfp_pooling head on 512x7x7 (f16 / bf16: under that autocast;
widened: the head on x.float()).

Each way is captured in a CUDA graph of NBUF forward + backward iterations that rotate over NBUF inputs holding > 2 x
the 126 MB L2 in all (x comes from HBM, not L2), timed with CUDA events over whole replays after warm-up; the median of
WINDOWS windows is reported per iteration.

    python tools/time_f16.py [B]
"""
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from neighbour_feature_pooling_b200 import NFPPooling, nfp_pooling, functional as NF  # noqa: E402

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


def nbuf_for(nbytes):
    return max(2, min(64, -(-2 * L2_BYTES // nbytes)))


class MapCase:
    """nfp_similarity fwd + bwd on a (B, C, H, W) map in NCHW or channels-last."""

    def __init__(self, dev, B, C, H, W, channels_last):
        self.name = f"{C}x{H}x{W} {'channels-last' if channels_last else 'NCHW'}"
        self.cfg = NFPPooling(C, R=1, measure="cosine", padding=1).config
        self.shape, self.cl = (B, C, H, W), channels_last
        self.nbuf = nbuf_for(B * C * H * W * 2)
        gen = torch.Generator(device=dev).manual_seed(C)
        fmt = torch.channels_last if channels_last else torch.contiguous_format
        base = [torch.randn(B, C, H, W, device=dev, generator=gen) for _ in range(self.nbuf)]
        self.x = {"f16": [b.half().contiguous(memory_format=fmt).requires_grad_(True) for b in base],
                  "bf16": [b.bfloat16().contiguous(memory_format=fmt).requires_grad_(True) for b in base]}
        self.x["widened"] = self.x["f16"]
        self.g = torch.randn(B, 8, H, W, device=dev, generator=gen).half()
        del base

    def path(self, way):
        dt = {"f16": torch.float16, "bf16": torch.bfloat16, "widened": torch.float32}[way]
        return NF.describe(self.shape, dt, self.cfg, layout=int(self.cl and way != "widened"))

    def step(self, way, i):
        x = self.x[way][i % self.nbuf]
        y = NF.nfp_similarity(x.float() if way == "widened" else x, self.cfg)
        if way == "widened":
            y = y.half()
        torch.autograd.grad(y, x, self.g.to(y.dtype))


class VitCase:
    """The ViT head: fp32 LayerNorm tokens (B, 1 + H W, C), their (B, C, H, W) view, under autocast."""

    def __init__(self, dev, B, C=192, H=14, W=14):
        self.name = f"ViT {C}x{H}x{W} token view, fp32 tokens"
        self.cfg = NFPPooling(C, R=1, measure="cosine", padding=1).config
        self.dims = (B, C, H, W)
        self.nbuf = nbuf_for(B * (H * W + 1) * C * 4)
        gen = torch.Generator(device=dev).manual_seed(C)
        self.feats = [torch.randn(B, H * W + 1, C, device=dev, generator=gen).requires_grad_(True)
                      for _ in range(self.nbuf)]
        self.g = torch.randn(B, 8, H, W, device=dev, generator=gen)

    def path(self, way):
        if way == "widened":
            return NF.describe(self.dims, torch.float32, self.cfg)
        return NF.describe(self.dims, torch.float16 if way == "f16" else torch.bfloat16, self.cfg, layout=1)

    def step(self, way, i):
        B, C, H, W = self.dims
        f = self.feats[i % self.nbuf]
        ac = {"f16": torch.float16, "bf16": torch.bfloat16, "widened": torch.float16}[way]
        # widened: what fp16 autocast did with fp32 tokens before (the NCHW repack and the fp32 kernels) is the call
        # without autocast
        with torch.autocast("cuda", dtype=ac, enabled=way != "widened", cache_enabled=False):
            y = NF.nfp_similarity(f[:, 1:].transpose(1, 2).reshape(B, C, H, W), self.cfg)
        torch.autograd.grad(y, f, self.g)


class HeadCase:
    """nfp_pooling (GAP(x) * proj(GAP(NFP(x)))) fwd + bwd on a (B, C, H, W) NCHW map."""

    def __init__(self, dev, B, C=512, H=7, W=7):
        self.name = f"nfp_pooling head {C}x{H}x{W}"
        Params = {"num_ftrs": {"m": C}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 3}}
        torch.manual_seed(0)
        self.pool = nfp_pooling(Params=Params).to(dev)
        self.shape = (B, C, H, W)
        self.nbuf = nbuf_for(B * C * H * W * 2)
        gen = torch.Generator(device=dev).manual_seed(C)
        base = [torch.randn(B, C, H, W, device=dev, generator=gen) for _ in range(self.nbuf)]
        self.x = {"f16": [b.half().requires_grad_(True) for b in base],
                  "bf16": [b.bfloat16().requires_grad_(True) for b in base]}
        self.x["widened"] = self.x["f16"]
        self.g = torch.randn(B, C, device=dev, generator=gen)
        del base

    def path(self, way):
        dt = {"f16": torch.float16, "bf16": torch.bfloat16, "widened": torch.float32}[way]
        return NF.describe(self.shape, dt, self.pool.nfp_layer.config, NF._capi.OP_POOL_FORWARD)

    def step(self, way, i):
        x = self.x[way][i % self.nbuf]
        if way == "widened":
            out = self.pool(x.float()).half()
        else:
            with torch.autocast("cuda", dtype=torch.float16 if way == "f16" else torch.bfloat16, cache_enabled=False):
                out = self.pool(x)
        torch.autograd.grad(out, x, self.g.to(out.dtype))


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
    dev = torch.device("cuda:0")
    print(f"card: {card()}")
    print(f"B = {B}; forward + backward per call; inputs rotate over buffers holding > 2 x L2 (HBM-cold x); "
          f"median of {WINDOWS} graph replays; us per call")
    cases = [MapCase(dev, B, 512, 7, 7, False), MapCase(dev, B, 512, 7, 7, True), MapCase(dev, B, 960, 7, 7, False),
             VitCase(dev, B), HeadCase(dev, B)]
    ways = ("f16", "widened", "bf16")
    print(f"{'shape':>38} | {'f16':>8} {'widened':>8} {'bf16':>8} | {'widened/f16':>11} | path f16 / widened / bf16")
    for c in cases:
        t = {w: graph_time(lambda i, w=w: c.step(w, i), c.nbuf) for w in ways}
        paths = " / ".join(c.path(w) for w in ways)
        print(f"{c.name:>38} | {t['f16'] * 1e6:8.1f} {t['widened'] * 1e6:8.1f} {t['bf16'] * 1e6:8.1f} | "
              f"{t['widened'] / t['f16']:10.2f}x | {paths}", flush=True)
        del c
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
