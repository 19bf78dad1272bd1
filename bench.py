#!/usr/bin/env python
"""NFP hot-path benchmark (BASELINE.json metric: NFP fwd+bwd feature-maps/s & % of the HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--shape l4|l3|mbv3|vit|eurosat] [--R 1|2] [--dtype fp32|bf16] [--batch 256] [--no-sweep]
                    [--dump-outputs DIR]

One "step" = one forward + one backward of the NFP layer (cosine, pad = R, reflect) over one batch
of synthetic feature maps.  Default workload: BASELINE.json configs[1], ResNet18 layer4 maps
(B=256, 512x7x7, 3x3, fp32).  Prints ONE JSON line (rank 0).

* ``value``    -- maps/s, inputs resident in HBM, the C-ABI entry points launched back to back from a
                  CUDA graph; buffers rotate over > 2x the L2 capacity so every step reads from HBM.
* ``e2e``      -- the same metric through the public nn.Module API (``NFPPooling`` + autograd) with
                  HOST pinned buffers: H2D of x and grad_y and D2H of y and grad_x inside the timed region.
* ``roofline`` -- the dominant kernel (backward): algorithmic bytes per launch / its average launch
                  duration (CUDA events around a graph of back-to-back launches on rotating buffers).
* ``cpu_baseline`` -- the reference's own operator (NFP_REFERENCE_ROOT, or the copy build() staged unmodified under
                  oracle/_ref) on the host cores; the conv-form port (oracle/nfp_convform.py) only if those files are missing.
* ``--impl reference`` -- that CPU path as its own arm, same metric / config.
* ``--dump-outputs DIR`` -- y and grad_x of the last timed step as DIR/*.npy (seeded inputs: two builds can be
                  compared output for output).

Multi-GPU (torchrun): the batch dimension is sharded, one process per GPU, no data-path collective;
weak scaling (B maps per GPU per step); time = max over ranks.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

SHAPES = {  # name -> (C, H, W, where it comes from)
    "l4": (512, 7, 7, "ResNet18 layer4"),
    "l3": (256, 14, 14, "ResNet18 layer3"),
    "mbv3": (960, 7, 7, "MobileNetV3-large last stage"),
    "vit": (192, 14, 14, "ViT-Tiny token grid"),
    "eurosat": (512, 2, 2, "ResNet18 layer4 at 64x64 input"),
}
L2_BYTES = 126 * 1024 * 1024
METRIC = "nfp_fwd_bwd_feature_maps_per_s"
UNIT = "maps/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--shape", default="l4", choices=sorted(SHAPES))
    ap.add_argument("--R", type=int, default=1)
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--windows", type=int, default=11, help="timed windows of --steps steps each; the median is reported")
    ap.add_argument("--no-sweep", action="store_true", help="skip the table over the other configs[1] cases")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the ResNet18+NFP training-step measurement")
    ap.add_argument("--train-config", default="eurosat", choices=["eurosat", "ucmerced", "gtos_mbv3", "plantvillage_vit"])
    ap.add_argument("--train-more", default="gtos_mbv3,plantvillage_vit,ucmerced",
                    help="further BASELINE.json configs measured as training steps (comma separated, '' = none)")
    ap.add_argument("--train-batch", type=int, default=256, help="images per GPU per training step")
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU-baseline budget (seconds of CPU work)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write y and grad_x of the last timed step as DIR/<name>.npy")
    return ap.parse_args()


def algorithmic_bytes(B, C, H, W, R, esz):
    """SURVEY.md 8(d3).  Per launch: forward reads x, writes y; backward reads x and grad_y, writes grad_x."""
    K = (2 * R + 1) ** 2 - 1
    fwd = B * (C * H * W + K * H * W) * esz
    bwd = B * (2 * C * H * W + K * H * W) * esz
    return fwd, bwd


def workload_name(B, C, H, W, R, dtype):
    k = 2 * R + 1
    return f"nfp_cosine_fwd_bwd B={B} {C}x{H}x{W} {k}x{k} pad={R} reflect {dtype}"


# ----------------------------------------------------------------------------------------------
# clocks: NVML polled from a thread while a timed region runs
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, dev):
        self.ok = False
        self.samples = []   # (tag, sm_mhz, reasons_mask)
        self.tag = None
        self._stop = threading.Event()
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            try:   # CUDA ordinal != NVML index under CUDA_VISIBLE_DEVICES: resolve by UUID
                uuid = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(dev.index or 0)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # NVML missing: report that, do not fake numbers
            self.err = repr(e)
            self.sm_max = None
        self.thread = None

    def _poll(self):
        nv = self.nv
        while not self._stop.is_set():
            tag = self.tag
            if tag is not None:
                try:
                    mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    try:
                        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.samples.append((tag, mhz, mask))
                except Exception:
                    pass
            time.sleep(0.001)

    def start(self):
        if self.ok:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()

    def stop(self):
        self._stop.set()
        if self.thread:
            self.thread.join(timeout=1.0)

    def summary(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": self.err}
        main = [s for s in self.samples if s[0] == "timed"]
        window = "timed region"
        if len(main) < 3:
            main = [s for s in self.samples if s[0] is not None]
            window = "all timed regions (value, kernel passes, e2e)"
        mhz = sorted(s[1] for s in main)
        mask = 0
        for s in main:
            mask |= s[2]
        reasons = [name for bit, name in self.REASONS.items() if mask & bit and name != "gpu_idle"]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": self.sm_max, "reasons": reasons,
                "samples": len(main), "window": window}


# ----------------------------------------------------------------------------------------------
# the B200 arm
# ----------------------------------------------------------------------------------------------
class LayerBench:
    """Rotating device buffers + C-ABI launches for one (shape, R, dtype) configuration."""

    def __init__(self, dev, B, C, H, W, R, dtype_name, seed=0, layout="nchw", inner_R=0):
        from neighbour_feature_pooling_b200 import _capi
        self.capi = _capi
        self.lib = _capi.load()
        self.dev = dev
        self.B, self.C, self.H, self.W, self.R = B, C, H, W, R
        # inner_R > 0: the multi-radius launch (SURVEY 8 f3) -- y / gy carry the radius-inner_R map in front
        self.K = (2 * R + 1) ** 2 - 1 + ((2 * inner_R + 1) ** 2 - 1 if inner_R else 0)
        self.tdtype = torch.float32 if dtype_name == "fp32" else torch.bfloat16
        self.esz = 4 if dtype_name == "fp32" else 2
        lay = _capi.LAYOUT_NHWC if layout == "nhwc" else _capi.LAYOUT_NCHW   # nhwc: channels_last x / grad_x, in place
        self.layout = layout
        self.desc = _capi.make_desc(_capi.F32 if dtype_name == "fp32" else _capi.BF16, B, C, H, W, R, 1, R, 1,
                                    "reflect", "cosine", True, False, 1e-6, 1, 1e-6, "auto", layout=lay, inner_R=inner_R)
        # backward entry points: x is a saved activation, not an output of the preceding launch (what autograd passes)
        self.desc_bwd = _capi.make_desc(_capi.F32 if dtype_name == "fp32" else _capi.BF16, B, C, H, W, R, 1, R, 1,
                                        "reflect", "cosine", True, False, 1e-6, 1, 1e-6, "auto", layout=lay,
                                        inner_R=inner_R)
        if os.environ.get("NFPB200_BENCH_NO_HINT", "0") != "1":
            self.desc_bwd.path |= _capi.HINT_X_STABLE
        self.path_fwd = _capi.describe_path(self.desc, _capi.OP_FORWARD)
        self.path_bwd = _capi.describe_path(self.desc, _capi.OP_BACKWARD)
        self.launches = _capi.launch_count(self.desc, _capi.OP_FORWARD) + _capi.launch_count(self.desc, _capi.OP_BACKWARD)
        set_bytes = (2 * B * C * H * W + 2 * B * self.K * H * W) * self.esz
        self.set_bytes = set_bytes
        self.nbuf = max(4, math.ceil(2.2 * L2_BYTES / set_bytes))
        gen = torch.Generator(device=dev).manual_seed(seed)
        mk = lambda *s: torch.randn(*s, device=dev, generator=gen).to(self.tdtype)
        fmt = torch.channels_last if layout == "nhwc" else torch.contiguous_format
        self.x = [mk(B, C, H, W).contiguous(memory_format=fmt) for _ in range(self.nbuf)]
        self.gy = [mk(B, self.K, H, W) for _ in range(self.nbuf)]
        self.y = [torch.empty(B, self.K, H, W, device=dev, dtype=self.tdtype) for _ in range(self.nbuf)]
        self.gx = [torch.empty(B, C, H, W, device=dev, dtype=self.tdtype).contiguous(memory_format=fmt)
                   for _ in range(self.nbuf)]
        wsf = _capi.workspace_bytes(self.desc, _capi.OP_FORWARD)
        wsb = _capi.workspace_bytes(self.desc, _capi.OP_BACKWARD)
        self.ws = torch.empty(max(wsf, wsb, 1), dtype=torch.uint8, device=dev)
        self.ws_n = max(wsf, wsb)

    def fwd(self, i):
        s = torch.cuda.current_stream(self.dev).cuda_stream
        rc = self.lib.nfpb200_forward(ctypes.byref(self.desc), self.x[i].data_ptr(), self.y[i].data_ptr(),
                                      self.ws.data_ptr() if self.ws_n else None, self.ws_n, s)
        self.capi.check(rc, "nfpb200_forward")

    def bwd(self, i):
        s = torch.cuda.current_stream(self.dev).cuda_stream
        rc = self.lib.nfpb200_backward(ctypes.byref(self.desc_bwd), self.x[i].data_ptr(), self.gy[i].data_ptr(),
                                       self.gx[i].data_ptr(), self.ws.data_ptr() if self.ws_n else None,
                                       self.ws_n, s)
        self.capi.check(rc, "nfpb200_backward")

    def cold(self, i):
        """buffer set the backward of step i works on: not the one the step's forward has just read, so that x is
        HBM-cold for the backward too (in a network the backward of a layer runs long after its forward)"""
        return (i + self.nbuf // 2) % self.nbuf

    def step(self, i):                # the headline step: conservative backward (no x-stable hint)
        self.fwd(i)
        self.bwd_conservative(self.cold(i))

    def step_r1(self, i):             # round 1's definition: hinted backward on the buffers its forward has just read
        self.fwd(i)
        self.bwd(i)

    def step_hinted(self, i):         # backward with NFPB200_HINT_X_STABLE, as the autograd function passes it
        self.fwd(i)
        self.bwd(self.cold(i))

    def bwd_conservative(self, i):   # without NFPB200_HINT_X_STABLE: the backward waits for the preceding launch first
        s = torch.cuda.current_stream(self.dev).cuda_stream
        rc = self.lib.nfpb200_backward(ctypes.byref(self.desc), self.x[i].data_ptr(), self.gy[i].data_ptr(),
                                       self.gx[i].data_ptr(), self.ws.data_ptr() if self.ws_n else None,
                                       self.ws_n, s)
        self.capi.check(rc, "nfpb200_backward")

    def step_conservative(self, i):
        self.step(i)

    # pooled mode (the nfp_pooling head, models/NFP_Pooling.py:25-36): GAP(x) and GAP(NFP(x)) from one pass over x,
    # backward from their two gradients; the similarity map is never written
    def pool_setup(self):
        mkf = lambda *s: torch.randn(*s, device=self.dev, dtype=torch.float32)
        self.gap_x = [torch.empty(self.B, self.C, device=self.dev) for _ in range(self.nbuf)]
        self.gap_n = [torch.empty(self.B, self.K, device=self.dev) for _ in range(self.nbuf)]
        self.g_gap_x = [mkf(self.B, self.C) for _ in range(self.nbuf)]
        self.g_gap_n = [mkf(self.B, self.K) for _ in range(self.nbuf)]
        c = self.capi
        self.path_pool = c.describe_path(self.desc, c.OP_POOL_FORWARD), c.describe_path(self.desc, c.OP_POOL_BACKWARD)
        wsn = max(c.workspace_bytes(self.desc, c.OP_POOL_FORWARD), c.workspace_bytes(self.desc, c.OP_POOL_BACKWARD))
        if wsn > self.ws_n:
            self.ws = torch.empty(wsn, dtype=torch.uint8, device=self.dev)
            self.ws_n = wsn

    def pool_fwd(self, i):
        s = torch.cuda.current_stream(self.dev).cuda_stream
        rc = self.lib.nfpb200_pool_forward(ctypes.byref(self.desc), self.x[i].data_ptr(), self.gap_x[i].data_ptr(),
                                           self.gap_n[i].data_ptr(), self.ws.data_ptr() if self.ws_n else None,
                                           self.ws_n, s)
        self.capi.check(rc, "nfpb200_pool_forward")

    def pool_bwd(self, i):
        s = torch.cuda.current_stream(self.dev).cuda_stream
        rc = self.lib.nfpb200_pool_backward(ctypes.byref(self.desc_bwd), self.x[i].data_ptr(), self.g_gap_x[i].data_ptr(),
                                            self.g_gap_n[i].data_ptr(), self.gx[i].data_ptr(),
                                            self.ws.data_ptr() if self.ws_n else None, self.ws_n, s)
        self.capi.check(rc, "nfpb200_pool_backward")

    def pool_step(self, i):
        self.pool_fwd(i)
        self.pool_bwd(self.cold(i))

    def _graph(self, fn, n, start):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for j in range(n):
                fn((start + j) % self.nbuf)
        return g

    def timed(self, fn, steps, warmup, sampler=None, tag=None, barrier=None, chunk=250, windows=1, reduce=None):
        """Run `warmup` untimed calls, then `windows` timed windows of EXACTLY `steps` calls of fn each (graph
        replays, CUDA events on the launching stream, barrier + synchronize on both sides of every window).
        Returns the seconds of the MEDIAN window (after `reduce`, e.g. max over ranks, was applied to every window);
        with windows > 1 also leaves the per-window list in self.last_windows."""
        for j in range(max(warmup, 3)):
            fn(j % self.nbuf)
        torch.cuda.synchronize(self.dev)
        plan, done = [], 0
        graphs = {}
        while done < steps:
            n = min(chunk, steps - done)
            key = (n, done % self.nbuf)
            if key not in graphs:
                graphs[key] = self._graph(fn, n, done % self.nbuf)
            plan.append(graphs[key])
            done += n
        plan[0].replay()     # graph upload / first-replay cost stays outside the timed region
        torch.cuda.synchronize(self.dev)
        times = []
        for w in range(windows):
            if barrier:
                barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if sampler:
                sampler.tag = tag
            torch.cuda.synchronize(self.dev)
            e0.record()
            for g in plan:
                g.replay()
            e1.record()
            e1.synchronize()
            if sampler:
                sampler.tag = None
            torch.cuda.synchronize(self.dev)
            t = e0.elapsed_time(e1) * 1e-3
            times.append(reduce(t) if reduce else t)
        self.last_windows = times
        return sorted(times)[len(times) // 2]


def e2e_through_module(dev, B, C, H, W, R, dtype_name, steps, warmup, sampler, barrier):
    """Public-API path with host buffers: H2D(x, gy) -> NFPPooling fwd -> autograd bwd -> D2H(y, gx), every step.

    The three legs run on three CUDA streams over three device buffer sets, so the host->device copy of step i+1,
    the kernels of step i and the device->host copy of step i-1 overlap (PCIe is full duplex); every step still
    moves all of its inputs and results through pinned host memory inside the timed region."""
    import neighbour_feature_pooling_b200 as nfpb
    tdtype = torch.float32 if dtype_name == "fp32" else torch.bfloat16
    K = (2 * R + 1) ** 2 - 1
    layer = nfpb.NFPPooling(C, R=R, measure="cosine", padding=R).to(dev)
    gen = torch.Generator().manual_seed(1)
    nh, nd = 2, 3  # host buffer sets (alternated), device buffer sets (pipeline depth)
    hx = [torch.randn(B, C, H, W, generator=gen).to(tdtype).pin_memory() for _ in range(nh)]
    hg = [torch.randn(B, K, H, W, generator=gen).to(tdtype).pin_memory() for _ in range(nh)]
    hy = [torch.empty(B, K, H, W, dtype=tdtype).pin_memory() for _ in range(nh)]
    hgx = [torch.empty(B, C, H, W, dtype=tdtype).pin_memory() for _ in range(nh)]
    dx = [torch.empty(B, C, H, W, dtype=tdtype, device=dev) for _ in range(nd)]
    dg = [torch.empty(B, K, H, W, dtype=tdtype, device=dev) for _ in range(nd)]
    s_in, s_cmp, s_out = (torch.cuda.Stream(dev) for _ in range(3))
    ev_in = [torch.cuda.Event() for _ in range(nd)]
    ev_cmp = [None] * nd   # kernels of the step that last used device set j
    ev_out = [None] * nd   # D2H of the step that last used device set j
    keep = [None] * nd     # that step's y / grad_x: alive until its D2H is ordered before any reuse of their memory

    def one(i):
        j, h = i % nd, i % nh
        with torch.cuda.stream(s_in):
            if ev_cmp[j] is not None:
                s_in.wait_event(ev_cmp[j])          # the kernels that read this device set are done
            dx[j].copy_(hx[h], non_blocking=True)
            dg[j].copy_(hg[h], non_blocking=True)
            ev_in[j].record(s_in)
        with torch.cuda.stream(s_cmp):
            s_cmp.wait_event(ev_in[j])
            if ev_out[j] is not None:
                s_cmp.wait_event(ev_out[j])         # outputs of step i - nd have left the device:
            keep[j] = None                          # their blocks may be reused by this stream from here on
            x = dx[j].detach().requires_grad_(True)
            y = layer(x)
            y.backward(dg[j])
            keep[j] = (y.detach(), x.grad)
            ev_cmp[j] = torch.cuda.Event()
            ev_cmp[j].record(s_cmp)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_cmp[j])
            hy[h].copy_(keep[j][0], non_blocking=True)
            hgx[h].copy_(keep[j][1], non_blocking=True)
            ev_out[j] = torch.cuda.Event()
            ev_out[j].record(s_out)

    def drain():
        cur = torch.cuda.current_stream(dev)
        for st in (s_in, s_cmp, s_out):
            cur.wait_stream(st)

    for i in range(max(3, warmup)):
        one(i)
    torch.cuda.synchronize(dev)
    if barrier:
        barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.tag = "e2e"
    e0.record()
    for st in (s_in, s_cmp, s_out):
        st.wait_event(e0)
    for i in range(steps):
        one(i)
    drain()
    e1.record()
    e1.synchronize()
    sampler.tag = None
    esz = 4 if dtype_name == "fp32" else 2
    h2d = (B * C * H * W + B * K * H * W) * esz
    d2h = h2d
    t_e2e = e0.elapsed_time(e1) * 1e-3
    # the host-link ceiling of this step: the same pinned buffers copied in and out concurrently, no kernels, every rank
    # at once (all ranks share the host's memory / PCIe fabric, so the per-rank rate drops as ranks are added)
    dy_ = [torch.empty(B, K, H, W, dtype=tdtype, device=dev) for _ in range(nd)]
    dgx_ = [torch.empty(B, C, H, W, dtype=tdtype, device=dev) for _ in range(nd)]

    def copies(i):
        j, h = i % nd, i % nh
        with torch.cuda.stream(s_in):
            dx[j].copy_(hx[h], non_blocking=True)
            dg[j].copy_(hg[h], non_blocking=True)
        with torch.cuda.stream(s_out):
            hy[h].copy_(dy_[j], non_blocking=True)
            hgx[h].copy_(dgx_[j], non_blocking=True)
    for i in range(3):
        copies(i)
    torch.cuda.synchronize(dev)
    if barrier:
        barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for st in (s_in, s_out):
        st.wait_event(c0)
    for i in range(steps):
        copies(i)
    drain()
    c1.record()
    c1.synchronize()
    t_link = c0.elapsed_time(c1) * 1e-3
    link = {"seconds_per_step_copies_only": t_link / steps, "h2d_gbs_per_rank": h2d * steps / t_link / 1e9,
            "d2h_gbs_per_rank": d2h * steps / t_link / 1e9}
    return t_e2e, h2d, d2h, link


# ----------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the conv-form port of the reference on the host cores
# ----------------------------------------------------------------------------------------------
def cpu_model_name():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    import platform
    return platform.processor() or "unknown"


def cpu_ref_setup(C, H, W, R, dtype_name, B):
    """-> (callable running one fwd+bwd of the CPU arm on B maps, kind, description).

    kind "reference": the UNMODIFIED reference operator (models/pooling/nfp.py, read from NFP_REFERENCE_ROOT or from the
    copy __graft_entry__.build() staged under the git-ignored oracle/_ref/) -- NFPPooling(C, R, 'cosine', padding=R) forward
    + autograd backward.  kind "port": the same ATen operator sequence restated (oracle/nfp_convform.py), used only
    when the reference files are not there.  (bench.py's CPU legs are the only product-side use of oracle/.)"""
    tdtype = torch.float32 if dtype_name == "fp32" else torch.bfloat16
    K = (2 * R + 1) ** 2 - 1
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(B, C, H, W, generator=gen).to(tdtype)
    g = torch.randn(B, K, H, W, generator=gen).to(tdtype)
    from oracle import ref_loader
    if ref_loader.reference_available():
        RefNFP, _ = ref_loader.load_reference()
        layer = RefNFP(C, R=R, measure="cosine", padding=R).to(tdtype)

        def run():
            xr = x.detach().requires_grad_(True)
            y = layer(xr)
            y.backward(g)
            return y, xr.grad
        return run, "reference", ("the unmodified reference NFPPooling (models/pooling/nfp.py via oracle/ref_loader): "
                                  "reflect-pad + one-hot depthwise convs + F.cosine_similarity + autograd")
    from oracle.nfp_convform import ConvFormCosineNFP, forward_backward
    layer = ConvFormCosineNFP(C, R=R, padding=R).to(tdtype)
    return (lambda: forward_backward(layer, x, g)), "port", ("conv-form port of the reference's ATen chain "
                                                             "(oracle/nfp_convform.py; reference files not staged)")


def cpu_threads():
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    torch.set_num_threads(n)
    return n


def cpu_baseline(C, H, W, R, dtype_name, B, budget_s):
    cores = cpu_threads()
    Bs = min(B, 32)
    run, kind, what = cpu_ref_setup(C, H, W, R, dtype_name, Bs)
    run()
    t0 = time.perf_counter(); run(); dt = time.perf_counter() - t0
    rate = Bs / dt
    # size the timed sample to ~budget_s of wall time (x cores of CPU work), at most the full batch
    Bt = int(max(1, min(B, rate * budget_s / 3)))
    run, kind, what = cpu_ref_setup(C, H, W, R, dtype_name, Bt)
    run()
    reps, t = 0, 0.0
    while reps < 3 or (t < budget_s and reps < 10):
        t0 = time.perf_counter(); run(); t += time.perf_counter() - t0
        reps += 1
        if t > 2 * budget_s:
            break
    return {"value": reps * Bt / t, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model_name(),
            "sample": f"{reps} x fwd+bwd of B={Bt} maps (same shape/dtype), {what}, "
                      f"torch {torch.__version__} CPU, {cores} threads, {t:.1f} s"}


def run_reference_arm(args, C, H, W, where):
    """--impl reference: the reference's own CPU implementation of the path on the host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = cpu_threads()
    B = args.batch
    probe, kind, what = cpu_ref_setup(C, H, W, args.R, args.dtype, min(B, 16))
    probe()
    t0 = time.perf_counter(); probe(); rate = min(B, 16) / (time.perf_counter() - t0)
    total = args.steps + args.warmup
    Bs = int(max(1, min(B, rate * 150.0 / max(total, 1))))   # whole run within a few minutes
    run, kind, what = cpu_ref_setup(C, H, W, args.R, args.dtype, Bs)
    for _ in range(args.warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run()
    dt = time.perf_counter() - t0
    value = args.steps * Bs / dt
    sample = (f"each step = fwd+bwd of B={Bs} maps (bounded sample of the B={B} batch), {what}, "
              f"torch {torch.__version__} CPU, {cores} threads")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.dtype == "fp32" else "bf16", "data": "synthetic",
            "config": {"workload": workload_name(B, C, H, W, args.R, args.dtype), "source": where,
                       "batch_per_step": Bs, "cpu": cpu_model_name(),
                       "note": "the reference's CPU path on the host cores only (kind=reference: its own operator "
                               "files, unmodified; kind=port: the same ATen sequence restated)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model_name(),
                             "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, lb, step):
    """What a caller of the timed path receives from step `step` of a window (LayerBench.step): y of its forward and
    grad_x of its backward, as float32 DIR/y.npy and DIR/grad_x.npy.  Above DUMP_BYTES in all, the same seeded sample
    of batch rows is kept from both, their indices in DIR/batch_rows.npy."""
    import numpy as np
    i = step % lb.nbuf
    arrays = {"y": lb.y[i], "grad_x": lb.gx[lb.cold(i)]}
    n = min(lb.B, DUMP_BYTES // (sum(a[0].numel() for a in arrays.values()) * 4))
    if n == 0:
        raise SystemExit(f"--dump-outputs: one batch row of y and grad_x is larger than {DUMP_BYTES} bytes")
    os.makedirs(out_dir, exist_ok=True)
    if n < lb.B:
        rows = torch.randperm(lb.B, generator=torch.Generator().manual_seed(0))[:n].sort().values
        arrays = {k: a[rows.to(a.device)] for k, a in arrays.items()}
        np.save(os.path.join(out_dir, "batch_rows.npy"), rows.double().numpy())
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())


# ----------------------------------------------------------------------------------------------
_JSON_OUT = None


def claim_stdout():
    """stdout must carry exactly ONE JSON line: keep a private handle on it and point fd 1 at stderr, so that
    banners printed by libraries (NCCL prints its version on stdout) cannot get in front of the line."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    return _JSON_OUT


def emit(line):
    out = claim_stdout()
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    args = parse_args()
    claim_stdout()
    C, H, W, where = SHAPES[args.shape]
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs dumps the b200 arm; the reference arm sizes its batch by timing")
        run_reference_arm(args, C, H, W, where)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=b200) needs a CUDA device: the NFP operator has no CPU fallback")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"   # NCCL prints its version banner on stdout; stdout carries ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)

    def barrier():
        if dist is not None:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize(dev)

    def max_over_ranks(t):
        if dist is None:
            return t
        v = torch.tensor([t], device=dev, dtype=torch.float64)
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        return float(v.item())

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    B, R = args.batch, args.R
    sampler = ClockSampler(dev)
    sampler.start()

    lb = LayerBench(dev, B, C, H, W, R, args.dtype)
    # ---- value: K steps of fwd+bwd, device resident, HBM-cold via buffer rotation.  The K-step window is timed
    # `--windows` times (each bracketed by barrier + synchronize, max over ranks) and the MEDIAN window is reported:
    # at the driver's --steps 20 one window is 0.4 ms, where one late launch on one rank moves the number by 10 %.
    t_step_total = lb.timed(lb.step, args.steps, args.warmup, sampler, "timed", barrier, windows=args.windows,
                            reduce=max_over_ranks)
    window_ms = [t * 1e3 for t in lb.last_windows]
    if args.dump_outputs and rank == 0:   # before the passes below reuse the buffers
        dump_outputs(args.dump_outputs, lb, args.steps - 1)
    value = world * args.steps * B / t_step_total
    # ---- per-kernel launch durations (same rotation, back-to-back launches of one kernel) ---------
    sampler_tag = "kernels"
    nk = max(args.steps, 100)
    t_fwd = lb.timed(lb.fwd, nk, args.warmup, sampler, sampler_tag, windows=3) / nk
    t_bwd = lb.timed(lb.bwd_conservative, nk, args.warmup, sampler, sampler_tag, windows=3) / nk
    fwd_bytes, bwd_bytes = algorithmic_bytes(B, C, H, W, R, lb.esz)
    # the same with the x-stable hint (the backward may stream x while the preceding launch drains)
    n_cons = max(min(args.steps, 300), 100)
    t_step_hint = lb.timed(lb.step_hinted, n_cons, 5, sampler, "kernels", windows=3) / n_cons
    t_bwd_hint = lb.timed(lb.bwd, n_cons, 5, sampler, "kernels", windows=3) / n_cons
    t_step_r1 = lb.timed(lb.step_r1, n_cons, 5, sampler, "kernels", windows=3) / n_cons
    # ---- e2e through the nn.Module API with host buffers ------------------------------------------------
    e2e_steps = min(args.steps, 50)
    t_e2e, h2d, d2h, link = e2e_through_module(dev, B, C, H, W, R, args.dtype, e2e_steps, min(args.warmup, 5),
                                               sampler, barrier)
    t_e2e = max_over_ranks(t_e2e)
    e2e_value = world * e2e_steps * B / t_e2e
    t_link = max_over_ranks(link["seconds_per_step_copies_only"])
    link["ceiling_maps_per_s"] = world * B / t_link      # what the host link alone allows at this rank count
    link["e2e_fraction_of_ceiling"] = e2e_value / link["ceiling_maps_per_s"]
    link["note"] = ("copies only (same pinned buffers, both directions at once, all ranks concurrently): the e2e number "
                    "is bound by this, not by the kernels; pinned memory is not NUMA-bound per rank")

    # ---- pooled mode: the nfp_pooling head path (SURVEY 8 a6 / f1), same shape, device resident -----------------
    lb.pool_setup()
    n_pool = min(args.steps, 300)
    t_pool = lb.timed(lb.pool_step, n_pool, 5, sampler, "pooled") / n_pool
    t_pool_f = lb.timed(lb.pool_fwd, n_pool, 5, sampler, "pooled") / n_pool
    t_pool_b = lb.timed(lb.pool_bwd, n_pool, 5, sampler, "pooled") / n_pool
    pool_fb = B * (C * H * W * lb.esz + (C + lb.K) * 4)                # read x; write GAP(x), GAP(NFP(x))
    pool_bb = B * (2 * C * H * W * lb.esz + (C + lb.K) * 4)            # read x and the two gradients; write grad_x
    pooled = {"workload": "nfp_pooling head (GAP(x), GAP(NFP(x)) fwd + bwd) " + workload_name(B, C, H, W, R, args.dtype)[20:],
              "maps_per_s": B / t_pool, "us_per_step": t_pool * 1e6, "us_fwd": t_pool_f * 1e6, "us_bwd": t_pool_b * 1e6,
              "bytes_per_step": pool_fb + pool_bb, "step_frac": (pool_fb + pool_bb) / t_pool / 1e9 / hbm_peak,
              "fwd_frac": pool_fb / t_pool_f / 1e9 / hbm_peak, "bwd_frac": pool_bb / t_pool_b / 1e9 / hbm_peak,
              "path": {"forward": lb.path_pool[0], "backward": lb.path_pool[1]}}

    # ---- the other configs[1] cases (reported, not part of `value`) -------------------------------------
    sweep = []
    if not args.no_sweep and rank == 0:
        cases = [(shp, r, dt, "nchw") for shp in ("l4", "l3") for r in (1, 2) for dt in ("fp32", "bf16")]
        cases += [("mbv3", 1, "fp32", "nchw"), ("vit", 1, "bf16", "nchw"), ("eurosat", 1, "fp32", "nchw")]   # configs[3], [4], [2]
        # channels-last / token layout consumed in place by the tensor-core kernels (SURVEY 8 f2)
        cases += [("vit", 1, "bf16", "nhwc"), ("l4", 1, "bf16", "nhwc"), ("l4", 2, "bf16", "nhwc"), ("l3", 1, "bf16", "nhwc"),
                  ("mbv3", 1, "bf16", "nhwc")]
        for shp, r, dt, lay in cases:
            if True:
                if True:
                    c, h, w, _ = SHAPES[shp]
                    s = LayerBench(dev, B, c, h, w, r, dt, layout=lay)
                    n = max(min(args.steps, 200), 60)
                    tt = s.timed(s.step, n, 5, sampler, "sweep") / n
                    tf = s.timed(s.fwd, n, 5, sampler, "sweep") / n
                    tb = s.timed(s.bwd_conservative, n, 5, sampler, "sweep") / n
                    fb, bb = algorithmic_bytes(B, c, h, w, r, s.esz)
                    sweep.append({"workload": workload_name(B, c, h, w, r, dt) + (" channels-last" if lay == "nhwc" else ""),
                                  "maps_per_s": B / tt,
                                  "us_per_step": tt * 1e6, "us_fwd": tf * 1e6, "us_bwd": tb * 1e6,
                                  "step_gbs": (fb + bb) / tt / 1e9, "step_frac": (fb + bb) / tt / 1e9 / hbm_peak,
                                  "bwd_frac": bb / tb / 1e9 / hbm_peak, "fwd_frac": fb / tf / 1e9 / hbm_peak,
                                  "path": s.path_bwd})
                    del s
                    torch.cuda.empty_cache()
    # ---- SURVEY 8 f3: R = 1 and R = 2 on the same map (MultiRadiusNFPHead, models/nfp_heads.py:80-118) in ONE launch each
    # way (desc.inner_R) against the same kernels launched once per radius (the concatenation copies not even counted)
    multi = []
    if not args.no_sweep and rank == 0:
        by_name = {e["workload"]: e for e in sweep}
        for shp, dt, lay in (("l4", "fp32", "nchw"), ("l4", "bf16", "nhwc"), ("l3", "fp32", "nchw")):
            c, h, w, _ = SHAPES[shp]
            s = LayerBench(dev, B, c, h, w, 2, dt, layout=lay, inner_R=1)
            n = max(min(args.steps, 200), 60)
            tt = s.timed(s.step, n, 5, sampler, "sweep") / n
            sfx = " channels-last" if lay == "nhwc" else ""
            sep = [by_name.get(workload_name(B, c, h, w, r, dt) + sfx) for r in (1, 2)]
            multi.append({"workload": f"nfp_cosine_fwd_bwd B={B} {c}x{h}x{w} 3x3 + 5x5 maps (32 channels) {dt}{sfx}",
                          "us_per_step_one_launch": tt * 1e6, "path": s.path_bwd,
                          "us_per_step_launch_per_radius": (sep[0]["us_per_step"] + sep[1]["us_per_step"]) if all(sep) else None})
            del s
            torch.cuda.empty_cache()
    # ---- the five maps of MobileNetV3_MultiStageNFP (models/texture_pooling.py:211-268) fwd + bwd, B = 64: one CUDA-graph
    # replay of all ten calls (planar row-band kernels for the three large maps, ring kernels for the two small ones)
    multi_stage = None
    if not args.no_sweep and rank == 0:
        maps = [(16, 112, 112), (24, 56, 56), (40, 28, 28), (112, 14, 14), (960, 7, 7)]
        lbs = [LayerBench(dev, 64, c, h, w, 1, "fp32") for c, h, w in maps]

        def all_maps(i):
            for s_ in lbs:
                s_.fwd(i % s_.nbuf)
            for s_ in reversed(lbs):
                s_.bwd_conservative(i % s_.nbuf)
        for i in range(3):
            all_maps(i)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(4):
                all_maps(i)
        g.replay()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.tag = "sweep"
        e0.record()
        for _ in range(10):
            g.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        sampler.tag = None
        algo = sum(sum(algorithmic_bytes(64, c, h, w, 1, 4)) for c, h, w in maps)
        t_set = e0.elapsed_time(e1) * 1e-3 / 40
        multi_stage = {"workload": "nfp_cosine_fwd_bwd B=64 fp32, the five maps of MobileNetV3_MultiStageNFP "
                                   "(16x112x112, 24x56x56, 40x28x28, 112x14x14, 960x7x7)",
                       "us_per_set": t_set * 1e6, "launches_per_set": sum(s_.launches for s_ in lbs),
                       "paths": [s_.path_bwd for s_ in lbs], "set_frac": algo / t_set / 1e9 / hbm_peak}
        del lbs, g
        torch.cuda.empty_cache()
    # ---- metric part (ii): ResNet18 + NFP training images/s (DDP over NCCL when N > 1) ---------------------------
    train = None
    if not args.no_train:
        try:
            import bench_train
            sampler.tag = "train"
            train = bench_train.run_gpu(args.train_config, args.train_batch, args.train_steps, 5)
            sampler.tag = None
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                train["cpu_baseline"] = bench_train.run_cpu_baseline(args.train_config)
            # the other BASELINE.json configs: [3] MobileNetV3+NFP (64 per GPU = 512 over 8), [4] ViT-Tiny+NFP bf16,
            # [0] ResNet18+NFP batch 8 3x224x224 (beside the reference's CPU time for exactly that case)
            more = []
            for name in [c for c in args.train_more.split(",") if c]:
                cfgm = bench_train.CONFIGS[name]
                bsz = 8 if name == "ucmerced" else cfgm.get("batch", args.train_batch)
                sampler.tag = "train"
                r = bench_train.run_gpu(name, bsz, args.train_steps, 5)
                sampler.tag = None
                r["config"] = name
                if name == "ucmerced" and rank == 0 and world == 1 and not args.no_cpu_baseline:
                    r["cpu_baseline"] = bench_train.run_cpu_baseline("ucmerced", batch=8, steps=2)
                more.append(r)
            train["more_configs"] = more
        except Exception as e:  # e.g. torchvision missing: report it, keep the layer numbers
            sampler.tag = None
            train = {"unavailable": repr(e)[:300]}
    sampler.stop()
    barrier()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(C, H, W, R, args.dtype, B, args.cpu_seconds)

    if rank == 0:
        achieved = bwd_bytes / t_bwd / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_step_total / args.steps * 1e3, "higher_is_better": True,
            "windows": {"n": len(window_ms), "steps_each": args.steps, "reported": "median window, max over ranks per window",
                        "ms": [round(v, 5) for v in window_ms]},
            "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.dtype == "fp32" else "bf16",
            "data": "synthetic",
            "config": {"workload": workload_name(B, C, H, W, R, args.dtype), "source": where,
                       "batch_per_gpu": B, "global_batch": B * world, "sharding": f"batch over {world} GPU(s), no collective",
                       "l2_hygiene": f"inputs/outputs rotate over {lb.nbuf} buffer sets "
                                     f"({lb.nbuf * lb.set_bytes / 2**20:.0f} MiB > 2x the 126 MiB L2); a step's backward works "
                                     f"on the set {lb.nbuf // 2} positions away from its forward's, so every kernel reads "
                                     "HBM-cold inputs",
                       "launch": "CUDA graph of C-ABI launches (nfpb200_forward + nfpb200_backward per step; conservative "
                                 "backward: no NFPB200_HINT_X_STABLE -- see with_x_stable_hint for the hinted order)",
                       "kernel_path": {"forward": lb.path_fwd, "backward": lb.path_bwd}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": t_e2e / e2e_steps * 1e3, "host_link": link,
                    "api": "NFPPooling(C,R,'cosine',padding=R).forward + autograd backward; pinned host x, grad_y -> "
                           "device; y, grad_x -> pinned host, every step; copy-in / kernels / copy-out on three "
                           "streams over three device buffer sets (pipelined, PCIe full duplex)"},
            "gpu_launches": args.steps * lb.launches,
            "roofline": {"bound": "hbm", "kernel": "nfpb200_backward (" + lb.path_bwd + ")", "achieved": achieved,
                         "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": None,
                         "peak_source": peak_src, "bytes_per_launch": bwd_bytes, "us_per_launch": t_bwd * 1e6},
            "roofline_forward": {"kernel": "nfpb200_forward (" + lb.path_fwd + ")", "achieved": fwd_bytes / t_fwd / 1e9,
                                 "frac": fwd_bytes / t_fwd / 1e9 / hbm_peak, "bytes_per_launch": fwd_bytes,
                                 "us_per_launch": t_fwd * 1e6},
            "roofline_step": {"achieved": (fwd_bytes + bwd_bytes) * args.steps / t_step_total / 1e9,
                              "frac": (fwd_bytes + bwd_bytes) * args.steps / t_step_total / 1e9 / hbm_peak,
                              "bytes_per_step": fwd_bytes + bwd_bytes,
                              "bwd_share_of_step": t_bwd / (t_fwd + t_bwd)},
            "with_x_stable_hint": {"us_per_step": t_step_hint * 1e6, "us_bwd": t_bwd_hint * 1e6,
                                   "maps_per_s": world * B / t_step_hint,
                                   "step_frac": (fwd_bytes + bwd_bytes) / t_step_hint / 1e9 / hbm_peak,
                                   "bwd_frac": bwd_bytes / t_bwd_hint / 1e9 / hbm_peak,
                                   "us_per_step_round1_definition": t_step_r1 * 1e6,
                                   "round1_definition": "hinted backward on the buffer set its forward has just read (x L2-warm): "
                                                        "what BENCH_r01's `value` measured; kept for round-over-round comparison",
                                   "note": "NFPB200_HINT_X_STABLE (include/nfp_b200.h; what the autograd function passes: "
                                           "x is a saved activation) lets a fused backward stream x while the preceding "
                                           "launch drains; it only pays when NFP launches are adjacent on the stream, as "
                                           "in this microbenchmark, so it is NOT the headline"},
            "clocks": sampler.summary(),
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        line["pooled"] = pooled
        if sweep:
            line["sweep"] = sweep
        if multi:
            line["multi_radius"] = multi
        if multi_stage:
            line["multi_stage"] = multi_stage
        if train is not None:
            line["train"] = train
        traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
        try:  # dram bytes per launch from the committed ncu --set full capture of this kernel, if any
            with open(traffic_file) as f:
                tr = json.load(f)
            key = workload_name(B, C, H, W, R, args.dtype)
            if key in tr:
                line["roofline"]["traffic"] = tr[key]["backward_dram_bytes"]
                line["roofline"]["traffic_source"] = tr[key].get("source")
        except Exception:
            pass
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
