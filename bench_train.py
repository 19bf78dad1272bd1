"""End-to-end ResNet18 + NFP training step (BASELINE.json metric part ii: images/s at 1/2/4/8 GPU).

Imported by bench.py (`train` object of the JSON line) and runnable on its own:

    python bench_train.py [--config eurosat|ucmerced] [--batch 256] [--steps 20] [--warmup 5]
    torchrun --nproc-per-node N bench_train.py ...

The model mirrors the reference's `ResNet18_NFPPooling` (models/texture_pooling.py:153-167): backbone
`forward_features` -> `nfp_pooling` (this package's drop-in: fused GAP(x), GAP(NFP(x)) kernels) -> `fc`, trained with
the reference's step (`Lightning_Wrapper.training_step`, lightning_wrappers/Lightning_Wrapper.py:81-105 and :69-79):
CrossEntropyLoss(label_smoothing=0.05) + Adam(lr).  timm is not installed in this image, so the backbone is
torchvision's resnet18 with random weights (same architecture; first conv widened for the 13-band EuroSAT input, as timm's
`in_chans` does).  Data are synthetic.  Multi-GPU = DistributedDataParallel over NCCL, batch-sharded (weak scaling):
the NFP path itself has no collective; only backbone / nfp_proj / fc gradients are all-reduced.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

CONFIGS = {  # BASELINE.json configs[2] and configs[0]; `raw` = the dtype the dataset's pixels are stored in
    "eurosat": dict(in_chans=13, size=64, classes=10, raw=torch.int16, raw_max=10000.0,
                    name="ResNet18+NFP EuroSAT-shaped 13x64x64 (16-bit bands), 10 classes (layer4 map 512x2x2)"),
    "ucmerced": dict(in_chans=3, size=224, classes=21, raw=torch.uint8, raw_max=255.0,
                     name="ResNet18+NFP UCMerced-shaped 3x224x224 (8-bit RGB), 21 classes (layer4 map 512x7x7)"),
    # BASELINE.json configs[3]: MobileNetV3 + NFP head (models/texture_pooling.py:191-207), GTOS-Mobile-shaped, 31 classes;
    # global batch 512 over 8 GPUs = 64 per GPU
    "gtos_mbv3": dict(arch="mbv3", feat=960, in_chans=3, size=224, classes=31, raw=torch.uint8, raw_max=255.0, batch=64,
                      name="MobileNetV3-large+NFP GTOS-Mobile-shaped 3x224x224, 31 classes (last-stage map 960x7x7)"),
    # BASELINE.json configs[4]: ViT-Tiny + NFP over the 14x14x192 token grid (models/texture_pooling.py:169-189), bf16
    "plantvillage_vit": dict(arch="vit", feat=192, in_chans=3, size=224, classes=38, raw=torch.uint8, raw_max=255.0,
                             batch=64, name="ViT-Tiny/16+NFP PlantVillage-shaped 3x224x224, 38 classes "
                                            "(token grid 14x14x192, consumed as the reference's transpose/reshape VIEW)"),
}


class ResNet18Features(nn.Module):
    """torchvision resnet18 up to layer4 == timm's `forward_features` for resnet18."""

    def __init__(self, in_chans):
        super().__init__()
        import torchvision
        m = torchvision.models.resnet18(weights=None)
        if in_chans != 3:
            m.conv1 = nn.Conv2d(in_chans, 64, kernel_size=7, stride=2, padding=3, bias=False)
        self.body = nn.Sequential(m.conv1, m.bn1, m.relu, m.maxpool, m.layer1, m.layer2, m.layer3, m.layer4)

    def forward(self, x):
        return self.body(x)


class ResNet18_NFPPooling(nn.Module):
    """Same composition as the reference class of that name (models/texture_pooling.py:153-167)."""

    def __init__(self, num_classes, in_chans, pool):
        super().__init__()
        self.backbone = ResNet18Features(in_chans)
        self.pool = pool
        self.fc = nn.Linear(512, num_classes)

    def forward(self, x):
        return self.fc(self.pool(self.backbone(x)))


class MobileNetV3_NFPPooling(nn.Module):
    """models/texture_pooling.py:191-207 with torchvision's mobilenet_v3_large().features standing in for timm's
    mobilenetv3_large_100 forward_features (same 960 x 7 x 7 last-stage map; random init)."""

    def __init__(self, num_classes, pool):
        super().__init__()
        import torchvision
        self.backbone = torchvision.models.mobilenet_v3_large(weights=None).features
        self.pool = pool
        self.fc = nn.Linear(960, num_classes)

    def forward(self, x):
        return self.fc(self.pool(self.backbone(x)))


class ViTTiny_NFPPooling(nn.Module):
    """models/texture_pooling.py:169-189 with torchvision's VisionTransformer(224, 16, 12 layers, 3 heads, 192, 768)
    standing in for timm's vit_tiny_patch16_224 forward_features: tokens (B, 197, 192) -> drop the class token ->
    transpose(1, 2).reshape(B, C, H, W) (a VIEW: channels-last memory) -> nfp_pooling -> fc."""

    def __init__(self, num_classes, pool):
        super().__init__()
        import torchvision
        self.backbone = torchvision.models.VisionTransformer(image_size=224, patch_size=16, num_layers=12, num_heads=3,
                                                             hidden_dim=192, mlp_dim=768, num_classes=1)
        self.backbone.heads = nn.Identity()
        self.pool = pool
        self.fc = nn.Linear(192, num_classes)

    def forward_features(self, x):
        vt = self.backbone
        x = vt._process_input(x)
        x = torch.cat([vt.class_token.expand(x.shape[0], -1, -1), x], dim=1)
        return vt.encoder(x)

    def forward(self, x):
        feats = self.forward_features(x)
        patch_tokens = feats[:, 1:]
        B, N, C = patch_tokens.shape
        H = W = int(N ** 0.5)
        fmap = patch_tokens.transpose(1, 2).reshape(B, C, H, W)
        return self.fc(self.pool(fmap))


def make_model(cfg, device, impl="b200"):
    arch, feat = cfg.get("arch", "resnet18"), cfg.get("feat", 512)
    Params = {"num_ftrs": {arch: feat}, "Model_name": arch, "Dataset": "synthetic",
              "num_classes": {"synthetic": cfg["classes"]}, "input_size": cfg["size"] // 32 if arch != "vit" else 14}
    if impl == "b200":
        import neighbour_feature_pooling_b200 as nfpb
        pool = nfpb.nfp_pooling(Params=Params)
    else:  # CPU baseline: the reference's own nfp_pooling (staged under oracle/_ref), else its conv-form port
        from oracle import ref_loader
        if ref_loader.reference_available():
            _, ref_pool = ref_loader.load_reference()
            pool = ref_pool(Params=Params)
        else:
            from oracle.nfp_convform import ConvFormCosineNFP

            class RefPool(nn.Module):
                def __init__(self):
                    super().__init__()
                    self.nfp_layer = ConvFormCosineNFP(feat, R=1, padding=1)
                    self.nfp_proj = nn.Linear(8, feat)

                def forward(self, x):
                    return x.mean((2, 3)) * self.nfp_proj(self.nfp_layer(x).mean((2, 3)))
            pool = RefPool()
    if arch == "mbv3":
        return MobileNetV3_NFPPooling(cfg["classes"], pool).to(device)
    if arch == "vit":
        return ViTTiny_NFPPooling(cfg["classes"], pool).to(device)
    return ResNet18_NFPPooling(cfg["classes"], cfg["in_chans"], pool).to(device)


def run_gpu(config="eurosat", batch=256, steps=20, warmup=5, amp=True, use_graph=True):
    """Returns a dict with images/s of the (DDP) training step; uses the current process group if any.

    The whole step (forward, backward with DDP's bucketed NCCL all-reduce, Adam) is captured in ONE CUDA graph and
    replayed; if capture fails the eager step is timed instead and the reason is reported."""
    import torch.distributed as dist
    cfg = CONFIGS[config]
    loss_scale = 1.0
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(1234)
    torch.backends.cudnn.benchmark = True
    main = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(dev)   # DDP + graph capture: build and warm up on a side stream (PyTorch CUDA-graphs notes)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        model = make_model(cfg, dev).to(memory_format=torch.channels_last)
        if world > 1:
            # BatchNorm statistics stay per rank (the reference trains on one GPU; SURVEY 8 e1), so DDP's per-forward
            # buffer broadcast is off unless NFP_DDP_BROADCAST_BUFFERS=1
            model = nn.parallel.DistributedDataParallel(
                model, device_ids=[dev.index], gradient_as_bucket_view=True,
                bucket_cap_mb=int(os.environ.get("NFP_DDP_BUCKET_MB", "25")),
                broadcast_buffers=os.environ.get("NFP_DDP_BROADCAST_BUFFERS", "0") == "1",
                static_graph=os.environ.get("NFP_DDP_STATIC_GRAPH", "0") == "1")
            if os.environ.get("NFP_DDP_BF16_HOOK", "0") == "1":
                from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
                model.register_comm_hook(None, default_hooks.bf16_compress_hook)
            elif os.environ.get("NFP_DDP_SUM_HOOK", "0") == "1":
                # DDP's default path divides every parameter's gradient by the world size with its own small kernel
                # (56 launches, 155 us per step at N = 8: profiles/r02_train_timeline_n8.txt).  A SUM all-reduce of the
                # bucket with the 1/world factor folded into the loss is the same average with no extra kernel.
                def sum_hook(state, bucket):
                    return dist.all_reduce(bucket.buffer(), async_op=True).get_future().then(lambda f: f.value()[0])
                model.register_comm_hook(None, sum_hook)
                loss_scale = 1.0 / world
        opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-4, capturable=use_graph)
    crit = nn.CrossEntropyLoss(label_smoothing=0.05)
    gen = torch.Generator().manual_seed(100 + rank)
    nhost = 3  # pinned host batches, rotated: every step does its own H2D copy like a DataLoader would
    # synthetic batches in the dataset's storage dtype (EuroSAT: 16-bit digital numbers, UCMerced: 8-bit RGB);
    # normalisation to float happens on the GPU inside the step, as a GPU-side data pipeline would do it
    hx = [torch.randint(0, int(cfg["raw_max"]), (batch, cfg["in_chans"], cfg["size"], cfg["size"]), generator=gen,
                        dtype=torch.int32).to(cfg["raw"]).pin_memory() for _ in range(nhost)]
    hy = [torch.randint(0, cfg["classes"], (batch,), generator=gen).pin_memory() for _ in range(nhost)]
    scale, shift = 2.0 / cfg["raw_max"], -1.0

    # input pipeline: the next batch is copied host->device on a copy stream while the current step computes
    # (what a DataLoader with pin_memory + non_blocking copies does); every step still moves its own batch.
    copy_stream = torch.cuda.Stream(dev)
    dx = [torch.empty((batch, cfg["in_chans"], cfg["size"], cfg["size"]), device=dev, dtype=cfg["raw"]) for _ in range(2)]
    dy = [torch.empty((batch,), dtype=torch.long, device=dev) for _ in range(2)]
    sx, sy = torch.empty_like(dx[0]), torch.empty_like(dy[0])   # static inputs of the captured step
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        b = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])
            dx[b].copy_(hx[i % nhost], non_blocking=True)
            dy[b].copy_(hy[i % nhost], non_blocking=True)
            ready[b].record(copy_stream)

    def train_step(xraw, y):
        x = (xraw.float() * scale + shift).contiguous(memory_format=torch.channels_last)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            loss = crit(model(x).float(), y)
        opt.zero_grad(set_to_none=True)
        (loss * loss_scale if loss_scale != 1.0 else loss).backward()
        opt.step()
        return loss

    graph, graph_note, static_loss = None, None, None
    from neighbour_feature_pooling_b200 import functional as _NF
    _NF.PATH_TRACE = set()
    with torch.cuda.stream(side):
        sx.copy_(hx[0], non_blocking=True)
        sy.copy_(hy[0], non_blocking=True)
        for _ in range(11 if use_graph else 2):   # DDP needs >= 11 eager iterations before capture
            train_step(sx, sy)
    main.wait_stream(side)
    torch.cuda.synchronize(dev)
    nfp_paths, _NF.PATH_TRACE = sorted(_NF.PATH_TRACE), None
    if use_graph:
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_loss = train_step(sx, sy)
            graph.replay()
            torch.cuda.synchronize(dev)
        except Exception as e:  # report and fall back to the eager step
            graph, graph_note = None, repr(e)[:200]
            torch.cuda.synchronize(dev)

    for e in consumed:
        e.record(main)
    prefetch(0)

    def step(i):
        b = i % 2
        prefetch(i + 1)
        main.wait_event(ready[b])
        sx.copy_(dx[b], non_blocking=True)
        sy.copy_(dy[b], non_blocking=True)
        consumed[b].record(main)
        if graph is not None:
            graph.replay()
            return static_loss
        return train_step(sx, sy)

    for i in range(warmup):
        loss = step(i)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier(device_ids=[dev.index])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        loss = step(i)
    lossv = float(loss.item())  # device->host read of the step's result inside the timed region
    e1.record()
    e1.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    if world > 1:
        tt = torch.tensor([t], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t = float(tt.item())
    out = {"workload": cfg["name"], "images_per_s": world * steps * batch / t, "ms_per_step": t / steps * 1e3,
           "batch_per_gpu": batch, "global_batch": batch * world, "n_gpus": world, "steps": steps, "warmup": warmup,
           "dtype": "bf16 autocast (NFP kernels: bf16 I/O, fp32 accumulate)" if amp else "fp32",
           "parallelism": f"DDP over NCCL, dp{world}, weak scaling" if world > 1 else "single GPU",
           "optimizer": "Adam(lr=1e-4), CrossEntropy(label_smoothing=0.05)",
           "backbone": {"resnet18": "torchvision resnet18", "mbv3": "torchvision mobilenet_v3_large().features",
                        "vit": "torchvision VisionTransformer(224, 16, 12, 3, 192, 768)"}[cfg.get("arch", "resnet18")]
                       + " (random init; timm absent), channels_last",
           "cuda_graph": graph is not None, "nfp_kernel_paths": nfp_paths,
           "h2d_bytes_per_step": hx[0].numel() * hx[0].element_size() + hy[0].numel() * 8, "final_loss": lossv, "data": "synthetic"}
    if graph_note:
        out["cuda_graph_error"] = graph_note
    return out


def run_cpu_baseline(config="eurosat", batch=8, steps=2):
    """The reference's CPU path for the same step (conv-form NFP port, fp32), bounded sample."""
    cfg = CONFIGS[config]
    torch.manual_seed(1234)
    model = make_model(cfg, torch.device("cpu"), impl="reference")
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    crit = nn.CrossEntropyLoss(label_smoothing=0.05)
    x = torch.randn(batch, cfg["in_chans"], cfg["size"], cfg["size"])
    y = torch.randint(0, cfg["classes"], (batch,))

    def step():
        loss = crit(model(x), y)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    from oracle import ref_loader
    return {"images_per_s": steps * batch / dt, "cores": torch.get_num_threads(),
            "kind": "reference" if ref_loader.reference_available() else "port",
            "sample": f"{steps} x fwd+bwd+Adam of batch {batch}, fp32, torch {torch.__version__} CPU"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="eurosat", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--fp32", action="store_true")
    ap.add_argument("--cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    args = ap.parse_args()
    import bench
    bench.claim_stdout()
    import torch.distributed as dist
    from neighbour_feature_pooling_b200 import sharding
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    rank, _, world = sharding.init_from_env("nccl", torch.device("cuda", local))
    out = run_gpu(args.config, args.batch, args.steps, args.warmup, amp=not args.fp32, use_graph=not args.no_graph)
    if rank == 0:
        if args.cpu_baseline:
            out["cpu_baseline"] = run_cpu_baseline(args.config)
        import bench
        bench.emit(out)
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
