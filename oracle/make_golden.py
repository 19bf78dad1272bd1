"""TEST INFRASTRUCTURE ONLY -- generate golden vectors from the reference.

Needs a checkout of the original project:

    NFP_REFERENCE_ROOT=/path/to/Neighbour_Feature_Pooling python -m oracle.make_golden

Executes the *unmodified* reference ``NFPPooling`` / ``nfp_pooling`` modules on
seeded inputs and stores inputs, outputs and input-gradients as small ``.npz``
fixtures under ``tests/golden/``.  The reference cannot travel to the GPU box,
the fixtures can.  Inputs are fp32 values; the reference is evaluated in fp64 on
those values (the exact answer) and, for the cosine hot path, also in fp32 (the
reference's own rounding noise, used to size the tolerances).
"""
from __future__ import annotations

import json
import os

import numpy as np
import torch

from . import nfp_oracle as O
from .ref_loader import load_reference

OUT_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# name -> (B, C, H, W, R, stride, padding, dilation, padding_mode)
GEOMS = {
    "l4_3x3": (2, 8, 7, 7, 1, 1, 1, 1, "reflect"),      # layer4-shaped, the live nfp_pooling config
    "l3_5x5": (1, 6, 14, 14, 2, 1, 2, 1, "reflect"),    # layer3-shaped, 5x5 (hot-path measures only)
    "r2": (1, 4, 6, 5, 2, 1, 2, 1, "reflect"),          # small 5x5 case for every measure
    "odd": (2, 5, 6, 9, 1, 2, 2, 2, "reflect"),          # stride 2, dilation 2, pad > R... non-square
    "zeros": (2, 4, 5, 6, 1, 1, 1, 1, "zeros"),
    "eurosat": (3, 8, 2, 2, 1, 1, 1, 1, "reflect"),
}
MEASURE_SPELLINGS = list(O.MEASURES) + ["sharpened_cosine", "Norm", "RMSE"]


def _case(NFPPooling, measure, geom, similarity, p, seed, relu):
    B, C, H, W, R, s, pad, d, mode = geom
    gen = torch.Generator().manual_seed(seed)
    x32 = torch.randn(B, C, H, W, generator=gen, dtype=torch.float32)
    if relu:
        x32 = x32.relu()
    ref = NFPPooling(C, R=R, measure=measure, p=p, stride=s, padding=pad, dilation=d,
                     padding_mode=mode, similarity=similarity)
    out = {}
    for tag, dt in (("f64", torch.float64), ("f32", torch.float32)):
        m = ref.to(dt)
        xr = x32.to(dt).clone().requires_grad_(True)
        y = m(xr)
        if tag == "f64":
            g32 = torch.randn(y.shape, generator=gen, dtype=torch.float32)
        (gx,) = torch.autograd.grad(y, xr, g32.to(dt))
        out["y_" + tag] = y.detach().numpy()
        out["gx_" + tag] = gx.numpy()
    out["x"] = x32.numpy()
    out["g"] = g32.numpy()
    return out


def multi_radius(NFPPooling):
    """The operator inside the reference's MultiRadiusNFPHead (models/nfp_heads.py:86-93,111-112), executed with the
    reference's own NFPPooling (the head's EnhancedNFPPooling is the symbol the reference does not ship): R_list = (1, 2),
    padding = R, then torch.cat along the channels; fp64 on fp32 values, input gradient for a seeded upstream gradient."""
    arrays, index = {}, []
    for i, (B, C, H, W, mode, similarity) in enumerate([(3, 64, 7, 7, "reflect", True), (2, 16, 14, 14, "reflect", True),
                                                       (2, 64, 7, 7, "replicate", False), (2, 8, 7, 7, "zeros", True)]):
        gen = torch.Generator().manual_seed(4000 + i)
        x32 = torch.randn(B, C, H, W, generator=gen)
        if i % 2 == 0:
            x32 = x32.relu()
        blocks = [NFPPooling(C, R=R, measure="cosine", padding=R, padding_mode=mode, similarity=similarity).double()
                  for R in (1, 2)]
        xr = x32.double().requires_grad_(True)
        nfp_maps = [blk(xr) for blk in blocks]
        nfp_cat = torch.cat(nfp_maps, dim=1)
        g32 = torch.randn(nfp_cat.shape, generator=gen)
        (gx,) = torch.autograd.grad(nfp_cat, xr, g32.double())
        key = f"m{i}"
        arrays.update({f"{key}_x": x32.numpy(), f"{key}_g": g32.numpy(), f"{key}_y": nfp_cat.detach().numpy(),
                       f"{key}_gx": gx.numpy()})
        index.append(dict(key=key, B=B, C=C, H=H, W=W, padding_mode=mode, similarity=similarity))
    np.savez_compressed(os.path.join(OUT_DIR, "nfp_multi_radius.npz"), **arrays)
    with open(os.path.join(OUT_DIR, "nfp_multi_radius.json"), "w") as f:
        json.dump(dict(generator="oracle/make_golden.py --multi-radius", torch=torch.__version__,
                       reference="models/pooling/nfp.py NFPPooling x 2 (R = 1, 2; padding = R) + torch.cat, as "
                                 "models/nfp_heads.py:86-93,111-112 composes them (unmodified, CPU, fp64)",
                       cases=index), f, indent=1)


def main():
    NFPPooling, nfp_pooling = load_reference()
    os.makedirs(OUT_DIR, exist_ok=True)
    import sys
    if "--multi-radius" in sys.argv:   # only this fixture (the others stay byte-identical)
        multi_radius(NFPPooling)
        print("multi-radius fixture written to", OUT_DIR)
        return
    arrays, index = {}, []
    cid = 0
    for measure in MEASURE_SPELLINGS:
        for gname, geom in GEOMS.items():
            for similarity in (True, False):
                if similarity is False and gname not in ("l4_3x3", "zeros"):
                    continue
                if gname == "l3_5x5" and measure not in ("cosine", "dot", "norm"):
                    continue
                ps = (1, 2) if measure.lower() in ("norm", "scs", "sharpened_cosine") else (1,)
                for p in ps:
                    relu = (cid % 3 == 2)
                    c = _case(NFPPooling, measure, geom, similarity, p, seed=1000 + cid, relu=relu)
                    key = f"c{cid:03d}"
                    for k, v in c.items():
                        if k.endswith("f32") and measure.lower() != "cosine":
                            continue  # fp32 noise is only recorded for the hot-path measure
                        arrays[f"{key}_{k}"] = v
                    index.append(dict(key=key, measure=measure, geom=gname, B=geom[0], C=geom[1],
                                      H=geom[2], W=geom[3], R=geom[4], stride=geom[5],
                                      padding=geom[6], dilation=geom[7], padding_mode=geom[8],
                                      similarity=similarity, p=p, relu=relu))
                    cid += 1
    half = len(index) // 2   # two files by case, each under 1 MB (tests/_util.py merges them)
    for part, cases in ((1, index[:half]), (2, index[half:])):
        keys = {c["key"] for c in cases}
        np.savez_compressed(os.path.join(OUT_DIR, f"nfp_measures_{part}.npz"),
                            **{k: v for k, v in arrays.items() if k.split("_")[0] in keys})
    with open(os.path.join(OUT_DIR, "nfp_measures.json"), "w") as f:
        json.dump(dict(generator="oracle/make_golden.py", torch=torch.__version__,
                       reference="models/pooling/nfp.py NFPPooling (unmodified, CPU)",
                       cases=index), f, indent=1)

    # the pooling wrapper, NFP_Pooling.py:25-36 (ResNet18-like C, layer4 7x7 and ViT 14x14 maps)
    arrays, index = {}, []
    for i, (B, C, H, W) in enumerate([(3, 16, 7, 7), (2, 12, 14, 14), (4, 8, 2, 2)]):
        Params = {"num_ftrs": {"m": C}, "Model_name": "m", "Dataset": "d", "num_classes": {"d": 5}}
        torch.manual_seed(2000 + i)
        pool = nfp_pooling(Params=Params)
        gen = torch.Generator().manual_seed(3000 + i)
        x32 = torch.randn(B, C, H, W, generator=gen).relu()
        g32 = torch.randn(B, C, generator=gen)
        pool64 = pool.double()
        xr = x32.double().requires_grad_(True)
        out = pool64(xr)
        gx, gw, gb = torch.autograd.grad(out, (xr, pool64.nfp_proj.weight, pool64.nfp_proj.bias),
                                         g32.double())
        key = f"p{i}"
        arrays.update({f"{key}_x": x32.numpy(), f"{key}_g": g32.numpy(),
                       f"{key}_w": pool.nfp_proj.weight.detach().float().numpy(),
                       f"{key}_b": pool.nfp_proj.bias.detach().float().numpy(),
                       f"{key}_out": out.detach().numpy(), f"{key}_gx": gx.numpy(),
                       f"{key}_gw": gw.numpy(), f"{key}_gb": gb.numpy()})
        index.append(dict(key=key, B=B, C=C, H=H, W=W))
    np.savez_compressed(os.path.join(OUT_DIR, "nfp_pooling_wrapper.npz"), **arrays)
    with open(os.path.join(OUT_DIR, "nfp_pooling_wrapper.json"), "w") as f:
        json.dump(dict(generator="oracle/make_golden.py", torch=torch.__version__,
                       reference="models/NFP_Pooling.py nfp_pooling (unmodified, CPU)",
                       cases=index), f, indent=1)

    # reference state_dict layout (SURVEY.md 3.4): keys, shapes and the one-hot contents
    sd = NFPPooling(3, R=1, measure="cosine", padding=1).state_dict()
    sdn = NFPPooling(3, R=1, measure="norm", padding=1).state_dict()
    np.savez_compressed(os.path.join(OUT_DIR, "nfp_state_dict.npz"),
                        **{"cosine_" + k: v.numpy() for k, v in sd.items()},
                        **{"norm_" + k: v.numpy() for k, v in sdn.items()})
    multi_radius(NFPPooling)
    print("golden fixtures written to", OUT_DIR)
    for fn in sorted(os.listdir(OUT_DIR)):
        print(f"  {fn}: {os.path.getsize(os.path.join(OUT_DIR, fn))} bytes")


if __name__ == "__main__":
    main()
