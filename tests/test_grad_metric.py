"""CPU: the input-gradient error norm of the GPU suite (grad_err, tests/_util.py) can see the bugs it is meant to
catch, passes an honest fp32 evaluation, and the grid of tests/test_grad_parity_gpu.py reaches every (kernel family,
op, padding mode, similarity, dtype) cell it is meant to cover.  No GPU: the oracle runs on the CPU, and the kernel
paths come from the library's host-only nfpb200_describe_path."""
import numpy as np
import pytest
import torch

from oracle import nfp_oracle as O

import test_grad_parity_gpu as G
from _util import grad_err, grad_errs, pixel_regions, rel_err

FP32_TOL = 1e-5
EPS = 1e-6
SHAPES = [(5, 64, 7, 7, 1), (2, 10, 5, 9, 2)]


def _oracle(x, g, R, mode, sim):
    _, gx = O.nfp_forward_backward(x.double(), g.double(), R=R, measure="cosine", padding=R, padding_mode=mode,
                                   similarity=sim)
    return torch.as_tensor(np.asarray(gx))


def _inputs(shape, kind="degenerate", seed=0):
    B, C, H, W, R = shape
    x, _ = G.make_inputs(kind, shape, torch.float32, seed)
    g = torch.randn(B, (2 * R + 1) ** 2 - 1, H, W, generator=torch.Generator().manual_seed(seed + 1))
    return x, g


def _backward_clamp_term_dropped(x, g, R, mode, sim):
    """The gradient a kernel gets when it differentiates max(||v||, eps) as the constant eps below eps: the term
    -y v / (N ||v||) that ATen keeps at a sub-eps pixel is missing there (and only there)."""
    xr = x.double().clone().requires_grad_(True)
    geo = O.geometry(x.shape[2], x.shape[3], R, 1, R, 1, mode)
    c, n = O.gather_centre_neighbours(xr, geo)
    nc = torch.linalg.vector_norm(c, dim=1).clamp_min(EPS)
    nn = torch.linalg.vector_norm(n, dim=1).clamp_min(EPS)
    y = (c * n).sum(1) / (nc * nn)
    (gx,) = torch.autograd.grad(y if sim else 1 - y, xr, g.double())
    return gx


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[:4])) + f"_r{s[4]}")
@pytest.mark.parametrize("mode", G.MODES)
@pytest.mark.parametrize("sim", [True, False], ids=["sim", "dist"])
def test_grad_err_flags_each_mutation(shape, mode, sim):
    """Every mutation of the fp64 gradient of the degenerate input is flagged at the fp32 bound."""
    B, C, H, W, R = shape
    x, g = _inputs(shape)
    want = _oracle(x, g, R, mode, sim)
    assert grad_err(want, want, x) == 0.0
    lab = pixel_regions(x)
    ordinary = (lab == 2)[:, None].expand_as(want)
    assert (lab == 0).any() and (lab == 1).any() and ordinary.any()
    mutations = {}
    mutations["ordinary pixels zeroed"] = torch.where(ordinary, torch.zeros_like(want), want)
    mutations["ordinary pixels sign-flipped"] = torch.where(ordinary, -want, want)
    # the interior ordinary pixel with the largest gradient, off by 1e-4 relative
    mag = want.abs().amax(1)
    inner = torch.zeros_like(lab, dtype=torch.bool)
    inner[:, 1:H - 1, 1:W - 1] = True
    b, h, w = np.unravel_index(int(torch.where(inner & (lab == 2), mag, torch.zeros_like(mag)).argmax()), mag.shape)
    m = want.clone()
    m[b, :, h, w] *= 1 + 1e-4
    mutations["one interior pixel x (1 + 1e-4)"] = m
    # the channel holding the largest ordinary gradient, scaled by 1 + 1e-4
    ch = int(torch.where(ordinary, want.abs(), torch.zeros_like(want)).amax((0, 2, 3)).argmax())
    m = want.clone()
    m[:, ch] *= 1 + 1e-4
    mutations["one channel x (1 + 1e-4)"] = m
    for other in G.MODES:   # the border handled with another padding rule
        if other != mode:
            mutations[f"{other} padding at the border"] = _oracle(x, g, R, other, sim)
    mutations["similarity sign flipped in the backward"] = _oracle(x, g, R, mode, not sim)
    mutations["norm-clamp term dropped below eps"] = _backward_clamp_term_dropped(x, g, R, mode, sim)
    missed = {k: grad_err(v, want, x) for k, v in mutations.items() if not grad_err(v, want, x) >= FP32_TOL}
    assert not missed, missed


def test_clamp_term_variant_differs_only_below_eps():
    """The mutation above is the intended one: equal to the oracle except at pixels with 0 < ||x|| < eps."""
    shape = SHAPES[0]
    x, g = _inputs(shape)
    want = _oracle(x, g, 1, "reflect", True)
    got = _backward_clamp_term_dropped(x, g, 1, "reflect", True)
    n = torch.linalg.vector_norm(x.double(), dim=1)
    sub = (n > 0) & (n < EPS)
    diff = (got - want).abs().amax(1)
    assert diff[~sub].max() <= 1e-12 * want.abs().max()
    assert (diff[sub] > 1e-5 * want.abs().amax(1)[sub]).all()   # its size goes with ||x|| / eps: 1e-4 at 1e-9 pixels


def test_whole_tensor_scale_misses_zeroed_gradients():
    """Why the GPU suite scores input gradients with grad_err: on the input the fused-kernel tests plant (an exact
    zero pixel and a pixel scaled by 1e-9), zeroing the gradient of every other pixel passes rel_err's whole-tensor
    1e-5 bound; grad_err reports an error of 1."""
    B, C, H, W = 3, 512, 7, 7
    gen = torch.Generator().manual_seed(B * 1000 + C + H + 1)
    x = torch.randn(B, C, H, W, generator=gen).relu()
    x[0, :, 0, 0] = 0.0
    x[-1, :, H - 1, W - 1] *= 1e-9
    g = torch.randn(B, 8, H, W, generator=gen)
    want = _oracle(x, g, 1, "zeros", True)
    keep = torch.zeros(B, 1, H, W, dtype=torch.bool)
    keep[0, :, 0, 0] = keep[-1, :, H - 1, W - 1] = True
    got = torch.where(keep, want, torch.zeros_like(want))
    assert rel_err(got, want) < FP32_TOL
    assert grad_err(got, want, x) == pytest.approx(1.0)


@pytest.mark.parametrize("shape", [(5, 64, 7, 7, 1), (3, 512, 7, 7, 2), (6, 512, 2, 2, 1), (2, 16, 28, 28, 1),
                                   (2, 10, 5, 9, 2), (2, 5, 3, 3, 1), (1, 4, 5, 8, 2)],
                         ids=lambda s: "x".join(map(str, s[:4])) + f"_r{s[4]}")
@pytest.mark.parametrize("kind", G.KINDS)
def test_fp32_evaluation_passes_every_region(shape, kind):
    """Specificity: the oracle evaluated in fp32 against itself in fp64 passes every image and region at 1e-5, in
    every padding mode and for both similarity flags."""
    B, C, H, W, R = shape
    x, g = _inputs(shape, kind, seed=sum(shape))
    for mode in G.MODES:
        if mode == "reflect" and R >= min(H, W):
            continue
        for sim in (True, False):
            kw = dict(R=R, measure="cosine", padding=R, padding_mode=mode, similarity=sim)
            _, gx32 = O.nfp_forward_backward(x.float(), g.float(), **kw)
            want = _oracle(x, g, R, mode, sim)
            errs = grad_errs(gx32, want, x)
            assert max(errs.values()) < FP32_TOL, (mode, sim, sorted(errs.items(), key=lambda kv: -kv[1])[:3])


def _required_cells():
    cells = set()

    def add(family, op, dtypes):
        cells.update((family, op, m, s, dt) for m in G.MODES for s in G.SIMS for dt in dtypes)
    for family in ("stream", "split"):
        add(family, "map", G.BOTH)
        add(family, "pooled", G.BOTH)
    add("band", "map", G.BOTH)
    add("table", "map", G.BOTH)
    add("token", "map", G.BF16)
    add("token", "pooled", G.BF16)
    add("stream", "head", G.BOTH)      # the fused head on NCHW maps
    add("token", "head", G.BF16)       # ... and on channels-last bf16 maps
    add("stream", "multi", G.BOTH)
    add("band", "multi", G.BOTH)
    add("token", "multi", G.BF16)
    return cells


def test_grid_reaches_every_cell():
    """Every case of the GPU grid takes the kernel family it is filed under (forward and backward launch), and
    together they reach every required cell; a dispatch change that empties a cell fails here, without a GPU."""
    reached = set()
    wrong = []
    for c in G.GRID:
        paths = G.case_paths(c)
        if all(p.startswith(G.FAMILIES[c.family][0]) for p in paths):
            reached.add((c.family, c.op, c.mode, c.sim, c.dtype))
        else:
            wrong.append((G.case_id(c), paths))
    assert not wrong, wrong[:5]
    missing = _required_cells() - reached
    assert not missing, sorted(missing, key=str)[:5]
    # the persistent image loops: more images than resident CTAs, in the map, pooled and token kernels
    for family, op in (("stream", "map"), ("split", "map"), ("stream", "pooled"), ("token", "map")):
        assert any(c.family == family and c.op == op and c.shape[0] >= 300 for c in G.GRID), (family, op)
    assert any(c.family == "stream" and c.op == "map" and c.shape[:2] == (300, 512) for c in G.GRID)
