"""GPU: the BEV backward reads each window's winning cell from the table the forward records, and writes every element
of grad_feats itself.  Output and gradient must equal oracle/bev.py bit for bit on the cases that stress that table:
ties inside a window (two equal maxima, a voxel value equal to an empty cell's zero), all-negative features (empty
cells win), dense occupancy (cells on window borders in 2 x 2 windows, padding edges), rows outside the image, several
rows per pixel under both policies, C not a multiple of 4, both gradient layouts, other pooling shapes and the
full-scale KITTI batch of 8.  Outputs and gradients are NaN and the workspace holds small junk bytes before the
calls, so an element that is not written, or a table entry that is read without having been written, shows up."""
import numpy as np
import pytest
import torch

from oracle import bev as ob

pytestmark = pytest.mark.gpu


def _run(cuda, coords, feats, B, bound, policy, layout, pool=(5, 3, 1), seed=0):
    """Forward and backward through the C ABI; returns (out, grad_feats, grad_out) as numpy, out in NCHW order."""
    from lidog_b200 import cabi
    L = cabi.lib()
    pk, ps, pp = pool
    n, C = feats.shape
    H = W = ob.image_size(bound)
    h, w = (H + 2 * pp - pk) // ps + 1, (W + 2 * pp - pk) // ps + 1
    fmt = torch.channels_last if layout else torch.contiguous_format
    c = torch.from_numpy(coords).to(cuda).contiguous()
    f = torch.from_numpy(feats).to(cuda).contiguous()
    pol = cabi.BEV_LAST if policy == "last" else cabi.BEV_MAX
    ws_bytes = L.lg_bev_workspace(n, C, B, H, W, pk, ps, pp)
    g = torch.Generator(device=cuda).manual_seed(seed)
    ws = torch.randint(0, pk * pk, (ws_bytes,), dtype=torch.uint8, device=cuda, generator=g)
    out = torch.full((B, C, h, w), float("nan"), device=cuda).contiguous(memory_format=fmt)
    cabi.check(L.lg_bev_forward(cabi.ptr(c), cabi.ptr(f), n, C, B, float(bound), 0.05, H, W, pk, ps, pp, pol, layout,
                                cabi.ptr(out), cabi.ptr(ws), ws_bytes, cabi.stream()), "lg_bev_forward")
    gout = torch.randn((B, C, h, w), device=cuda, generator=g).contiguous(memory_format=fmt)
    gf = torch.full((n, C), float("nan"), device=cuda)
    cabi.check(L.lg_bev_backward(cabi.ptr(c), cabi.ptr(f), n, C, B, H, W, pk, ps, pp, pol, layout, cabi.ptr(gout),
                                 cabi.ptr(gf), cabi.ptr(ws), ws_bytes, cabi.stream()), "lg_bev_backward")
    torch.cuda.synchronize()
    return out.contiguous().cpu().numpy(), gf.cpu().numpy(), gout.contiguous().cpu().numpy()


def _check(cuda, coords, feats, B, bound, policy, layout, pool=(5, 3, 1)):
    out, g, gout = _run(cuda, coords, feats, B, bound, policy, layout, pool)
    ref, ctx = ob.bev_forward(coords, feats, B, bound, pool=pool, policy=policy)
    gref = ob.bev_backward(gout, ctx)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
    assert np.array_equal(g.view(np.uint32), gref.view(np.uint32))
    return g


def _dense_case(rng, B, bound, C, occupancy, values, rows_per_pixel=2):
    """Most pixels of a small image occupied (every window border and padding edge is reached), a margin of voxels
    outside the strict bound, up to `rows_per_pixel` z-voxels per pixel.  values: 'ties' = integers in [-2, 2]
    (equal maxima, voxel zeros against empty zeros), 'negative' = all below zero."""
    lim = int(round(bound / 0.05)) + 2
    xs, ys = np.meshgrid(np.arange(-lim, lim), np.arange(-lim, lim), indexing="ij")
    xy = np.stack([xs.ravel(), ys.ravel()], 1)
    rows = []
    for b in range(B):
        keep = xy[rng.random(len(xy)) < occupancy]
        for z in range(rows_per_pixel):
            sel = keep[rng.random(len(keep)) < (1.0 if z == 0 else 0.5)]
            rows.append(np.concatenate([np.full((len(sel), 1), b), sel, np.full((len(sel), 1), z)], 1))
    coords = np.concatenate(rows).astype(np.int32)
    coords = coords[rng.permutation(len(coords))]  # rows of a pixel in any order: the chains and winners vary
    n = len(coords)
    if values == "ties":
        feats = rng.integers(-2, 3, size=(n, C)).astype(np.float32)
    else:
        feats = (-1.0 - rng.random((n, C))).astype(np.float32)
    return coords, feats


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("policy", ["last", "max"])
@pytest.mark.parametrize("C", [3, 37])
def test_ties_and_zero_ties_dense(cuda, C, policy, layout):
    rng = np.random.default_rng(100 + C)
    coords, feats = _dense_case(rng, 2, 1.0, C, 0.7, "ties", rows_per_pixel=3)
    g = _check(cuda, coords, feats, 2, 1.0, policy, layout)
    inb, _, _ = ob.pixel_indices(coords[:, 1:], 1.0)
    assert (~inb).any() and not g[~inb].any()  # rows outside the image come back as zeros


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("policy", ["last", "max"])
def test_all_negative_features_empty_cells_win(cuda, policy, layout):
    rng = np.random.default_rng(7)
    coords, feats = _dense_case(rng, 2, 1.0, 5, 0.85, "negative")
    g = _check(cuda, coords, feats, 2, 1.0, policy, layout)
    assert g.any()  # fully occupied windows still route gradient to a voxel


@pytest.mark.parametrize("policy", ["last", "max"])
@pytest.mark.parametrize("pool", [(3, 2, 1), (4, 2, 0), (2, 3, 0)])
def test_other_pooling_shapes(cuda, pool, policy):
    """Windows of other sizes and strides, including pk < ps (cells no window covers get zero)."""
    rng = np.random.default_rng(21)
    coords, feats = _dense_case(rng, 1, 1.0, 6, 0.6, "ties")
    _check(cuda, coords, feats, 1, 1.0, policy, 1, pool)


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("policy", ["last", "max"])
def test_sparse_many_rows_per_pixel(cuda, policy, layout):
    import tests.golden.make_bev_golden as mk
    rng = np.random.default_rng(31)
    coords, feats = mk.make_case(rng, 4000, 3, 3.0, 10, dup_frac=0.6)
    _check(cuda, coords, feats, 3, 3.0, policy, layout)


def test_kitti_batch8_full_scale(cuda):
    """The bench's shape: 8 KITTI-like scans at stride 1, 96 channels, 2000 x 2000 -> 666 x 666, channels_last."""
    from lidog_b200 import me as ME
    from lidog_b200.lidog import synth
    scans = synth.make_batch(8, 1234, "kitti", 7)
    res = ME.utils.sparse_quantize_batch([torch.from_numpy(p).to(cuda) for p, _ in scans], None, 0.05)
    coords = ME.CoordinateManager.from_quantized(res).get_coords(1).cpu().numpy().astype(np.int32)
    rng = np.random.default_rng(8)
    feats = np.maximum(rng.standard_normal((len(coords), 96)), 0).astype(np.float32)  # post-ReLU: many zero ties
    _check(cuda, coords, feats, 8, 50.0, "last", 1)
