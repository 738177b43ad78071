"""GPU: the BEV projection at every max-pool geometry of its envelope -- overlapping windows (a cell in up to
ceil(pk/ps)^2 of them), strides up to 16, windows of 1 to 15 cells, images wider than 1024 windows -- bit for bit
against oracle/bev.py, forward and backward, both policies and both layouts.  As in tests/test_gpu_bev_argmax.py,
outputs and gradients are NaN and the workspace holds junk bytes before the calls, so an element that is not written,
or a table entry read without having been written, shows up.  Also: the reference's scaling factor through
`patch_reference_model`, and a training step of the mirror model at a scaled BEV resolution."""
import numpy as np
import pytest
import torch

from oracle import bev as ob
from tests.test_gpu_bev_argmax import _dense_case

pytestmark = pytest.mark.gpu

POOLS = [(5, 1, 1), (5, 2, 1), (5, 3, 1), (5, 4, 1), (5, 6, 1), (5, 5, 2), (3, 1, 1), (2, 1, 0), (1, 1, 0), (7, 2, 3),
         (15, 1, 7), (15, 16, 0)]


def _run(cuda, coords, feats, B, bound, policy, layout, pool, voxel=0.05, seed=0):
    """Forward and backward through the C ABI; returns device tensors (out, grad_feats, grad_out), out in `layout`."""
    from lidog_b200 import cabi
    L = cabi.lib()
    pk, ps, pp = pool
    n, C = feats.shape
    H = W = ob.image_size(bound, voxel)
    h, w = (H + 2 * pp - pk) // ps + 1, (W + 2 * pp - pk) // ps + 1
    fmt = torch.channels_last if layout else torch.contiguous_format
    c = torch.from_numpy(coords).to(cuda).contiguous()
    f = torch.from_numpy(feats).to(cuda).contiguous()
    pol = cabi.BEV_LAST if policy == "last" else cabi.BEV_MAX
    ws_bytes = L.lg_bev_workspace(n, C, B, H, W, pk, ps, pp)
    g = torch.Generator(device=cuda).manual_seed(seed)
    ws = torch.randint(0, pk * pk, (ws_bytes,), dtype=torch.uint8, device=cuda, generator=g)
    out = torch.full((B, C, h, w), float("nan"), device=cuda).contiguous(memory_format=fmt)
    cabi.check(L.lg_bev_forward(cabi.ptr(c), cabi.ptr(f), n, C, B, float(bound), voxel, H, W, pk, ps, pp, pol, layout,
                                cabi.ptr(out), cabi.ptr(ws), ws_bytes, cabi.stream()), "lg_bev_forward")
    gout = torch.randn((B, C, h, w), device=cuda, generator=g).contiguous(memory_format=fmt)
    gf = torch.full((n, C), float("nan"), device=cuda)
    cabi.check(L.lg_bev_backward(cabi.ptr(c), cabi.ptr(f), n, C, B, H, W, pk, ps, pp, pol, layout, cabi.ptr(gout),
                                 cabi.ptr(gf), cabi.ptr(ws), ws_bytes, cabi.stream()), "lg_bev_backward")
    torch.cuda.synchronize()
    return out, gf, gout


def _same(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


def _check(cuda, coords, feats, B, bound, policy, layout, pool, voxel=0.05):
    out, gf, gout = _run(cuda, coords, feats, B, bound, policy, layout, pool, voxel)
    ref, ctx = ob.bev_forward(coords, feats, B, bound, voxel, pool=pool, policy=policy)
    gref = ob.bev_backward(gout.contiguous().cpu().numpy(), ctx)
    assert _same(out.contiguous().cpu().numpy(), ref), (pool, policy, layout)
    g = gf.cpu().numpy()
    assert _same(g, gref), (pool, policy, layout)
    return g


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("policy", ["last", "max"])
@pytest.mark.parametrize("C", [1, 3, 5, 32, 37, 96, 128, 256])
@pytest.mark.parametrize("pool", POOLS, ids=lambda p: "%d-%d-%d" % p)
def test_dense_ties_many_rows_per_pixel(cuda, pool, C, policy, layout):
    """Integer features in [-2, 2] (equal maxima, voxel zeros against empty zeros), most pixels occupied (every window
    border and padding edge reached), up to three rows per pixel, a margin of rows outside the image."""
    rng = np.random.default_rng(1000 + 7 * C + pool[0] * 31 + pool[1])
    coords, feats = _dense_case(rng, 2, 1.0, C, 0.7, "ties", rows_per_pixel=3)
    g = _check(cuda, coords, feats, 2, 1.0, policy, layout, pool)
    inb, _, _ = ob.pixel_indices(coords[:, 1:], 1.0)
    assert (~inb).any() and not g[~inb].any()  # rows outside the image come back as zeros


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("policy", ["last", "max"])
@pytest.mark.parametrize("pool", POOLS, ids=lambda p: "%d-%d-%d" % p)
def test_all_negative_features(cuda, pool, policy, layout):
    """Empty cells (zeros) win wherever a window holds one; fully occupied windows route to a voxel."""
    rng = np.random.default_rng(77 + pool[0] * 31 + pool[1])
    coords, feats = _dense_case(rng, 2, 1.0, 37, 0.85, "negative")
    _check(cuda, coords, feats, 2, 1.0, policy, layout, pool)


@pytest.mark.parametrize("policy", ["last", "max"])
@pytest.mark.parametrize("pool", [(5, 3, 1), (5, 1, 1), (15, 16, 0)], ids=lambda p: "%d-%d-%d" % p)
def test_image_wider_than_1024_windows(cuda, pool, policy):
    """Bound 50 m at 0.025 m: a 4000 x 4000 image, 1333 windows wide at ps = 3 and 3998 at ps = 1 -- more than 32
    tile column blocks per occupancy word.  Sparse voxels over the whole image plus a dense patch at the far edge."""
    import tests.golden.make_bev_golden as mk
    rng = np.random.default_rng(5)
    coords, feats = mk.make_case(rng, 30000, 1, 50.0, 3, dup_frac=0.3, voxel=0.025)
    patch = np.stack(np.meshgrid(np.arange(1900, 2003), np.arange(-2003, -1900), indexing="ij"), -1).reshape(-1, 2)
    patch = patch[rng.random(len(patch)) < 0.6]
    extra = np.concatenate([np.zeros((len(patch), 1)), patch, np.full((len(patch), 1), 50)], 1).astype(np.int32)
    coords = np.concatenate([coords, extra])
    feats = np.concatenate([feats, rng.integers(-2, 3, size=(len(extra), 3)).astype(np.float32)])
    _check(cuda, coords, feats, 1, 50.0, policy, 1, pool, voxel=0.025)


@pytest.mark.parametrize("pool", [(5, 1, 1), (5, 2, 1), (5, 6, 1)], ids=lambda p: "%d-%d-%d" % p)
def test_kitti_batch8_full_scale(cuda, pool):
    """The bench's batch (8 KITTI-like scans, stride 1, 96 channels, 2000 x 2000, channels_last) at scaled pools;
    compared one sample at a time, which keeps the oracle's dense images and indices to one sample."""
    from lidog_b200 import me as ME
    from lidog_b200.lidog import synth
    scans = synth.make_batch(8, 1234, "kitti", 7)
    res = ME.utils.sparse_quantize_batch([torch.from_numpy(p).to(cuda) for p, _ in scans], None, 0.05)
    coords = ME.CoordinateManager.from_quantized(res).get_coords(1).cpu().numpy().astype(np.int32)
    rng = np.random.default_rng(8)
    feats = np.maximum(rng.standard_normal((len(coords), 96)), 0).astype(np.float32)  # post-ReLU: many zero ties
    out, gf, gout = _run(cuda, coords, feats, 8, 50.0, "last", 1, pool)
    gf = gf.cpu().numpy()
    for b in range(8):
        rows = np.nonzero(coords[:, 0] == b)[0]
        cb = coords[rows].copy()
        cb[:, 0] = 0
        ref, ctx = ob.bev_forward(cb, feats[rows], 1, 50.0, pool=pool, policy="last")
        assert _same(out[b].contiguous().cpu().numpy(), ref[0]), b
        del ref
        gref = ob.bev_backward(gout[b:b + 1].contiguous().cpu().numpy(), ctx)
        assert _same(gf[rows], gref), b


def test_scaled_pool_matches_the_dense_torch_twin(cuda):
    """An anchor independent of oracle.bev_forward: the reference's own torch code at pool 5/2/1."""
    import tests.golden.make_bev_golden as mk
    rng = np.random.default_rng(12)
    coords, feats = mk.make_case(rng, 4000, 2, 4.0, 10, dup_frac=0.0)
    inb, px, py = ob.pixel_indices(coords[:, 1:], 4.0)  # one row per pixel: the twin's index_put_ has no ties to break
    _, keep = np.unique(coords[:, 0].astype(np.int64) * 10 ** 6 + py * 1000 + px, return_index=True)
    coords, feats = coords[np.sort(keep)], feats[np.sort(keep)]
    out, _, _ = _run(cuda, coords, feats, 2, 4.0, "last", 0, (5, 2, 1))
    threads = torch.get_num_threads()
    try:  # the twin runs single-threaded, as the reference's index_put_ does on the CPU
        twin = ob.bev_forward_sparse_reference(torch.from_numpy(coords), torch.from_numpy(feats), 2, 4.0,
                                               pool=(5, 2, 1))
    finally:
        torch.set_num_threads(threads)
    assert _same(out.cpu().numpy(), twin)


@pytest.mark.parametrize("s", [0.5, 1.5, 2.0, 3.0])
def test_patch_reference_model_scaling_factor(cuda, s):
    """sparse2super(x, scaling_factor=s) of a patched reference-shaped module: pool (5, int(3/s), 1), bit for bit."""
    import tests.golden.make_bev_golden as mk
    from lidog_b200 import me as ME
    from lidog_b200.lidog.bev import patch_reference_model

    class Stub(torch.nn.Module):
        mapping_bound_2d = 3.0

    m = patch_reference_model(Stub())
    rng = np.random.default_rng(int(s * 10))
    coords, feats = mk.make_case(rng, 3000, 2, 3.0, 16, dup_frac=0.3)
    x = ME.SparseTensor(coordinates=torch.from_numpy(coords).to(cuda), features=torch.from_numpy(feats).to(cuda))
    out = m.sparse2super(x, 0.05, scaling_factor=s)
    ref, _ = ob.bev_forward(coords, feats, 2, 3.0, pool=(5, int(3 / s), 1), policy="last")
    assert tuple(out.shape) == ref.shape and _same(out.contiguous().cpu().numpy(), ref)


def test_training_step_at_scaled_bev_resolution_matches_oracle(cuda):
    """MinkUNet34BEV(bev_scaling_factor=1.5): pool 5/2/1, a 600 x 600 projection and a 150 x 150 label image, one
    training step against the CPU oracle with the bars of tests/test_gpu_trainer.py (exact-fp32 kernels, fp32 head)."""
    from lidog_b200.me import conv as meconv
    from lidog_b200.lidog import model as M, step
    from oracle import me_cpu
    from oracle.me_cpu.bevfn import sparse2super as o_s2s
    from tests.test_gpu_trainer import GRAD_TOL, LOSS_TOL, _batch

    pts, lab = _batch()
    torch.manual_seed(0)
    ref_net = M.MinkUNet34BEV(1, 7, ME=me_cpu, bev_fn=o_s2s, mapping_bound_2d=30.0, bev_scaling_factor=1.5)
    state = {k: v.clone() for k, v in ref_net.state_dict().items()}
    ref = step.LidogTrainer(ref_net, num_classes=7, shape="nuscenes", ME=me_cpu)
    assert ref.bev_img == 150
    P, L = [torch.from_numpy(p) for p in pts], [torch.from_numpy(l) for l in lab]
    c_o, f_o, sem_o, bev_o, cm_o = ref.voxelize(P, L)
    tot_o, l3_o, l2_o = ref.forward_loss(c_o, f_o, sem_o, bev_o, len(P), cm_o)
    ref.optimizer.zero_grad(set_to_none=True)
    tot_o.backward()
    ref.optimizer.step()

    old_conf, old_tf32 = dict(meconv.CONFIG), torch.backends.cudnn.allow_tf32
    meconv.CONFIG["tc"] = "off"
    torch.backends.cudnn.allow_tf32 = False
    try:
        net = M.MinkUNet34BEV(1, 7, mapping_bound_2d=30.0, bev_scaling_factor=1.5)
        net.load_state_dict(state)
        net = net.to(cuda)
        tr = step.LidogTrainer(net, num_classes=7, shape="nuscenes")
        c, f, sem, bev, cm = tr.voxelize([p.to(cuda) for p in P], [l.to(cuda) for l in L])
        assert torch.equal(bev.cpu(), bev_o) and bev.shape[-1] == 150
        tot, l3, l2 = tr.forward_loss(c, f, sem, bev, len(P), cm)
        tr.optimizer.zero_grad(set_to_none=True)
        tot.backward()
        tr.optimizer.step()
        torch.cuda.synchronize()
    finally:
        meconv.CONFIG.update(old_conf)
        torch.backends.cudnn.allow_tf32 = old_tf32

    for name, a, b in (("3d", l3, l3_o), ("bev", l2, l2_o), ("total", tot, tot_o)):
        assert abs(float(a) - float(b)) <= LOSS_TOL * max(1.0, abs(float(b))), (name, float(a), float(b))
    ref_params = dict(ref_net.named_parameters())
    top = max(float(p.grad.norm()) for p in ref_params.values())
    bad = []
    for name, p in net.named_parameters():
        g, go = p.grad, ref_params[name].grad
        assert g is not None and go is not None and torch.isfinite(g).all(), name
        if float(go.norm()) > 1e-6 * top:
            e = float((g.detach().cpu().double() - go.double()).norm() / go.double().norm().clamp_min(1e-30))
            if e > GRAD_TOL[("off", False)]:
                bad.append((name, e))
    assert not bad, (top, bad[:8])
