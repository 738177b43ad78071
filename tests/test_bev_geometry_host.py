"""Host side of the BEV projection at every pooling geometry: the scaling-factor -> pool and label-image-size helpers,
the oracle's backward at overlapping pools against torch autograd of the reference's own formulation, and the C ABI's
rejection of pools outside the envelope (1 <= pk <= 15, 1 <= ps <= 16, 0 <= 2 pp <= pk) before any CUDA call."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bev as ob


def test_pool_for_scaling_is_the_reference_mapping():
    from lidog_b200.lidog.bev import pool_for_scaling
    assert pool_for_scaling() == pool_for_scaling(1.0) == (5, 3, 1)
    assert [pool_for_scaling(s) for s in (0.5, 0.75, 1.5, 2.0, 3.0)] == [(5, 6, 1), (5, 4, 1), (5, 2, 1), (5, 1, 1),
                                                                       (5, 1, 1)]


def test_label_image_size_reproduces_shapes_and_follows_the_pool():
    from lidog_b200.lidog.bev import label_image_size
    from lidog_b200.lidog.synth import SHAPES
    assert label_image_size(50.0, 0.05) == 167 == SHAPES["kitti"]["bev_img"]
    assert label_image_size(30.0, 0.05) == 100 == SHAPES["nuscenes"]["bev_img"]
    # 2000 -> pooled 5/2/1: 999 -> Encoder2D 500 -> 250; 5/1/1: 1998 -> 999 -> 500; 5/6/1: 333 -> 167 -> 84
    assert [label_image_size(50.0, 0.05, p) for p in ((5, 2, 1), (5, 1, 1), (5, 6, 1))] == [250, 500, 84]
    # the size the dense head really produces on a pooled image of that side
    for pool in ((5, 3, 1), (5, 2, 1), (5, 4, 1), (5, 1, 1)):
        pk, ps, pp = pool
        h = (ob.image_size(8.0) + 2 * pp - pk) // ps + 1
        y = F.conv2d(F.conv2d(torch.zeros(1, 1, h, h), torch.zeros(1, 1, 3, 3), stride=2, padding=1),
                     torch.zeros(1, 1, 3, 3), stride=2, padding=1)
        assert y.shape[-1] == label_image_size(8.0, 0.05, pool), pool


def test_trainer_label_image_follows_the_model_pool():
    from lidog_b200.lidog import model as M, step
    from oracle import me_cpu
    from oracle.me_cpu.bevfn import sparse2super
    for s, want in ((1.0, 100), (1.5, 150)):
        net = M.MinkUNet34BEV(1, 7, ME=me_cpu, bev_fn=sparse2super, mapping_bound_2d=30.0, layers=(1,) * 8,
                              bev_scaling_factor=s)
        assert step.LidogTrainer(net, shape="nuscenes", ME=me_cpu).bev_img == want
    default = M.MinkUNet34BEV(1, 7, ME=me_cpu, bev_fn=sparse2super, layers=(1,) * 8)
    scaled = M.MinkUNet34BEV(1, 7, ME=me_cpu, bev_fn=sparse2super, layers=(1,) * 8, bev_scaling_factor=2.0)
    assert default.bev_pool == (5, 3, 1) and scaled.bev_pool == (5, 1, 1)
    assert list(default.state_dict()) == list(scaled.state_dict())


def _autograd_reference(coords, feats, batch_size, bound, pool):
    """`bev_forward_sparse_reference` with autograd: the reference's torch code (index_put_ + max_pool2d)."""
    C = feats.shape[1]
    H = ob.image_size(bound)
    c = torch.as_tensor(coords)
    xyz = c[:, 1:] * 0.05
    outs = []
    for b in range(batch_size):
        m = c[:, 0] == b
        fb, xb = feats[m], xyz[m]
        inb = (-bound < xb[:, 0]) & (xb[:, 0] < bound) & (-bound < xb[:, 1]) & (xb[:, 1] < bound)
        fb, xb = fb[inb], xb[inb]
        img = torch.zeros((H, H, C))
        px = torch.floor((xb[:, 0] - (-bound)) / 0.05).long()
        py = torch.floor(torch.tensor(H).int() - (xb[:, 1] - (-bound)) / 0.05).long() - 1
        img = img.index_put((py, px), fb)
        outs.append(F.max_pool2d(img.view(1, -1, H, H), pool[0], pool[1], pool[2]))
    return torch.cat(outs, 0)


@pytest.mark.parametrize("pool", [(5, 1, 1), (5, 2, 1), (3, 1, 1), (7, 2, 3), (15, 1, 7)])
def test_oracle_backward_at_overlapping_pools_is_torch_autograd(pool):
    """A cell sits in up to ceil(pk/ps)^2 windows here: the oracle's per-cell sums must be torch's, bit for bit."""
    torch.set_num_threads(1)
    rng = np.random.default_rng(40 + pool[0] * 17 + pool[1])
    lim = 30  # voxels at +-1.5 m on a 2 m bound: dense, with ties between neighbours; one voxel per pixel
    xy = rng.permutation((2 * lim) ** 2)[:1500]
    coords = np.stack([rng.integers(0, 2, 1500), xy // (2 * lim) - lim, xy % (2 * lim) - lim,
                       np.zeros(1500)], 1).astype(np.int32)
    inb, px, py = ob.pixel_indices(coords[:, 1:], 2.0)
    _, keep = np.unique(coords[:, 0] * 10 ** 6 + py * 1000 + px, return_index=True)
    coords = coords[np.sort(keep)]
    feats = rng.integers(-2, 3, size=(len(coords), 6)).astype(np.float32)
    f = torch.from_numpy(feats).requires_grad_(True)
    out = _autograd_reference(coords, f, 2, 2.0, pool)
    ref, ctx = ob.bev_forward(coords, feats, 2, 2.0, pool=pool, policy="last")
    assert np.array_equal(out.detach().numpy().view(np.uint32), ref.view(np.uint32))
    assert np.array_equal(ref, ob.bev_forward_sparse_reference(coords, feats, 2, 2.0, pool=pool))
    g = rng.standard_normal(ref.shape).astype(np.float32)
    out.backward(torch.from_numpy(g))
    assert np.array_equal(f.grad.numpy().view(np.uint32), ob.bev_backward(g, ctx).view(np.uint32))


def test_cabi_rejects_pools_outside_the_envelope():
    """Rejected before any CUDA call: this runs without a device."""
    from lidog_b200 import build, cabi
    build.build()
    L = cabi.lib()
    buf = ctypes.create_string_buffer(1 << 12)
    a16 = (ctypes.addressof(buf) + 15) & ~15
    ok = dict(pk=5, ps=3, pp=1, H=40)

    def fwd(**kw):
        d = dict(ok, **kw)
        return L.lg_bev_forward(a16, a16, 4, 8, 1, 1.0, 0.05, d["H"], d["H"], d["pk"], d["ps"], d["pp"], cabi.BEV_LAST,
                                0, a16, a16, 1 << 40, None)

    def bwd(**kw):
        d = dict(ok, **kw)
        return L.lg_bev_backward(a16, a16, 4, 8, 1, d["H"], d["H"], d["pk"], d["ps"], d["pp"], cabi.BEV_LAST, 0, a16,
                                 a16, a16, 1 << 40, None)

    for bad, word in ((dict(pk=16), b"kernel 16"), (dict(pk=0), b"kernel 0"), (dict(pk=5, pp=3), b"padding 3"),
                      (dict(pk=2, pp=2), b"padding 2"), (dict(ps=0), b"stride 0"), (dict(ps=17), b"stride 17"),
                      (dict(H=3, pk=15, pp=5), b"smaller than the pool window")):
        for fn, who in ((fwd, b"lg_bev_forward"), (bwd, b"lg_bev_backward")):
            assert fn(**bad) == -1, (bad, who)
            msg = L.lg_last_error_string()
            assert who in msg and word in msg, (bad, msg)
