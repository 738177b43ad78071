"""GPU: per-scan feature covariance on csrc/isw.cu (lg_inst_cov_forward / _backward) against the float64 oracle
(oracle/isw.py), the statistic and gradient of RobustNet's instance-whitening loss.

Outputs are filled with NaN before each call, so an element the kernels leave unwritten fails.  cov and dx are
checked element by element, each against a bar scaled by the sum of absolute products that forms it:
sum_rows |x_i| |x_j| / (n_b - 1) for cov_ij, sum_i |x_r[i]| |S_ij| for dx_rj.  Cases: batch-sorted and permuted
rows, an absent scan, a one-row scan, rows outside [0, B), B = 1, 8, 64, 256, C = 1, 3, 32, 37, 128, 256, data with
mean 1e3; bit-identical runs; the KITTI batch-8 level shapes; a conv -> InstanceNorm -> ReLU -> covariance -> loss
chain against the same chain on oracle/me_cpu; no host synchronisation inside a step."""
import numpy as np
import pytest
import torch

from oracle import isw as oisw
from tests.helpers import random_voxels, record

pytestmark = pytest.mark.gpu

EPS = 1e-5
COV_TOL = 1e-5  # float sums over 32 rows (worst case 32 * 2^-24 = 1.9e-6 of the bar), merged in double


def _dx_tol(C):
    return 2.0 * (C + 4) * 2.0 ** -24  # one float fmaf chain over C terms, S rounded to float once


def _layout(kind, C, B=8, seed=0, mean=0.0, n=2000):
    g = torch.Generator().manual_seed(seed)
    bidx = torch.randint(0, B, (n,), generator=g)
    if kind == "absent":
        bidx[bidx == 5] = 6
    if kind == "one_row":
        bidx[bidx == 7] = 6
        bidx[123] = 7
    if kind == "outside":  # rows with a batch index outside [0, B): left out of cov, NaN in dx
        bidx[::97] = B
        bidx[1::101] = -1
    if kind == "sorted":
        bidx = bidx.sort().values
    coords = torch.randint(-50, 50, (n, 4), generator=g, dtype=torch.int32)
    coords[:, 0] = bidx.to(torch.int32)
    x = torch.randn(n, C, generator=g) + mean
    G = torch.randn(B, C, C, generator=g)
    return x, coords, B, G


def _gpu(x, coords, B, G, dev):
    from lidog_b200 import cabi
    L = cabi.lib()
    n, C = x.shape
    x, coords, G = x.to(dev).contiguous(), coords.to(dev).contiguous(), G.to(dev).contiguous()
    cov = torch.full((B, C, C), float("nan"), device=dev)
    counts = torch.full((B,), -7, dtype=torch.int32, device=dev)
    dx = torch.full((n, C), float("nan"), device=dev)
    s = cabi.stream_of(x)
    cabi.check(L.lg_inst_cov_forward(x.data_ptr(), coords.data_ptr(), n, C, B, EPS, cov.data_ptr(), counts.data_ptr(),
                                     s), "lg_inst_cov_forward")
    cabi.check(L.lg_inst_cov_backward(x.data_ptr(), coords.data_ptr(), n, C, B, G.data_ptr(), counts.data_ptr(),
                                      dx.data_ptr(), s), "lg_inst_cov_backward")
    torch.cuda.synchronize()
    return cov.cpu(), counts.cpu(), dx.cpu()


def _check(cuda, x, coords, B, G):
    cov, counts, dx = _gpu(x, coords, B, G, cuda)
    n, C = x.shape
    b = coords[:, 0].long()
    xd = x.double()
    ref = oisw.instance_covariance(xd, b, B, EPS)
    want_counts = torch.stack([(b == i).sum() for i in range(B)]).to(torch.int32)
    assert torch.equal(counts, want_counts)
    assert torch.equal(cov, cov.transpose(1, 2))  # mirrored, not computed twice
    errs = dict(cov=0.0, dx=0.0)
    for i in range(B):
        r = b == i
        nb = int(r.sum())
        if nb <= 1:  # eps * I exactly, and no gradient
            assert torch.equal(cov[i], (EPS * torch.eye(C)).float()), i
            assert torch.equal(dx[r], torch.zeros(nb, C)), i
            continue
        xa = xd[r].abs()
        scale = xa.t() @ xa / (nb - 1) + EPS * torch.eye(C, dtype=torch.float64)
        e = ((cov[i].double() - ref[i]).abs() / scale.clamp_min(1e-30)).max()
        errs["cov"] = max(errs["cov"], float(e))
        S = (G[i].double() + G[i].double().t()) / (nb - 1)
        dscale = xa @ S.abs()
        e = ((dx[r].double() - xd[r] @ S).abs() / dscale.clamp_min(1e-30)).max()
        errs["dx"] = max(errs["dx"], float(e))
    valid = (b >= 0) & (b < B)
    assert torch.isnan(dx[~valid]).all() and not torch.isnan(dx[valid]).any()
    record("isw_oracle", rows=n, channels=C, scans=B, **errs)
    assert errs["cov"] <= COV_TOL and errs["dx"] <= _dx_tol(C), errs
    return errs


@pytest.mark.parametrize("C", [1, 3, 32, 37, 128, 256])
@pytest.mark.parametrize("kind", ["sorted", "permuted", "absent", "one_row", "outside"])
def test_matches_float64_oracle(cuda, kind, C):
    x, coords, B, G = _layout(kind, C, seed=C)
    _check(cuda, x, coords, B, G)


@pytest.mark.parametrize("C", [3, 32, 128])
@pytest.mark.parametrize("kind", ["sorted", "permuted"])
@pytest.mark.parametrize("B", [1, 64, 256])
def test_scan_counts(cuda, B, kind, C):
    x, coords, B, G = _layout(kind, C, B=B, seed=B + C, n=4000)
    _check(cuda, x, coords, B, G)


@pytest.mark.parametrize("C", [3, 32, 128])
@pytest.mark.parametrize("kind", ["sorted", "permuted"])
def test_large_mean(cuda, kind, C):
    """mean 1e3: every product is ~1e6 and the covariance is dominated by the mean (it is not centred)."""
    x, coords, B, G = _layout(kind, C, seed=7 + C, mean=1e3)
    _check(cuda, x, coords, B, G)


@pytest.mark.parametrize("C", [32, 37])
def test_many_chunks(cuda, C):
    """Enough rows for hundreds of position chunks, scans beginning inside chunks, several rank chunks per scan."""
    x, coords, B, G = _layout("permuted", C, seed=11, mean=0.5, n=300_000)
    _check(cuda, x, coords, B, G)


def test_runs_are_bit_identical(cuda):
    x, coords, B, G = _layout("permuted", 48, seed=5, mean=3.0, n=200_000)
    r1 = _gpu(x, coords, B, G, cuda)
    r2 = _gpu(x, coords, B, G, cuda)
    for a, c in zip(r1, r2):
        assert torch.equal(a, c)


def test_kitti_batch8_levels(cuda):
    """The stride-1 (32 channels) and stride-8 (128 channels) levels of the KITTI-shaped batch of 8 scans."""
    from lidog_b200 import me as ME
    from lidog_b200.lidog import synth
    scans = synth.make_batch(8, shape="kitti")
    pts = [torch.from_numpy(p).to(cuda) for p, _ in scans]
    cm = ME.CoordinateManager.from_quantized(ME.utils.sparse_quantize_batch(pts, None, 0.05))
    g = torch.Generator().manual_seed(0)
    for ts, C in ((1, 32), (8, 128)):
        coords = cm.get_coords(ts).cpu()
        n = coords.shape[0]
        x = torch.randn(n, C, generator=g)
        G = torch.randn(8, C, C, generator=g)
        errs = _check(cuda, x, coords, 8, G)
        record("isw_kitti_level", tensor_stride=ts, rows=n, channels=C, **errs)


def test_tensor_without_rows(cuda):
    """No rows: eps * I for each of the manager's batch_size scans and a zero gradient; without a batch_size there is
    no way to tell how many scans there are, and the call says so."""
    import MinkowskiEngine as ME
    from lidog_b200.me.sparse_tensor import SparseTensor

    class Manager:
        batch_size = 3

    f = torch.empty(0, 5, device=cuda, requires_grad=True)
    cov = ME.instance_covariance(SparseTensor(f, coordinate_manager=Manager(), tensor_stride=2))
    assert cov.shape == (3, 5, 5) and torch.equal(cov.detach().cpu(), (EPS * torch.eye(5)).expand(3, 5, 5))
    ME.instance_whitening_loss(cov, torch.ones(5, 5, device=cuda), -1.0, 1.0).backward()
    assert f.grad is not None and f.grad.shape == (0, 5)
    with pytest.raises(ValueError, match="batch_size"):
        ME.instance_covariance(SparseTensor(torch.empty(0, 5, device=cuda), coordinate_manager=object()))


def test_no_host_synchronisation(cuda):
    """instance_covariance -> loss -> backward, with B known to the manager, synchronises nothing that torch sees (the
    library's own calls are outside what set_sync_debug_mode watches; INTEGRATION.md says when they synchronise)."""
    import MinkowskiEngine as ME
    rng = np.random.default_rng(3)
    c = torch.from_numpy(random_voxels(rng, 5000, span=30, batch=4)).to(cuda)
    f = torch.randn(c.shape[0], 32, device=cuda, requires_grad=True)
    x = ME.SparseTensor(features=f, coordinates=c)
    x.coordinate_manager.batch_size = 4
    mask = torch.triu(torch.ones(32, 32, device=cuda), 1)
    x.C  # the coordinates exist before the step
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        cov = ME.instance_covariance(x)
        loss = ME.instance_whitening_loss(cov, mask, 0.0, 10.0)
        loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert f.grad is not None and bool(torch.isfinite(f.grad).all())


# conv -> IN -> ReLU -> covariance -> loss: with exact-fp32 convolutions a tight bar; with fp16 tensor-core operands
# the bars of the instance-norm chain (tests/test_gpu_instnorm.py), whose numbers this chain inherits
CHAIN_BARS = {"off": dict(out=2e-5, grad=1e-4), "fp16": dict(out=4e-3, grad=2.5e-2)}


@pytest.mark.parametrize("mode", ["off", "fp16"])
def test_chain_conv_in_relu_covariance_loss_matches_oracle(cuda, mode):
    import MinkowskiEngine as ME
    from lidog_b200.me import conv as meconv
    from oracle import me_cpu
    from oracle.instnorm import MinkowskiInstanceNorm as CpuInstanceNorm
    rng = np.random.default_rng(9)
    coords = random_voxels(rng, 4000, span=25, batch=3)
    feats = rng.standard_normal((coords.shape[0], 32)).astype(np.float32)  # 32 | Cin: the tensor-core path
    torch.manual_seed(0)
    C = 32
    mask = torch.triu(torch.from_numpy(rng.random((C, C)) > 0.5).double(), 1)

    def build(M, InstanceNorm):
        return torch.nn.ModuleList([M.MinkowskiConvolution(32, C, kernel_size=3, dimension=3), InstanceNorm(C),
                                    M.MinkowskiReLU()])

    ref = build(me_cpu, CpuInstanceNorm)
    with torch.no_grad():
        ref[1].weight.uniform_(0.5, 1.5)
        ref[1].bias.uniform_(-0.5, 0.5)
    ref = ref.double()
    fo = torch.from_numpy(feats).double().requires_grad_(True)
    t = me_cpu.SparseTensor(coordinates=torch.from_numpy(coords), features=fo)
    for layer in ref:
        t = layer(t)
    cov_o = oisw.instance_covariance(t.F, t.C[:, 0], 3, EPS)
    margin = float((cov_o.detach() * mask).abs().sum(dim=(1, 2)).sort().values[:2].mean())  # one scan clamped
    loss_o = oisw.instance_whitening_loss(cov_o, mask, margin, 20.0)
    loss_o.backward()

    old = dict(meconv.CONFIG)
    meconv.CONFIG["tc"] = mode
    try:
        net = build(ME, ME.MinkowskiInstanceNorm)
        net.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
        net = net.to(cuda)
        fg = torch.from_numpy(feats).to(cuda).requires_grad_(True)
        g = ME.SparseTensor(coordinates=torch.from_numpy(coords).to(cuda), features=fg)
        for layer in net:
            g = layer(g)
        cov = ME.instance_covariance(g)
        loss = ME.instance_whitening_loss(cov, mask.float().to(cuda), margin, 20.0)
        loss.backward()
        torch.cuda.synchronize()
    finally:
        meconv.CONFIG.update(old)

    def rel(a, b):
        a, b = a.detach().cpu().double(), b.detach().cpu().double()
        return float((a - b).norm() / b.norm().clamp_min(1e-30))

    errs = dict(cov=rel(cov, cov_o), loss=rel(loss, loss_o), dfeat=rel(fg.grad, fo.grad))
    for (k, p), (_, po) in zip(net.named_parameters(), ref.named_parameters()):
        errs[k] = rel(p.grad, po.grad)
    record("isw_chain", mode=mode, **errs)
    bars = CHAIN_BARS[mode]
    assert errs["cov"] <= bars["out"] and errs["loss"] <= bars["out"], (mode, errs)
    assert all(v <= bars["grad"] for k, v in errs.items() if k not in ("cov", "loss")), (mode, errs)
