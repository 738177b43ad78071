"""GPU: MinkowskiInstanceNorm on csrc/instnorm.cu against the float64 oracle (oracle/instnorm.py).

Forward and the three gradients within 1e-5 relative (Frobenius), the fused BN's bar, over row layouts (batch-sorted,
permuted, an absent instance, a one-row instance, B = 1, B = 64, many chunks), channel counts from 1 to 256, data with
a large mean and a small spread, ReLU on and off.  Also: the 16-bit copy equals lg_cast_rows(y) bit for bit, runs are
bit-identical, eval equals train, stride-4 tensors of the coordinate pyramid, the IBN channel split, and an autograd
chain convolution -> IN -> ReLU -> convolution against the same chain on oracle/me_cpu."""
import numpy as np
import pytest
import torch

from oracle.instnorm import instance_norm
from tests.helpers import random_voxels, record

pytestmark = pytest.mark.gpu

EPS = 1e-8


def rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


LAYOUTS = ("sorted", "permuted", "absent", "one_row", "B1", "B64")


def _layout(kind, C, seed=0, mean=0.0, std=1.0, n=2000):
    g = torch.Generator().manual_seed(seed)
    B = {"B1": 1, "B64": 64}.get(kind, 8)
    if kind == "B64":
        n = 3000
    bidx = torch.randint(0, B, (n,), generator=g)
    if kind == "absent":
        bidx[bidx == 5] = 6
    if kind == "one_row":
        bidx[bidx == 7] = 6
        bidx[123] = 7
    if kind == "sorted":
        bidx = bidx.sort().values
    coords = torch.randint(-50, 50, (n, 4), generator=g, dtype=torch.int32)
    coords[:, 0] = bidx.to(torch.int32)
    x = torch.randn(n, C, generator=g) * std + mean
    w = torch.randn(1, C, generator=g) * 0.5 + 1.0
    b = torch.randn(1, C, generator=g)
    dy = torch.randn(n, C, generator=g)
    return x, coords, B, w, b, dy


def _gpu(x, coords, B, w, b, dy, relu, dev, box=None):
    from lidog_b200.me.norm import InstanceNormFunction
    x = x.to(dev).requires_grad_(True)
    w = w.to(dev).requires_grad_(True)
    b = b.to(dev).requires_grad_(True)
    y = InstanceNormFunction.apply(x, w, b, coords.to(dev), B, relu, {} if box is None else box)
    y.backward(dy.to(dev))
    torch.cuda.synchronize()
    return y.detach(), x.grad, w.grad, b.grad


def _oracle(x, coords, w, b, dy, relu):
    xo, wo, bo = (t.double().requires_grad_(True) for t in (x, w, b))
    yo = instance_norm(xo, coords[:, 0], wo, bo, EPS)
    if relu:
        yo = torch.relu(yo)
    yo.backward(dy.double())
    return yo.detach(), xo.grad, wo.grad, bo.grad


def _check(cuda, x, coords, B, w, b, dy, relu, bar=1e-5):
    got = _gpu(x, coords, B, w, b, dy, relu, cuda)
    ref = _oracle(x, coords, w, b, dy, relu)
    errs = {k: rel(g, r) for k, g, r in zip(("y", "dx", "dweight", "dbias"), got, ref)}
    assert all(v <= bar for v in errs.values()), errs
    assert got[2].shape == w.shape and got[3].shape == b.shape
    return got


@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("C", [1, 3, 16, 32, 48, 96, 128, 256])
@pytest.mark.parametrize("kind", LAYOUTS)
def test_matches_float64_oracle(cuda, kind, C, relu):
    x, coords, B, w, b, dy = _layout(kind, C, seed=C)
    got = _check(cuda, x, coords, B, w, b, dy, relu)
    if kind == "one_row":  # a one-row instance normalises to 0: y = act(bias), dx = 0
        r = (coords[:, 0] == 7).nonzero().flatten()
        want = torch.relu(b) if relu else b
        assert torch.equal(got[0][r].cpu(), want.expand(len(r), -1))
        assert torch.equal(got[1][r].cpu(), torch.zeros(len(r), C))


@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("C", [3, 32, 128])
@pytest.mark.parametrize("kind", ["sorted", "permuted", "B64"])
def test_large_mean_small_spread(cuda, kind, C, relu):
    """mean 1e3, std 1: statistics that subtract the square of the mean from the mean square lose every digit here."""
    x, coords, B, w, b, dy = _layout(kind, C, seed=7 + C, mean=1e3, std=1.0)
    _check(cuda, x, coords, B, w, b, dy, relu)


@pytest.mark.parametrize("C", [32, 35])
def test_many_chunks(cuda, C):
    """Enough rows for hundreds of statistics blocks and several rows of partials per tail thread."""
    x, coords, B, w, b, dy = _layout("permuted", C, seed=11, mean=5.0, std=2.0, n=300_000)
    _check(cuda, x, coords, B, w, b, dy, True)


@pytest.mark.parametrize("fmt_name", ["fp16", "bf16"])
@pytest.mark.parametrize("C", [32, 3])
def test_16bit_copy_equals_cast_rows(cuda, fmt_name, C):
    from lidog_b200 import cabi
    L = cabi.lib()
    fmt = cabi.FMT_FP16 if fmt_name == "fp16" else cabi.FMT_BF16
    dt = torch.float16 if fmt_name == "fp16" else torch.bfloat16
    x, coords, B, w, b, _ = _layout("permuted", C, seed=3, std=4e4)  # fp16 copies saturate at +-65504 like lg_cast_rows
    x, coords, w, b = x.to(cuda), coords.to(cuda), w.to(cuda) * 3e4, b.to(cuda)
    n = x.shape[0]
    for relu in (0, 1):
        y = torch.empty_like(x)
        y16 = torch.empty((n, C), dtype=dt, device=cuda)
        st = torch.empty((2, B, C), dtype=torch.float64, device=cuda)
        cabi.check(L.lg_instnorm_forward(x.data_ptr(), coords.data_ptr(), n, C, B, w.data_ptr(), b.data_ptr(), EPS,
                                         relu, y.data_ptr(), y16.data_ptr(), fmt, st.data_ptr(), cabi.stream_of(x)))
        ref = torch.empty_like(y16)
        cabi.check(L.lg_cast_rows(y.data_ptr(), ref.data_ptr(), y.numel(), fmt, None, cabi.stream_of(y)))
        torch.cuda.synchronize()
        assert torch.equal(y16.view(torch.int16), ref.view(torch.int16)), (fmt_name, relu)


def test_runs_are_bit_identical(cuda):
    x, coords, B, w, b, dy = _layout("permuted", 48, seed=5, mean=3.0, n=200_000)
    box1, box2 = {}, {}
    r1 = _gpu(x, coords, B, w, b, dy, True, cuda, box1)
    r2 = _gpu(x, coords, B, w, b, dy, True, cuda, box2)
    for a, c in zip(r1, r2):
        assert torch.equal(a, c)
    if box1.get("y16") is not None:
        assert torch.equal(box1["y16"], box2["y16"])


def _sparse(cuda, n=3000, C=32, batch=3, seed=0):
    import MinkowskiEngine as ME
    rng = np.random.default_rng(seed)
    c = torch.from_numpy(random_voxels(rng, n, span=30, batch=batch)).to(cuda)
    f = torch.from_numpy(rng.standard_normal((c.shape[0], C)).astype(np.float32)).to(cuda)
    return ME.SparseTensor(features=f, coordinates=c)


def test_module_eval_equals_train_and_fuses_relu(cuda):
    import MinkowskiEngine as ME
    x = _sparse(cuda)
    m = ME.MinkowskiInstanceNorm(32).to(cuda)
    with torch.no_grad():
        m.weight.uniform_(0.5, 1.5)
        m.bias.uniform_(-0.5, 0.5)
    y_train = ME.MinkowskiReLU()(m(x))
    m.eval()
    y_eval = ME.MinkowskiReLU()(m(x))
    assert torch.equal(y_train.F, y_eval.F)
    assert y_train._f16_cache is not None  # the ReLU ran inside the launch and left the operand copy
    ref = torch.relu(instance_norm(x.F.cpu(), x.C[:, 0].cpu(), m.weight.cpu(), m.bias.cpu(), EPS))
    assert rel(y_train.F, ref) <= 1e-5
    # B from the manager's batch_size when set: trailing absent instances change nothing
    x.coordinate_manager.batch_size = 7
    assert torch.equal(ME.MinkowskiReLU()(m(x)).F, y_train.F)


def test_empty_tensor_launches_nothing(cuda):
    import MinkowskiEngine as ME
    from lidog_b200.me.sparse_tensor import SparseTensor
    st = SparseTensor(torch.empty(0, 8, device=cuda), coordinate_manager=object(), tensor_stride=2)
    y = ME.MinkowskiInstanceNorm(8).to(cuda)(st)
    assert y.F.shape == (0, 8) and y.tensor_stride == [2, 2, 2]


def test_stride4_tensor_of_the_pyramid(cuda):
    """Batch indices are read from the coarse coordinates of the tensor's own stride."""
    import MinkowskiEngine as ME
    x1 = _sparse(cuda, n=6000, batch=4, seed=2)
    cm = x1.coordinate_manager
    c4 = cm.get_coords(4)
    f = torch.randn(c4.shape[0], 48, device=cuda) * 2 + 7
    x4 = ME.SparseTensor(features=f, coordinate_manager=cm, tensor_stride=4)
    m = ME.MinkowskiInstanceNorm(48).to(cuda)
    y = m(x4)
    assert y.tensor_stride == [4, 4, 4] and torch.equal(y.C, c4)
    ref = instance_norm(f.cpu(), c4[:, 0].cpu(), m.weight.cpu(), m.bias.cpu(), EPS)
    assert rel(y.F, ref) <= 1e-5


def test_ibn_split_keeps_coordinates(cuda):
    """IBN-Net's block: half the channels through IN, half through BN, ME.cat, ReLU -- at stride 4."""
    import MinkowskiEngine as ME
    x1 = _sparse(cuda, n=6000, batch=4, seed=4)
    cm = x1.coordinate_manager
    c4 = cm.get_coords(4)
    f = torch.randn(c4.shape[0], 64, device=cuda)
    x = ME.SparseTensor(features=f, coordinate_manager=cm, tensor_stride=4)
    h = 32
    a = ME.SparseTensor(features=x.F[:, :h], coordinate_map_key=x.coordinate_map_key, coordinate_manager=x.coordinate_manager)
    b = ME.SparseTensor(features=x.F[:, h:], coordinate_map_key=x.coordinate_map_key, coordinate_manager=x.coordinate_manager)
    assert a.tensor_stride == [4, 4, 4] and b.coordinate_map_key == x.coordinate_map_key
    inn, bn = ME.MinkowskiInstanceNorm(h).to(cuda), ME.MinkowskiBatchNorm(64 - h).to(cuda)
    out = ME.MinkowskiReLU()(ME.cat(inn(a), bn(b)))
    assert out.tensor_stride == [4, 4, 4] and torch.equal(out.C, c4)
    fo = f.cpu().double()
    ref_a = instance_norm(fo[:, :h], c4[:, 0].cpu(), inn.weight.cpu(), inn.bias.cpu(), EPS)
    ref_b = torch.nn.functional.batch_norm(fo[:, h:], None, None, bn.bn.weight.detach().cpu().double(),
                                           bn.bn.bias.detach().cpu().double(), True, 0.0, bn.bn.eps)
    assert rel(out.F, torch.relu(torch.cat([ref_a, ref_b], 1))) <= 1e-5


# conv -> IN -> ReLU -> conv: with fp16 tensor-core operands the whole-model output bar of tests/test_gpu_model.py
# (4e-3; measured 4.1e-4 here) and, for the gradients, about twice the measured worst (1.2e-2: the fp16 dgrad / wgrad
# operands, unit round-off 2^-11, on a 2-layer chain); with the exact-fp32 convolutions tight bars
CHAIN_BARS = {"fp16": dict(out=4e-3, grad=2.5e-2), "off": dict(out=2e-5, grad=1e-4)}


@pytest.mark.parametrize("mode", ["off", "fp16"])
def test_chain_conv_in_relu_conv_matches_oracle(cuda, mode):
    import MinkowskiEngine as ME
    from lidog_b200.me import conv as meconv
    from oracle import me_cpu
    from oracle.instnorm import MinkowskiInstanceNorm as CpuInstanceNorm
    rng = np.random.default_rng(9)
    coords = random_voxels(rng, 4000, span=25, batch=3)
    feats = rng.standard_normal((coords.shape[0], 32)).astype(np.float32)
    torch.manual_seed(0)

    def build(M, InstanceNorm):
        return torch.nn.ModuleList([M.MinkowskiConvolution(32, 64, kernel_size=3, dimension=3),
                                    InstanceNorm(64), M.MinkowskiReLU(),
                                    M.MinkowskiConvolution(64, 32, kernel_size=3, dimension=3)])

    ref = build(me_cpu, CpuInstanceNorm)
    with torch.no_grad():
        ref[1].weight.uniform_(0.5, 1.5)
        ref[1].bias.uniform_(-0.5, 0.5)
    ref = ref.double()
    R = torch.from_numpy(rng.standard_normal((coords.shape[0], 32)))
    fo = torch.from_numpy(feats).double().requires_grad_(True)
    t = me_cpu.SparseTensor(coordinates=torch.from_numpy(coords), features=fo)
    for layer in ref:
        t = layer(t)
    (t.F * R).sum().backward()

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
        (g.F * R.float().to(cuda)).sum().backward()
        torch.cuda.synchronize()
    finally:
        meconv.CONFIG.update(old)
    errs = dict(out=rel(g.F, t.F), dfeat=rel(fg.grad, fo.grad))
    for (k, p), (_, po) in zip(net.named_parameters(), ref.named_parameters()):
        errs[k] = rel(p.grad, po.grad)
    record("instnorm_chain", mode=mode, **errs)
    bars = CHAIN_BARS[mode]
    assert errs["out"] <= bars["out"], (mode, errs)
    assert all(v <= bars["grad"] for k, v in errs.items() if k != "out"), (mode, errs)
