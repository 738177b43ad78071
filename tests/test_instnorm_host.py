"""CPU: MinkowskiInstanceNorm's module surface, the float64 oracle it is checked against, C-ABI argument validation of
lg_instnorm_forward / lg_instnorm_backward, and the coordinate_map_key round trip of IBN-style channel splits."""
import ctypes

import pytest
import torch

from oracle.instnorm import instance_norm

EPS = 1e-8


def _loop_oracle(x, bidx, w, b, eps):
    """Per-instance Python loop in float64: the definition, spelled out."""
    x = x.double()
    out = torch.empty_like(x)
    for i in torch.unique(bidx).tolist():
        rows = (bidx == i).nonzero().flatten()
        xi = x[rows]
        mu = xi.mean(0, keepdim=True)
        var = ((xi - mu) ** 2).mean(0, keepdim=True)
        out[rows] = (xi - mu) / torch.sqrt(var + eps) * w.double().reshape(1, -1) + b.double().reshape(1, -1)
    return out


def test_module_surface():
    import MinkowskiEngine as ME
    from lidog_b200 import me
    from lidog_b200.me.norm import INSTANCE_NORM_EPS
    assert ME.MinkowskiInstanceNorm is me.MinkowskiInstanceNorm
    assert INSTANCE_NORM_EPS == 1e-8
    m = ME.MinkowskiInstanceNorm(48)
    assert tuple(m.weight.shape) == (1, 48) and tuple(m.bias.shape) == (1, 48)
    assert torch.equal(m.weight.detach(), torch.ones(1, 48)) and torch.equal(m.bias.detach(), torch.zeros(1, 48))
    assert sorted(m.state_dict()) == ["bias", "weight"]
    assert list(dict(m.named_buffers())) == []
    from oracle.instnorm import MinkowskiInstanceNorm as CpuInstanceNorm
    o = CpuInstanceNorm(48)
    assert sorted(o.state_dict()) == ["bias", "weight"]
    o.load_state_dict(m.state_dict())


def test_module_refuses_cpu_features():
    from lidog_b200.me.sparse_tensor import SparseTensor
    import MinkowskiEngine as ME
    st = SparseTensor(torch.ones(3, 2), coordinate_manager=object(), tensor_stride=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        ME.MinkowskiInstanceNorm(2)(st)


@pytest.mark.parametrize("sorted_rows", [True, False])
def test_oracle_equals_per_instance_loop(sorted_rows):
    g = torch.Generator().manual_seed(0)
    n, C = 200, 7
    bidx = torch.randint(0, 5, (n,), generator=g)
    bidx[bidx == 3] = 4  # instance 3 absent
    bidx[0] = 2
    bidx[bidx == 2] = 1
    bidx[17] = 2  # one-row instance: y = bias
    if sorted_rows:
        bidx = bidx.sort().values
    x = torch.randn(n, C, generator=g, dtype=torch.float64) * 3 + 1e3
    w, b = torch.randn(C, generator=g), torch.randn(C, generator=g)
    got = instance_norm(x, bidx, w, b, EPS)
    ref = _loop_oracle(x, bidx, w, b, EPS)
    assert got.dtype == torch.float64
    assert torch.allclose(got, ref, rtol=1e-12, atol=1e-10)
    one = (bidx == 2).nonzero().flatten()
    assert torch.allclose(got[one], b.double().reshape(1, -1).expand(len(one), -1), rtol=0, atol=1e-12)


def test_oracle_equals_torch_instance_norm_on_the_dense_view():
    g = torch.Generator().manual_seed(1)
    B, C, nb = 4, 6, 37
    x = torch.randn(B, C, nb, generator=g, dtype=torch.float64)
    w, b = torch.randn(C, generator=g, dtype=torch.float64), torch.randn(C, generator=g, dtype=torch.float64)
    ref = torch.nn.functional.instance_norm(x, weight=w, bias=b, eps=EPS)  # [B, C, nb]
    rows = x.permute(0, 2, 1).reshape(B * nb, C)
    bidx = torch.arange(B).repeat_interleave(nb)
    got = instance_norm(rows, bidx, w, b, EPS)
    assert torch.allclose(got, ref.permute(0, 2, 1).reshape(B * nb, C), rtol=1e-12, atol=1e-12)


def test_oracle_gradcheck():
    g = torch.Generator().manual_seed(2)
    n, C = 23, 3
    bidx = torch.tensor([0] * 9 + [2] * 13 + [3])  # absent instance 1, one-row instance 3
    x = torch.randn(n, C, generator=g, dtype=torch.float64, requires_grad=True)
    w = torch.randn(1, C, generator=g, dtype=torch.float64, requires_grad=True)
    b = torch.randn(1, C, generator=g, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(lambda x, w, b: instance_norm(x, bidx, w, b, 1e-3), (x, w, b))


def test_oracle_backward_matches_the_closed_form():
    """The formulas csrc/instnorm.cu implements: dx = invstd (g - mean_b g - xhat mean_b(g xhat)), g = dy w."""
    g = torch.Generator().manual_seed(3)
    n, C = 60, 4
    bidx = torch.randint(0, 3, (n,), generator=g)
    x = torch.randn(n, C, generator=g, dtype=torch.float64, requires_grad=True)
    w = torch.randn(1, C, generator=g, dtype=torch.float64, requires_grad=True)
    b = torch.randn(1, C, generator=g, dtype=torch.float64, requires_grad=True)
    dy = torch.randn(n, C, generator=g, dtype=torch.float64)
    instance_norm(x, bidx, w, b, EPS).backward(dy)
    with torch.no_grad():
        dx = torch.empty_like(x)
        xhat_all = torch.empty_like(x)
        for i in range(3):
            r = bidx == i
            xi = x[r]
            mu, var = xi.mean(0), xi.var(0, unbiased=False)
            invstd = 1 / torch.sqrt(var + EPS)
            xhat = (xi - mu) * invstd
            gg = dy[r] * w
            dx[r] = invstd * (gg - gg.mean(0) - xhat * (gg * xhat).mean(0))
            xhat_all[r] = xhat
    assert torch.allclose(x.grad, dx, rtol=1e-9, atol=1e-9)
    assert torch.allclose(w.grad, (dy * xhat_all).sum(0, keepdim=True), rtol=1e-10)
    assert torch.allclose(b.grad, dy.sum(0, keepdim=True), rtol=1e-12)


def test_cabi_argument_validation():
    """Rejected before any CUDA call: this runs without a device."""
    from lidog_b200 import build, cabi
    build.build()
    L = cabi.lib()
    buf = ctypes.create_string_buffer(1 << 12)
    a = ctypes.addressof(buf)
    a16 = (a + 15) & ~15
    fwd = L.lg_instnorm_forward
    ok = dict(x=a16, coords=a16, n=4, C=8, B=2, w=a16, b=a16, eps=1e-8, relu=1, y=a16, y16=None, fmt=0, st=a16)

    def f(**kw):
        d = dict(ok, **kw)
        return fwd(d["x"], d["coords"], d["n"], d["C"], d["B"], d["w"], d["b"], d["eps"], d["relu"], d["y"], d["y16"],
                   d["fmt"], d["st"], None)

    for bad in (dict(x=None), dict(coords=None), dict(w=None), dict(b=None), dict(y=None), dict(st=None),
                dict(n=-1), dict(C=0), dict(B=0), dict(x=a16 + 4), dict(y=a16 + 8), dict(st=a16 + 4),
                dict(y16=a16 + 2), dict(y16=a16, fmt=7)):
        assert f(**bad) == -1, bad
        assert b"lg_instnorm_forward" in L.lg_last_error_string()
    assert f(B=257) == -4  # LG_ERR_UNSUPPORTED: more instances than the kernels take
    assert f(C=3, x=a16 + 4, y=a16 + 4, n=0) == 0  # C % 4 != 0 needs 4-byte alignment only; n = 0 launches nothing
    bwd = L.lg_instnorm_backward
    okb = dict(dy=a16, x=a16, y=a16, coords=a16, n=4, C=8, B=2, w=a16, relu=1, st=a16, dx=a16, dw=a16, db=a16)

    def g(**kw):
        d = dict(okb, **kw)
        return bwd(d["dy"], d["x"], d["y"], d["coords"], d["n"], d["C"], d["B"], d["w"], d["relu"], d["st"], d["dx"],
                   d["dw"], d["db"], None)

    for bad in (dict(dy=None), dict(x=None), dict(y=None), dict(coords=None), dict(w=None), dict(st=None),
                dict(dx=None), dict(dw=None), dict(db=None), dict(n=-1), dict(C=0), dict(B=0), dict(dy=a16 + 4),
                dict(dx=a16 + 8)):
        assert g(**bad) == -1, bad
        assert b"lg_instnorm_backward" in L.lg_last_error_string()
    assert g(B=300) == -4


def test_coordinate_map_key_round_trip():
    """IBN splits channels as ME.SparseTensor(features=x.F[:, :h], coordinate_map_key=x.coordinate_map_key,
    coordinate_manager=x.coordinate_manager): the new tensor must sit at x's stride, not at stride 1."""
    import MinkowskiEngine as ME
    cm = object()
    x = ME.SparseTensor(torch.ones(5, 6), coordinate_manager=cm, tensor_stride=4)
    key = x.coordinate_map_key
    assert isinstance(key, ME.CoordinateMapKey) and key.get_tensor_stride() == [4, 4, 4]
    assert key == ME.CoordinateMapKey(4) and key != ME.CoordinateMapKey(2) and hash(key) == hash(ME.CoordinateMapKey(4))
    h = x.F[:, :3]
    y = ME.SparseTensor(features=h, coordinate_map_key=key, coordinate_manager=x.coordinate_manager)
    assert y.tensor_stride == [4, 4, 4] and y.coordinate_manager is cm and y.F is h
    # without a key nothing changes: the stride argument (default 1) decides
    assert ME.SparseTensor(h, coordinate_manager=cm).tensor_stride == [1, 1, 1]
    assert ME.SparseTensor(h, coordinate_manager=cm, tensor_stride=2).tensor_stride == [2, 2, 2]
