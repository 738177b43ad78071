"""CPU: the float64 oracle of RobustNet's instance-whitening loss on sparse tensors (oracle/isw.py), the closed-form
backward csrc/isw.cu implements, the n_b <= 1 rule, inactive scans, sign(0), C-ABI argument validation of
lg_inst_cov_forward / lg_inst_cov_backward, and the host module's surface."""
import ctypes
import importlib.util
import os

import pytest
import torch

from oracle.isw import instance_covariance, instance_whitening_loss

EPS = 1e-5


def _rows(B=5, C=6, n=120, seed=0, sorted_rows=False):
    g = torch.Generator().manual_seed(seed)
    bidx = torch.randint(0, B, (n,), generator=g)
    bidx[bidx == 3] = 4  # scan 3 absent
    bidx[bidx == 1] = 0
    bidx[17] = 1  # scan 1 has one row
    if sorted_rows:
        bidx = bidx.sort().values
    x = torch.randn(n, C, generator=g, dtype=torch.float64)
    return x, bidx


def _closed_form_dx(x, bidx, B, cov, mask, margin, num_sensitive):
    """dX_b = X_b (G_b + G_b^T) / (n_b - 1), G_b = (1/B) [term_b > 0] / num_sensitive * sign(cov_b) * M."""
    dx = torch.zeros_like(x)
    for b in range(B):
        r = bidx == b
        nb = int(r.sum())
        if nb <= 1:
            continue
        term = ((cov[b] * mask).abs().sum() - margin) / num_sensitive
        Gb = (term > 0).double() / B / num_sensitive * torch.sign(cov[b]) * mask
        dx[r] = x[r] @ (Gb + Gb.t()) / (nb - 1)
    return dx


@pytest.mark.parametrize("sorted_rows", [True, False])
def test_oracle_equals_literal_per_scan_bmm(sorted_rows):
    B, C = 5, 6
    x, bidx = _rows(B, C, sorted_rows=sorted_rows)
    got = instance_covariance(x, bidx, B, EPS)
    for b in range(B):
        rows = x[bidx == b]
        nb = rows.shape[0]
        if nb <= 1:
            want = EPS * torch.eye(C, dtype=torch.float64)
        else:
            f = rows.t().unsqueeze(0)
            want = torch.bmm(f, f.transpose(1, 2)).div(nb - 1)[0] + EPS * torch.eye(C, dtype=torch.float64)
        assert torch.allclose(got[b], want, rtol=1e-13, atol=1e-15), b


def test_oracle_equals_robustnet_dense_formula_on_a_feature_map():
    """RobustNet's get_covariance_matrix on a B x C x H x W map == the oracle on the same values as sparse rows."""
    g = torch.Generator().manual_seed(1)
    B, C, H, W = 3, 5, 4, 7
    fmap = torch.randn(B, C, H, W, generator=g, dtype=torch.float64)
    f = fmap.view(B, C, -1)
    dense = torch.bmm(f, f.transpose(1, 2)).div(H * W - 1) + EPS * torch.eye(C, dtype=torch.float64)
    rows = fmap.permute(0, 2, 3, 1).reshape(-1, C)
    bidx = torch.arange(B).repeat_interleave(H * W)
    perm = torch.randperm(rows.shape[0], generator=g)
    assert torch.allclose(instance_covariance(rows[perm], bidx[perm], B, EPS), dense, rtol=1e-13, atol=1e-15)


def test_oracle_gradcheck():
    x, bidx = _rows(B=4, C=3, n=25, seed=2)
    x.requires_grad_(True)
    mask = (torch.rand(3, 3, generator=torch.Generator().manual_seed(3)) > 0.4).double()
    mask = torch.triu(mask, 1)
    assert torch.autograd.gradcheck(
        lambda x: instance_whitening_loss(instance_covariance(x, bidx, 4, EPS), mask, 0.1, 3.0), (x,))
    assert torch.autograd.gradcheck(lambda x: instance_covariance(x, bidx, 4, EPS), (x,))


def test_autograd_equals_the_closed_form_backward():
    B, C = 5, 7
    x, bidx = _rows(B, C, n=200, seed=4)
    x.requires_grad_(True)
    mask = torch.triu(torch.ones(C, C, dtype=torch.float64), 1)
    cov = instance_covariance(x, bidx, B, EPS)
    # margin between the scans' masked sums: some scans are clamped (no gradient), some are not
    sums = (cov.detach() * mask).abs().sum(dim=(1, 2))
    margin = float(sums[[0, 2, 4]].sort().values[:2].mean())  # strictly between two scans' sums: off the kink
    instance_whitening_loss(cov, mask, margin, 4.0).backward()
    want = _closed_form_dx(x.detach(), bidx, B, cov.detach(), mask, margin, 4.0)
    assert torch.allclose(x.grad, want, rtol=1e-12, atol=1e-15)
    active = [b for b in (0, 2, 4) if float(sums[b]) > margin]
    assert 0 < len(active) < 3
    for b in (0, 2, 4):
        r = bidx == b
        assert bool((x.grad[r] != 0).any()) == (b in active), b  # a clamped scan passes exactly zero


def test_scans_with_at_most_one_row():
    B, C = 5, 4
    x, bidx = _rows(B, C, n=80, seed=5)
    x.requires_grad_(True)
    cov = instance_covariance(x, bidx, B, EPS)
    eye = EPS * torch.eye(C, dtype=torch.float64)
    assert torch.equal(cov[1].detach(), eye) and torch.equal(cov[3].detach(), eye)  # one row; absent
    instance_whitening_loss(cov, torch.ones(C, C, dtype=torch.float64), -1.0, 1.0).backward()
    assert torch.equal(x.grad[bidx == 1], torch.zeros(1, C, dtype=torch.float64))
    assert bool((x.grad[bidx == 0] != 0).all())


def test_sign_of_zero_passes_no_gradient():
    """cov_ij exactly 0 (channels with disjoint support): |.|'s gradient there is 0, as torch's abs backward gives."""
    B, C = 2, 4
    n = 40
    bidx = torch.arange(n) % B
    x = torch.randn(n, C, dtype=torch.float64, generator=torch.Generator().manual_seed(6))
    x[: n // 2, 0] = 0.0
    x[n // 2:, 1] = 0.0
    x.requires_grad_(True)
    cov = instance_covariance(x, bidx, B, EPS)
    assert float(cov[0, 0, 1].detach()) == 0.0 and float(cov[1, 0, 1].detach()) == 0.0
    mask = torch.zeros(C, C, dtype=torch.float64)
    mask[0, 1] = mask[1, 0] = 1.0  # only the zero entries are selected
    loss = instance_whitening_loss(cov, mask, -1.0, 2.0)  # active: term = 1 / 2 > 0
    loss.backward()
    assert float(loss.detach()) == 0.5 * 2 / B and torch.equal(x.grad, torch.zeros_like(x))


def test_host_loss_equals_oracle_loss():
    from lidog_b200.me.isw import instance_whitening_loss as host_loss
    g = torch.Generator().manual_seed(7)
    cov = torch.randn(6, 5, 5, generator=g, dtype=torch.float64)
    cov = (cov + cov.transpose(1, 2)).requires_grad_(True)
    mask = (torch.rand(5, 5, generator=g) > 0.5).double()
    margin = float((cov.detach() * mask).abs().sum(dim=(1, 2)).sort().values[2:4].mean())
    a = host_loss(cov, mask, margin, 3)
    ga, = torch.autograd.grad(a, cov)
    b = instance_whitening_loss(cov, mask, margin, 3)
    gb, = torch.autograd.grad(b, cov)
    assert torch.allclose(a, b, rtol=1e-15) and torch.equal(ga, gb)


def test_module_surface():
    import MinkowskiEngine as ME
    from lidog_b200 import me
    from lidog_b200.me.isw import COVARIANCE_EPS
    assert COVARIANCE_EPS == 1e-5
    assert me.instance_covariance is ME.instance_covariance
    assert me.instance_whitening_loss is ME.instance_whitening_loss
    from lidog_b200.me.sparse_tensor import SparseTensor
    st = SparseTensor(torch.ones(3, 2), coordinate_manager=object(), tensor_stride=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        me.instance_covariance(st)


def test_cabi_argument_validation():
    """Rejected before any CUDA call: this runs without a device."""
    from lidog_b200 import build, cabi
    build.build()
    L = cabi.lib()
    buf = ctypes.create_string_buffer(1 << 12)
    a16 = (ctypes.addressof(buf) + 15) & ~15
    ok = dict(x=a16, coords=a16, n=4, C=8, B=2, eps=1e-5, cov=a16, counts=a16)

    def f(**kw):
        d = dict(ok, **kw)
        return L.lg_inst_cov_forward(d["x"], d["coords"], d["n"], d["C"], d["B"], d["eps"], d["cov"], d["counts"], None)

    for bad in (dict(x=None), dict(coords=None), dict(cov=None), dict(counts=None), dict(n=-1), dict(n=1 << 31),
                dict(C=0), dict(B=0), dict(x=a16 + 4), dict(coords=a16 + 2), dict(cov=a16 + 2), dict(counts=a16 + 1),
                dict(eps=-1.0)):
        assert f(**bad) == -1, bad
        assert b"lg_inst_cov_forward" in L.lg_last_error_string()
    assert f(B=257) == -4 and f(C=257) == -4  # LG_ERR_UNSUPPORTED
    okb = dict(x=a16, coords=a16, n=4, C=8, B=2, G=a16, counts=a16, dx=a16)

    def g(**kw):
        d = dict(okb, **kw)
        return L.lg_inst_cov_backward(d["x"], d["coords"], d["n"], d["C"], d["B"], d["G"], d["counts"], d["dx"], None)

    for bad in (dict(x=None), dict(coords=None), dict(G=None), dict(counts=None), dict(dx=None), dict(n=-1),
                dict(C=0), dict(B=0), dict(x=a16 + 4), dict(dx=a16 + 8), dict(G=a16 + 1)):
        assert g(**bad) == -1, bad
        assert b"lg_inst_cov_backward" in L.lg_last_error_string()
    assert g(B=300) == -4 and g(C=300) == -4
    assert g(n=0, C=3, x=a16 + 4, dx=a16 + 4) == 0  # C % 4 != 0 needs 4-byte alignment only; n = 0 launches nothing


def _reference_loss():
    """RobustNet's own instance_whitening_loss from a reference checkout at oracle/_ref, if it has one."""
    from tests import refharness as rh
    for dirpath, _, files in os.walk(rh.REF):
        for name in files:
            if not name.endswith(".py"):
                continue
            path = os.path.join(dirpath, name)
            with open(path, errors="ignore") as fh:
                if "def instance_whitening_loss" not in fh.read():
                    continue
            spec = importlib.util.spec_from_file_location("_isw_ref_" + name[:-3], path)
            mod = importlib.util.module_from_spec(spec)
            try:
                spec.loader.exec_module(mod)
            except Exception:  # the file needs modules this checkout does not have
                continue
            return mod.instance_whitening_loss
    return None


def test_reference_function_on_the_oracle_shim():
    fn = _reference_loss()
    if fn is None:
        pytest.skip("no reference checkout defining instance_whitening_loss at oracle/_ref")
    B, C = 4, 5
    x, bidx = _rows(B, C, n=90, seed=8, sorted_rows=True)
    mask = torch.triu(torch.ones(C, C, dtype=torch.float64), 1)
    for b in (0, 2, 4):
        rows = x[bidx == b]
        fmap = rows.t().reshape(1, C, rows.shape[0], 1)  # (1, C, n_b) as an image of n_b x 1 pixels
        ref = fn(fmap, torch.eye(C, dtype=torch.float64), mask, 0.1, 3)
        ours = instance_whitening_loss(instance_covariance(rows, torch.zeros(rows.shape[0]), 1, EPS), mask, 0.1, 3)
        assert torch.allclose(torch.as_tensor(ref, dtype=torch.float64).reshape(()), ours, rtol=1e-12), b
