"""Instance-selective whitening loss of RobustNet on sparse tensors (oracle, float64 torch-CPU).

[RobustNet-recalled] `get_covariance_matrix` and `instance_whitening_loss` (SURVEY.md 2.2) with "image" read as
"scan" (the rows whose batch index is b) and H*W as the scan's row count n_b: for each scan, the dense formula
    f = X_b^T viewed as (1, C, n_b);  cov_b = bmm(f, f^T) / (n_b - 1) + eps * I
on the features as given (not centred).  A scan with n_b <= 1 (the dense formula divides by zero there) is defined
as cov_b = eps * I with no gradient.  Written with differentiable torch ops, so autograd gives the reference
gradients (gradcheck in tests/test_isw_host.py)."""
from __future__ import annotations

import torch


def instance_covariance(x: torch.Tensor, batch_idx: torch.Tensor, B: int, eps: float) -> torch.Tensor:
    """x [n, C], batch_idx int [n] (rows outside [0, B) are left out) -> float64 [B, C, C]."""
    x = x.double()
    C = x.shape[1]
    b = batch_idx.long()
    eye = torch.eye(C, dtype=torch.float64)
    out = []
    for i in range(B):
        rows = x[b == i]
        nb = rows.shape[0]
        if nb <= 1:
            out.append(eps * eye + 0.0 * rows.sum())  # keeps the graph: the rows' gradient is exactly 0
            continue
        f = rows.t().reshape(1, C, nb)
        out.append((torch.bmm(f, f.transpose(1, 2)).div(nb - 1) + eps * eye)[0])
    return torch.stack(out)


def instance_whitening_loss(cov: torch.Tensor, mask: torch.Tensor, margin: float, num_sensitive) -> torch.Tensor:
    """(1/B) sum_b max(0, (sum_ij |cov_b * mask|_ij - margin) / num_sensitive), as RobustNet writes it."""
    off = torch.sum(torch.abs(cov * mask), dim=(1, 2), keepdim=True) - margin
    return torch.sum(torch.clamp(torch.div(off, num_sensitive), min=0)) / cov.shape[0]
