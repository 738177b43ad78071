"""Instance-selective whitening (ISW) loss of RobustNet, one of the normalisation baselines LiDOG is compared against
(SURVEY.md 2.2), with "image" read as "scan" (batch index of `.C`) and H*W as the scan's row count n_b.

    cov = instance_covariance(x)                            # [B, C, C], csrc/isw.cu, autograd
    loss = instance_whitening_loss(cov, mask, margin, num_sensitive)

`instance_covariance` is RobustNet's `get_covariance_matrix` on a sparse tensor: per scan, X_b^T X_b / (n_b - 1)
+ eps * I on the features as given (not centred); a scan with n_b <= 1 gets eps * I and passes no gradient.  Choosing
the mask (RobustNet's `CovMatrix_ISW`) is host code on covariances this returns and is not part of this module."""
from __future__ import annotations

import torch

from .. import cabi
from .norm import _instance_count
from .sparse_tensor import SparseTensor

# RobustNet's eps of get_covariance_matrix
COVARIANCE_EPS = 1e-5


class InstanceCovarianceFunction(torch.autograd.Function):
    """cov [B, C, C] of the rows of each scan (csrc/isw.cu), ONE library call each way; the backward forms
    (G_b + G_b^T) / (n_b - 1) once per scan and multiplies every row by it."""

    @staticmethod
    def forward(ctx, x, coords, B, eps):
        x = x.contiguous()
        n, C = x.shape
        cov = torch.empty((B, C, C), dtype=torch.float32, device=x.device)
        counts = torch.empty((B,), dtype=torch.int32, device=x.device)
        cabi.check(cabi.lib().lg_inst_cov_forward(x.data_ptr(), coords.data_ptr(), n, C, B, eps, cov.data_ptr(),
                                                  counts.data_ptr(), cabi.stream_of(x)), "lg_inst_cov_forward")
        ctx.save_for_backward(x, coords, counts)
        return cov

    @staticmethod
    def backward(ctx, dcov):
        x, coords, counts = ctx.saved_tensors
        n, C = x.shape
        B = counts.shape[0]
        dcov = dcov.contiguous()
        dx = torch.empty_like(x)
        cabi.check(cabi.lib().lg_inst_cov_backward(x.data_ptr(), coords.data_ptr(), n, C, B, dcov.data_ptr(),
                                                   counts.data_ptr(), dx.data_ptr(), cabi.stream_of(x)),
                   "lg_inst_cov_backward")
        return dx, None, None, None


def instance_covariance(x: SparseTensor, eps: float = COVARIANCE_EPS) -> torch.Tensor:
    """Per-scan covariance [B, C, C] (float32, exactly symmetric) of `x.F`, B from `coordinate_manager.batch_size`
    or one cached max()+1 read, as MinkowskiInstanceNorm does.  A deferred MinkowskiBatchNorm / InstanceNorm output
    is evaluated by reading `.F` (without a ReLU: apply MinkowskiReLU first to get one).  A tensor without rows gives
    eps * I for each of the manager's `batch_size` scans (which must then be set: there is no batch index to read)
    and a zero gradient."""
    f = x.F
    if not (f.is_cuda and f.dtype == torch.float32 and f.dim() == 2):
        raise RuntimeError("instance_covariance runs on CUDA float32 features only (csrc/isw.cu)")
    if f.shape[0] == 0:
        B = getattr(x.coordinate_manager, "batch_size", None)
        if B is None:
            raise ValueError("instance_covariance of a tensor without rows needs coordinate_manager.batch_size")
        C = f.shape[1]
        return (eps * torch.eye(C, device=f.device)).expand(int(B), C, C) + f.sum() * 0.0
    return InstanceCovarianceFunction.apply(f, x.C.contiguous(), _instance_count(x), float(eps))


def instance_whitening_loss(cov: torch.Tensor, mask: torch.Tensor, margin: float, num_sensitive) -> torch.Tensor:
    """RobustNet's instance_whitening_loss: (1/B) sum_b max(0, (sum_ij |cov_b * mask|_ij - margin) / num_sensitive),
    torch ops on the device, no host read."""
    off = (cov * mask).abs().sum(dim=(1, 2)) - margin
    return torch.clamp(off / num_sensitive, min=0).sum() / cov.shape[0]
