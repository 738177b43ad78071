"""Instance normalisation of a sparse tensor's feature matrix (oracle, float64 torch-CPU).

ME.MinkowskiInstanceNorm (SURVEY.md Appendix C): instance b = the rows whose batch index is b, statistics per
(instance, channel) with the biased variance, y = (x - mean_b) / sqrt(var_b + eps) * weight + bias.  Two passes
(mean, then centred squares) in float64, written with differentiable torch ops so autograd gives the reference
gradients (gradcheck in tests/test_instnorm_host.py).  `MinkowskiInstanceNorm` wraps it as a module for the sparse
tensors of oracle.me_cpu, so a small model built from both runs on the CPU stand-in too."""
from __future__ import annotations

import torch


def instance_norm(x: torch.Tensor, batch_idx: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor,
                  eps: float) -> torch.Tensor:
    """x [n, C], batch_idx int [n], weight / bias [C] or [1, C] -> float64 [n, C]."""
    x = x.double()
    b = batch_idx.long()
    if x.shape[0] == 0:
        return x.clone()
    B = int(b.max()) + 1
    onehot = torch.nn.functional.one_hot(b, B).double()  # [n, B]
    count = onehot.sum(0).clamp_min(1.0)[:, None]
    mean = onehot.t() @ x / count
    xc = x - mean[b]
    var = onehot.t() @ (xc * xc) / count
    return xc * torch.rsqrt(var[b] + eps) * weight.double().reshape(1, -1) + bias.double().reshape(1, -1)


class MinkowskiInstanceNorm(torch.nn.Module):
    """CPU stand-in of ME.MinkowskiInstanceNorm for oracle.me_cpu sparse tensors (`.F`, `.C`, `._like`): parameters
    `weight` [1, C] (ones) and `bias` [1, C] (zeros), no buffers; computes in float64 and returns the input's dtype."""

    def __init__(self, num_features):
        super().__init__()
        self.weight = torch.nn.Parameter(torch.ones(1, num_features))
        self.bias = torch.nn.Parameter(torch.zeros(1, num_features))

    def forward(self, x):
        # the one eps both implementations use (ME's constant): a shared number, not shared arithmetic
        from lidog_b200.me.norm import INSTANCE_NORM_EPS
        y = instance_norm(x.F, x.C[:, 0], self.weight, self.bias, INSTANCE_NORM_EPS)
        return x._like(y.to(x.F.dtype))
