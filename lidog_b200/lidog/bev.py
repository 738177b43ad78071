"""Fused point-to-BEV projection operator (CUDA, csrc/bev.cu) with autograd.

Replaces `MinkUNetBaseBEV.sparse2super` + `filter_bounds` of the reference
(utils/models/minkunet_bev.py:158-230) without the D2H copy of the coordinates,
the per-sample Python loop and the dense 2000 x 2000 x C tensor.
`patch_reference_model` swaps it into an instance of the reference's own class.
"""
from __future__ import annotations

import os
import types

import torch

from .. import cabi

POLICIES = {"last": cabi.BEV_LAST, "max": cabi.BEV_MAX}

# Memory format of the projected image handed to the dense 2D head (logical shape stays (B, C, h, w)):
# channels_last lets cuDNN's tensor-op convolutions run without their NCHW<->NHWC staging copies.
CONFIG = {"channels_last": int(os.environ.get("LIDOG_BEV_CHANNELS_LAST", "1"))}


def image_size(bound: float, voxel_size: float) -> int:
    # max_height / max_width exactly as minkunet_bev.py:184-185 computes them
    return int(torch.tensor((bound - (-bound)) / voxel_size).int())


def pool_for_scaling(scaling_factor: float = 1.0) -> tuple:
    """MaxPool2d (kernel, stride, padding) of the reference's `sparse2super(x, input_voxel_size, scaling_factor)`
    (minkunet_bev.py:151-156, 222-224): stride 3 at s = 1, else int(3 / s).  The fused operator takes strides 1..16."""
    return (5, 3, 1) if scaling_factor == 1.0 else (5, int(3 / scaling_factor), 1)


def label_image_size(bound: float, voxel_size: float, pool=(5, 3, 1)) -> int:
    """Side of the BEV label image: the output of `Encoder2D` (two stride-2 3x3 convolutions, each ceil(h / 2)) on the
    pooled projection.  167 for the KITTI bound of 50 m and 100 for nuScenes' 30 m, at voxel 0.05 and pool 5/3/1."""
    pk, ps, pp = pool
    h = (image_size(bound, voxel_size) + 2 * pp - pk) // ps + 1
    for _ in range(2):
        h = (h + 1) // 2
    return h


class BevProjectFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, coords, batch_size, bound, voxel_size, pool, policy, channels_last):
        L = cabi.lib()
        feats_c = feats.detach().contiguous()
        coords = coords.contiguous()
        n, C = feats_c.shape
        H = W = image_size(bound, voxel_size)
        pk, ps, pp = pool
        h = (H + 2 * pp - pk) // ps + 1
        w = (W + 2 * pp - pk) // ps + 1
        out = torch.empty((batch_size, C, h, w), dtype=torch.float32, device=feats.device,
                          memory_format=torch.channels_last if channels_last else torch.contiguous_format)
        ws_bytes = L.lg_bev_workspace(n, C, batch_size, H, W, pk, ps, pp)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=feats.device)
        cabi.check(L.lg_bev_forward(cabi.ptr(coords), cabi.ptr(feats_c), n, C, batch_size, float(bound),
                                    float(voxel_size), H, W, pk, ps, pp, policy, 1 if channels_last else 0,
                                    cabi.ptr(out), cabi.ptr(ws), ws_bytes, cabi.stream()), "lg_bev_forward")
        ctx.save_for_backward(feats_c, coords, ws)
        ctx.args = (n, C, batch_size, H, W, pk, ps, pp, policy, ws_bytes)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        feats, coords, ws = ctx.saved_tensors
        n, C, batch_size, H, W, pk, ps, pp, policy, ws_bytes = ctx.args
        # consume the gradient in the memory order it arrives in (cuDNN hands back channels_last)
        nhwc = grad_out.dim() == 4 and grad_out.is_contiguous(memory_format=torch.channels_last) \
            and not grad_out.is_contiguous()
        if not nhwc:
            grad_out = grad_out.contiguous()
        grad_feats = torch.empty((n, C), dtype=torch.float32, device=feats.device)
        cabi.check(cabi.lib().lg_bev_backward(cabi.ptr(coords), cabi.ptr(feats), n, C, batch_size, H, W, pk, ps, pp,
                                              policy, 1 if nhwc else 0, cabi.ptr(grad_out), cabi.ptr(grad_feats),
                                              cabi.ptr(ws), ws_bytes, cabi.stream()), "lg_bev_backward")
        return grad_feats, None, None, None, None, None, None, None


def bev_project(coords, feats, batch_size, bound=50.0, voxel_size=0.05, pool=(5, 3, 1), policy="last",
                channels_last=False):
    return BevProjectFunction.apply(feats, coords, int(batch_size), float(bound), float(voxel_size), tuple(pool),
                                    POLICIES[policy], bool(channels_last))


def sparse2super(x, bound=50.0, voxel_size=0.05, pool=(5, 3, 1), policy="last", batch_size=None):
    """x: SparseTensor (any tensor stride; coordinates in stride-1 voxel units) -> [B, C, h, w]."""
    cm = x.coordinate_manager
    if batch_size is None:
        batch_size = getattr(cm, "batch_size", None)
    if batch_size is None:  # reference: batch_bottle_idx.max()+1 (minkunet_bev.py:193); one host sync, cached
        batch_size = int(x.C[:, 0].max().item()) + 1
        cm.batch_size = batch_size
    return bev_project(x.C, x.F, batch_size, bound, voxel_size, pool, policy, CONFIG["channels_last"])


def patch_reference_model(model, policy="last"):
    """Route an instance of the reference's MinkUNetBaseBEV (unchanged class) to the fused operator."""

    def _s2s(self, x, input_voxel_size=0.05, scaling_factor=1.0):
        return sparse2super(x, bound=self.mapping_bound_2d, voxel_size=input_voxel_size,
                            pool=pool_for_scaling(scaling_factor), policy=policy)

    model.sparse2super = types.MethodType(_s2s, model)

    # the dense head's DoubleConv (utils/models/conv2d.py:9-25): BN + ReLU pairs on the fused kernels
    def _double_conv(self, x):
        from lidog_b200.me.norm import double_conv_forward
        return double_conv_forward(self.double_conv, x)

    for m in model.modules():
        seq = getattr(m, "double_conv", None)
        if (isinstance(seq, torch.nn.Sequential) and len(seq) == 6 and isinstance(seq[1], torch.nn.BatchNorm2d)
                and isinstance(seq[2], torch.nn.ReLU) and isinstance(seq[4], torch.nn.BatchNorm2d)
                and isinstance(seq[5], torch.nn.ReLU)):
            m.forward = types.MethodType(_double_conv, m)
    return model
