"""MinkUNet34 + BEV head, assembled from a layer table on the MinkowskiEngine-shaped API.

Host-side mirror of the reference's model interface
(utils/models/minkunet_bev.py:44-157 layer graph, :302-399 forward, :401-408
init, :410-442 `_make_layer`; utils/models/conv2d.py:9-25,42-52,180-197 for
the dense 2D head).  Module attribute names, parameter shapes and therefore
state-dict keys match the reference (SURVEY.md Appendix C.10), so its Lightning
checkpoints load here and vice versa.  The reference file itself also runs
unchanged on `MinkowskiEngine` (see INTEGRATION.md); this file exists because
/root/reference is not available on the GPU box and because the BEV projection
is routed to the fused CUDA operator instead of the dense torch formulation.

`ME` is the namespace providing the sparse layers: `lidog_b200.me` in the
product (default); tests pass the CPU oracle's stand-in to obtain the reference
result for the same weights.
"""
from __future__ import annotations

import torch
import torch.nn as nn

PLANES = (32, 64, 128, 256, 256, 128, 96, 96)
LAYERS34 = (2, 3, 4, 6, 2, 2, 2, 2)
INIT_DIM = 32
BLOCK_OUT = {"block8": 96, "block7": 96, "block6": 128, "bottle": 256}


class _DoubleConv(nn.Module):
    def __init__(self, cin, cout, k, s, p):
        super().__init__()
        self.double_conv = nn.Sequential(
            nn.Conv2d(cin, cout, kernel_size=k, padding=p, stride=s, bias=False), nn.BatchNorm2d(cout),
            nn.ReLU(inplace=True),
            nn.Conv2d(cout, cout, kernel_size=k, padding=p, stride=s, bias=False), nn.BatchNorm2d(cout),
            nn.ReLU(inplace=True))

    def forward(self, x):
        if x.is_cuda:  # BN + ReLU pairs on the fused kernels (the CPU oracle build of this model never gets here)
            from lidog_b200.me.norm import double_conv_forward
            return double_conv_forward(self.double_conv, x)
        return self.double_conv(x)


class _Down(nn.Module):
    def __init__(self, cin, cout):
        super().__init__()
        self.maxpool_conv = nn.Sequential(_DoubleConv(cin, cout, 3, 2, 1))

    def forward(self, x):
        return self.maxpool_conv(x)


class _OutConv(nn.Module):
    def __init__(self, cin, cout):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, kernel_size=1)

    def forward(self, x):
        return self.conv(x)


class Encoder2D(nn.Module):
    """Dense BEV head (cuDNN): two stride-2 3x3 conv+BN+ReLU, then 1x1 to classes."""

    def __init__(self, input_size, n_classes=7):
        super().__init__()
        self.down1 = _Down(input_size, 256)
        self.out_conv = _OutConv(256, n_classes)

    def forward(self, x):
        return self.out_conv(self.down1(x))


class MinkUNet34BEV(nn.Module):
    def __init__(self, in_channels, out_channels, D=3, initial_kernel_size=5, decoder_2d_level=("block8",),
                 mapping_bound_2d=50.0, ME=None, bev_fn=None, bev_policy="last", layers=LAYERS34,
                 bev_scaling_factor=1.0):
        super().__init__()
        from lidog_b200.lidog.bev import pool_for_scaling
        if ME is None:
            from lidog_b200 import me as ME
        if bev_fn is None:
            from lidog_b200.lidog.bev import sparse2super as bev_fn
        self._ME, self._bev_fn, self.bev_policy = ME, bev_fn, bev_policy
        self.D = D
        self.mapping_bound_2d = mapping_bound_2d
        # the reference's sparse2super scaling factor as a MaxPool2d (kernel, stride, padding); no parameters depend
        # on it, so the state dict is the same at every factor
        self.bev_pool = pool_for_scaling(bev_scaling_factor)
        self.decoder_2d_level = list(decoder_2d_level)
        Block = ME.modules.resnet_block.BasicBlock
        conv, convtr, bn = ME.MinkowskiConvolution, ME.MinkowskiConvolutionTranspose, ME.MinkowskiBatchNorm

        self.inplanes = INIT_DIM
        self.conv0p1s1 = conv(in_channels, INIT_DIM, kernel_size=initial_kernel_size, dimension=D)
        self.bn0 = bn(INIT_DIM)
        # encoder: stride-2 conv + BN, then a residual stage
        for i, ts in enumerate((1, 2, 4, 8)):
            setattr(self, f"conv{i + 1}p{ts}s2", conv(self.inplanes, self.inplanes, kernel_size=2, stride=2, dimension=D))
            setattr(self, f"bn{i + 1}", bn(self.inplanes))
            setattr(self, f"block{i + 1}", self._stage(Block, PLANES[i], layers[i]))
        # decoder: transposed conv + BN, concat skip, residual stage
        skips = (PLANES[2], PLANES[1], PLANES[0], INIT_DIM)
        for j, ts in enumerate((16, 8, 4, 2)):
            i = 4 + j
            setattr(self, f"convtr{i}p{ts}s2", convtr(self.inplanes, PLANES[i], kernel_size=2, stride=2, dimension=D))
            setattr(self, f"bntr{i}", bn(PLANES[i]))
            self.inplanes = PLANES[i] + skips[j] * Block.expansion
            setattr(self, f"block{i + 1}", self._stage(Block, PLANES[i], layers[i]))
        self.final = conv(PLANES[7] * Block.expansion, out_channels, kernel_size=1, bias=True, dimension=D)
        self.relu = ME.MinkowskiReLU(inplace=True)
        self.dropout = ME.MinkowskiDropout(p=0.5)  # constructed, never called (reference :126)
        self.encoders2d = nn.ModuleDict({k: Encoder2D(BLOCK_OUT[k], out_channels) for k in self.decoder_2d_level})
        self._init_weights()

    def _stage(self, Block, planes, n):
        ME = self._ME
        downsample = None
        if self.inplanes != planes * Block.expansion:
            downsample = nn.Sequential(
                ME.MinkowskiConvolution(self.inplanes, planes * Block.expansion, kernel_size=1, stride=1,
                                        dimension=self.D),
                ME.MinkowskiBatchNorm(planes * Block.expansion))
        blocks = [Block(self.inplanes, planes, stride=1, dilation=1, downsample=downsample, dimension=self.D)]
        self.inplanes = planes * Block.expansion
        blocks += [Block(self.inplanes, planes, stride=1, dilation=1, dimension=self.D) for _ in range(1, n)]
        return nn.Sequential(*blocks)

    def _init_weights(self):
        ME = self._ME
        for m in self.modules():
            if isinstance(m, ME.MinkowskiConvolution):  # transposed convs keep the default init (App. B.6)
                ME.utils.kaiming_normal_(m.kernel, mode="fan_out", nonlinearity="relu")
            if isinstance(m, ME.MinkowskiBatchNorm):
                nn.init.constant_(m.bn.weight, 1)
                nn.init.constant_(m.bn.bias, 0)

    def sparse2super(self, x, input_voxel_size=0.05):
        return self._bev_fn(x, bound=self.mapping_bound_2d, voxel_size=input_voxel_size, pool=self.bev_pool,
                            policy=self.bev_policy)

    def forward(self, x, is_seg=True, is_train=False):
        ME, relu = self._ME, self.relu
        out_p1 = relu(self.bn0(self.conv0p1s1(x)))
        skips = [out_p1]
        out = out_p1
        for i, ts in enumerate((1, 2, 4, 8)):
            out = relu(getattr(self, f"bn{i + 1}")(getattr(self, f"conv{i + 1}p{ts}s2")(out)))
            out = getattr(self, f"block{i + 1}")(out)
            skips.append(out)
        out_bottle = skips.pop()
        feats = {}
        names = ("bottle", "block6", "block7", "block8")
        for j, ts in enumerate((16, 8, 4, 2)):
            i = 4 + j
            out = relu(getattr(self, f"bntr{i}")(getattr(self, f"convtr{i}p{ts}s2")(out)))
            out = ME.cat(out, skips.pop())
            out = getattr(self, f"block{i + 1}")(out)
            feats[names[j]] = out
        out_block8 = out
        img_pred = None
        if is_train:
            img_pred = {k: self.encoders2d[k](self.sparse2super(feats[k])) for k in self.encoders2d.keys()}
        logits = self.final(out_block8)
        if is_seg:
            return logits, img_pred
        return logits, img_pred, out_bottle, None
