"""MinkowskiBatchNorm / MinkowskiSyncBatchNorm / ReLU / Dropout.

ME implements these as torch modules applied to the N x C feature matrix
(`.bn` attribute: utils/models/minkunet_bev.py:407-408; recursive
`convert_sync_batchnorm`: train_lidog.py:228).  The parameters and buffers still live in
`self.bn` (a torch BatchNorm1d / SyncBatchNorm, so state dicts stay ME-compatible), but in
training mode the arithmetic runs in liblidog_b200 (csrc/bn.cu), fused with what the
reference chains around it (utils/models/minkunet_bev.py:308-368, ME's BasicBlock):

    conv -> BN -> ReLU                         one statistics pass + one apply pass
    conv -> BN -> (+= residual) -> ReLU        the residual (a plain tensor or a second,
                                               not yet applied BN: the block's downsample)
                                               joins the same apply pass

The module API is unchanged, so the fusion is done lazily: `MinkowskiBatchNorm.forward`
returns a `DeferredBN` sparse tensor that only remembers its inputs; `+=` attaches the
residual, `MinkowskiReLU` (or any read of `.F`) runs the fused kernels.  The apply pass
also writes the 16-bit operand copy the next tensor-core convolution gathers, and the
backward pass hands the scaled 16-bit gradient straight to the convolution's dgrad / wgrad.
SyncBN exchanges the (2C+1) sums of the statistics pass (forward) and the 2C sums of the
backward pass with one all-reduce each.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn

from .. import cabi
from .conv import DeferredConv
from .sparse_tensor import SparseTensor

import ctypes as _C

CONFIG = {"fused": int(os.environ.get("LIDOG_FUSED_BN", "1")),
          # 1 = one library call per layer each way (lg_bn_layer_forward / _backward); 0 = fine-grained calls
          "layer_calls": int(os.environ.get("LIDOG_LAYER_CALLS", "1")),
          # 1 = layers without a residual recompute the ReLU mask from x in the backward instead of reading y
          "recompute_mask": int(os.environ.get("LIDOG_BN_RECOMPUTE_MASK", "1")),
          # 1 = BatchNorm2d + ReLU of the dense BEV head on the fused kernels too (channels_last memory)
          "head2d": int(os.environ.get("LIDOG_FUSED_HEAD_BN", "1")),
          # 1 = where the BN input came straight out of a tensor-core convolution, the backward writes dx in 16 bits
          # only (that convolution's backward reads nothing else); see me/_grad16.py for the guards
          "skip_dx32": int(os.environ.get("LIDOG_BN_SKIP_DX32", "1"))}
C_byref = _C.byref

from ._grad16 import publish_grad16


def _fmt16():
    from . import conv as meconv
    return meconv._fmt()


def _dtype16(fmt):
    return torch.float16 if fmt == cabi.FMT_FP16 else torch.bfloat16


def _group(bn):
    """(process group, world size) for a SyncBatchNorm in a live process group, else (None, 1)."""
    if isinstance(bn, nn.SyncBatchNorm) and torch.distributed.is_available() and torch.distributed.is_initialized():
        pg = bn.process_group if bn.process_group is not None else torch.distributed.group.WORLD
        ws = torch.distributed.get_world_size(pg)
        if ws > 1:
            return pg, ws
    return None, 1


def _all_sum(v: torch.Tensor, pg) -> torch.Tensor:
    """Sum of a float64 vector over the ranks of `pg`: the one-kernel peer-memory exchange (me/peer.py) when the
    node offers symmetric memory, an NCCL all-reduce otherwise.  Returns a new tensor."""
    from . import peer
    ex = peer.get(pg)
    out = torch.empty_like(v)
    if ex is not None:
        return ex.sum(v, out)
    out.copy_(v)
    torch.distributed.all_reduce(out, group=pg)
    return out


def _bn_statistics(x: torch.Tensor, bn, ws, ws_bytes):
    """Training-mode statistics of one BN: returns (stats [4C] = mean, invstd, scale, shift; global count; group)."""
    L = cabi.lib()
    n, C = x.shape
    dev = x.device
    sums = torch.empty(2 * C + 1, dtype=torch.float64, device=dev)
    cabi.check(L.lg_bn_stats(cabi.ptr(x), n, C, cabi.ptr(sums), cabi.ptr(ws), ws_bytes, cabi.stream()), "lg_bn_stats")
    pg, world = _group(bn)
    count = float(n)  # a host number without SyncBN, a device scalar (never read back) with it
    if pg is not None:  # SyncBN: one exchange of [sum x, sum x^2, n]
        sums = _all_sum(sums, pg)
        count = sums[2 * C:]
    count_host, count_dev = (count, None) if isinstance(count, float) else (0.0, count)
    stats = torch.empty(4 * C, dtype=torch.float32, device=dev)
    track = bn.track_running_stats and bn.running_mean is not None
    momentum = 0.1 if bn.momentum is None else float(bn.momentum)
    cabi.check(L.lg_bn_finalize(cabi.ptr(sums), count_host, cabi.ptr(count_dev), C,
                                cabi.ptr(bn.weight.detach() if bn.affine else None),
                                cabi.ptr(bn.bias.detach() if bn.affine else None), float(bn.eps), momentum,
                                cabi.ptr(bn.running_mean if track else None),
                                cabi.ptr(bn.running_var if track else None),
                                cabi.ptr(bn.num_batches_tracked if track else None), cabi.ptr(stats), cabi.stream()),
               "lg_bn_finalize")
    return stats, count, pg


class FusedBNFunction(torch.autograd.Function):
    """y = act(BN_a(x) [+ BN_b(x2)] [+ res]) with ONE library call each way (lg_bn_layer_forward / _backward): the
    statistics pass (skipped when the convolution epilogue already wrote its partials), a tail kernel that finishes the
    reduction, runs the SyncBN exchange over NVLink peer memory and finalises the statistics, and the apply pass.
    The 16-bit copy of y travels in `box`; `aux` = (bn_a, bn_b, stat partials of x, of x2, peer exchange or None)."""

    @staticmethod
    def forward(ctx, x, w, b, x2, w2, b2, res, aux, relu, box):
        bn_a, bn_b, sp_a, sp_b, ex = aux
        L = cabi.lib()
        x = x.contiguous()
        n, C = x.shape
        dev = x.device
        fmt = None if box.get("no16") else _fmt16()  # no16: no convolution of this library consumes y (dense 2D head)
        y = torch.empty_like(x)
        y16 = torch.empty((n, C), dtype=_dtype16(fmt), device=dev) if fmt is not None else None
        n_st = 4 * C + 4  # [4C + 2] used; rows of the two-branch tensor must stay 16-byte aligned (float4 reads)

        def branch(xt, bn, sp, stats):
            track = bn.track_running_stats and bn.running_mean is not None
            sp_ptr, sp_rows = (sp.data_ptr(), sp.shape[0]) if sp is not None else (None, 0)
            return cabi.BnBranch(xt.data_ptr(), sp_ptr, sp_rows, bn.weight.data_ptr(), bn.bias.data_ptr(),
                                 bn.running_mean.data_ptr() if track else None,
                                 bn.running_var.data_ptr() if track else None,
                                 bn.num_batches_tracked.data_ptr() if track else None, bn.eps,
                                 0.1 if bn.momentum is None else bn.momentum, stats.data_ptr())

        if x2 is not None:
            x2 = x2.contiguous()
            stats = torch.empty((2, n_st), dtype=torch.float32, device=dev)
            st_a, st_b = stats[0], stats[1]
            br_b = C_byref(branch(x2, bn_b, sp_b, st_b))
        else:
            st_a, st_b, br_b = torch.empty(n_st, dtype=torch.float32, device=dev), None, None
        if res is not None:
            res = res.contiguous()
        cabi.check(L.lg_bn_layer_forward(C_byref(branch(x, bn_a, sp_a, st_a)), br_b, cabi.ptr(res), 1 if relu else 0,
                                         n, C, y.data_ptr(), cabi.ptr(y16), fmt if fmt is not None else 0,
                                         cabi.peer_ctx(ex, 2 if x2 is not None else 1), cabi.stream_of(x)),
                   "lg_bn_layer_forward")
        if cabi.is_counting():
            cabi.count_launches("lg_bn_layer_forward", 1 + (1 if sp_a is not None else 2) +
                                (0 if x2 is None else (1 if sp_b is not None else 2)))
        box["y16"], box["fmt"] = y16, fmt
        # y is saved only where the backward needs it for the ReLU mask: without a residual the library recomputes
        # the mask from x (lg_bn_layer_backward with y = NULL; the two-branch form of that kernel spills registers,
        # so the three downsample layers keep reading y)
        keep_y = relu and (res is not None or x2 is not None or not CONFIG["recompute_mask"])
        ctx.save_for_backward(x, x2, y if keep_y else None, st_a, st_b, w, w2)
        ctx.meta = (relu, res is not None, fmt, ex)
        # fp32 dx / dx2 are skipped where the input is the output of a tensor-core convolution (it carried epilogue
        # statistics) and a 16-bit copy is published for that convolution's backward
        skip = bool(CONFIG["skip_dx32"]) and fmt is not None
        ctx.skip32 = (skip and sp_a is not None, skip and sp_b is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        L = cabi.lib()
        x, x2, y, st_a, st_b, w, w2 = ctx.saved_tensors
        relu, has_res, fmt, ex = ctx.meta
        n, C = x.shape
        # the gradient of one input of ME.cat is a column slice of the concatenated gradient: consumed in place
        if not (dy.stride(1) == 1 and dy.stride(0) >= C and dy.stride(0) % 4 == 0 and dy.data_ptr() % 16 == 0):
            dy = dy.contiguous()
        dev = x.device
        use16 = fmt is not None
        d16 = _dtype16(fmt) if use16 else None
        scales = torch.empty(12, dtype=torch.float32, device=dev)

        def branch(xt, st, gamma, skip32):
            dx = torch.empty_like(xt)  # autograd's handle; its values are written unless skip32
            dx16 = torch.empty((n, C), dtype=d16, device=dev) if use16 else None
            dgb = torch.empty((2, C), dtype=torch.float32, device=dev)
            return dx, dx16, dgb, cabi.BnBwdBranch(xt.data_ptr(), st.data_ptr(), gamma.data_ptr(),
                                                   None if skip32 else dx.data_ptr(),
                                                   cabi.ptr(dx16), dgb.data_ptr(), dgb.data_ptr() + 4 * C)

        skip_a, skip_b = ctx.skip32[0] and use16, ctx.skip32[1] and use16
        dx, dx16, dgb, br_a = branch(x, st_a, w, skip_a)
        dx2 = dx2_16 = dgb2 = br_b = None
        if x2 is not None:
            dx2, dx2_16, dgb2, br_b = branch(x2, st_b, w2, skip_b)
            br_b = C_byref(br_b)
        dres = torch.empty_like(x) if (has_res and ctx.needs_input_grad[6]) else None
        cabi.check(L.lg_bn_layer_backward(dy.data_ptr(), dy.stride(0) if n > 1 else C, cabi.ptr(y), 1 if relu else 0, n, C,
                                          C_byref(br_a), br_b,
                                          cabi.ptr(dres), fmt if use16 else 0, scales.data_ptr(),
                                          cabi.peer_ctx(ex, 1), cabi.stream_of(x)), "lg_bn_layer_backward")
        dw, db = dgb[0], dgb[1]
        dw2 = db2 = None
        if use16:
            publish_grad16(dx, dx16, scales, fmt, fp32_valid=not skip_a)
        if x2 is not None:
            dw2, db2 = dgb2[0], dgb2[1]
            if use16:
                publish_grad16(dx2, dx2_16, scales[4:], fmt, fp32_valid=not skip_b)
        return dx, dw, db, dx2, dw2, db2, dres, None, None, None


def bn_relu_2d(x: torch.Tensor, bn) -> torch.Tensor:
    """`nn.BatchNorm2d` -> `nn.ReLU` of the dense BEV head (`utils/models/conv2d.py:9-25`, DoubleConv) on the
    fused kernels: a channels_last [B, C, H, W] tensor IS a row-major [B*H*W, C] matrix.  One statistics pass, the
    tail kernel and one apply pass with the ReLU inside (12 B/element instead of cuDNN BN + in-place clamp = 20), and a
    backward that recomputes the mask (20 B/element instead of threshold_backward + cuDNN BN backward ~ 32).  Anything
    else (eval mode, NCHW memory, CPU) takes the torch modules."""
    if not (CONFIG["fused"] and CONFIG["head2d"] and bn.training and x.is_cuda and x.dtype == torch.float32
            and x.dim() == 4 and x.shape[1] % 4 == 0 and x.shape[1] <= 1024 and bn.affine
            and (bn.momentum is not None or not bn.track_running_stats)
            and x.is_contiguous(memory_format=torch.channels_last)):
        return torch.relu_(bn(x))
    B, C, H, W = x.shape
    rows = x.permute(0, 2, 3, 1).reshape(B * H * W, C)  # a view: channels_last memory is [B, H, W, C] row-major
    y = FusedBNFunction.apply(rows, bn.weight, bn.bias, None, None, None, None, (bn, None, None, None, None), True,
                              {"no16": True})
    return y.view(B, H, W, C).permute(0, 3, 1, 2)


def double_conv_forward(seq: nn.Sequential, x: torch.Tensor) -> torch.Tensor:
    """Forward of the reference's `DoubleConv.double_conv` = Sequential(Conv2d, BatchNorm2d, ReLU, Conv2d, BatchNorm2d,
    ReLU) with the two BN + ReLU pairs on the fused kernels (same modules, same parameters, same state-dict keys)."""
    if x.is_cuda and seq[1].training:
        return bn_relu_2d(seq[3](bn_relu_2d(seq[0](x), seq[1])), seq[4])
    return seq(x)


class FusedBNFunctionFine(torch.autograd.Function):
    """Fine-grained form of FusedBNFunction (5-9 library calls per layer each way): SyncBN over NCCL when the peer-memory
    exchange is unavailable, and LIDOG_LAYER_CALLS=0 for A/B runs.  Same arithmetic, same kernels for the two passes."""

    @staticmethod
    def forward(ctx, x, w, b, x2, w2, b2, res, bn_a, bn_b, relu, box):
        L = cabi.lib()
        x = x.contiguous()
        n, C = x.shape
        dev = x.device
        ws_bytes = L.lg_bn_workspace(n, C)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        st_a, count_a, pg_a = _bn_statistics(x, bn_a, ws, ws_bytes)
        st_b = count_b = pg_b = None
        if x2 is not None:
            x2 = x2.contiguous()
            st_b, count_b, pg_b = _bn_statistics(x2, bn_b, ws, ws_bytes)
        if res is not None:
            res = res.contiguous()
        fmt = _fmt16()
        y = torch.empty_like(x)
        y16 = torch.empty(x.shape, dtype=_dtype16(fmt), device=dev) if fmt is not None else None
        cabi.check(L.lg_bn_apply(cabi.ptr(x), cabi.ptr(st_a), cabi.ptr(x2), cabi.ptr(st_b), cabi.ptr(res), int(relu), n, C,
                                 cabi.ptr(y), cabi.ptr(y16), fmt if fmt is not None else 0, cabi.stream()), "lg_bn_apply")
        box["y16"], box["fmt"] = y16, fmt
        ctx.save_for_backward(x, x2, y if relu else None, st_a, st_b,
                              w.detach() if w is not None else None, w2.detach() if w2 is not None else None)
        ctx.meta = (relu, count_a, pg_a, count_b, pg_b, res is not None, fmt)
        return y

    @staticmethod
    def backward(ctx, dy):
        L = cabi.lib()
        x, x2, y, st_a, st_b, w, w2 = ctx.saved_tensors
        relu, count_a, pg_a, count_b, pg_b, has_res, fmt = ctx.meta
        dy = dy.contiguous()
        n, C = x.shape
        dev = x.device
        ws_bytes = L.lg_bn_workspace(n, C)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        sums = torch.empty(3 * C, dtype=torch.float64, device=dev)
        maxes = torch.empty(3 * C, dtype=torch.float32, device=dev)
        cabi.check(L.lg_bn_bwd_stats(cabi.ptr(dy), cabi.ptr(y), cabi.ptr(x), cabi.ptr(st_a), cabi.ptr(x2),
                                     cabi.ptr(st_b), int(relu), n, C, cabi.ptr(sums), cabi.ptr(maxes), cabi.ptr(ws),
                                     ws_bytes, cabi.stream()), "lg_bn_bwd_stats")
        sums_g = sums
        pg = pg_a if pg_a is not None else pg_b
        if pg is not None:  # SyncBN: dx needs the sums over every rank; dgamma / dbeta stay local (DDP reduces them)
            sums_g = _all_sum(sums, pg)  # (the fp16 bound only has to hold on this rank: maxes stay local)
        use16 = fmt is not None
        d16 = _dtype16(fmt) if use16 else None

        def branch(k, st, gamma, count, want_param_grads):
            coef = torch.empty(3 * C, dtype=torch.float32, device=dev)
            scale = torch.empty(4, dtype=torch.float32, device=dev)
            dgamma = torch.empty(C, dtype=torch.float32, device=dev) if want_param_grads else None
            dbeta = torch.empty(C, dtype=torch.float32, device=dev) if want_param_grads else None
            count_host, count_dev = (count, None) if isinstance(count, float) else (0.0, count)
            cabi.check(L.lg_bn_bwd_finalize(cabi.ptr(sums), cabi.ptr(sums_g), cabi.ptr(maxes), count_host,
                                            cabi.ptr(count_dev), C, k,
                                            cabi.ptr(gamma), cabi.ptr(st), cabi.ptr(coef), cabi.ptr(dgamma),
                                            cabi.ptr(dbeta), cabi.ptr(scale), cabi.stream()), "lg_bn_bwd_finalize")
            return coef, scale, dgamma, dbeta

        coef_a, scale_a, dw, db = branch(0, st_a, w, count_a, w is not None)
        dx = torch.empty_like(x)
        dx16 = torch.empty(x.shape, dtype=d16, device=dev) if use16 else None
        coef_b = scale_b = dw2 = db2 = dx2 = dx2_16 = None
        if x2 is not None:
            coef_b, scale_b, dw2, db2 = branch(1, st_b, w2, count_b, w2 is not None)
            dx2 = torch.empty_like(x2)
            dx2_16 = torch.empty(x2.shape, dtype=d16, device=dev) if use16 else None
        dres = dres16 = scale_r = None  # (no 16-bit copy of the residual gradient: no convolution consumes it)
        if has_res and ctx.needs_input_grad[6]:
            dres = torch.empty_like(x)
        cabi.check(L.lg_bn_bwd_apply(cabi.ptr(dy), cabi.ptr(y), cabi.ptr(x), cabi.ptr(st_a), cabi.ptr(coef_a),
                                     cabi.ptr(x2), cabi.ptr(st_b), cabi.ptr(coef_b), int(relu), n, C, cabi.ptr(dx),
                                     cabi.ptr(dx16), cabi.ptr(scale_a), cabi.ptr(dx2), cabi.ptr(dx2_16),
                                     cabi.ptr(scale_b), cabi.ptr(dres), cabi.ptr(dres16), cabi.ptr(scale_r),
                                     fmt if use16 else 0, cabi.stream()), "lg_bn_bwd_apply")
        if use16:
            publish_grad16(dx, dx16, scale_a, fmt)
            if dx2 is not None:
                publish_grad16(dx2, dx2_16, scale_b, fmt)
        return dx, dw, db, dx2, dw2, db2, dres, None, None, None, None


def _fusable(bn, feats: torch.Tensor) -> bool:
    """Decided from properties every rank of a SyncBN group shares (module configuration, dtype, channel count) --
    never from the local row count: a rank whose scan leaves 0 or 1 voxels at some stride must still take part in
    the same exchange as its peers (the kernels handle n = 0)."""
    return (CONFIG["fused"] and bn.training and feats.is_cuda and feats.dtype == torch.float32 and feats.dim() == 2
            and feats.shape[1] % 4 == 0 and feats.shape[1] <= 1024 and bn.affine
            and (bn.momentum is not None or not bn.track_running_stats))


def _partials_of(t: SparseTensor):
    """Epilogue statistics of the convolution that produced `t` (me/conv.py), if they still describe t.F."""
    sp = getattr(t, "_stat_partials", None)
    if sp is None or sp[1] != t.F._version:
        return None
    return sp[0]


class DeferredBN(SparseTensor):
    """BN output that has not been computed yet (see the module docstring).  Behaves as a SparseTensor; the first
    read of `.F` evaluates BN(src) [+ residual] without activation."""

    def __init__(self, src: SparseTensor, bn):
        self.coordinate_manager = src.coordinate_manager
        self._ts = src._ts
        self._f16_cache = None
        self._src, self._bn = src, bn
        self._residual = None
        self._value = None

    @property
    def _F(self):
        if self._value is None:
            self._evaluate(False)
        return self._value

    @_F.setter
    def _F(self, v):
        self._value = v

    def _evaluate(self, relu: bool):
        bn = self._bn
        x2 = w2 = b2 = res = bn_b = None
        r = self._residual
        if isinstance(r, DeferredBN) and r._value is None and r._residual is None:
            x2, w2, b2, bn_b = r._src.F, r._bn.weight, r._bn.bias, r._bn
        elif r is not None:
            res = r.F if isinstance(r, SparseTensor) else r
        box = {}
        src = self._src
        pg, _ = _group(bn)
        ex = None
        if pg is not None:
            from . import peer
            ex = peer.get(pg)
        if CONFIG["layer_calls"] and (pg is None or ex is not None):
            sp_a = _partials_of(src)
            sp_b = _partials_of(r._src) if x2 is not None else None
            self._value = FusedBNFunction.apply(src.F, bn.weight, bn.bias, x2, w2, b2, res, (bn, bn_b, sp_a, sp_b, ex),
                                                bool(relu), box)
        else:
            self._value = FusedBNFunctionFine.apply(src.F, bn.weight, bn.bias, x2, w2, b2, res, bn, bn_b, bool(relu), box)
        if box.get("y16") is not None:  # the next convolution's operand: no separate cast pass
            f = self._value
            self._f16_cache = ((box["fmt"], f._version, f.data_ptr()), box["y16"])
        self._src = self._residual = None
        return self

    def __iadd__(self, other):
        if self._value is None and self._residual is None and isinstance(other, SparseTensor):
            self._same_map(other)
            self._residual = other
            return self
        return SparseTensor.__iadd__(self, other)


def eval_bn_stats(bn) -> torch.Tensor:
    """Eval-mode coefficients of a BatchNorm1d in the lg_bn_apply layout, float32 [4C] = [mean, invstd, scale, shift]:
    scale = gamma / sqrt(running_var + eps), shift = beta - running_mean * scale, computed in float64 and rounded once."""
    mean, var = bn.running_mean.detach().double(), bn.running_var.detach().double()
    std = torch.sqrt(var + bn.eps)
    invstd = 1.0 / std
    scale = bn.weight.detach().double() / std if bn.affine else invstd
    shift = -mean * scale
    if bn.affine:
        shift = shift + bn.bias.detach().double()
    return torch.cat([mean, invstd, scale, shift]).float().contiguous()


def _infer_attachable(bn) -> bool:
    """An eval-mode BN that normalises with its running statistics can join the preceding convolution's launch."""
    return (not bn.training and bn.track_running_stats and bn.running_mean is not None
            and bn.running_var is not None)


class MinkowskiBatchNorm(nn.Module):
    def __init__(self, num_features, eps=1e-5, momentum=0.1, affine=True, track_running_stats=True):
        super().__init__()
        self.bn = nn.BatchNorm1d(num_features, eps=eps, momentum=momentum, affine=affine,
                                 track_running_stats=track_running_stats)

    def forward(self, input: SparseTensor) -> SparseTensor:
        if isinstance(input, DeferredConv) and _infer_attachable(self.bn) and input.accepts_bn(self.bn.num_features):
            input._bn_stats = self._eval_stats()
            return input
        if _fusable(self.bn, input.F):
            return DeferredBN(input, self.bn)
        return input._like(self.bn(input.F))

    def _eval_stats(self) -> torch.Tensor:
        """eval_bn_stats(self.bn), cached until a parameter or buffer is replaced or modified by torch, or the module
        goes back to training mode (the training kernels update the running buffers in place, invisibly to
        `_version`)."""
        b = self.bn
        key = tuple((t._version, t.data_ptr()) for t in (b.weight, b.bias, b.running_mean, b.running_var)
                    if t is not None)
        cache = self.__dict__.get("_eval_cache")
        if cache is None or cache[0] != key:
            cache = (key, eval_bn_stats(b))
            self.__dict__["_eval_cache"] = cache
        return cache[1]

    def train(self, mode: bool = True):
        if mode:  # running statistics change only in training mode
            self.__dict__.pop("_eval_cache", None)
        return super().train(mode)

    def __repr__(self):
        b = self.bn
        return f"{self.__class__.__name__}({b.num_features}, eps={b.eps}, momentum={b.momentum}, affine={b.affine})"


class MinkowskiSyncBatchNorm(MinkowskiBatchNorm):
    def __init__(self, num_features, eps=1e-5, momentum=0.1, affine=True, track_running_stats=True,
                 process_group=None):
        nn.Module.__init__(self)
        self.bn = nn.SyncBatchNorm(num_features, eps=eps, momentum=momentum, affine=affine,
                                   track_running_stats=track_running_stats, process_group=process_group)

    @classmethod
    def convert_sync_batchnorm(cls, module, process_group=None):
        """Recursively swap MinkowskiBatchNorm for MinkowskiSyncBatchNorm, keeping parameters and buffers."""
        out = module
        if isinstance(module, MinkowskiBatchNorm) and not isinstance(module, MinkowskiSyncBatchNorm):
            b = module.bn
            out = cls(b.num_features, b.eps, b.momentum, b.affine, b.track_running_stats, process_group)
            if b.affine:
                with torch.no_grad():
                    out.bn.weight, out.bn.bias = b.weight, b.bias
            out.bn.running_mean, out.bn.running_var = b.running_mean, b.running_var
            out.bn.num_batches_tracked = b.num_batches_tracked
            if hasattr(b, "qconfig"):
                out.bn.qconfig = b.qconfig
            return out
        for name, child in module.named_children():
            out.add_module(name, cls.convert_sync_batchnorm(child, process_group))
        return out


# ME's eps of MinkowskiInstanceNorm (SURVEY.md Appendix C); the CPU oracle's stand-in normalises with this value too
INSTANCE_NORM_EPS = 1e-8


def _instance_count(t: SparseTensor) -> int:
    """Instances B of a batch: `coordinate_manager.batch_size` when set, else max batch index + 1 (one host sync,
    cached on the manager, as lidog/bev.py:sparse2super does)."""
    cm = t.coordinate_manager
    B = getattr(cm, "batch_size", None)
    if B is None:
        B = int(t.C[:, 0].max().item()) + 1
        cm.batch_size = B
    return int(B)


class InstanceNormFunction(torch.autograd.Function):
    """y = act(IN(x) * weight + bias) per instance (csrc/instnorm.cu), ONE library call each way.  The 16-bit copy of
    y travels in `box`."""

    @staticmethod
    def forward(ctx, x, weight, bias, coords, B, relu, box):
        L = cabi.lib()
        x = x.contiguous()
        n, C = x.shape
        dev = x.device
        fmt = _fmt16()
        y = torch.empty_like(x)
        y16 = torch.empty((n, C), dtype=_dtype16(fmt), device=dev) if fmt is not None else None
        stats = torch.empty((2, B, C), dtype=torch.float64, device=dev)
        w, b = weight.detach().reshape(C).contiguous(), bias.detach().reshape(C).contiguous()
        cabi.check(L.lg_instnorm_forward(x.data_ptr(), coords.data_ptr(), n, C, B, w.data_ptr(), b.data_ptr(),
                                         INSTANCE_NORM_EPS, 1 if relu else 0, y.data_ptr(), cabi.ptr(y16),
                                         fmt if fmt is not None else 0, stats.data_ptr(), cabi.stream_of(x)),
                   "lg_instnorm_forward")
        box["y16"], box["fmt"] = y16, fmt
        ctx.save_for_backward(x, y if relu else None, coords, stats, w)
        ctx.meta = (B, bool(relu), tuple(weight.shape))
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y, coords, stats, w = ctx.saved_tensors
        B, relu, wshape = ctx.meta
        dy = dy.contiguous()
        n, C = x.shape
        dx = torch.empty_like(x)
        dwb = torch.empty((2, C), dtype=torch.float32, device=x.device)
        cabi.check(cabi.lib().lg_instnorm_backward(dy.data_ptr(), x.data_ptr(), cabi.ptr(y), coords.data_ptr(), n, C,
                                                   B, w.data_ptr(), 1 if relu else 0, stats.data_ptr(), dx.data_ptr(),
                                                   dwb[0].data_ptr(), dwb[1].data_ptr(), cabi.stream_of(x)),
                   "lg_instnorm_backward")
        return dx, dwb[0].view(wshape), dwb[1].view(wshape), None, None, None, None


class DeferredIN(SparseTensor):
    """MinkowskiInstanceNorm output not computed yet: `MinkowskiReLU` evaluates it with the ReLU fused, any other read
    of `.F` without.  Either way the result carries the 16-bit operand copy for the next convolution."""

    def __init__(self, src: SparseTensor, module):
        self.coordinate_manager = src.coordinate_manager
        self._ts = src._ts
        self._f16_cache = None
        self._src, self._in = src, module
        self._value = None

    @property
    def _F(self):
        if self._value is None:
            self._evaluate(False)
        return self._value

    @_F.setter
    def _F(self, v):
        self._value = v

    def _evaluate(self, relu: bool):
        src, m = self._src, self._in
        feats = src.F
        box = {}
        self._value = InstanceNormFunction.apply(feats, m.weight, m.bias, src.C.contiguous(), _instance_count(src),
                                                 bool(relu), box)
        if box.get("y16") is not None:
            f = self._value
            self._f16_cache = ((box["fmt"], f._version, f.data_ptr()), box["y16"])
        self._src = None
        return self


class MinkowskiInstanceNorm(nn.Module):
    """ME.MinkowskiInstanceNorm: per (instance = batch index, channel) normalisation with the biased variance and
    eps = INSTANCE_NORM_EPS, then `weight` [1, C] and `bias` [1, C]; no running statistics, so train and eval mode
    compute the same.  On CUDA float32 features it runs on csrc/instnorm.cu and defers like MinkowskiBatchNorm, so
    a following MinkowskiReLU joins the same launch."""

    def __init__(self, num_features):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(1, num_features))
        self.bias = nn.Parameter(torch.zeros(1, num_features))

    def forward(self, input: SparseTensor) -> SparseTensor:
        f = input.F
        if not (f.is_cuda and f.dtype == torch.float32 and f.dim() == 2):
            raise RuntimeError("MinkowskiInstanceNorm runs on CUDA float32 features only (csrc/instnorm.cu)")
        if f.shape[0] == 0:
            return input._like(torch.empty_like(f))
        return DeferredIN(input, self)

    def __repr__(self):
        return f"{self.__class__.__name__}({self.weight.shape[1]})"


class MinkowskiReLU(nn.Module):
    def __init__(self, inplace=False):
        super().__init__()
        self.inplace = inplace

    def forward(self, input: SparseTensor) -> SparseTensor:
        if isinstance(input, (DeferredBN, DeferredIN)) and input._value is None:
            return input._evaluate(True)
        if isinstance(input, DeferredConv) and input._value is None and input._bn_stats is not None:
            return input._launch(True)
        return input._like(torch.relu_(input.F) if self.inplace else torch.relu(input.F))


class MinkowskiDropout(nn.Module):
    def __init__(self, p=0.5, inplace=False):
        super().__init__()
        self.module = nn.Dropout(p, inplace)

    def forward(self, input: SparseTensor) -> SparseTensor:
        return input._like(self.module(input.F))
