"""MinkowskiConvolution / MinkowskiConvolutionTranspose on liblidog_b200.

Mirror of the reference-facing layer interface (ctor arguments, `.kernel`
(K, Cin, Cout) / (Cin, Cout), `.bias` (1, Cout); utils/models/minkunet_bev.py:57-123,
:404).  Forward, dgrad and wgrad call the C ABI: the tcgen05 gather-GEMM kernels for
channel counts that are multiples of 32, the exact-fp32 SIMT kernels otherwise
(1-channel stem, class head).  There is no CPU or torch fallback.
"""
from __future__ import annotations

import math
import os

import torch
import torch.nn as nn

from .. import cabi
from ._grad16 import take_grad16, require_fp32
from .sparse_tensor import SparseTensor

# operand format of the tensor-core path: "fp16" (default; 2^-11 unit round-off meets the 1e-3 bar),
# "bf16", or "off" (SIMT fp32 everywhere).
CONFIG = {
    "tc": os.environ.get("LIDOG_TC", "fp16"),
    # mask-sorted gather plans (lg_kernel_map_sorted) for the 3x3x3 and stride-2 layers; 0 = natural row order
    "sorted": int(os.environ.get("LIDOG_SORTED_PLANS", "1")),
    # the GEMM epilogue also writes per-tile column sums / sums of squares for the batch norm that follows
    # (lg_conv_layer_forward's stat_partials): the statistics pass over the convolution output disappears
    "epi_stats": int(os.environ.get("LIDOG_EPI_STATS", "1")),
    # 1 = one library call per layer each way (lg_conv_layer_forward / _backward); 0 = the fine-grained entry points
    # (lg_prep_weights + lg_conv_gemm_tc + lg_conv_wgrad_tc, workspaces from torch) kept for A/B runs
    "layer_calls": int(os.environ.get("LIDOG_LAYER_CALLS", "1")),
}


# Instrumentation for bench.py / tools (never on in a timed headline loop): per-launch CUDA events + algorithmic FLOPs
# (2 * pairs * Cin * Cout).  A census pass (events=False) counts the pairs of every plan once; an instrumented pass
# (events=True) brackets every launch with events and looks the pairs up by key.
PROFILE = {"enabled": False, "events": False, "records": [], "pairs": {}}


def _profiled(kernel, plan, cin, cout, launch):
    if not PROFILE["events"]:
        if plan.key not in PROFILE["pairs"]:
            PROFILE["pairs"][plan.key] = plan.count_pairs()
        out = launch()
        PROFILE["records"].append(dict(kernel=kernel, key=plan.key, cin=cin, cout=cout,
                                       flops=2.0 * PROFILE["pairs"][plan.key] * cin * cout))
        return out
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = launch()
    e1.record()
    PROFILE["records"].append(dict(kernel=kernel, key=plan.key, cin=cin, cout=cout, e0=e0, e1=e1,
                                   flops=2.0 * PROFILE["pairs"].get(plan.key, 0) * cin * cout))
    return out


def _fmt():
    return {"fp16": cabi.FMT_FP16, "bf16": cabi.FMT_BF16}.get(CONFIG["tc"])


# The tensor-core wgrad (k_wgrad2) takes at most 64 kernel offsets (two mask words); a layer with more (kernel size 5:
# 125 offsets) runs forward and backward on the SIMT kernels.  The whole layer moves: the tensor-core forward keeps only
# the 16-bit copy of x, and the SIMT wgrad needs the fp32 x.
TC_MAX_KERNEL_VOLUME = 64


def _tc_ok(cin, cout, kernel_volume):
    return (_fmt() is not None and cin % 32 == 0 and cout % 32 == 0
            and kernel_volume <= TC_MAX_KERNEL_VOLUME)


def _dt16(fmt):
    return torch.float16 if fmt == cabi.FMT_FP16 else torch.bfloat16


def _cast16(x: torch.Tensor, fmt: int, scale: torch.Tensor | None = None) -> torch.Tensor:
    out = torch.empty(x.shape, dtype=_dt16(fmt), device=x.device)
    cabi.check(cabi.lib().lg_cast_rows(cabi.ptr(x), cabi.ptr(out), x.numel(), fmt, cabi.ptr(scale), cabi.stream_of(x)),
               "lg_cast_rows")
    return out


def _gemm_simt(plan, A, W3, N, w_transposed, flip, bias):
    Y = torch.empty((plan.n_out, N), dtype=torch.float32, device=A.device)
    cabi.check(cabi.lib().lg_conv_gemm_simt(plan.cref, cabi.ptr(A), A.shape[1], cabi.ptr(W3), N, w_transposed, flip,
                                            cabi.ptr(bias), cabi.ptr(Y), cabi.stream_of(A)), "lg_conv_gemm_simt")
    return Y


def _gemm_tc(plan, A16, B16, N, flip, fmt, out_scale, bias):
    """Fine-grained path (LIDOG_LAYER_CALLS=0, instrumented passes, tools)."""
    Y = torch.empty((plan.n_out, N), dtype=torch.float32, device=A16.device)

    def launch():
        cabi.check(cabi.lib().lg_conv_gemm_tc(plan.cref, cabi.ptr(A16), A16.shape[1], cabi.ptr(B16), N, flip, fmt,
                                              cabi.ptr(out_scale), cabi.ptr(bias), cabi.ptr(Y),
                                              cabi.stream_of(A16)), "lg_conv_gemm_tc")
    if PROFILE["enabled"]:
        _profiled("k_gemm_tc", plan, A16.shape[1], N, launch)
    else:
        launch()
    return Y


class WeightCache:
    """16-bit copies of one layer's kernel, refreshed only when the parameter changed (optimizer step, load):
    round 1 ran lg_prep_weights for all 61 layers on every forward."""
    __slots__ = ("key", "w16", "w16t")

    def __init__(self):
        self.key = None

    def get(self, kernel: torch.Tensor, K, cin, cout, fmt):
        """-> (w16 [K][Cin][Cout], w16t [K][Cout][Cin], stale) -- `stale` = the copies must be rewritten."""
        key = (kernel._version, kernel.data_ptr(), fmt)
        stale = key != self.key
        if stale:
            if self.key is None or self.w16.device != kernel.device or self.key[2] != fmt:
                dt = _dt16(fmt)
                self.w16 = torch.empty((K, cin, cout), dtype=dt, device=kernel.device)
                self.w16t = torch.empty((K, cout, cin), dtype=dt, device=kernel.device)
            self.key = key
        return self.w16, self.w16t, stale


class SparseConvFunction(torch.autograd.Function):
    """y = conv(x, kernel) over the gather plans of one layer.

    plans = (fwd, dgrad, wgrad, flip_dgrad): see MinkowskiConvolutionBase._plans.
    `src` (optional SparseTensor) provides the cached 16-bit operand copy of x, `wcache` the cached 16-bit weights,
    `box` (dict) receives the epilogue statistics for the batch norm that follows ("stats": [4 * tiles, 2 * Cout]).
    """

    @staticmethod
    def forward(ctx, x, kernel, bias, plans, src, wcache, box):
        p_fwd = plans[0]
        if kernel.dim() == 3:
            K, cin, cout = kernel.shape
        else:
            K, (cin, cout) = 1, kernel.shape
        x = x.contiguous()
        ctx.plans, ctx.shape, ctx.kdim = plans, (K, cin, cout), kernel.dim()
        ctx.has_bias = bias is not None
        ctx.tc = _tc_ok(cin, cout, K) and x.shape[0] > 0
        L = cabi.lib()
        if ctx.tc:
            fmt = _fmt()
            x16 = src._f16(fmt) if src is not None else _cast16(x.detach(), fmt)
            Wc = kernel.detach()
            if not Wc.is_contiguous():
                Wc = Wc.contiguous()
            b = None if bias is None else bias.detach().reshape(-1)
            if wcache is None:
                wcache = WeightCache()
            w16, w16t, stale = wcache.get(Wc, K, cin, cout, fmt)
            if CONFIG["layer_calls"] and not PROFILE["enabled"]:
                y = torch.empty((p_fwd.n_out, cout), dtype=torch.float32, device=x.device)
                stats = None
                if box is not None and CONFIG["epi_stats"] and b is None:
                    stats = torch.empty((4 * p_fwd.n_tiles, 2 * cout), dtype=torch.float32, device=x.device)
                    box["stats"] = stats
                cabi.check(L.lg_conv_layer_forward(p_fwd.cref, x16.data_ptr(), cin, Wc.data_ptr(), cout, w16.data_ptr(),
                                                   w16t.data_ptr(), 1 if stale else 0, fmt, cabi.ptr(b), y.data_ptr(),
                                                   cabi.ptr(stats), cabi.stream_of(x)), "lg_conv_layer_forward")
                cabi.count_launches("lg_conv_layer_forward", 2 if stale else 1)
            else:
                if stale:
                    cabi.check(L.lg_prep_weights(Wc.data_ptr(), K, cin, cout, w16.data_ptr(), w16t.data_ptr(), fmt,
                                                 cabi.stream_of(x)), "lg_prep_weights")
                y = _gemm_tc(p_fwd, x16, w16t, cout, 0, fmt, None, b)
            # `kernel` is saved for autograd's version check only: a parameter update between this forward and its
            # backward (which would also have refreshed the cached 16-bit copy) then fails loudly
            ctx.fmt, ctx.w16 = fmt, w16
            ctx.save_for_backward(x16, kernel)
        else:
            W3c = (kernel if kernel.dim() == 3 else kernel.unsqueeze(0)).detach().contiguous()
            b = None if bias is None else bias.detach().reshape(-1).contiguous()
            y = _gemm_simt(p_fwd, x.detach(), W3c, cout, 0, 0, b)
            ctx.save_for_backward(x.detach(), W3c)
        return y

    @staticmethod
    def backward(ctx, dy):
        _, p_dgrad, p_wgrad, flip = ctx.plans
        K, cin, cout = ctx.shape
        L = cabi.lib()
        dy = dy.contiguous()
        dx = dw = db = None
        if ctx.has_bias and ctx.needs_input_grad[2]:
            require_fp32(dy, "convolution bias gradient")
            db = dy.sum(0, keepdim=True)
        if ctx.tc:
            x16, _ = ctx.saved_tensors
            fmt = ctx.fmt
            w16 = ctx.w16
            hit = take_grad16(dy, fmt)  # the fused BN backward already wrote the scaled 16-bit gradient
            if hit is not None:
                dy16, scale = hit
            else:
                require_fp32(dy, "convolution backward (16-bit copy not usable)")
                scale = None
                if fmt == cabi.FMT_FP16:  # bring the gradient into fp16's normal range (power-of-two scale)
                    scale = torch.empty(4, dtype=torch.float32, device=dy.device)
                    cabi.check(L.lg_absmax_scale(cabi.ptr(dy), dy.numel(), cabi.ptr(scale), cabi.stream_of(dy)),
                               "lg_absmax_scale")
                dy16 = _cast16(dy, fmt, scale)
            inv_ptr = None if scale is None else scale.data_ptr() + 4  # scale = {2^k, 2^-k, ...}
            want_dx, want_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
            if CONFIG["layer_calls"] and not PROFILE["enabled"]:
                if want_dx:
                    dx = torch.empty((p_dgrad.n_out, cin), dtype=torch.float32, device=dy.device)
                if want_dw:
                    dw = torch.empty((K, cin, cout), dtype=torch.float32, device=dy.device)
                cabi.check(L.lg_conv_layer_backward(p_dgrad.cref, p_wgrad.cref, flip, x16.data_ptr(), cin,
                                                    dy16.data_ptr(), cout, w16.data_ptr(), fmt, inv_ptr, cabi.ptr(dx),
                                                    cabi.ptr(dw), cabi.stream_of(dy)), "lg_conv_layer_backward")
                cabi.count_launches("lg_conv_layer_backward", (1 if want_dx else 0) + (2 if want_dw else 0))
            else:
                inv = None if scale is None else scale[1:]
                if want_dx:
                    dx = _gemm_tc(p_dgrad, dy16, w16, cin, flip, fmt, inv, None)
                if want_dw:
                    dw = torch.empty((K, cin, cout), dtype=torch.float32, device=dy.device)
                    ws_bytes = L.lg_conv_wgrad_tc_workspace(p_wgrad.cref, cin, cout)
                    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dy.device)

                    def launch():
                        cabi.check(L.lg_conv_wgrad_tc(p_wgrad.cref, cabi.ptr(x16), cin, cabi.ptr(dy16), cout, fmt,
                                                      cabi.ptr(inv), cabi.ptr(dw), cabi.ptr(ws), ws_bytes,
                                                      cabi.stream_of(dy)), "lg_conv_wgrad_tc")
                    if PROFILE["enabled"]:
                        _profiled("k_wgrad_tc", p_wgrad, cin, cout, launch)
                    else:
                        launch()
        else:
            require_fp32(dy, "fp32 convolution backward")
            x, W3c = ctx.saved_tensors
            if ctx.needs_input_grad[0]:
                dx = _gemm_simt(p_dgrad, dy, W3c, cin, 1, flip, None)
            if ctx.needs_input_grad[1]:
                dw = torch.empty((K, cin, cout), dtype=torch.float32, device=dy.device)
                ws_bytes = L.lg_conv_wgrad_workspace(p_wgrad.cref, cin, cout)
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dy.device)
                cabi.check(L.lg_conv_wgrad_simt(p_wgrad.cref, cabi.ptr(x), cin, cabi.ptr(dy), cout, cabi.ptr(dw),
                                                cabi.ptr(ws), ws_bytes, cabi.stream_of(dy)), "lg_conv_wgrad_simt")
        if dw is not None and ctx.kdim == 2:
            dw = dw[0]
        return dx, dw, db, None, None, None, None


class MinkowskiConvolutionBase(nn.Module):
    is_transpose = False

    def __init__(self, in_channels, out_channels, kernel_size=-1, stride=1, dilation=1, bias=False,
                 kernel_generator=None, expand_coordinates=False, convolution_mode=None, dimension=3):
        super().__init__()
        if dimension != 3:
            raise ValueError("only dimension=3 is on the LiDOG path")
        if dilation != 1 or kernel_generator is not None or expand_coordinates:
            raise NotImplementedError("dilation / kernel_generator / expand_coordinates are outside the LiDOG path")
        kernel_size, stride = int(kernel_size), int(stride)
        if (kernel_size, stride) not in ((1, 1), (3, 1), (5, 1), (2, 2)):
            raise NotImplementedError(f"kernel_size={kernel_size}, stride={stride} is outside the LiDOG path")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.dilation, self.dimension = kernel_size, stride, 1, dimension
        self.kernel_volume = kernel_size ** 3
        shape = (in_channels, out_channels) if self.kernel_volume == 1 else (self.kernel_volume, in_channels, out_channels)
        self.kernel = nn.Parameter(torch.empty(shape))
        self.bias = nn.Parameter(torch.empty(1, out_channels)) if bias else None
        self._wcache = WeightCache()
        self.reset_parameters()

    def reset_parameters(self, is_transpose=None):
        # ME default: uniform(+-1/sqrt(fan)), fan = Cin*K (Cout*K when transposed)  [SURVEY App. C.9]
        n = (self.out_channels if self.is_transpose else self.in_channels) * self.kernel_volume
        stdv = 1.0 / math.sqrt(n)
        with torch.no_grad():
            self.kernel.uniform_(-stdv, stdv)
            if self.bias is not None:
                self.bias.uniform_(-stdv, stdv)

    def _plans(self, cm, ts_in):
        k, s = self.kernel_size, self.stride
        if self.is_transpose:
            ts_out = ts_in // s
            if s != 2 or ts_in % 2:
                raise NotImplementedError("transposed convolution is implemented for kernel 2 / stride 2")
            if ts_out not in cm.levels:
                raise RuntimeError("transposed convolution needs the finer coordinate map created by the encoder")
            up, down = cm.plan("up", ts_in, ts_out, 2), cm.plan(self._kind("down"), ts_out, ts_in, 2)
            return ts_out, (up, down, up, 0)
        ts_out = ts_in * s
        if s == 2:
            down, up = cm.plan(self._kind("down"), ts_in, ts_out, 2), cm.plan("up", ts_out, ts_in, 2)
            return ts_out, (down, up, down, 0)
        if k == 1:
            p = cm.plan("identity", ts_in, ts_in, 1)
            return ts_out, (p, p, p, 0)
        p = cm.plan(self._kind("same") if k == 3 else "same", ts_in, ts_in, k)
        return ts_out, (p, p, p, 1)

    @staticmethod
    def _kind(kind):
        return kind + "_sorted" if CONFIG["sorted"] else kind

    def forward(self, input: SparseTensor) -> SparseTensor:
        assert isinstance(input, SparseTensor)
        cm = input.coordinate_manager
        ts_out, plans = self._plans(cm, input._ts)
        if not self.training and infer_fast_path(False, torch.is_grad_enabled(), self.bias is not None,
                                                 self.in_channels, self.out_channels, input.F.is_cuda, plans[0].n_out,
                                                 self.kernel_volume):
            return DeferredConv(self, input, plans, ts_out)
        box = {} if self.training else None
        y = SparseConvFunction.apply(input.F, self.kernel, self.bias, plans, input, self._wcache, box)
        out = SparseTensor(y, tensor_stride=ts_out, coordinate_manager=cm)
        if box:
            out._stat_partials = (box["stats"], y._version)
        return out

    def _forward_now(self, input: SparseTensor, plans, ts_out) -> SparseTensor:
        """Today's forward of an eval-mode layer: the convolution alone (no epilogue statistics)."""
        y = SparseConvFunction.apply(input.F, self.kernel, self.bias, plans, input, self._wcache, None)
        return SparseTensor(y, tensor_stride=ts_out, coordinate_manager=input.coordinate_manager)

    def __repr__(self):
        return (f"{self.__class__.__name__}(in={self.in_channels}, out={self.out_channels}, "
                f"kernel_size={[self.kernel_size] * 3}, stride={[self.stride] * 3}, dilation=[1, 1, 1])")


def infer_fast_path(training, grad_enabled, has_bias, cin, cout, is_cuda, n_out, kernel_volume=1) -> bool:
    """Whether a convolution forward returns a DeferredConv (inference epilogue, lg_conv_layer_infer): only in eval mode
    without autograd, on the tensor-core path (kernel_volume <= TC_MAX_KERNEL_VOLUME; the layers pass theirs) with one
    library call per layer and no instrumentation, for a layer without bias whose column blocks are multiples of 32, on
    a non-empty output.  Everything else runs the forward of training and of eval with gradients unchanged."""
    return (not training and not grad_enabled and not has_bias and _tc_ok(cin, cout, kernel_volume)
            and (cout // ((cout + 255) // 256)) % 32 == 0 and bool(CONFIG["layer_calls"]) and not PROFILE["enabled"]
            and is_cuda and n_out > 0)


class DeferredConv(SparseTensor):
    """Output of an eval-mode tensor-core convolution that has not been launched yet (the inference counterpart of
    me/norm.py's DeferredBN, one step earlier).  An eval-mode MinkowskiBatchNorm attaches its running-statistics
    coefficients, `+=` a residual, and MinkowskiReLU launches conv -> BN [-> + residual] -> ReLU as ONE library call
    that also writes the 16-bit operand copy of the next convolution.  Any other read of `.F` launches without ReLU
    (and without anything, when no batch norm was attached: the plain convolution)."""

    def __init__(self, conv: MinkowskiConvolutionBase, src: SparseTensor, plans, ts_out: int):
        self.coordinate_manager = src.coordinate_manager
        self._ts = ts_out
        self._f16_cache = None
        self._conv, self._src, self._plans = conv, src, plans
        self._bn_stats = None   # float32 [4 * Cout] in the lg_bn_apply layout, set by MinkowskiBatchNorm
        self._residual = None   # fp32 [n_out, Cout] features of the residual, set by +=
        self._value = None

    @property
    def _F(self):
        if self._value is None:
            self._launch(False)
        return self._value

    @_F.setter
    def _F(self, v):
        self._value = v

    def accepts_bn(self, num_features: int) -> bool:
        """A batch norm of `num_features` channels can still be attached: not launched, nothing attached yet."""
        return (self._value is None and self._bn_stats is None and self._residual is None
                and num_features == self._conv.out_channels)

    def __iadd__(self, other):
        if self._value is None and self._bn_stats is not None and self._residual is None and isinstance(other, SparseTensor):
            self._same_map(other)
            if isinstance(other, DeferredConv) and other._value is None:
                other._launch(False)  # the block's downsample (1x1 conv + BN): launched first, without ReLU
            r = other.F
            if (r.dtype == torch.float32 and r.is_contiguous() and r.data_ptr() % 16 == 0
                    and tuple(r.shape) == (self._plans[0].n_out, self._conv.out_channels)):
                self._residual = r
                return self
        return SparseTensor.__iadd__(self, other)

    def _launch(self, relu: bool):
        conv, src = self._conv, self._src
        if self._bn_stats is None:  # nothing to fuse: the plain convolution
            self._value = conv._forward_now(src, self._plans, self._ts).F
            self._src = None
            return self
        p = self._plans[0]
        kernel = conv.kernel.detach()
        if kernel.dim() == 3:
            K, cin, cout = kernel.shape
        else:
            K, (cin, cout) = 1, kernel.shape
        fmt = _fmt()
        x16 = src._f16(fmt)
        Wc = kernel if kernel.is_contiguous() else kernel.contiguous()
        w16, w16t, stale = conv._wcache.get(Wc, K, cin, cout, fmt)
        res = self._residual
        y = torch.empty((p.n_out, cout), dtype=torch.float32, device=x16.device)
        y16 = torch.empty((p.n_out, cout), dtype=_dt16(fmt), device=x16.device)
        cabi.check(cabi.lib().lg_conv_layer_infer(p.cref, x16.data_ptr(), cin, Wc.data_ptr(), cout, w16.data_ptr(),
                                                  w16t.data_ptr(), 1 if stale else 0, fmt, self._bn_stats.data_ptr(),
                                                  cabi.ptr(res), 1 if relu else 0, y.data_ptr(), y16.data_ptr(),
                                                  cabi.stream_of(y)), "lg_conv_layer_infer")
        cabi.count_launches("lg_conv_layer_infer", 1 if stale else 0)
        self._value = y
        self._f16_cache = ((fmt, y._version, y.data_ptr()), y16)  # the next convolution's operand: no cast pass
        self._src = self._residual = self._bn_stats = None
        return self


class MinkowskiConvolution(MinkowskiConvolutionBase):
    is_transpose = False


class MinkowskiConvolutionTranspose(MinkowskiConvolutionBase):
    is_transpose = True
