"""ctypes binding of liblidog_b200.so (the C ABI declared in include/lidog_b200.h).

PyTorch is used only for device memory and streams: tensors are passed as raw
`data_ptr()`s, the stream as `torch.cuda.current_stream().cuda_stream`.
There is NO CPU fallback: if the library is missing or a call fails, a
RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_LIB = None
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "liblidog_b200.so")

TILE = 128
FMT_BF16, FMT_FP16 = 0, 1
BEV_LAST, BEV_MAX = 0, 1
ERR_RANGE = -3

_vp, _i32, _i64, _f32, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t


class ConvPlan(C.Structure):
    _fields_ = [("nbr", _vp), ("k_stride", _i64), ("out_row", _vp), ("tile_mask", _vp), ("kernel_volume", _i32),
                ("mask_words", _i32), ("n_slots", _i64), ("n_out", _i64), ("n_in", _i64)]


_PP = C.POINTER(ConvPlan)


class PeerCtx(C.Structure):
    _fields_ = [("bufs", C.POINTER(C.c_void_p)), ("world", _i32), ("rank", _i32), ("epoch", C.c_uint64)]


class BnBranch(C.Structure):
    _fields_ = [("x", _vp), ("stat_partials", _vp), ("n_stat_rows", _i64), ("gamma", _vp), ("beta", _vp),
                ("running_mean", _vp), ("running_var", _vp), ("num_batches_tracked", _vp), ("eps", _f32),
                ("momentum", _f32), ("stats", _vp)]


class BnBwdBranch(C.Structure):
    _fields_ = [("x", _vp), ("stats", _vp), ("gamma", _vp), ("dx", _vp), ("dx16", _vp), ("dgamma", _vp), ("dbeta", _vp)]


class LevelOut(C.Structure):
    _fields_ = [("table", _vp), ("capacity", _i64), ("coords4", _vp), ("unique_map", _vp), ("inverse_map", _vp)]


_PB, _PBB, _PPC = C.POINTER(BnBranch), C.POINTER(BnBwdBranch), C.POINTER(PeerCtx)

SIGNATURES = {
    "lg_version": (C.c_int, []),
    "lg_last_error_string": (C.c_char_p, []),
    "lg_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "lg_hash_capacity": (_i64, [_i64]),
    "lg_hash_bytes": (_sz, [_i64]),
    "lg_quantize_points": (C.c_int, [_vp, _vp, _i64, _f32, _f32, _f32, _vp, _vp]),
    "lg_quantize_points_f64": (C.c_int, [_vp, _vp, _i64, C.c_double, C.c_double, C.c_double, _vp, _vp]),
    "lg_coords_unique_workspace": (_sz, [_i64]),
    "lg_coords_unique": (C.c_int, [_vp, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _sz, _vp]),
    "lg_coords_pyramid": (C.c_int, [_vp, _i64, _vp, _i32, _vp, _i32, C.POINTER(_i32), C.POINTER(LevelOut), _vp, _vp, _vp]),
    "lg_kernel_map": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _i64, _vp, _vp]),
    "lg_kernel_map_sorted_workspace": (_sz, [_i64, _i32]),
    "lg_kernel_map_sorted": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "lg_scan_workspace": (_sz, [_i64]),
    "lg_kernel_map_pairs": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "lg_kernel_map_up2": (C.c_int, [_vp, _vp, _i64, _i32, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "lg_conv_gemm_simt": (C.c_int, [_PP, _vp, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _vp]),
    "lg_conv_wgrad_workspace": (_sz, [_PP, _i32, _i32]),
    "lg_conv_wgrad_simt": (C.c_int, [_PP, _vp, _i32, _vp, _i32, _vp, _vp, _sz, _vp]),
    "lg_cast_rows": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "lg_absmax_scale": (C.c_int, [_vp, _i64, _vp, _vp]),
    "lg_prep_weights": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp, _i32, _vp]),
    "lg_conv_gemm_tc": (C.c_int, [_PP, _vp, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "lg_conv_wgrad_tc_workspace": (_sz, [_PP, _i32, _i32]),
    "lg_conv_wgrad_tc": (C.c_int, [_PP, _vp, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "lg_conv_layer_forward": (C.c_int, [_PP, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "lg_conv_layer_backward": (C.c_int, [_PP, _PP, _i32, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _vp, _vp, _vp]),
    "lg_conv_layer_infer": (C.c_int, [_PP, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    "lg_confusion_matrix": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp]),
    "lg_arena_bytes": (_sz, []),
    "lg_arena_release": (C.c_int, []),
    "lg_bn_layer_forward": (C.c_int, [_PB, _PB, _vp, _i32, _i64, _i32, _vp, _vp, _i32, _PPC, _vp]),
    "lg_bn_layer_backward": (C.c_int, [_vp, _i64, _vp, _i32, _i64, _i32, _PBB, _PBB, _vp, _i32, _vp, _PPC, _vp]),
    "lg_bn_workspace": (_sz, [_i64, _i32]),
    "lg_bn_stats": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _sz, _vp]),
    "lg_bn_finalize": (C.c_int, [_vp, C.c_double, _vp, _i32, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp]),
    "lg_bn_apply": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp, _vp, _i32, _vp]),
    "lg_bn_bwd_stats": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _sz, _vp]),
    "lg_bn_bwd_finalize": (C.c_int, [_vp, _vp, _vp, C.c_double, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lg_bn_bwd_gscale": (C.c_int, [_vp, _i32, _vp, _vp]),
    "lg_bn_bwd_apply": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp,
                                  _vp, _vp, _vp, _vp, _i32, _vp]),
    "lg_instnorm_forward": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _f32, _i32, _vp, _vp, _i32, _vp, _vp]),
    "lg_instnorm_backward": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "lg_inst_cov_forward": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _f32, _vp, _vp, _vp]),
    "lg_inst_cov_backward": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp]),
    "lg_peer_exchange_bytes": (_sz, []),
    "lg_peer_sum": (C.c_int, [_vp, _i32, C.POINTER(C.c_void_p), _i32, _i32, C.c_uint64, _vp, _vp]),
    "lg_dice_forward": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _f32, _i32, _vp, _vp, _vp]),
    "lg_dice_backward": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _f32, _i32, _vp, _vp, _vp, _vp]),
    "lg_bev_workspace": (_sz, [_i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32]),
    "lg_bev_forward": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _f32, _f32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp,
                                 _vp, _sz, _vp]),
    "lg_bev_backward": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp,
                                  _sz, _vp]),
}


# CUDA kernels launched by one call of each entry point (memsets not counted; variable ones are counted by the
# caller through `count_launches`).  bench.py runs one CENSUS step with counting on to report `gpu_launches`; the
# timed steps go straight to the CDLL.
KERNELS_PER_CALL = {
    "lg_quantize_points": 1, "lg_quantize_points_f64": 1, "lg_coords_unique": 7, "lg_kernel_map": 1, "lg_kernel_map_sorted": 7, "lg_kernel_map_pairs": 3,
    "lg_kernel_map_up2": 9, "lg_conv_gemm_simt": 1, "lg_conv_wgrad_simt": 2, "lg_cast_rows": 1,
    "lg_absmax_scale": 2, "lg_prep_weights": 1, "lg_conv_gemm_tc": 1, "lg_conv_wgrad_tc": 2,
    "lg_bev_forward": 2, "lg_bev_backward": 1,
    "lg_bn_stats": 2, "lg_bn_finalize": 1, "lg_bn_apply": 1, "lg_bn_bwd_stats": 2, "lg_bn_bwd_finalize": 1,
    "lg_bn_bwd_gscale": 1, "lg_bn_bwd_apply": 1, "lg_peer_sum": 1,
    "lg_bn_layer_backward": 3, "lg_dice_forward": 2, "lg_dice_backward": 1,
    # + 1 (lg_prep_weights) when the call refreshes the 16-bit weights: counted by the caller
    "lg_conv_layer_infer": 1, "lg_confusion_matrix": 1,
    "lg_instnorm_forward": 3, "lg_instnorm_backward": 3,
    "lg_inst_cov_forward": 5, "lg_inst_cov_backward": 2,
}
COUNTS: dict = {}
_RAW = None


class _Counting:
    """Proxy over the CDLL that counts calls per entry point (census passes only)."""

    def __init__(self, cdll):
        self._cdll = cdll
        self._fns = {}

    def __getattr__(self, name):
        fn = self._fns.get(name)
        if fn is None:
            raw = getattr(self._cdll, name)
            if name in KERNELS_PER_CALL:
                def fn(*a, _raw=raw, _name=name):
                    COUNTS[_name] = COUNTS.get(_name, 0) + 1
                    return _raw(*a)
            else:
                fn = raw
            self._fns[name] = fn
        return fn


def counting(on: bool) -> None:
    """Census mode: count library calls (and the launches callers report through `count_launches`)."""
    global _LIB
    lib()
    _LIB = _Counting(_RAW) if on else _RAW
    if on:
        COUNTS.clear()


def is_counting() -> bool:
    return _LIB is not None and _LIB is not _RAW


def count_launches(name: str, n: int) -> None:
    """Launch count of a call whose kernel count depends on its arguments (the fused layer entry points)."""
    if _LIB is not _RAW:
        COUNTS["#" + name] = COUNTS.get("#" + name, 0) + n


def kernel_launches() -> int:
    return sum(v if k.startswith("#") else KERNELS_PER_CALL[k] * v for k, v in COUNTS.items())


def lib():
    """Load the shared library once; fail loudly when it is not there."""
    global _LIB, _RAW
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not built: run `python -m lidog_b200.build` (no CPU fallback exists)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _RAW = _LIB = L
    return _LIB


def check(rc: int, what: str = ""):
    if rc != 0:
        raise RuntimeError(f"liblidog_b200 {what} failed ({rc}): {lib().lg_last_error_string().decode()}")


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_of(t):
    """Raw handle of torch's current stream on the device of tensor `t` (not the thread's current device)."""
    return torch._C._cuda_getCurrentRawStream(t.device.index)


def stream():
    """Raw handle of torch's current CUDA stream on the current device.  `torch.cuda.current_stream()` builds a
    Python Stream object through three layers of device-index helpers (16 us per call, 640 calls per training
    step = 10 ms of host time, tools/host_profile.py); the private raw getter is ~50x cheaper."""
    try:
        return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())
    except AttributeError:  # older / newer torch without the private getters
        return torch.cuda.current_stream().cuda_stream


def device_info():
    a, b, c = C.c_int(), C.c_int(), C.c_int()
    check(lib().lg_device_info(C.byref(a), C.byref(b), C.byref(c)), "lg_device_info")
    return a.value, b.value, c.value


def peer_ctx(ex, n_epochs: int):
    """lgPeerCtx of a me.peer.PeerExchange for a call that consumes `n_epochs` exchanges (None -> NULL)."""
    if ex is None:
        return None
    ctx = PeerCtx(ex.ptrs, ex.world, ex.rank, ex.epoch + 1)
    ex.epoch += n_epochs
    return C.byref(ctx)


def make_plan(nbr, k_stride, out_row, tile_mask, K, n_slots, n_out, n_in) -> ConvPlan:
    return ConvPlan(ptr(nbr), k_stride, ptr(out_row), ptr(tile_mask), K, (K + 31) // 32, n_slots, n_out, n_in)
