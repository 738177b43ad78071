"""SparseTensor: features + a handle on the batch's CoordinateManager.

Mirror of the part of ME.SparseTensor LiDOG touches: construction from
(coordinates int [N,4] = (b,x,y,z), features [N,C]) at
utils/pipelines/trainer_lighting_2d.py:151, `.F`, `.C`, `.device`
(utils/models/minkunet_bev.py:172,211) and `out += residual` in BasicBlock.
Row order of a stride-1 tensor equals the input row order (labels are matched
row by row at trainer_lighting_2d.py:169,194).
"""
from __future__ import annotations

import torch

from .. import cabi
from .coords import CoordinateManager


class CoordinateMapKey:
    """Names the coordinate map of a tensor within its manager, as ME's key does: here the tensor stride is all there
    is to it.  `SparseTensor(features=..., coordinate_map_key=t.coordinate_map_key,
    coordinate_manager=t.coordinate_manager)` puts new features on t's coordinates (IBN-style channel splits)."""

    def __init__(self, tensor_stride):
        self._ts = int(tensor_stride[0] if isinstance(tensor_stride, (list, tuple)) else tensor_stride)

    def get_tensor_stride(self):
        return [self._ts] * 3

    def __eq__(self, other):
        return isinstance(other, CoordinateMapKey) and other._ts == self._ts

    def __hash__(self):
        return hash(("CoordinateMapKey", self._ts))

    def __repr__(self):
        return f"CoordinateMapKey(tensor_stride={self.get_tensor_stride()})"


class SparseTensor:
    _stat_partials = None  # (per-tile column statistics written by the producing convolution's epilogue, F version)

    def __init__(self, features, coordinates=None, tensor_stride=1, coordinate_map_key=None,
                 coordinate_manager=None, quantization_mode=None, device=None, **unused):
        if not isinstance(features, torch.Tensor):
            raise ValueError("features must be a torch.Tensor")
        if isinstance(tensor_stride, (list, tuple)):
            tensor_stride = tensor_stride[0]
        if device is not None:
            features = features.to(device)
        if coordinate_map_key is not None and coordinate_manager is not None:
            tensor_stride = coordinate_map_key._ts
        if coordinate_manager is None:
            if coordinates is None:
                raise ValueError("either coordinates or a coordinate_manager is required")
            if not features.is_cuda:
                raise RuntimeError("lidog_b200 has no CPU path: move features/coordinates to a CUDA device")
            if coordinates.dim() != 2 or coordinates.shape[1] != 4 or coordinates.shape[0] != features.shape[0]:
                raise ValueError("coordinates must be [N, 4] = (batch, x, y, z) with one row per feature row")
            coords = coordinates.to(device=features.device, dtype=torch.int32)
            coordinate_manager = CoordinateManager(coords)
            if coordinate_manager.had_duplicates:
                # duplicate coordinates: keep the first occurrence of each voxel
                features = features.index_select(0, coordinate_manager.input_unique_map)
        self._F = features
        self.coordinate_manager = coordinate_manager
        self._ts = int(tensor_stride)
        self._f16_cache = None

    # ---- ME-facing attributes
    @property
    def F(self):
        return self._F

    @property
    def C(self):
        return self.coordinate_manager.get_coords(self._ts)

    coordinates = C
    features = F

    @property
    def tensor_stride(self):
        return [self._ts] * 3

    @property
    def coordinate_map_key(self):
        return CoordinateMapKey(self._ts)

    @property
    def device(self):
        return self._F.device

    @property
    def dtype(self):
        return self._F.dtype

    @property
    def shape(self):
        return self._F.shape

    def size(self, *a):
        return self._F.size(*a)

    def __len__(self):
        return self._F.shape[0]

    def __repr__(self):
        return f"SparseTensor(F={tuple(self._F.shape)}, tensor_stride={self._ts}, device={self.device})"

    # ---- internals
    def _like(self, feats):
        return SparseTensor(feats, tensor_stride=self._ts, coordinate_manager=self.coordinate_manager)

    def _f16(self, fmt):
        """16-bit copy of the features for the tensor-core kernels, cached per tensor version
        (a tensor often feeds two convolutions: conv1 and the block's 1x1 downsample)."""
        f = self._F
        key = (fmt, f._version, f.data_ptr())
        if self._f16_cache is None or self._f16_cache[0] != key:
            src = f.detach().contiguous()
            out = torch.empty(src.shape, dtype=torch.float16 if fmt == cabi.FMT_FP16 else torch.bfloat16,
                              device=src.device)
            cabi.check(cabi.lib().lg_cast_rows(cabi.ptr(src), cabi.ptr(out), src.numel(), fmt, None, cabi.stream_of(src)),
                       "lg_cast_rows")
            self._f16_cache = (key, out)
        return self._f16_cache[1]

    def _same_map(self, other):
        if other.coordinate_manager is not self.coordinate_manager or other._ts != self._ts:
            raise ValueError("sparse tensors must share the coordinate map")

    def __add__(self, other):
        if isinstance(other, SparseTensor):
            self._same_map(other)
            return self._like(self._F + other._F)
        return self._like(self._F + other)

    def __iadd__(self, other):
        if isinstance(other, SparseTensor):
            self._same_map(other)
            self._F += other._F
        else:
            self._F += other
        return self


def cat(*tensors):
    """Concatenate features of tensors on the same coordinate map (utils/models/minkunet_bev.py:337-370)."""
    t0 = tensors[0]
    for t in tensors[1:]:
        t0._same_map(t)
    out = t0._like(torch.cat([t.F for t in tensors], dim=1))
    caches = [t._f16_cache for t in tensors]
    if all(c is not None and c[0] == (caches[0][0][0], t.F._version, t.F.data_ptr()) for c, t in zip(caches, tensors)):
        f = out._F  # the 16-bit operand copies concatenate too: no cast pass for the block that follows
        out._f16_cache = ((caches[0][0][0], f._version, f.data_ptr()), torch.cat([c[1] for c in caches], dim=1))
    return out
