"""One LiDOG training step on the GPU hot path.

Mirror of `PLTTrainer2D.training_step` + `configure_optimizers`
(utils/pipelines/trainer_lighting_2d.py:141-293, 349-360) minus logging/metrics:
voxelise -> ME.SparseTensor -> MinkUNet34BEV(is_train=True) -> SoftDICE (3D) + DICE (BEV)
-> backward -> Adam(lr 1e-3, weight_decay 1e-4).  Reference quirks kept on purpose:
the (B,C,h,w) BEV logits are re-viewed as (-1, C) without a permute (`:181`), the 3D loss
uses the first point's label per voxel and the BEV image the agree-or-ignore colabel
(semantickitti_bev.py:242,249).
"""
from __future__ import annotations

import contextlib
import os

import torch

from . import losses
from .bev import label_image_size
from .synth import SHAPES


_NVTX = int(os.environ.get("LIDOG_NVTX", "0"))


def _range(name: str):
    """NVTX range around a phase of the step (LIDOG_NVTX=1; SURVEY.md section 5): shows up in ncu / nsys timelines."""
    return torch.cuda.nvtx.range(name) if _NVTX and torch.cuda.is_available() else contextlib.nullcontext()


def bev_label_image(coords4: torch.Tensor, colabels: torch.Tensor, batch_size: int, bound: float, img: int,
                    voxel_size: float = 0.05) -> torch.Tensor:
    """Device version of PC2ImgConverter.getBEVImageNew (semantickitti_bev.py:433-464) for a whole
    batch: int64 [B, img, img], -1 = ignore.  Duplicate pixels: highest row wins (deterministic)."""
    dev = coords4.device
    # `(quantized_coords * voxel_size).astype(np.float32)` (semantickitti_bev.py:244): an int32 array times a python
    # float is a DOUBLE product rounded once to float32 -- not float32(c) * float32(0.05) as in sparse2super
    pts = (coords4[:, 1:].to(torch.float64) * voxel_size).to(torch.float32)
    grid = (bound - (-bound)) / img
    valid = (colabels != -1) & (-bound < pts[:, 0]) & (pts[:, 0] < bound) & (-bound < pts[:, 1]) & \
            (pts[:, 1] < bound) & (-10 < pts[:, 2]) & (pts[:, 2] < 8)
    # torch's CUDA kernel for `tensor / python_scalar` multiplies by the reciprocal; the reference divides (numpy
    # float32, IEEE), and floor() of the two differs on cell boundaries -- divide by a TENSOR to get the true quotient
    # (found by tests/test_gpu_trainer.py against the CPU evaluation of this same function)
    grid_t = torch.full((), grid, dtype=torch.float32, device=dev)  # (a fill kernel: no host-to-device copy / sync)
    px = torch.floor(torch.div(pts[:, 0] - (-bound), grid_t)).long()
    py = torch.floor(img - torch.div(pts[:, 1] - (-bound), grid_t)).long() - 1
    py = torch.where(py < 0, py + img, py)
    pix = coords4[:, 0].long() * (img * img) + py.clamp(0, img - 1) * img + px.clamp(0, img - 1)
    rows = torch.arange(coords4.shape[0], device=dev)
    rows = torch.where(valid, rows, torch.full_like(rows, -1))
    win = torch.full((batch_size * img * img,), -1, dtype=torch.long, device=dev)
    win.scatter_reduce_(0, pix, rows, reduce="amax", include_self=True)
    lab = torch.where(win >= 0, colabels.long()[win.clamp_min(0)], torch.full_like(win, -1))
    return lab.view(batch_size, img, img)


class LidogTrainer:
    """Owns model + Adam; `training_step` takes raw device point clouds."""

    def __init__(self, model, num_classes=7, voxel_size=0.05, ignore_label=-1, lr=1e-3, weight_decay=1e-4,
                 source_weights=(0.5, 0.5), shape="kitti", ME=None, buffer_sync=None):
        if ME is None:
            from lidog_b200 import me as ME
        self.ME, self.model = ME, model
        self.buffer_sync = buffer_sync  # lidog/ddp.py FlatBuffers: rank 0's BN buffers broadcast at the start of a step
        self.num_classes, self.voxel_size, self.ignore_label = num_classes, voxel_size, ignore_label
        self.source_weights = source_weights
        # the label image has the size of the BEV head's output at the model's pooling (SHAPES' bev_img at the default)
        pool = getattr(getattr(model, "module", model), "bev_pool", (5, 3, 1))
        self.bound = SHAPES[shape]["bound"]
        self.bev_img = label_image_size(self.bound, voxel_size, pool)
        params = list(model.parameters())
        # same update rule as the reference's torch.optim.Adam (trainer_lighting_2d.py:349-360); on the GPU the
        # ~190 parameter tensors are updated by the fused multi-tensor kernels instead of one launch per op
        fused = len(params) > 0 and all(p.is_cuda for p in params)
        self.optimizer = torch.optim.Adam(params, lr=lr, weight_decay=weight_decay, fused=fused)

    def voxelize(self, points_list, labels_list):
        """GPU sparse_quantize of the whole batch (one hash build) + the dataset-side label products."""
        q = self.ME.utils.sparse_quantize_batch(points_list, labels_list, self.voxel_size, self.ignore_label)
        labels = torch.cat(labels_list, 0)
        sem_labels = labels[q["unique_map"]].long()  # first point's label per voxel
        bev_labels = bev_label_image(q["coords"], q["colabels"], len(points_list), self.bound, self.bev_img,
                                     self.voxel_size)
        feats = torch.ones((q["coords"].shape[0], 1), dtype=torch.float32, device=labels.device)
        cm = None
        if hasattr(self.ME, "CoordinateManager") and hasattr(self.ME.CoordinateManager, "from_quantized"):
            cm = self.ME.CoordinateManager.from_quantized(q)  # share the voxelisation hash with the network
        return q["coords"], feats, sem_labels, bev_labels, cm

    def voxelize_multi(self, sources):
        """All source batches through ONE voxelisation / coordinate pyramid (one hashed voxel index and one host round
        trip for the whole step), then one view of the shared coordinate manager per source
        (`CoordinateManager.split`; SURVEY.md 8f-4).  Backends without `split` (the CPU oracle) voxelise per source.
        -> [(coords, feats, sem_labels, bev_labels, manager, batch_size), ...]"""
        CM = getattr(self.ME, "CoordinateManager", None)
        if CM is None or not hasattr(CM, "split"):
            return [self.voxelize(p, l) + (len(p),) for p, l in sources]
        sizes = [len(p) for p, _ in sources]
        pts = [x for p, _ in sources for x in p]
        lab = [x for _, l in sources for x in l]
        coords, feats, sem_labels, bev_labels, cm = self.voxelize(pts, lab)
        out, r0, b0 = [], 0, 0
        for view, nb in zip(cm.split(sizes), sizes):
            n = view.levels[1].n
            out.append((view.levels[1].coords, feats[r0:r0 + n], sem_labels[r0:r0 + n], bev_labels[b0:b0 + nb], view, nb))
            r0, b0 = r0 + n, b0 + nb
        return out

    def forward_loss(self, coords, feats, sem_labels, bev_labels, batch_size=None, coordinate_manager=None):
        if coordinate_manager is not None:
            stensor = self.ME.SparseTensor(features=feats, coordinate_manager=coordinate_manager)
        else:
            stensor = self.ME.SparseTensor(coordinates=coords, features=feats)
        if batch_size is not None:
            stensor.coordinate_manager.batch_size = batch_size
        out, bev_preds = self.model(stensor, is_train=True)
        loss_bev = 0.0
        for key, pred in bev_preds.items():
            loss_bev = loss_bev + losses.dice_loss(pred.reshape(-1, self.num_classes), bev_labels.reshape(-1),
                                                   self.ignore_label) / len(bev_preds)
        loss_3d = losses.soft_dice_loss(out.F, sem_labels, self.ignore_label, is_kitti=self.num_classes == 19)
        return self.source_weights[0] * loss_3d + self.source_weights[1] * loss_bev, loss_3d, loss_bev

    def training_step(self, points_list, labels_list):
        if self.buffer_sync is not None:
            self.buffer_sync.broadcast()
        with _range("lidog/voxelize"):
            coords, feats, sem_labels, bev_labels, cm = self.voxelize(points_list, labels_list)
        self.optimizer.zero_grad(set_to_none=True)
        with _range("lidog/forward+loss"):
            total, l3, l2 = self.forward_loss(coords, feats, sem_labels, bev_labels, len(points_list), cm)
        with _range("lidog/backward"):
            total.backward()
        with _range("lidog/adam"):
            self.optimizer.step()
        return total.detach()

    def training_step_multi(self, sources):
        """Multi-source step (PLTTrainer2DMulti.training_step, utils/pipelines/trainer_lighting_2d_multi.py:135-199):
        one forward pass per source domain through the SAME model, each on its own batch / coordinate manager,
        total = sum_i source_weights[i] * (loss_3d_i + loss_bev_i), one backward, one optimizer step.
        `sources` = [(points_list, labels_list), ...] (two in the reference)."""
        assert len(sources) == len(self.source_weights), "one weight per source domain"
        if self.buffer_sync is not None:
            self.buffer_sync.broadcast()
        batches = self.voxelize_multi(sources)
        self.optimizer.zero_grad(set_to_none=True)
        total = None
        for w, (coords, feats, sem_labels, bev_labels, cm, n) in zip(self.source_weights, batches):
            _, l3, l2 = self.forward_loss(coords, feats, sem_labels, bev_labels, n, cm)
            term = w * (l3 + l2)
            total = term if total is None else total + term
        total.backward()
        self.optimizer.step()
        return total.detach()
