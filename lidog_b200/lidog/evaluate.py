"""LiDOG evaluation on the GPU: eval-mode forward and per-class IoU / mIoU from a device confusion matrix.

The reference evaluates with `sklearn.metrics.jaccard_score(..., average=None)` on the CPU (trainer_lighting_bev.py:
265-323) and logs a torchmetrics `JaccardIndex(ignore_index)` in the training step.  Both are functions of one
(C + 1) x C matrix of counts that `lg_confusion_matrix` accumulates on the device (row C: targets outside [0, C),
the ignore label included); `iou_from_confusion` turns it into either convention.

The forward runs with the model in eval mode under `torch.no_grad()`, which is where the tensor-core layers take the
inference epilogue (conv -> batch norm -> residual -> ReLU in one launch, me/conv.py `DeferredConv`).
"""
from __future__ import annotations

import numpy as np
import torch

from .. import cabi


def iou_from_confusion(conf, ignore_rows: bool):
    """Per-class IoU (float64 [C]) from a (C + 1) x C (or C x C) confusion matrix, rows = target, columns = prediction.

    ignore_rows=False: sklearn `jaccard_score(labels=range(C), average=None, zero_division=0)` on all voxels -- a voxel
    whose target is outside [0, C) still enlarges the union of the class predicted for it (row C).
    ignore_rows=True: torchmetrics `JaccardIndex(ignore_index)` -- voxels with such targets are dropped (row C is not
    read).  A class absent from both targets and predictions gets IoU 0."""
    conf = np.asarray(conf, dtype=np.int64)
    C = conf.shape[1]
    m = conf[:C] if ignore_rows else conf
    tp = np.diagonal(m[:C]).astype(np.float64)
    pred = m.sum(0).astype(np.float64)          # column sums over the rows in use
    true = m[:C].sum(1).astype(np.float64)      # rows 0..C-1 only: row C is no class
    union = pred + true - tp
    return np.where(union > 0, tp / np.where(union > 0, union, 1.0), 0.0)


class LidogEvaluator:
    """Accumulates the confusion matrix of `model(x, is_train=False)` over batches of raw device point clouds.

    `step` voxelises like the training step (first point's label per voxel), runs the eval forward and adds the batch
    into a device int64 matrix; it does not wait for the device.  `result` copies the matrix to the host once and
    returns per-class IoU / mIoU in both conventions."""

    def __init__(self, model, num_classes, ignore_label=-1, voxel_size=0.05, ME=None):
        if ME is None:
            from lidog_b200 import me as ME
        if not 1 <= num_classes <= 32:
            raise ValueError("lg_confusion_matrix supports 1 <= num_classes <= 32")
        self.ME, self.model = ME, model
        self.num_classes, self.ignore_label, self.voxel_size = num_classes, ignore_label, voxel_size
        self.conf = None

    def reset(self):
        self.conf = None

    def voxelize(self, points_list, labels_list):
        q = self.ME.utils.sparse_quantize_batch(points_list, labels_list, self.voxel_size, self.ignore_label)
        sem_labels = torch.cat(labels_list, 0)[q["unique_map"]].long()  # first point's label per voxel
        feats = torch.ones((q["coords"].shape[0], 1), dtype=torch.float32, device=sem_labels.device)
        return feats, sem_labels, self.ME.CoordinateManager.from_quantized(q)

    def logits(self, points_list, labels_list):
        """Eval-mode logits [U, C] of one batch and the voxel labels [U]; restores the model's training flag."""
        feats, sem_labels, cm = self.voxelize(points_list, labels_list)
        was_training = self.model.training
        self.model.eval()
        try:
            with torch.no_grad():
                x = self.ME.SparseTensor(features=feats, coordinate_manager=cm)
                x.coordinate_manager.batch_size = len(points_list)
                out, _ = self.model(x, is_train=False)
                logits = out.F
        finally:
            self.model.train(was_training)
        return logits, sem_labels

    def add(self, logits: torch.Tensor, target: torch.Tensor):
        """Add a batch of logits [n, C] (float32) and targets [n] (int64), both on the same CUDA device, to the matrix."""
        if not (logits.is_cuda and target.device == logits.device):
            raise ValueError("logits and target must be on the same CUDA device")
        if self.conf is not None and self.conf.device != logits.device:
            raise ValueError(f"the matrix is accumulated on {self.conf.device}, the batch is on {logits.device}")
        if self.conf is None:
            self.conf = torch.zeros((self.num_classes + 1, self.num_classes), dtype=torch.int64, device=logits.device)
        logits = logits.detach().float().contiguous()
        target = target.detach().long().contiguous()
        if logits.dim() != 2 or logits.shape[1] != self.num_classes or target.shape != logits.shape[:1]:
            raise ValueError(f"logits must be [n, {self.num_classes}] and target [n]")
        cabi.check(cabi.lib().lg_confusion_matrix(cabi.ptr(logits), logits.shape[0], self.num_classes,
                                                  cabi.ptr(target), cabi.ptr(self.conf), cabi.stream_of(logits)),
                   "lg_confusion_matrix")

    def step(self, points_list, labels_list):
        logits, sem_labels = self.logits(points_list, labels_list)
        self.add(logits, sem_labels)
        return logits

    def result(self, process_group=None):
        """-> dict(iou, miou: sklearn convention (all voxels); iou_ignore, miou_ignore: torchmetrics convention
        (voxels with an ignored target dropped); confusion: the int64 (C + 1) x C matrix).  With `process_group`, the
        matrices of all its ranks are summed first (one all_reduce)."""
        C = self.num_classes
        conf = self.conf
        if conf is None:
            dev = torch.device("cuda", torch.cuda.current_device())
            conf = torch.zeros((C + 1, C), dtype=torch.int64, device=dev)
        if process_group is not None:
            conf = conf.clone()
            torch.distributed.all_reduce(conf, group=process_group)
        host = conf.cpu().numpy()
        iou = iou_from_confusion(host, ignore_rows=False)
        iou_ig = iou_from_confusion(host, ignore_rows=True)
        return dict(iou=iou, miou=float(iou.mean()), iou_ignore=iou_ig, miou_ignore=float(iou_ig.mean()),
                    confusion=host)
