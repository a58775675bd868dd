"""Segmentation metrics of the reference (utilities/metrics.py:8-61) on a device-side confusion matrix.

``pixel_accuracy / mIoU / mDice(logits, mask)`` are drop-ins (same arguments, python float results, one host
sync each -- as the reference).  ``MetricAccumulator`` is what a training loop should use instead of the
reference's per-iteration ``.item()`` calls (UAPS_train.py:295-306): it keeps per-batch metric sums on the
device and syncs once when ``result()`` is called.
"""
from __future__ import annotations

import torch

from . import _lib as L


def confusion(logits: torch.Tensor, mask: torch.Tensor, out: torch.Tensor = None) -> torch.Tensor:
    """[C, C] int64 counts, row = label, column = argmax(softmax(logits)); accumulated into ``out`` if given."""
    L.require_cuda(logits, mask)
    if logits.dtype != torch.float32 or logits.dim() != 4:
        raise RuntimeError("logits must be fp32 [B, C, H, W]")
    B, C, H, W = logits.shape
    logits, mask = logits.contiguous(), mask.reshape(B, H, W).long().contiguous()
    conf = out if out is not None else torch.zeros((C, C), dtype=torch.int64, device=logits.device)
    with L.on_device(logits.device):
        L.check(L.lib().uaps_confusion(logits.data_ptr(), mask.data_ptr(), B, C, H * W, conf.data_ptr(), L.stream_ptr()),
                "uaps_confusion")
    return conf


def metrics_from_confusion(conf: torch.Tensor, smooth: float = 1e-10, n_pixels: int = None):
    """(pixel_accuracy, mIoU, mDice) as 0-dim device tensors, the reference's formulas: classes 1..C-1, classes
    absent from the labels skipped (np.nanmean), smooth 1e-10.  n_pixels: the accuracy's denominator -- the reference
    divides by ``mask.numel()`` (utilities/metrics.py:12), so a pixel whose label lies outside [0, C) (an ignore
    index) counts as WRONG there; the confusion matrix does not hold such pixels, hence the explicit total.
    conf may also be a stack [..., C, C] of matrices (n_pixels then a number or a tensor of shape [...]); the results are
    then tensors of shape [...], one value per matrix."""
    c = conf.double()
    diag = c.diagonal(dim1=-2, dim2=-1)
    acc = diag.sum(-1) / (c.sum((-2, -1)) if n_pixels is None else
                          (n_pixels.double() if torch.is_tensor(n_pixels) else float(n_pixels)))
    inter = diag[..., 1:]
    label_n, pred_n = c.sum(-1)[..., 1:], c.sum(-2)[..., 1:]
    union = label_n + pred_n - inter
    present = label_n > 0
    iou = (inter + smooth) / (union + smooth)
    dice = 2 * (inter + smooth) / (union + inter + smooth)
    n = present.sum(-1)
    nan = torch.full((), float("nan"), dtype=torch.float64, device=conf.device)
    miou = torch.where(n > 0, (iou * present).sum(-1) / n.clamp(min=1), nan)
    mdice = torch.where(n > 0, (dice * present).sum(-1) / n.clamp(min=1), nan)
    return acc, miou, mdice


def pixel_accuracy(output: torch.Tensor, mask: torch.Tensor) -> float:
    return float(metrics_from_confusion(confusion(output, mask), n_pixels=mask.numel())[0])


def mIoU(pred_mask: torch.Tensor, mask: torch.Tensor, smooth: float = 1e-10, n_classes: int = 4) -> float:
    return float(metrics_from_confusion(confusion(pred_mask, mask)[:n_classes, :n_classes], smooth)[1])


def mDice(pred_mask: torch.Tensor, mask: torch.Tensor, smooth: float = 1e-10, n_classes: int = 4) -> float:
    return float(metrics_from_confusion(confusion(pred_mask, mask)[:n_classes, :n_classes], smooth)[2])


class MetricAccumulator:
    """Running per-batch means of (accuracy, mIoU, mDice), kept on the device (the reference averages per-batch
    values, UAPS_train.py:316-327 / :395-400)."""

    def __init__(self, device):
        self.sums = torch.zeros(3, dtype=torch.float64, device=device)
        self.batches = 0

    def update(self, logits: torch.Tensor, mask: torch.Tensor) -> None:
        self.sums += torch.stack(metrics_from_confusion(confusion(logits, mask), n_pixels=mask.numel()))
        self.batches += 1

    def result(self):
        acc, miou, mdice = (self.sums / max(self.batches, 1)).tolist()      # the only host sync
        return {"pixel_accuracy": acc, "mIoU": miou, "mDice": mdice}
