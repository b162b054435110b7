"""Loss and metric surface of the hot path.

`RobustBCEDiceLoss()` is interchangeable with the reference's `criterion = nn.BCELoss()`
(Main_Final.py:551,580): with the default weights (w_bce=1, w_dice=0) it is exactly torch's BCELoss on
probabilities (log clamp at -100 forward, (p-y)/max(p(1-p),1e-12)/N backward).  `w_dice > 0` adds the
build-defined Dice term (SURVEY.md §8c).  The same kernel pass also produces the per-image integer
confusion counts behind `ModelEvaluator.calculate_metrics` (Main_Final.py:519-547); they are kept on the
module as `last_counts` ([B,4] int64 TP,FP,FN,TN, device tensor) so a validation loop needs no second pass.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops

METRIC_KEYS = ("accuracy", "iou", "precision", "recall", "f1_score")


class _BceDice(torch.autograd.Function):
    @staticmethod
    def forward(ctx, probs, target, mod):
        p = probs.detach().contiguous().float()
        y = target.detach().contiguous().float()
        loss, sums, counts = ops.loss_forward(p, y, mod.threshold, mod.w_bce, mod.w_dice, mod.smooth)
        mod.last_counts = counts
        ctx.save_for_backward(p, y, sums)
        ctx.cfg = (mod.w_bce, mod.w_dice, mod.smooth)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        p, y, sums = ctx.saved_tensors
        w_bce, w_dice, smooth = ctx.cfg
        g = grad_out.detach().contiguous().float().reshape(1)
        dp = ops.loss_backward(p, y, g, sums, w_bce, w_dice, smooth)
        return dp, None, None


class RobustBCEDiceLoss(nn.Module):
    def __init__(self, w_bce: float = 1.0, w_dice: float = 0.0, smooth: float = 1.0, threshold: float = 0.5):
        super().__init__()
        self.w_bce, self.w_dice, self.smooth, self.threshold = float(w_bce), float(w_dice), float(smooth), float(threshold)
        self.last_counts = None

    def forward(self, outputs: torch.Tensor, masks: torch.Tensor) -> torch.Tensor:
        if not outputs.is_cuda or not masks.is_cuda:
            raise RuntimeError("rbunet.RobustBCEDiceLoss runs on CUDA tensors only (no CPU fallback)")
        if outputs.shape != masks.shape:
            raise ValueError(f"outputs {tuple(outputs.shape)} and masks {tuple(masks.shape)} differ "
                             "(the reference resizes with F.interpolate before the loss, Main_Final.py:577-578)")
        return _BceDice.apply(outputs, masks, self)


def metrics_from_counts(tp, fp, fn, tn) -> dict:
    """float64 ratios of ModelEvaluator.calculate_metrics (Main_Final.py:525-547) from integer counts."""
    tp, fp, fn, tn = float(tp), float(fp), float(fn), float(tn)
    precision = tp / (tp + fp + 1e-8)
    recall = tp / (tp + fn + 1e-8)
    return {"accuracy": (tp + tn) / (tp + fp + fn + tn), "iou": tp / (tp + fp + fn + 1e-8), "precision": precision,
            "recall": recall, "f1_score": 2 * precision * recall / (precision + recall + 1e-8)}


def confusion_counts(pred: torch.Tensor, target: torch.Tensor, threshold: float = 0.5) -> torch.Tensor:
    """[B,...] probabilities / 0-1 masks on the GPU -> int64 [B,4] = TP, FP, FN, TN (pred > threshold, strict)."""
    if not pred.is_cuda:
        raise RuntimeError("rbunet.confusion_counts runs on CUDA tensors only (no CPU fallback)")
    return ops.confusion_counts(pred.detach().contiguous().float(), target.detach().contiguous().float(), threshold)


def calculate_metrics(pred: torch.Tensor, target: torch.Tensor, threshold: float = 0.5) -> dict:
    """Same signature and keys as ModelEvaluator.calculate_metrics (Main_Final.py:519): pred/target [H,W]."""
    c = confusion_counts(pred.reshape(1, -1), target.reshape(1, -1), threshold).cpu().tolist()[0]
    return metrics_from_counts(*c)


def batch_metrics(pred: torch.Tensor, target: torch.Tensor, threshold: float = 0.5) -> list:
    """Per-image metric dicts for a whole batch with ONE device->host copy of [B,4] counts (the reference
    copies every image to the host, Main_Final.py:604-606,655-657)."""
    return [metrics_from_counts(*c) for c in confusion_counts(pred, target, threshold).cpu().tolist()]


def class_confusion_counts(pred: torch.Tensor, target: torch.Tensor, threshold: float = 0.5) -> torch.Tensor:
    """[B,K,H,W] per-class probabilities (a K-class RobustUNet's output) / 0-1 masks on the GPU -> int64 [B,K,4] =
    TP, FP, FN, TN of each class (pred > threshold, strict), from one counting pass over the B*K planes."""
    if not pred.is_cuda:
        raise RuntimeError("rbunet.class_confusion_counts runs on CUDA tensors only (no CPU fallback)")
    if pred.dim() < 3 or pred.shape != target.shape:
        raise ValueError(f"expected pred and target of the same shape [B,K,H,W], got {tuple(pred.shape)} and "
                         f"{tuple(target.shape)}")
    B, K = pred.shape[0], pred.shape[1]
    if B * K > 65535:
        raise ValueError(f"B*K = {B * K} planes; at most 65535 per call")
    p = pred.detach().contiguous().float().reshape(B * K, -1)
    t = target.detach().contiguous().float().reshape(B * K, -1)
    return ops.confusion_counts(p, t, threshold).reshape(B, K, 4)


def class_metrics(pred: torch.Tensor, target: torch.Tensor, threshold: float = 0.5) -> list:
    """For each image, K metric dicts (metrics_from_counts of each class plane) with ONE device->host copy."""
    return [[metrics_from_counts(*c) for c in img] for img in class_confusion_counts(pred, target, threshold).cpu().tolist()]
