"""Per-class confusion-count references for the K-class heads, built on the oracle's single-class helpers
(oracle.unet_ref.argmax_counts, oracle.robust_unet_ref.confusion_counts).  Test infrastructure only."""
import numpy as np

from oracle import robust_unet_ref as R


def argmax_class_counts(logits: np.ndarray, target: np.ndarray) -> np.ndarray:
    """Integer TP/FP/FN/TN per image and class of the K-class arg-max (ties -> lowest class index, as torch.argmax)
    against class-index targets [B,H,W].  Targets outside [0, K) are left out of every count.  Returns int64 [B,K,4]."""
    B, K = logits.shape[0], logits.shape[1]
    pred = np.argmax(logits, axis=1).reshape(B, -1)
    t = target.reshape(B, -1)
    valid = (t >= 0) & (t < K)
    out = np.zeros((B, K, 4), dtype=np.int64)
    for k in range(K):
        pk, tk = (pred == k) & valid, (t == k) & valid
        out[:, k, 0] = (pk & tk).sum(1)
        out[:, k, 1] = (pk & ~tk).sum(1)
        out[:, k, 2] = (~pk & tk).sum(1)
        out[:, k, 3] = valid.sum(1) - out[:, k, :3].sum(1)
    return out


def class_confusion_counts(pred: np.ndarray, target: np.ndarray, threshold: float = 0.5) -> np.ndarray:
    """confusion_counts of each class plane of [B,K,H,W] per-class probabilities against [B,K,H,W] 0/1 masks.
    Returns int64 [B,K,4]."""
    B, K = pred.shape[0], pred.shape[1]
    return R.confusion_counts(np.asarray(pred).reshape(B * K, -1), np.asarray(target).reshape(B * K, -1),
                              threshold).reshape(B, K, 4)
