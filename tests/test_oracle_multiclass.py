"""CPU checks of the per-class count references (tests/multiclass_ref.py) (K-class UNet arg-max, K-class RobustUNet thresholded planes)
against brute-force loops, and of their two-class slices against the existing single-class helpers."""
import numpy as np
import pytest

from oracle import robust_unet_ref as R
from oracle import unet_ref as U
from multiclass_ref import argmax_class_counts, class_confusion_counts


def _brute_argmax(logits, target):
    B, K = logits.shape[:2]
    out = np.zeros((B, K, 4), dtype=np.int64)
    for b in range(B):
        for i in range(logits.shape[2]):
            for j in range(logits.shape[3]):
                y = int(target[b, i, j])
                if not 0 <= y < K:
                    continue
                z = logits[b, :, i, j]
                a = 0
                for k in range(1, K):            # first maximum wins
                    if z[k] > z[a]:
                        a = k
                for k in range(K):
                    p, t = a == k, y == k
                    out[b, k, 0 if p and t else 1 if p else 2 if t else 3] += 1
    return out


@pytest.mark.parametrize("K", [2, 3, 5])
def test_argmax_class_counts_brute_force_with_ties(K):
    rng = np.random.default_rng(K)
    z = rng.integers(-2, 3, size=(2, K, 7, 9)).astype(np.float32)      # small integers: many exact ties
    t = rng.integers(0, K, size=(2, 7, 9))
    t[0, 0, :4] = [-1, K, -100, K + 3]                                  # outside [0, K): no counts
    got = argmax_class_counts(z, t)
    assert got.dtype == np.int64 and got.shape == (2, K, 4)
    assert (got == _brute_argmax(z, t)).all()
    assert (got.sum(2) == ((t >= 0) & (t < K)).reshape(2, -1).sum(1)[:, None]).all()


def test_argmax_class_counts_two_class_slice_is_argmax_counts():
    rng = np.random.default_rng(0)
    z = rng.integers(-1, 2, size=(3, 2, 8, 8)).astype(np.float32)
    t = rng.integers(0, 2, size=(3, 8, 8))
    got = argmax_class_counts(z, t)
    assert (got[:, 1] == U.argmax_counts(z, t)).all()
    assert (got[:, 0] == U.argmax_counts(z, t)[:, ::-1]).all()          # class 0 = [TN, FN, FP, TP] of class 1


def test_class_confusion_counts_brute_force_and_single_class_slice():
    rng = np.random.default_rng(1)
    p = rng.integers(0, 5, size=(2, 4, 6, 5)).astype(np.float32) / 8    # includes p == 0.5 exactly: strict threshold
    y = (rng.random((2, 4, 6, 5)) > 0.5).astype(np.float32)
    got = class_confusion_counts(p, y)
    assert got.shape == (2, 4, 4) and got.dtype == np.int64
    for b in range(2):
        for k in range(4):
            pb, tb = p[b, k] > 0.5, y[b, k] != 0
            want = [(pb & tb).sum(), (pb & ~tb).sum(), (~pb & tb).sum(), (~pb & ~tb).sum()]
            assert list(got[b, k]) == want
    p1, y1 = p[:, :1], y[:, :1]
    assert (class_confusion_counts(p1, y1)[:, 0] == R.confusion_counts(p1, y1)).all()
