"""CPU: the numpy restatement of the reference's image operations (oracle/imageops_ref.py) against the committed
fixtures generated from the reference's own enhance_image and from OpenCV (tests/golden/imageops.npz), against numpy's
percentile, and -- when cv2 is installed -- against live OpenCV."""
import os

import numpy as np
import pytest

from oracle import imageops_ref as I

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "imageops.npz"))


@pytest.mark.parametrize("tag", ["u16", "u8", "u16full", "tiny"])
def test_enhance_matches_reference_fixture(tag):
    rgb = GOLD[f"enh_{tag}_in"]
    for ew in (0, 1):
        assert np.array_equal(I.enhance_image(rgb, bool(ew)), GOLD[f"enh_{tag}_out{ew}"])
    pct = GOLD[f"enh_{tag}_pct"]
    for i in range(rgb.shape[2]):
        assert I.percentile_linear(rgb[:, :, i], 2) == pct[i, 0]
        assert I.percentile_linear(rgb[:, :, i], 98) == pct[i, 1]


def test_percentile_equals_numpy_on_random_bands():
    rng = np.random.default_rng(5)
    for dt, hi in ((np.uint8, 256), (np.uint16, 65536), (np.uint16, 700)):
        for n in (1, 2, 3, 50, 51, 101, 4096, 9999):
            band = rng.integers(0, hi, size=n).astype(dt)
            for q in (2, 98):
                assert I.percentile_linear(band, q) == np.percentile(band, q), (dt, n, q)


def test_enhance_constant_band_is_zero_not_garbage():
    rgb = np.full((8, 8, 3), 77, dtype=np.uint8)
    rgb[:, :, 1] = np.arange(64, dtype=np.uint8).reshape(8, 8)
    out = I.enhance_image(rgb, True)
    assert (out[:, :, 0] == 0).all() and (out[:, :, 2] == 0).all()
    assert out[:, :, 1].max() == 255 and out[:, :, 1].min() == 0


@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 20, 31])
def test_ellipse_matches_opencv_fixture(k):
    assert np.array_equal(I.structuring_ellipse(k), GOLD[f"ellipse_{k}"])


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_coastline_matches_opencv_fixture(tag):
    mask = GOLD[f"mask_{tag}"]
    for k in (5, 20, 3):
        assert np.array_equal(I.coastline_mask(mask, k), GOLD[f"coast_{tag}_k{k}"])
        assert np.array_equal(I.coastline_mask(mask // 255, k), GOLD[f"coast01_{tag}_k{k}"])
    assert np.array_equal(I.dilate(GOLD[f"gray_{tag}"], I.structuring_ellipse(5)), GOLD[f"graydil_{tag}_k5"])


def test_against_live_opencv_when_present():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(9)
    for k in range(1, 34):
        assert np.array_equal(I.structuring_ellipse(k), cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k))), k
    for k in (4, 5, 9, 20):
        m = ((rng.random((37, 53)) > 0.93) * 255).astype(np.uint8)
        ref = cv2.dilate(m, cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k)), iterations=1) - m
        assert np.array_equal(I.coastline_mask(m, k), ref)
