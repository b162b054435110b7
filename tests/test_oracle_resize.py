"""CPU: the numpy restatement of Pillow's BILINEAR / NEAREST resize, OpenCV's INTER_NEAREST resize and torchvision's
Resize output size (oracle/resize_ref.py) against the fixtures generated from those libraries
(tests/golden/resize.npz) and, when they are installed, against the live libraries on a seeded sweep."""
import os

import numpy as np
import pytest

from oracle import resize_ref as I

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "resize.npz"))
CASES = sorted({k[:-3] for k in GOLD.files if k.endswith("_in") and not k.startswith("tv_")})
TV_CASES = sorted({k[:-3] for k in GOLD.files if k.startswith("tv_") and k.endswith("_in")})


def _oracle(img, size, mode):
    return I.cv2_resize_nearest(img, size) if mode == "cv2_nearest" else I.pil_resize(img, size, mode)


@pytest.mark.parametrize("case", CASES)
def test_oracle_matches_library_fixture(case):
    img = GOLD[f"{case}_in"]
    modes = [m for m in ("bilinear", "nearest", "cv2_nearest") if f"{case}_{m}" in GOLD.files]
    assert modes
    for mode in modes:
        want = GOLD[f"{case}_{mode}"]
        assert np.array_equal(_oracle(img, want.shape[:2], mode), want), mode


@pytest.mark.parametrize("case", TV_CASES)
def test_torchvision_int_size_fixture(case):
    img, want = GOLD[f"{case}_in"], GOLD[f"{case}_out"]
    size = int(GOLD[f"{case}_size"])
    assert I.torchvision_output_size(img.shape[:2], size) == want.shape[:2]
    assert np.array_equal(I.pil_resize(img, want.shape[:2], "bilinear"), want)


def test_discriminating_sizes_differ_from_the_closed_forms():
    """The accumulated Pillow coordinate and OpenCV's double reciprocal are not the textbook formulas."""
    for n_in, n_out in ((4, 333), (16, 100), (40, 100)):
        closed = np.array([int(n_in / n_out * (o + 0.5)) for o in range(n_out)])
        assert not np.array_equal(I._pil_nearest_index(n_in, n_out), closed)
    for n_in, n_out in ((22, 100), (36, 1000), (141, 333)):
        exact = np.minimum(np.arange(n_out) * n_in // n_out, n_in - 1)
        assert not np.array_equal(I.cv2_nearest_index(n_in, n_out), exact)


def test_against_live_libraries_when_present():
    Image = pytest.importorskip("PIL.Image")
    cv2 = pytest.importorskip("cv2")
    transforms = pytest.importorskip("torchvision.transforms")
    rng = np.random.default_rng(2026)
    for _ in range(60):
        H, W = (int(v) for v in rng.integers(1, 200, 2))
        h, w = (int(v) for v in rng.integers(1, 400, 2))
        for C in (1, 3):
            img = rng.integers(0, 256, size=(H, W, C) if C == 3 else (H, W)).astype(np.uint8)
            pil = Image.fromarray(img)
            assert np.array_equal(I.pil_resize(img, (h, w), "bilinear"), np.asarray(pil.resize((w, h), Image.BILINEAR)))
            assert np.array_equal(I.pil_resize(img, (h, w), "nearest"), np.asarray(pil.resize((w, h), Image.NEAREST)))
            assert np.array_equal(I.cv2_resize_nearest(img, (h, w)),
                                  cv2.resize(img, (w, h), interpolation=cv2.INTER_NEAREST))
    for hw in ((100, 50), (50, 100), (77, 77), (3, 1000)):
        for size in (1, 7, 64, 512):
            o = transforms.Resize(size)(Image.fromarray(np.zeros(hw + (3,), np.uint8)))
            assert I.torchvision_output_size(hw, size) == (o.size[1], o.size[0])
