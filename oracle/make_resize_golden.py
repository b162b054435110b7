"""TEST INFRASTRUCTURE — generate `tests/golden/resize.npz` from live Pillow, OpenCV and torchvision (the third-party
calls of Main_Final.py:44-54,697-701 and predict_coastline.py:386-392,583-602; no reference scripts needed).  Run:

    python oracle/make_resize_golden.py

The library versions are stored in the file.
"""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


# (name, source h, w, output h, w, modes), each with C = 1 and C = 3.  The first six are the sizes where Pillow's
# accumulated nearest coordinate and OpenCV's double form differ from their closed / exact-rational forms.
_ALL = ("bilinear", "nearest", "cv2_nearest")
RESIZE_CASES = [
    ("pil_nn_4_333", 4, 4, 333, 333, ("nearest",)), ("pil_nn_16_100", 16, 16, 100, 100, ("nearest",)),
    ("pil_nn_40_100", 40, 40, 100, 100, ("nearest",)), ("cv_nn_22_100", 22, 22, 100, 100, ("cv2_nearest",)),
    ("cv_nn_36_1000", 36, 36, 1000, 1000, ("cv2_nearest",)), ("cv_nn_141_333", 141, 141, 333, 333, ("cv2_nearest",)),
    ("up_1x1", 1, 1, 512, 512, _ALL), ("up_2x3", 2, 3, 512, 511, _ALL), ("down_3000x40", 3000, 40, 128, 40, _ALL),
    ("identity", 37, 53, 37, 53, _ALL), ("odd", 97, 61, 45, 130, _ALL), ("down_2x", 256, 256, 128, 128, _ALL),
    ("mixed", 300, 77, 64, 256, _ALL),
]
# torchvision Resize(int) on portrait and landscape inputs: (name, source h, w, size)
RESIZE_TV_CASES = [("tv_portrait", 300, 200, 64), ("tv_landscape", 123, 457, 50), ("tv_square", 80, 80, 33)]


def resize_golden():
    """Live Pillow Image.resize (BILINEAR / NEAREST), torchvision transforms.Resize on PIL images and cv2.resize
    (INTER_NEAREST) -- the third-party calls of Main_Final.py:44-54,697-701 and predict_coastline.py:386-392,583-602."""
    import PIL
    import cv2
    import torchvision
    from PIL import Image
    from torchvision import transforms
    rng = np.random.default_rng(512)
    out = {"pil_version": np.array(PIL.__version__), "cv2_version": np.array(cv2.__version__),
           "torchvision_version": np.array(torchvision.__version__)}
    def source(H, W, C):       # uniform noise on small sources; 8x8-pixel random blocks on large ones (the file stays small)
        if H * W <= 4096:
            return rng.integers(0, 256, size=(H, W, C)).astype(np.uint8)
        low = rng.integers(0, 256, size=(H // 8 + 2, W // 8 + 2, C)).astype(np.uint8)
        return np.kron(low, np.ones((8, 8, 1), np.uint8))[:H, :W].copy()

    for name, H, W, h, w, modes in RESIZE_CASES:
        for C in (1, 3):
            img = source(H, W, C)
            img = img[:, :, 0].copy() if C == 1 else img
            key = f"{name}_c{C}"
            out[f"{key}_in"] = img
            if "bilinear" in modes:
                out[f"{key}_bilinear"] = np.asarray(Image.fromarray(img).resize((w, h), Image.BILINEAR))
            if "nearest" in modes:
                out[f"{key}_nearest"] = np.asarray(Image.fromarray(img).resize((w, h), Image.NEAREST))
            if "cv2_nearest" in modes:
                out[f"{key}_cv2_nearest"] = cv2.resize(img, (w, h), interpolation=cv2.INTER_NEAREST)
    for name, H, W, size in RESIZE_TV_CASES:
        img = source(H, W, 3)
        out[f"{name}_in"] = img
        out[f"{name}_size"] = np.array(size)
        out[f"{name}_out"] = np.asarray(transforms.Resize(size)(Image.fromarray(img)))
    np.savez_compressed(os.path.join(OUT, "resize.npz"), **out)
    print("resize goldens:", len(out), "arrays")


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    resize_golden()
