"""GPU parity (bit-exact) of rbu_resize_u8 through rbunet.resize and rbunet.preprocess(size=):
Pillow BILINEAR / NEAREST (torchvision Resize on PIL images) and OpenCV INTER_NEAREST, against the library fixtures
(tests/golden/resize.npz), the numpy oracle and, where installed, the live libraries."""
import os

import numpy as np
import pytest
import torch

import rbunet
from rbunet import _lib
from oracle import resize_ref as I
from oracle import robust_unet_ref as R

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "resize.npz"))
CASES = sorted({k[:-3] for k in GOLD.files if k.endswith("_in") and not k.startswith("tv_")})
DEV = "cuda:0"


def _oracle(img, size, mode):
    return I.cv2_resize_nearest(img, size) if mode == "cv2_nearest" else I.pil_resize(img, size, mode)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.mark.parametrize("case", CASES)
def test_golden_cases(case):
    img = GOLD[f"{case}_in"]
    for mode in ("bilinear", "nearest", "cv2_nearest"):
        if f"{case}_{mode}" in GOLD.files:
            want = GOLD[f"{case}_{mode}"]
            got = rbunet.resize(_dev(img), want.shape[:2], mode).cpu().numpy()
            assert got.shape == want.shape and np.array_equal(got, want), mode


@pytest.mark.parametrize("case", ["tv_portrait", "tv_landscape", "tv_square"])
def test_torchvision_int_size(case):
    want = GOLD[f"{case}_out"]
    got = rbunet.resize(_dev(GOLD[f"{case}_in"]), int(GOLD[f"{case}_size"])).cpu().numpy()
    assert np.array_equal(got, want)


RAGGED = [(1, 1), (5, 9), (300, 200), (1024, 777), (64, 64), (999, 1500), (17, 530)]


@pytest.mark.parametrize("mode", ["bilinear", "nearest", "cv2_nearest"])
@pytest.mark.parametrize("C", [1, 3])
def test_ragged_batch(mode, C):
    """Seven sources of different sizes, up- and downscaled to one size in one call, each equal to its own oracle."""
    rng = np.random.default_rng(C * 10 + len(mode))
    imgs = [rng.integers(0, 256, size=(h, w, C) if C == 3 else (h, w)).astype(np.uint8) for h, w in RAGGED]
    got = rbunet.resize([_dev(a) for a in imgs], (200, 256), mode).cpu().numpy()
    assert got.shape == ((7, 200, 256, 3) if C == 3 else (7, 200, 256))
    for i, a in enumerate(imgs):
        assert np.array_equal(got[i], _oracle(a, (200, 256), mode)), (i, a.shape)


def test_strided_crop_source():
    rng = np.random.default_rng(3)
    full = rng.integers(0, 256, size=(400, 500, 3)).astype(np.uint8)
    crop = _dev(full)[37:337, 101:451]                  # rows strided by 1500 bytes, pixels dense
    assert not crop.is_contiguous()
    for mode in ("bilinear", "nearest", "cv2_nearest"):
        got = rbunet.resize(crop, (123, 211), mode).cpu().numpy()
        assert np.array_equal(got, _oracle(full[37:337, 101:451], (123, 211), mode)), mode


def test_batch_of_64_1024_to_512_against_pillow():
    rng = np.random.default_rng(64)
    x = rng.integers(0, 256, size=(64, 1024, 1024, 3)).astype(np.uint8)
    got = rbunet.resize(_dev(x), (512, 512)).cpu().numpy()
    try:
        from PIL import Image
        ref = lambda a: np.asarray(Image.fromarray(a).resize((512, 512), Image.BILINEAR))   # noqa: E731
    except ImportError:
        ref = lambda a: I.pil_resize(a, (512, 512))                                             # noqa: E731
    for b in range(64):
        assert np.array_equal(got[b], ref(x[b])), b


def test_mask_to_scene_size_cv2_nearest():
    rng = np.random.default_rng(5)
    m = ((rng.random((512, 512)) > 0.5) * 255).astype(np.uint8)
    got = rbunet.resize(_dev(m), (4000, 3000), "cv2_nearest").cpu().numpy()
    assert np.array_equal(got, I.cv2_resize_nearest(m, (4000, 3000)))


def test_extreme_nearest_upscale():
    """Pillow's accumulated coordinate can reach the source size on large upscales (those pixels stay 0 in Pillow)."""
    rng = np.random.default_rng(6)
    for (H, W), (h, w) in (((3, 7), (2000, 3584)), ((1, 5), (7, 4097))):
        a = rng.integers(1, 256, size=(H, W)).astype(np.uint8)
        got = rbunet.resize(_dev(a), (h, w), "nearest").cpu().numpy()
        assert np.array_equal(got, I.pil_resize(a, (h, w), "nearest"))


def test_large_downscale_loops_over_row_chunks():
    """A 10 980-row scene to 512 rows: 45 vertical taps, the tile's source rows span several shared-memory chunks."""
    rng = np.random.default_rng(7)
    a = rng.integers(0, 256, size=(10980, 150, 3)).astype(np.uint8)
    got = rbunet.resize(_dev(a), (512, 64)).cpu().numpy()
    assert np.array_equal(got, I.pil_resize(a, (512, 64)))


@pytest.mark.parametrize("nc", [3, 4, 6])
def test_preprocess_with_size(nc):
    """preprocess(size=) == preprocess(resize(...)) == the oracle's preprocess(pil_resize(...)), as raw fp32 bits."""
    rng = np.random.default_rng(nc)
    imgs = [rng.integers(0, 256, size=(h, w, 3)).astype(np.uint8) for h, w in RAGGED]
    imgs[2][0, :6] = [[0, 0, 0], [255, 255, 255], [128, 128, 128], [255, 0, 0], [0, 255, 0], [0, 0, 255]]
    dev = [_dev(a) for a in imgs]
    one_call = rbunet.preprocess(dev, nc, size=(96, 80)).cpu().numpy()
    composed = rbunet.preprocess(rbunet.resize(dev, (96, 80)), nc).cpu().numpy()
    want = R.preprocess(np.stack([I.pil_resize(a, (96, 80)) for a in imgs]), nc)
    assert one_call.shape == want.shape == (7, nc, 96, 80) and one_call.dtype == np.float32
    assert np.array_equal(one_call.view(np.uint32), composed.view(np.uint32))
    assert np.array_equal(one_call.view(np.uint32), want.view(np.uint32))
    batch = _dev(np.stack([imgs[4]] * 3))                          # a dense [B,H,W,3] batch and an int size
    got = rbunet.preprocess(batch, nc, size=32).cpu().numpy()
    assert np.array_equal(got.view(np.uint32), R.preprocess(np.stack([I.pil_resize(imgs[4], (32, 32))] * 3), nc).view(np.uint32))


def test_launch_count_does_not_depend_on_the_batch():
    rng = np.random.default_rng(8)
    imgs = [_dev(rng.integers(0, 256, size=(h, w, 3)).astype(np.uint8)) for h, w in RAGGED]
    for B in (1, 7):
        for fn, launches in ((lambda: rbunet.resize(imgs[:B], (64, 64)), 1),
                             (lambda: rbunet.resize(imgs[:B], (64, 64), "cv2_nearest"), 1),
                             (lambda: rbunet.preprocess(imgs[:B], 6, size=(64, 64)), 2)):
            n0 = _lib.launch_count()
            fn()
            assert _lib.launch_count() - n0 == launches, B


def test_largest_supported_downscale_and_beyond():
    rng = np.random.default_rng(9)
    a = rng.integers(0, 256, size=(2, 508, 3)).astype(np.uint8)              # 127x: 255 taps per output
    got = rbunet.resize(_dev(a), (2, 4)).cpu().numpy()
    assert np.array_equal(got, I.pil_resize(a, (2, 4)))
    b = _dev(rng.integers(0, 256, size=(2, 512, 3)).astype(np.uint8))        # 128x: 257 taps
    with pytest.raises(RuntimeError, match="taps"):
        rbunet.resize(b, (2, 4))
    with pytest.raises(RuntimeError, match="taps"):
        rbunet.preprocess(b.unsqueeze(0), 3, size=(2, 4))
    assert np.array_equal(rbunet.resize(b, (2, 4), "nearest").cpu().numpy(),
                          I.pil_resize(b.cpu().numpy(), (2, 4), "nearest"))   # the gathers have no tap limit
    torch.cuda.synchronize()


def test_errors():
    x = torch.zeros((8, 8, 3), dtype=torch.uint8, device=DEV)
    with pytest.raises(RuntimeError):
        rbunet.resize(torch.zeros((8, 8, 3), dtype=torch.uint8), (4, 4))               # CPU tensor
    with pytest.raises(RuntimeError):
        rbunet.resize(x.float(), (4, 4))                                                # dtype
    with pytest.raises(RuntimeError):
        rbunet.resize([x, torch.zeros((8, 8), dtype=torch.uint8, device=DEV)], (4, 4))   # mixed band counts
    with pytest.raises(RuntimeError):
        rbunet.resize([x, torch.zeros((8, 8, 3), dtype=torch.uint8)], (4, 4))            # mixed devices
    with pytest.raises(RuntimeError):
        rbunet.resize(torch.zeros((8, 8, 4), dtype=torch.uint8, device=DEV)[None], (4, 4))  # 4 bands
    with pytest.raises(RuntimeError):
        rbunet.resize(x, (0, 4))
    with pytest.raises(RuntimeError):
        rbunet.resize(x, (4, -1))
    with pytest.raises(RuntimeError):
        rbunet.resize(x, (4, 4), "bicubic")
    with pytest.raises(RuntimeError):
        rbunet.resize(x.permute(1, 0, 2), (4, 4)).cpu()        # dense rows required: pixel stride != 3
    with pytest.raises(RuntimeError):
        rbunet.resize([x, torch.zeros((8, 16, 3), dtype=torch.uint8, device=DEV)], 4)    # int size, different shapes
    with pytest.raises(RuntimeError):
        rbunet.preprocess([torch.zeros((8, 8), dtype=torch.uint8, device=DEV)], 3, size=(4, 4))   # not RGB
    torch.cuda.synchronize()
