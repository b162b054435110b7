"""Thin Python wrappers: torch tensors -> C-ABI calls (device pointers + sizes)."""
from __future__ import annotations

import ctypes
from ctypes import c_void_p
from dataclasses import dataclass

import torch

from . import _lib
from ._lib import ConvGemmArgs, call, stream_ptr


@dataclass
class View:
    """A channel slice of an NHWC bf16 activation buffer [N,H,W,ld]."""
    base: torch.Tensor      # contiguous bf16 [N,H,W,ld] (or [P,ld])
    off: int = 0            # first channel of the slice
    C: int = -1             # channels in the slice

    def __post_init__(self):
        if self.C < 0:
            self.C = self.base.shape[-1] - self.off
        assert self.base.dtype == torch.bfloat16 and self.base.is_contiguous() and self.base.is_cuda
        assert self.off % 8 == 0 and self.C % 8 == 0 and self.ld % 8 == 0

    @property
    def ld(self) -> int:
        return self.base.shape[-1]

    @property
    def ptr(self) -> int:
        return self.base.data_ptr() + 2 * self.off

    def slice(self, off, C):
        return View(self.base, self.off + off, C)

    def dense(self) -> torch.Tensor:
        return self.base[..., self.off:self.off + self.C]


def _p(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def pack_dims(w: torch.Tensor, mode: int):
    """(Nn, T, K, Cout, destination shape) of the bf16 GEMM operand that rbu_pack_weight / rbu_pack_weights_multi build
    from the fp32 torch-layout weight `w` in pack mode `mode`."""
    if mode == 0:            # Conv2d [Cout,Cin,kh,kw] forward
        Nn, T, K, cout = w.shape[0], w.shape[2] * w.shape[3], w.shape[1], 0
    elif mode == 1:          # Conv2d data gradient
        Nn, T, K, cout = w.shape[1], w.shape[2] * w.shape[3], w.shape[0], 0
    elif mode == 2:          # ConvTranspose2d [Cin,Cout,2,2] forward
        Nn, T, K, cout = 4 * w.shape[1], 1, w.shape[0], w.shape[1]
    elif mode == 3:          # ConvTranspose2d data gradient
        Nn, T, K, cout = w.shape[0], 4, w.shape[1], 0
    elif mode in (4, 5):     # stem Conv2d [C,nc,3,3] on the rbu_stem_im2col patches: [Nn][1][Kp] with T = nc; mode 4
        nc = w.shape[1]      # also holds the 1x1 shortcut (second source) in rows C..2C-1
        Nn, T, K, cout = (2 if mode == 4 else 1) * w.shape[0], nc, (9 * nc + 7) // 8 * 8, 0
    else:
        raise ValueError(mode)
    return Nn, T, K, cout, ((Nn, 1, K) if mode >= 4 else (Nn, T, K))


def pack_weight(w: torch.Tensor, mode: int) -> torch.Tensor:
    """fp32 torch-layout weight -> bf16 GEMM operand [Ncols][taps][K] (see rbu_pack_weight; modes 0-3)."""
    assert w.is_cuda and w.dtype == torch.float32 and w.is_contiguous()
    Nn, T, K, cout, shape = pack_dims(w, mode)
    out = torch.empty(shape, dtype=torch.bfloat16, device=w.device)
    call("rbu_pack_weight", _p(w), _p(out), Nn, T, K, mode, cout, stream_ptr())
    return out


def conv_gemm(N, H, W, segs, Ncols, y: View, scatter=False, Cout=0, bias=None, addend: View = None, tag="conv_gemm",
              flops=None, stats: torch.Tensor = None, scale: torch.Tensor = None, relu: int = 0,
              tile_stats: torch.Tensor = None):
    """segs: list of (x: View, w_packed, taps, dil, gather).  `flops`: algorithmic FLOPs of the call when they
    differ from the GEMM's own 2*M*N*K (e.g. the zero-padded stem)."""
    a = ConvGemmArgs()
    a.N, a.H, a.W, a.nseg = N, H, W, len(segs)
    keep = []
    for i, (x, wp, taps, dil, gather) in enumerate(segs):
        a.seg[i].x = x.ptr
        a.seg[i].x_ld = x.ld
        a.seg[i].C = x.C
        a.seg[i].w = wp.data_ptr()
        a.seg[i].taps = taps
        a.seg[i].dil = dil
        a.seg[i].gather = int(gather)
        keep.append(wp)
    a.Ncols = Ncols
    a.y = y.ptr
    a.y_ld = y.ld
    a.scatter = int(scatter)
    a.Cout = Cout
    a.bias = bias.data_ptr() if bias is not None else None
    a.addend = addend.ptr if addend is not None else None
    a.addend_ld = addend.ld if addend is not None else 0
    a.stats = stats.data_ptr() if stats is not None else None
    a.tile_stats = tile_stats.data_ptr() if tile_stats is not None else None
    a.scale = scale.data_ptr() if scale is not None else None
    a.relu = int(relu)
    if flops is None:
        flops = 2.0 * N * H * W * Ncols * sum(t * x.C for (x, _, t, _, _) in segs)
    # algorithmic bytes: every input / output activation once, plus the packed weights
    nbytes = 2.0 * N * H * W * (sum(x.C for (x, _, _, _, _) in segs) + Ncols * (2 if addend is not None else 1)) + \
        2.0 * Ncols * sum(t * x.C for (x, _, t, _, _) in segs)
    if tag == "conv_gemm":
        # profiler classes: the halo kernel's 3x3 convolutions are tensor-pipe work; everything else that goes through
        # the generic kernel in this network (1x1, stem, ConvTranspose, 16x16 dilated) is bound by its activation bytes
        if any(t == 9 and d == 1 for (_, _, t, d, _) in segs) and H >= 16 and W >= 16 and not scatter:
            tag = "conv3x3"
        else:
            tag = "conv_small"
    label = None
    if _lib.PROFILER is not None:
        label = f"conv {N}x{H}x{W} " + "+".join(f"{x.C}t{t}{'g' if g else ''}d{d}" for (x, _, t, d, g) in segs) + \
            f"->{Ncols}{' scatter' if scatter else ''}"
    call("rbu_conv_gemm", ctypes.byref(a), stream_ptr(), tag=tag, flops=flops, nbytes=nbytes, label=label)


def conv_direct_ref(x: View, N, H, W, w, bias, ksz, dil):
    cout = w.shape[0]
    out = torch.empty((N, H, W, cout), dtype=torch.float32, device=w.device)
    call("rbu_conv_direct_ref", c_void_p(x.ptr), x.ld, N, H, W, x.C, _p(w), _p(bias), cout, ksz, dil, _p(out),
         stream_ptr())
    return out


def loss_forward(probs, target, threshold=0.5, w_bce=1.0, w_dice=0.0, smooth=1.0):
    """Returns (loss[1] f32, sums[4] f64, counts[B,4] i64) device tensors."""
    B = probs.shape[0]
    HW = probs.numel() // B
    dev = probs.device
    ws_bytes = _lib.lib().rbu_loss_workspace_bytes(B, HW)
    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    sums = torch.empty(4, dtype=torch.float64, device=dev)
    counts = torch.empty((B, 4), dtype=torch.int64, device=dev)
    call("rbu_loss_forward", _p(probs), _p(target), B, HW, threshold, w_bce, w_dice, smooth, _p(ws), ws_bytes,
         _p(loss), _p(sums), _p(counts), stream_ptr())
    return loss, sums, counts


def loss_backward(probs, target, grad_out, sums, w_bce=1.0, w_dice=0.0, smooth=1.0):
    dp = torch.empty_like(probs)
    call("rbu_loss_backward", _p(probs), _p(target), probs.numel(), _p(grad_out), _p(sums), w_bce, w_dice, smooth,
         _p(dp), stream_ptr())
    return dp


def confusion_counts(pred, target, threshold=0.5):
    B = pred.shape[0]
    HW = pred.numel() // B
    counts = torch.empty((B, 4), dtype=torch.int64, device=pred.device)
    call("rbu_confusion_counts", _p(pred), _p(target), B, HW, threshold, _p(counts), stream_ptr())
    return counts


def preprocess(img_u8, n_channels: int = 3, size=None) -> torch.Tensor:
    """uint8 RGB [B,H,W,3] CUDA tensor -> fp32 NCHW [B,n_channels,H,W] (Normalize of Main_Final.py:697-701; channels
    beyond 3 are the build-defined HSV planes).  With `size`, the images are first resized by `resize(img_u8, size)`
    (Pillow bilinear = torchvision Resize on PIL images): the reference's Compose([Resize(size), ToTensor(), Normalize]).
    `img_u8` may then also be an RGB [H,W,3] image or a list of RGB images of different sizes.  (Two launches: a fused
    single-pass form measured slower on B200, profiles/r03_resize_fused_ab.txt.)"""
    if size is not None:
        srcs, _, C, _ = _resize_sources(img_u8, "rbunet.preprocess")
        if C != 3:
            raise RuntimeError("rbunet.preprocess expects RGB images [..., 3]")
        img_u8 = resize(srcs, size)
    if not img_u8.is_cuda or img_u8.dtype != torch.uint8 or img_u8.dim() != 4 or img_u8.shape[-1] != 3:
        raise RuntimeError("rbunet.preprocess expects a uint8 CUDA tensor [B,H,W,3] (no CPU fallback)")
    img_u8 = img_u8.contiguous()
    B, H, W, _ = img_u8.shape
    out = torch.empty((B, n_channels, H, W), dtype=torch.float32, device=img_u8.device)
    call("rbu_preprocess", _p(img_u8), B, H, W, n_channels, _p(out), stream_ptr())
    return out


_RESIZE_MODES = {"bilinear": 0, "nearest": 1, "cv2_nearest": 2}
_DESC = None


def _resize_sources(images, who):
    """Normalise `images` to a list of [H,W,C] uint8 CUDA views (C 1 or 3, dense pixels, rows may be strided)."""
    single = False
    if isinstance(images, torch.Tensor):
        if images.dim() == 2 or (images.dim() == 3 and images.shape[-1] == 3):
            images, single = [images], True
        elif images.dim() in (3, 4):
            images = list(images.unbind(0))
        else:
            raise RuntimeError(f"{who} expects [H,W], [H,W,3], [B,H,W] or [B,H,W,3] uint8 CUDA tensors")
    images = list(images)
    if not images:
        raise RuntimeError(f"{who}: no images")
    srcs = []
    for im in images:
        if not isinstance(im, torch.Tensor) or not im.is_cuda or im.dtype != torch.uint8 or im.dim() not in (2, 3):
            raise RuntimeError(f"{who} expects uint8 CUDA images [H,W] or [H,W,3] (no CPU fallback)")
        x = im.unsqueeze(-1) if im.dim() == 2 else im
        if x.shape[2] not in (1, 3) or x.shape[0] <= 0 or x.shape[1] <= 0:
            raise RuntimeError(f"{who}: images must be non-empty with 1 or 3 bands, got {tuple(im.shape)}")
        if not ((x.shape[2] == 1 or x.stride(2) == 1) and (x.shape[1] == 1 or x.stride(1) == x.shape[2])):
            raise RuntimeError(f"{who}: the pixels of a row must be dense (rows may be strided)")
        srcs.append(x)
    if len({x.shape[2] for x in srcs}) != 1 or len({x.device for x in srcs}) != 1:
        raise RuntimeError(f"{who}: all images must have the same band count and device")
    return srcs, srcs[0].device, srcs[0].shape[2], single


def _output_size(srcs, size, who):
    """(oh, ow) shared by every source: (h, w) as given, or torchvision's Resize(int) rule (shorter side = size)."""
    if isinstance(size, int):
        sizes = set()
        for x in srcs:
            h, w = x.shape[0], x.shape[1]
            short, long = (w, h) if w <= h else (h, w)
            new_long = int(size * long / short)
            sizes.add((new_long, size) if w <= h else (size, new_long))
        if len(sizes) != 1:
            raise RuntimeError(f"{who}: Resize({size}) gives images of different sizes {sorted(sizes)}; pass (h, w)")
        oh, ow = sizes.pop()
    else:
        oh, ow = (int(v) for v in size)
    if oh <= 0 or ow <= 0:
        raise RuntimeError(f"{who}: output size must be positive, got {(oh, ow)}")
    return oh, ow


def _descriptor_table(srcs, dev):
    """rbu_resize_src[B] on the device, copied from a pinned host buffer on the current stream (no synchronisation)."""
    import numpy as np
    global _DESC
    if _DESC is None:
        _DESC = np.dtype([("src", "<u8"), ("row_pitch", "<i8"), ("H", "<i4"), ("W", "<i4")])
    tab = np.zeros(len(srcs), _DESC)
    tab["src"] = [x.data_ptr() for x in srcs]
    tab["row_pitch"] = [x.stride(0) for x in srcs]
    tab["H"] = [x.shape[0] for x in srcs]
    tab["W"] = [x.shape[1] for x in srcs]
    host = torch.empty(tab.nbytes, dtype=torch.uint8, pin_memory=True)
    host.numpy()[:] = tab.view(np.uint8)
    with torch.cuda.device(dev):
        table = host.to(dev, non_blocking=True)
    return table, int(tab["H"].max()), int(tab["W"].max())


def resize(images, size, interpolation: str = "bilinear") -> torch.Tensor:
    """Resize uint8 CUDA images or masks, bit-exact with the reference's library calls:
      "bilinear"     Pillow Image.resize(BILINEAR) = torchvision transforms.Resize on PIL images (Main_Final.py:697-701)
      "nearest"      Pillow Image.resize(NEAREST), the mask resize of Main_Final.py:44-54
      "cv2_nearest"  cv2.resize(INTER_NEAREST), the predicted mask back to scene size (predict_coastline.py:583-602)
    `images`: [H,W], [H,W,3], [B,H,W] or [B,H,W,3], or a list of [H,W] / [H,W,3] images of different sizes (rows may be
    strided, pixels dense).  `size`: (h, w), or an int for torchvision's shorter-side rule.  Returns uint8 [B,h,w(,3)]
    from one launch, or one image when one image came in."""
    if interpolation not in _RESIZE_MODES:
        raise RuntimeError(f"rbunet.resize: interpolation must be one of {sorted(_RESIZE_MODES)}")
    srcs, dev, C, single = _resize_sources(images, "rbunet.resize")
    oh, ow = _output_size(srcs, size, "rbunet.resize")
    table, max_h, max_w = _descriptor_table(srcs, dev)
    out = torch.empty((len(srcs), oh, ow, C), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        call("rbu_resize_u8", _p(table), len(srcs), C, max_h, max_w, oh, ow, _RESIZE_MODES[interpolation], _p(out),
             stream_ptr(), nbytes=float(sum(s.numel() for s in srcs) + out.numel()))
    if C == 1:
        out = out[..., 0]
    return out[0] if single else out


def enhance_image(img: torch.Tensor, enhance_water: bool = True, return_percentiles: bool = False):
    """tif_to_image.py:139-171 `enhance_image` on the GPU: [H,W,C] or [B,H,W,C] uint8 / uint16 CUDA tensor -> uint8 of the
    same shape (2-98 percentile stretch per image and band, band-0 darkening).  Bit-exact against the reference."""
    if not img.is_cuda or img.dtype not in (torch.uint8, torch.uint16) or img.dim() not in (3, 4):
        raise RuntimeError("rbunet.enhance_image expects a uint8 / uint16 CUDA tensor [H,W,C] or [B,H,W,C] (no CPU fallback)")
    single = img.dim() == 3
    x = (img.unsqueeze(0) if single else img).contiguous()
    B, H, W, C = x.shape
    bits = 8 if x.dtype == torch.uint8 else 16
    out = torch.empty((B, H, W, C), dtype=torch.uint8, device=x.device)
    pct = torch.empty((B, C, 2), dtype=torch.float64, device=x.device)
    nbytes = int(_lib.lib().rbu_enhance_workspace_bytes(B, C, bits))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    call("rbu_enhance_image", _p(x), bits, B, H, W, C, int(bool(enhance_water)), _p(out), _p(pct), _p(ws), nbytes,
         stream_ptr(), nbytes=float(x.numel() * x.element_size() * 2 + out.numel()))
    if single:
        out, pct = out[0], pct[0]
    return (out, pct) if return_percentiles else out


def coastline_mask(mask: torch.Tensor, ksize: int = 5) -> torch.Tensor:
    """predict_coastline.py:595-602 on the GPU: cv2.dilate(mask, ellipse(ksize)) - mask for a uint8 CUDA mask [H,W] or
    [B,H,W].  The contour tracing that follows in the reference is rbunet.find_contours."""
    if not mask.is_cuda or mask.dtype != torch.uint8 or mask.dim() not in (2, 3):
        raise RuntimeError("rbunet.coastline_mask expects a uint8 CUDA tensor [H,W] or [B,H,W] (no CPU fallback)")
    single = mask.dim() == 2
    m = (mask.unsqueeze(0) if single else mask).contiguous()
    B, H, W = m.shape
    out = torch.empty_like(m)
    call("rbu_coastline_mask", _p(m), B, H, W, int(ksize), _p(out), stream_ptr(), nbytes=float(2 * m.numel()))
    return out[0] if single else out
