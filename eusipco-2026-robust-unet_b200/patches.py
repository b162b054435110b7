"""Patch sampling for training at native resolution, the counterpart of `predict_tiled` on the training side.

The reference trains on whole images resized to 512² (Main_Final.py:44-54,697-701); a model trained that way learns at
scene/512 pixels and is then asked by `predict_tiled` to segment native pixels.  `PatchSampler` keeps whole scenes in
HBM and draws every training batch with one kernel launch: random crops at the network's input size under the eight
flips / 90-degree rotations, a fraction of them centred on a focus pixel, e.g. the coastline band (nnU-Net's foreground
oversampling, MONAI's RandCropByPosNegLabel).
"""
from __future__ import annotations

import numpy as np
import torch

from ._lib import call, stream_ptr
from .ops import _p, _resize_sources

_WHO = "rbunet.PatchSampler"
_SRC = np.dtype([("image", "<u8"), ("image_pitch", "<i8"), ("mask", "<u8"), ("mask_pitch", "<i8"), ("focus", "<u8"),
                 ("focus_pitch", "<i8"), ("focus_rows", "<u8"), ("H", "<i4"), ("W", "<i4")])
_JOB = np.dtype([("scene", "<i4"), ("op", "<i4"), ("y0", "<i4"), ("x0", "<i4"), ("focus", "<i4"), ("pad", "<i4"),
                 ("r", "<i8")])


def draw_jobs(B: int, sizes, ph: int, pw: int, n_focus: int, dihedral: bool, generator=None) -> np.ndarray:
    """The job table of one `sample(B)` call (rbu_patch_job[B]) from one torch.randint(0, 2**62, (B, 5)) on the CPU:
    scene = c0 % S; op = c1 % 8 (0 without dihedral); y0 = c2 % (H - wh + 1), x0 = c3 % (W - ww + 1) for the job's
    wh x ww window (pw x ph for ops 4-7); r = c4.  Jobs 0 .. n_focus-1 are focus jobs.  `sizes`: (H, W) per scene."""
    c = torch.randint(0, 2 ** 62, (B, 5), generator=generator, dtype=torch.int64).numpy()
    hw = np.asarray(sizes, dtype=np.int64).reshape(-1, 2)
    jobs = np.zeros(B, dtype=_JOB)
    scene = c[:, 0] % len(hw)
    op = c[:, 1] % 8 if dihedral else np.zeros(B, dtype=np.int64)
    tr = (op & 4) != 0
    wh, ww = np.where(tr, pw, ph), np.where(tr, ph, pw)
    jobs["scene"] = scene
    jobs["op"] = op
    jobs["y0"] = c[:, 2] % (hw[scene, 0] - wh + 1)
    jobs["x0"] = c[:, 3] % (hw[scene, 1] - ww + 1)
    jobs["focus"] = np.arange(B) < n_focus
    jobs["r"] = c[:, 4]
    return jobs


def _planes(tensors, name, bands):
    """Check a list of uint8 CUDA [H,W] (bands 1) or [H,W,3] (bands 3) tensors with dense pixels (rows may be strided)."""
    if isinstance(tensors, torch.Tensor) or not isinstance(tensors, (list, tuple)):
        raise TypeError(f"{_WHO}: {name} must be a list of tensors")
    shape = "[H,W,3]" if bands == 3 else "[H,W]"
    for t in tensors:
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{_WHO}: {name} must hold torch tensors, got {type(t).__name__}")
        if not t.is_cuda or t.dtype != torch.uint8:
            raise TypeError(f"{_WHO}: {name} must be uint8 CUDA tensors {shape} (no CPU fallback), got {t.dtype} on "
                            f"{t.device}")
        if t.dim() != (3 if bands == 3 else 2) or (bands == 3 and t.shape[-1] != 3):
            raise ValueError(f"{_WHO}: {name} must be {shape}, got {tuple(t.shape)}")
    try:
        srcs = _resize_sources(list(tensors), _WHO)[0]
    except RuntimeError as e:
        raise ValueError(f"{name}: {e}") from None
    return srcs


def _size(size):
    ph, pw = size if isinstance(size, (tuple, list)) and len(size) == 2 else (size, size)
    for v in (ph, pw):
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
            raise TypeError(f"{_WHO}: size must be an int or a pair of ints, got {size!r}")
    if ph < 1 or pw < 1:
        raise ValueError(f"{_WHO}: size must be positive, got {size!r}")
    return int(ph), int(pw)


class PatchSampler:
    """Random training patches of whole scenes resident on the GPU, one kernel launch per batch.

    images          list of uint8 CUDA RGB scenes [H,W,3] (sizes may differ; rows may be strided, pixels dense).
    masks           list of uint8 CUDA masks [H,W], one per scene, raw values (binarise with (y > 127) as the reference
                    does, or use them as class indices).
    size            patch size, int or (ph, pw).
    n_channels      3, 4 or 6: the planes of rbunet.preprocess.
    focus           None, or a list of uint8 CUDA [H,W] masks whose nonzero pixels are the focus pixels, e.g.
                    rbunet.coastline_mask((m > 127).to(torch.uint8) * 255, 5) for the coastline band.
    focus_fraction  in [0, 1]: the first round(focus_fraction * B) patches of a batch are centred on a uniformly drawn
                    focus pixel of their scene (clamped into the scene, so the patch holds that pixel); a scene without
                    focus pixels gets a uniform crop instead.  Needs `focus` when above 0.
    dihedral        draw one of the eight flips / 90-degree rotations per patch (each needs a scene of at least
                    max(ph, pw) in both axes); False keeps every patch as it is in the scene.
    generator       CPU torch.Generator for the host-side draws (torch's default generator when None).

    sample(B) returns (x, y): x fp32 [B,n_channels,ph,pw], equal bit for bit to rbunet.preprocess of the uint8 crops,
    and y uint8 [B,ph,pw]; `last_jobs` holds the int32 [B,4] device table (scene, y, x, op) of the resolved origins.
    A call draws its random numbers on the host (draw_jobs), copies the 32-byte jobs to the device from pinned memory
    without blocking and makes one launch; it never synchronises.  The same generator seed gives the same batches.
    The sampler keeps references to the scenes.  Under rbunet.DataParallel each rank builds its own sampler with its own
    seed."""

    def __init__(self, images, masks, size=256, n_channels: int = 3, focus=None, focus_fraction: float = 0.0,
                 dihedral: bool = True, generator=None):
        imgs = _planes(images, "images", 3)
        msks = _planes(masks, "masks", 1)
        fcs = _planes(focus, "focus", 1) if focus is not None else None
        if len(msks) != len(imgs) or (fcs is not None and len(fcs) != len(imgs)):
            raise ValueError(f"{_WHO}: images, masks and focus must hold one entry per scene, got {len(imgs)}, "
                             f"{len(msks)}" + (f", {len(fcs)}" if fcs is not None else ""))
        dev = imgs[0].device
        if any(t.device != dev for t in imgs + msks + (fcs or [])):
            raise ValueError(f"{_WHO}: every scene, mask and focus mask must be on one device")
        for s, (im, m) in enumerate(zip(imgs, msks)):
            for name, t in (("mask", m), ("focus", fcs[s] if fcs is not None else None)):
                if t is not None and tuple(t.shape[:2]) != tuple(im.shape[:2]):
                    raise ValueError(f"{_WHO}: scene {s} is {tuple(im.shape[:2])}, its {name} {tuple(t.shape[:2])}")
        if isinstance(n_channels, bool) or n_channels not in (3, 4, 6):
            raise ValueError(f"{_WHO}: n_channels must be 3, 4 or 6, got {n_channels!r}")
        ph, pw = _size(size)
        need = (max(ph, pw), max(ph, pw)) if dihedral else (ph, pw)
        for s, im in enumerate(imgs):
            if im.shape[0] < need[0] or im.shape[1] < need[1]:
                raise ValueError(f"{_WHO}: scene {s} ({im.shape[0]}x{im.shape[1]}) is smaller than the "
                                 f"{need[0]}x{need[1]} window" + (" that dihedral patches need" if dihedral else ""))
        if isinstance(focus_fraction, bool) or not isinstance(focus_fraction, (int, float)) or \
                not (0.0 <= focus_fraction <= 1.0):
            raise ValueError(f"{_WHO}: focus_fraction must be in [0, 1], got {focus_fraction!r}")
        if focus_fraction > 0 and fcs is None:
            raise ValueError(f"{_WHO}: focus_fraction > 0 needs focus masks")
        if generator is not None and (not isinstance(generator, torch.Generator) or generator.device.type != "cpu"):
            raise TypeError(f"{_WHO}: generator must be a CPU torch.Generator or None")

        self.size, self.n_channels, self.dihedral = (ph, pw), int(n_channels), bool(dihedral)
        self.focus_fraction, self.generator, self.device = float(focus_fraction), generator, dev
        self._sizes = [(int(im.shape[0]), int(im.shape[1])) for im in imgs]
        self.last_jobs = None
        tab = np.zeros(len(imgs), _SRC)
        with torch.cuda.device(dev):
            self._focus_rows = []
            if fcs is not None:
                for f in fcs:
                    rows = torch.zeros(f.shape[0] + 1, dtype=torch.int64, device=dev)
                    torch.cumsum(torch.count_nonzero(f[..., 0], dim=1), 0, out=rows[1:])
                    self._focus_rows.append(rows)
                tab["focus"] = [f.data_ptr() for f in fcs]
                tab["focus_pitch"] = [f.stride(0) for f in fcs]
                tab["focus_rows"] = [r.data_ptr() for r in self._focus_rows]
            tab["image"] = [t.data_ptr() for t in imgs]
            tab["image_pitch"] = [t.stride(0) for t in imgs]
            tab["mask"] = [t.data_ptr() for t in msks]
            tab["mask_pitch"] = [t.stride(0) for t in msks]
            tab["H"] = [h for h, _ in self._sizes]
            tab["W"] = [w for _, w in self._sizes]
            self._table = self._to_device(tab)
        self._scenes = (imgs, msks, fcs)                 # the descriptors point into these

    def _to_device(self, tab: np.ndarray) -> torch.Tensor:
        host = torch.empty(tab.nbytes, dtype=torch.uint8, pin_memory=True)
        host.numpy()[:] = tab.view(np.uint8)
        return host.to(self.device, non_blocking=True)

    def sample(self, B: int):
        """One batch: (x fp32 [B,n_channels,ph,pw], y uint8 [B,ph,pw]); see the class documentation."""
        if isinstance(B, bool) or not isinstance(B, (int, np.integer)) or B < 1:
            raise ValueError(f"{_WHO}: B must be a positive int, got {B!r}")
        B = int(B)
        (ph, pw), nc = self.size, self.n_channels
        jobs = draw_jobs(B, self._sizes, ph, pw, round(self.focus_fraction * B), self.dihedral, self.generator)
        with torch.cuda.device(self.device):
            table = self._to_device(jobs)
            x = torch.empty((B, nc, ph, pw), dtype=torch.float32, device=self.device)
            y = torch.empty((B, ph, pw), dtype=torch.uint8, device=self.device)
            out_jobs = torch.empty((B, 4), dtype=torch.int32, device=self.device)
            call("rbu_sample_patches", _p(self._table), len(self._sizes), _p(table), B, ph, pw, nc, _p(x), _p(y),
                 _p(out_jobs), stream_ptr(), nbytes=float(B * ph * pw * (3 + 1 + 4 * nc + 1)))
        self.last_jobs = out_jobs
        return x, y
