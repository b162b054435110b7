"""TEST INFRASTRUCTURE — CPU restatement (numpy / torch) of `rbunet.PatchSampler` and `rbu_sample_patches`: the host-side
draw of a job table, the focus-pixel origin, the dihedral op and the normalisation.  Only tests/ and tools/ may import
this file; the product package never does.

Functions
---------
draw_jobs      the job table of one sample(B) call from one torch.randint(0, 2**62, (B, 5))
apply_op       the op 0-7 on the last two axes: transpose (bit 2), then flip rows (bit 1), then flip columns (bit 0)
kth_focus      the k-th nonzero pixel of a focus mask in row-major order (np.flatnonzero)
origin         the resolved origin of one job: (y0, x0), or the clamped window around the chosen focus pixel
sample         images fp32 [B,nc,ph,pw] (robust_unet_ref.preprocess of the uint8 crops), masks uint8 [B,ph,pw] and the
               resolved jobs int32 [B,4] = (scene, y, x, op)
"""
import numpy as np
import torch

from . import robust_unet_ref as R


def draw_jobs(B, sizes, ph, pw, n_focus, dihedral, generator=None):
    """Columns (scene, op, y0, x0, focus, r) as int64 [B, 6]: c = torch.randint(0, 2**62, (B, 5)), scene = c0 % S,
    op = c1 % 8 or 0, y0 = c2 % (H - wh + 1), x0 = c3 % (W - ww + 1) with wh x ww = pw x ph for ops 4-7, r = c4; the first
    n_focus jobs are focus jobs."""
    c = torch.randint(0, 2 ** 62, (B, 5), generator=generator, dtype=torch.int64).tolist()
    out = []
    for b, (c0, c1, c2, c3, c4) in enumerate(c):
        scene = c0 % len(sizes)
        op = c1 % 8 if dihedral else 0
        wh, ww = (pw, ph) if op & 4 else (ph, pw)
        H, W = sizes[scene]
        out.append([scene, op, c2 % (H - wh + 1), c3 % (W - ww + 1), int(b < n_focus), c4])
    return np.array(out, dtype=np.int64).reshape(B, 6)


def apply_op(t: torch.Tensor, op: int) -> torch.Tensor:
    if op & 4:
        t = t.transpose(-2, -1)
    if op & 2:
        t = t.flip(-2)
    if op & 1:
        t = t.flip(-1)
    return t


def kth_focus(focus: np.ndarray, k: int):
    flat = np.flatnonzero(focus)
    return divmod(int(flat[k]), focus.shape[1])


def origin(job, H, W, ph, pw, focus=None):
    """(y, x) of a job (scene, op, y0, x0, focus, r) on an H x W scene with focus mask `focus` (or None)."""
    _, op, y0, x0, is_focus, r = (int(v) for v in job)
    wh, ww = (pw, ph) if op & 4 else (ph, pw)
    total = int(np.count_nonzero(focus)) if focus is not None else 0
    if not is_focus or total == 0:
        return y0, x0
    py, px = kth_focus(focus, (r % (1 << 64)) % total)
    return min(max(py - wh // 2, 0), H - wh), min(max(px - ww // 2, 0), W - ww)


def sample(images, masks, focus, jobs, ph, pw, nc):
    """images / masks / focus: per scene numpy uint8 [H,W,3] / [H,W] / [H,W] (focus may be None or hold None);
    jobs: [B, 6] as draw_jobs.  Returns (fp32 [B,nc,ph,pw], uint8 [B,ph,pw], int32 [B,4], uint8 crops [B,ph,pw,3])."""
    crops, mcrops, resolved = [], [], []
    for job in jobs:
        s, op = int(job[0]), int(job[1])
        H, W = masks[s].shape
        y, x = origin(job, H, W, ph, pw, focus[s] if focus is not None else None)
        wh, ww = (pw, ph) if op & 4 else (ph, pw)
        win = torch.from_numpy(np.ascontiguousarray(images[s][y:y + wh, x:x + ww])).permute(2, 0, 1)
        crops.append(apply_op(win, op).permute(1, 2, 0).numpy())
        mcrops.append(apply_op(torch.from_numpy(np.ascontiguousarray(masks[s][y:y + wh, x:x + ww])), op).numpy())
        resolved.append((s, y, x, op))
    crops = np.stack(crops)
    return (R.preprocess(crops, nc), np.stack(mcrops), np.array(resolved, dtype=np.int32).reshape(-1, 4), crops)
