"""GPU: patch sampling for native-resolution training (rbu_sample_patches, rbunet.PatchSampler) against the CPU oracle
(oracle/patch_ref.py), bit for bit."""
import types

import numpy as np
import pytest
import torch

import rbunet
from rbunet import _lib
from rbunet.ops import _p
from rbunet.patches import _JOB, _SRC
from oracle import patch_ref as P

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _blobs(rng, H, W, cell=8):
    """A land / water mask (0 / 255) of cell x cell blocks."""
    m = np.kron(rng.rand(H // cell + 1, W // cell + 1) > 0.5, np.ones((cell, cell), np.uint8))[:H, :W]
    return (m * 255).astype(np.uint8)


class Scene:
    """A scene on the host (numpy) and on the device; with pad > 0 the device rows are strided views of a wider buffer
    whose padding columns hold a sentinel."""

    def __init__(self, H, W, seed, pad=0, focus="random"):
        rng = np.random.RandomState(seed)
        self.img = rng.randint(0, 256, (H, W, 3)).astype(np.uint8)
        self.img[0, :min(W, 3)] = [[0, 0, 0], [255, 255, 255], [200, 10, 200]][:min(W, 3)]
        self.msk = _blobs(rng, H, W) ^ rng.randint(0, 2, (H, W)).astype(np.uint8)
        if isinstance(focus, str):
            focus = (rng.rand(H, W) < 0.01).astype(np.uint8) * rng.randint(1, 256, (H, W)).astype(np.uint8)
        self.foc = focus
        self.d_img = self._dev(self.img, pad)
        self.d_msk = self._dev(self.msk, pad)
        self.d_foc = self._dev(self.foc, pad) if self.foc is not None else None
        self.rows = None
        if self.d_foc is not None:
            self.rows = torch.zeros(H + 1, dtype=torch.int64, device=DEV)
            self.rows[1:] = torch.cumsum(torch.count_nonzero(self.d_foc, dim=1), 0)

    @staticmethod
    def _dev(a, pad):
        buf = torch.full((a.shape[0], a.shape[1] + pad) + a.shape[2:], 0xA5, dtype=torch.uint8)
        buf[:, :a.shape[1]] = torch.from_numpy(a)
        return buf.to(DEV)[:, :a.shape[1]]

    @property
    def HW(self):
        return self.msk.shape


def _table(scenes):
    tab = np.zeros(len(scenes), _SRC)
    for i, s in enumerate(scenes):
        tab[i] = (s.d_img.data_ptr(), s.d_img.stride(0), s.d_msk.data_ptr(), s.d_msk.stride(0),
                  s.d_foc.data_ptr() if s.d_foc is not None else 0, s.d_foc.stride(0) if s.d_foc is not None else 0,
                  s.rows.data_ptr() if s.rows is not None else 0, s.HW[0], s.HW[1])
    return torch.from_numpy(tab.view(np.uint8).copy()).to(DEV)


def _call(scenes, jobs, ph, pw, nc):
    """rbu_sample_patches on jobs [B, 6] (scene, op, y0, x0, focus, r) with every output inside a sentinel-filled buffer;
    checks the sentinels and returns (images, masks, jobs_out) on the host."""
    B = len(jobs)
    jt = np.zeros(B, _JOB)
    for k, name in enumerate(("scene", "op", "y0", "x0", "focus", "r")):
        jt[name] = jobs[:, k]
    table, jd = _table(scenes), torch.from_numpy(jt.view(np.uint8).copy()).to(DEV)
    ni, nm, g = B * nc * ph * pw, B * ph * pw, 37
    ibuf = torch.full((ni + 2 * g,), float("nan"), device=DEV)
    mbuf = torch.full((nm + 2 * g,), 0xCD, dtype=torch.uint8, device=DEV)
    jbuf = torch.full((4 * B + 2 * g,), -7, dtype=torch.int32, device=DEV)
    _lib.call("rbu_sample_patches", _p(table), len(scenes), _p(jd), B, ph, pw, nc, _p(ibuf[g:]), _p(mbuf[g:]),
              _p(jbuf[g:]), _lib.stream_ptr())
    ibuf, mbuf, jbuf = ibuf.cpu(), mbuf.cpu(), jbuf.cpu()
    for buf, n, sentinel in ((mbuf, nm, 0xCD), (jbuf, 4 * B, -7)):
        assert (buf[:g] == sentinel).all() and (buf[g + n:] == sentinel).all()
    assert ibuf[:g].isnan().all() and ibuf[g + ni:].isnan().all()
    return ibuf[g:g + ni].view(B, nc, ph, pw), mbuf[g:g + nm].view(B, ph, pw), jbuf[g:g + 4 * B].view(B, 4)


def _check(scenes, jobs, ph, pw, nc):
    images, masks, jout = _call(scenes, jobs, ph, pw, nc)
    want_i, want_m, want_j, _ = P.sample([s.img for s in scenes], [s.msk for s in scenes], [s.foc for s in scenes],
                                         jobs, ph, pw, nc)
    assert torch.equal(jout, torch.from_numpy(want_j))
    assert torch.equal(masks, torch.from_numpy(want_m))
    assert np.array_equal(images.numpy().view(np.uint32), want_i.view(np.uint32))
    return want_j


def _all_jobs(scenes, ph, pw, seed):
    """For every scene and every op whose window fits: one uniform job at a random origin and one focus job."""
    rng = np.random.RandomState(seed)
    jobs = []
    for s, sc in enumerate(scenes):
        H, W = sc.HW
        for op in range(8):
            wh, ww = (pw, ph) if op & 4 else (ph, pw)
            if wh > H or ww > W:
                continue
            for focus in (0, 1):
                jobs.append([s, op, rng.randint(0, H - wh + 1), rng.randint(0, W - ww + 1), focus,
                             rng.randint(0, 2 ** 62, dtype=np.int64)])
    return np.array(jobs, dtype=np.int64)


@pytest.mark.parametrize("ph,pw", [(64, 64), (48, 80), (37, 19)])
@pytest.mark.parametrize("nc", [3, 4, 6])
def test_sample_patches_is_bit_exact(ph, pw, nc):
    scenes = [Scene(ph, pw, 1, focus=None),                                # exactly the window; no focus mask
              Scene(pw, ph, 2, pad=5),                                     # exactly the transposed window, strided
              Scene(150, 131, 3, pad=3),
              Scene(max(ph, pw) + 3, max(ph, pw) + 70, 4)]
    jobs = _all_jobs(scenes, ph, pw, ph * pw + nc)
    assert set(jobs[:, 1].tolist()) == set(range(8))
    _check(scenes, jobs, ph, pw, nc)


def _focus_masks(H, W):
    out = {}
    for name, (y, x) in (("top-left", (0, 0)), ("top-right", (0, W - 1)), ("bottom-left", (H - 1, 0)),
                         ("bottom-right", (H - 1, W - 1)), ("centre", (H // 2, W // 2))):
        f = np.zeros((H, W), np.uint8)
        f[y, x] = 1
        out[name] = f
    f = np.zeros((H, W), np.uint8)
    f[H - 1, 5:] = 200
    out["last row"] = f
    f = np.zeros((H, W), np.uint8)
    f[3:, W - 1] = 1
    out["last column"] = f
    out["empty"] = np.zeros((H, W), np.uint8)
    out["dense"] = np.full((H, W), 255, np.uint8)
    return out


@pytest.mark.parametrize("name", list(_focus_masks(4, 4)))
def test_focus_origins(name):
    H, W, ph, pw = 70, 90, 16, 24
    f = _focus_masks(H, W)[name]
    scene = Scene(H, W, 9, pad=1, focus=f)
    rng = np.random.RandomState(len(name))
    jobs = []
    for op in range(8):
        wh, ww = (pw, ph) if op & 4 else (ph, pw)
        for r in (0, 1, 2 ** 62 - 1, int(rng.randint(0, 2 ** 62, dtype=np.int64))):
            jobs.append([0, op, rng.randint(0, H - wh + 1), rng.randint(0, W - ww + 1), 1, r])
    jobs = np.array(jobs, dtype=np.int64)
    got = _check([scene], jobs, ph, pw, 3)
    ys, xs = np.nonzero(f)
    for (_, y, x, op), job in zip(got, jobs):
        wh, ww = (pw, ph) if op & 4 else (ph, pw)
        if len(ys) == 0:
            assert (y, x) == (job[2], job[3])                                # falls back to the drawn origin
        else:
            k = int(job[5]) % len(ys)
            assert y <= ys[k] < y + wh and x <= xs[k] < x + ww


def test_a_scene_over_2_gib():
    """The only focus pixel and a uniform job at the far corner of a 30 000 x 24 000 x 3 scene (2.16 GB): 64-bit offsets."""
    H, W, ph, pw, R = 30000, 24000, 64, 48, 128
    assert H * W * 3 > 2 ** 31
    rng = np.random.RandomState(5)
    corner_img = rng.randint(0, 256, (R, R, 3)).astype(np.uint8)
    corner_msk = rng.randint(0, 256, (R, R)).astype(np.uint8)
    img = torch.zeros((H, W, 3), dtype=torch.uint8, device=DEV)
    msk = torch.zeros((H, W), dtype=torch.uint8, device=DEV)
    foc = torch.zeros((H, W), dtype=torch.uint8, device=DEV)
    img[H - R:, W - R:] = torch.from_numpy(corner_img).to(DEV)
    msk[H - R:, W - R:] = torch.from_numpy(corner_msk).to(DEV)
    foc[H - 1, W - 1] = 1
    rows = torch.zeros(H + 1, dtype=torch.int64, device=DEV)
    rows[1:] = torch.cumsum(torch.count_nonzero(foc, dim=1), 0)
    scene = types.SimpleNamespace(d_img=img, d_msk=msk, d_foc=foc, rows=rows, HW=(H, W))
    jobs = []
    for op in range(8):
        wh, ww = (pw, ph) if op & 4 else (ph, pw)
        jobs.append([0, op, H - wh, W - ww, 0, 0])                          # uniform, at the far corner
        jobs.append([0, op, 0, 0, 1, 2 ** 62 - 1])                          # focus, the pixel (H-1, W-1)
    jobs = np.array(jobs, dtype=np.int64)
    images, masks, jout = _call([scene], jobs, ph, pw, 3)
    local = jobs.copy()
    local[:, 2] -= H - R
    local[:, 3] -= W - R
    local[:, 4] = 0
    for b, (op, y0, x0) in enumerate(zip(jobs[:, 1], jobs[:, 2], jobs[:, 3])):
        wh, ww = (pw, ph) if op & 4 else (ph, pw)
        local[b, 2], local[b, 3] = R - wh, R - ww
        assert jout[b].tolist() == [0, H - wh, W - ww, op]
    want_i, want_m, _, _ = P.sample([corner_img], [corner_msk], None, local, ph, pw, 3)
    assert torch.equal(masks, torch.from_numpy(want_m))
    assert np.array_equal(images.numpy().view(np.uint32), want_i.view(np.uint32))


def _sampler_scenes():
    return [Scene(150, 131, 11, pad=3), Scene(96, 200, 12), Scene(64, 64, 13, pad=7)]


def _focus_of(scenes):
    return [rbunet.coastline_mask((s.d_msk > 127).to(torch.uint8) * 255, 5) for s in scenes]


def test_sampler_equals_preprocess_of_the_oracle_crops():
    scenes = _sampler_scenes()
    focus = _focus_of(scenes)
    ph, pw, nc = 48, 64, 4
    s = rbunet.PatchSampler([c.d_img for c in scenes], [c.d_msk for c in scenes], size=(ph, pw), n_channels=nc,
                            focus=focus, focus_fraction=0.4, generator=torch.Generator().manual_seed(21))
    g = torch.Generator().manual_seed(21)
    sizes = [c.HW for c in scenes]
    f_np = [f.cpu().numpy() for f in focus]
    for B in (10, 7):
        x, y = s.sample(B)
        jobs = P.draw_jobs(B, sizes, ph, pw, round(0.4 * B), True, g)
        want_i, want_m, want_j, crops = P.sample([c.img for c in scenes], [c.msk for c in scenes], f_np, jobs, ph, pw, nc)
        assert x.shape == (B, nc, ph, pw) and x.dtype == torch.float32 and y.shape == (B, ph, pw) and y.dtype == torch.uint8
        assert torch.equal(x, rbunet.preprocess(torch.from_numpy(crops).to(DEV), nc))
        assert np.array_equal(x.cpu().numpy().view(np.uint32), want_i.view(np.uint32))
        assert torch.equal(y.cpu(), torch.from_numpy(want_m))
        assert s.last_jobs.dtype == torch.int32 and torch.equal(s.last_jobs.cpu(), torch.from_numpy(want_j))
        for (sc, yy, xx, op), j in zip(want_j[:round(0.4 * B)], jobs):      # focus patches hold a coastline pixel
            wh, ww = (pw, ph) if op & 4 else (ph, pw)
            assert f_np[sc][yy:yy + wh, xx:xx + ww].any()


def test_same_seed_same_batches_and_calls_differ():
    scenes = _sampler_scenes()
    focus = _focus_of(scenes)

    def make():
        return rbunet.PatchSampler([c.d_img for c in scenes], [c.d_msk for c in scenes], size=32, focus=focus,
                                   focus_fraction=0.33, generator=torch.Generator().manual_seed(4))
    a, b = make(), make()
    xa, ya = a.sample(16)
    xb, yb = b.sample(16)
    assert torch.equal(xa, xb) and torch.equal(ya, yb) and torch.equal(a.last_jobs, b.last_jobs)
    xa2, _ = a.sample(16)
    assert not torch.equal(xa, xa2)
    torch.manual_seed(8)
    d1 = rbunet.PatchSampler([scenes[0].d_img], [scenes[0].d_msk], size=16, dihedral=False)
    x1, _ = d1.sample(8)
    assert (d1.last_jobs[:, 3] == 0).all()
    torch.manual_seed(8)
    x2, _ = d1.sample(8)
    assert torch.equal(x1, x2)                                               # torch's default generator


def test_one_launch_and_no_synchronisation():
    scenes = _sampler_scenes()
    focus = _focus_of(scenes)
    imgs, msks = [c.d_img for c in scenes], [c.d_msk for c in scenes]
    s = rbunet.PatchSampler(imgs, msks, size=64, focus=focus, focus_fraction=0.5)
    s.sample(8)
    n0 = _lib.launch_count()
    s.sample(32)
    assert _lib.launch_count() - n0 == 1
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        s2 = rbunet.PatchSampler(imgs, msks, size=64, n_channels=6, focus=focus, focus_fraction=0.25,
                                 generator=torch.Generator().manual_seed(1))
        x, y = s2.sample(12)
        s.sample(4)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert x.shape == (12, 6, 64, 64) and y.shape == (12, 64, 64)


def test_argument_errors_raise_before_any_launch():
    sc = Scene(64, 80, 3)
    img, msk, foc = sc.d_img, sc.d_msk, sc.d_foc
    ok = dict(images=[img], masks=[msk], size=(48, 80), dihedral=False)

    def with_(**kw):
        return lambda: rbunet.PatchSampler(**{**ok, **kw})
    s = rbunet.PatchSampler(**ok)
    cases = [
        (TypeError, with_(images=[img.cpu()])),
        (TypeError, with_(images=[img.float()])),
        (TypeError, with_(masks=[msk.cpu()])),
        (TypeError, with_(masks=[msk.to(torch.int16)])),
        (TypeError, with_(images=img)),
        (TypeError, with_(focus=[foc.cpu()], focus_fraction=0.5)),
        (ValueError, with_(images=[])),
        (ValueError, with_(images=[img[:, :, :2]])),
        (ValueError, with_(masks=[img])),
        (ValueError, with_(images=[img[:, ::2]], masks=[msk[:, ::2]])),                      # pixels not dense
        (ValueError, with_(masks=[msk, msk])),
        (ValueError, with_(masks=[msk[:63]])),
        (ValueError, with_(focus=[foc[:, :79]], focus_fraction=0.5)),
        (ValueError, with_(n_channels=5)),
        (ValueError, with_(size=(65, 64))),
        (ValueError, with_(size=(48, 81))),
        (ValueError, with_(size=(48, 80), dihedral=True)),                                   # 80 > H = 64
        (ValueError, with_(size=0)),
        (TypeError, with_(size=32.0)),
        (ValueError, with_(focus_fraction=1.5)),
        (ValueError, with_(focus_fraction=-0.1)),
        (ValueError, with_(focus_fraction=0.5)),                                             # no focus
        (TypeError, with_(generator=torch.Generator(device=DEV))),
        (ValueError, lambda: s.sample(0)),
        (ValueError, lambda: s.sample(-3)),
    ]
    if torch.cuda.device_count() > 1:
        cases.append((ValueError, with_(masks=[msk.to("cuda:1")])))
    for i, (exc, fn) in enumerate(cases):
        n0 = _lib.launch_count()
        with pytest.raises(exc, match="rbunet.PatchSampler"):
            fn()
        assert _lib.launch_count() == n0, i
    torch.cuda.synchronize()


def _train(batches, seed=0):
    torch.manual_seed(seed)
    model = rbunet.RobustUNet(3, 1, 16).to(DEV).train()
    opt = rbunet.FusedAdam(model.parameters(), lr=1e-3, weight_decay=1e-4)
    crit = rbunet.RobustBCEDiceLoss()
    torch.manual_seed(seed + 1)                                              # Dropout2d
    for x, y in batches:
        opt.zero_grad()
        loss = crit(model(x), (y > 127).float().unsqueeze(1))
        loss.backward()
        opt.step()
    torch.cuda.synchronize()
    return [p.detach().clone() for p in model.parameters()]


def test_training_on_sampled_batches_equals_training_on_oracle_batches():
    scenes = _sampler_scenes()
    focus = _focus_of(scenes)
    s = rbunet.PatchSampler([c.d_img for c in scenes], [c.d_msk for c in scenes], size=64, focus=focus,
                            focus_fraction=0.5, generator=torch.Generator().manual_seed(77))
    got = [tuple(t.clone() for t in s.sample(4)) for _ in range(3)]
    g = torch.Generator().manual_seed(77)
    f_np = [f.cpu().numpy() for f in focus]
    want = []
    for _ in range(3):
        jobs = P.draw_jobs(4, [c.HW for c in scenes], 64, 64, 2, True, g)
        i, m, _, _ = P.sample([c.img for c in scenes], [c.msk for c in scenes], f_np, jobs, 64, 64, 3)
        want.append((torch.from_numpy(i).to(DEV), torch.from_numpy(m).to(DEV)))
    pa, pb = _train(got), _train(want)
    assert all(torch.equal(a, b) for a, b in zip(pa, pb))
    assert not all(torch.equal(a, b) for a, b in zip(pa, _train(got[:1])))             # the steps did train
