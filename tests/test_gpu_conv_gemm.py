"""GPU parity: tcgen05 implicit-GEMM convolution (rbu_conv_gemm through the C ABI) against torch CPU fp32
convolutions on the same bf16-rounded operands (per-kernel bar: rel-L2 <= 1e-2 for bf16 storage; here the
only rounding is the bf16 output, so the bound used is much tighter)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _rel_l2(a, b):
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()


def _rand(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale)


def _nhwc_buffer(x_nchw, ld, off, dev):
    """Place x (NCHW fp32, CPU) as a channel slice at `off` of an NHWC bf16 buffer with pixel stride ld
    (other channels filled with a sentinel so slice handling errors show up)."""
    n, c, h, w = x_nchw.shape
    buf = torch.full((n, h, w, ld), 77.0, dtype=torch.bfloat16)
    buf[..., off:off + c] = x_nchw.permute(0, 2, 3, 1).to(torch.bfloat16)
    return buf.to(dev)


CASES = [
    # name, N, H, W, Cin, Cout, ksz, dil, x_ld, x_off, y_ld, y_off, bias, addend
    ("1x1_c64", 2, 16, 16, 64, 64, 1, 1, 64, 0, 64, 0, False, False),
    ("1x1_c128_2k", 2, 16, 16, 128, 128, 1, 1, 128, 0, 128, 0, True, False),
    ("3x3_c64", 2, 32, 32, 64, 64, 3, 1, 64, 0, 64, 0, False, False),
    ("3x3_d2_n256", 1, 16, 16, 128, 256, 3, 2, 128, 0, 256, 0, True, False),
    ("3x3_d4_slice", 2, 16, 16, 64, 128, 3, 4, 192, 64, 512, 128, True, False),
    ("3x3_ragged", 3, 24, 12, 64, 96, 3, 1, 64, 0, 96, 0, False, True),
    ("3x3_tiny_spatial", 5, 2, 2, 128, 64, 3, 1, 128, 0, 64, 0, False, False),
    ("1x1_cin32", 2, 8, 8, 32, 32, 1, 1, 32, 0, 32, 0, True, False),
    ("3x3_multi_tile", 4, 64, 64, 256, 512, 3, 1, 256, 0, 512, 0, False, False),
    ("3x3_1x1spatial", 130, 1, 1, 64, 64, 3, 1, 64, 0, 64, 0, False, False),
    # halo kernel (16x16 tiles, two accumulators per weight stage): ragged tile edges, channel slices, partial column
    # blocks, a one-tile image with a 256-column block, resident weights
    ("3x3_halo_ragged", 2, 20, 36, 64, 96, 3, 1, 64, 0, 96, 0, True, True),
    ("3x3_halo_slice", 2, 32, 48, 128, 160, 3, 1, 192, 64, 256, 32, True, False),
    ("3x3_one_tile_n256", 3, 16, 16, 128, 256, 3, 1, 128, 0, 256, 0, False, True),
    ("3x3_halo_resident", 2, 48, 32, 64, 64, 3, 1, 64, 0, 64, 0, True, False),
    # odd numbers of spatial tiles: the second CTA of the last CTA pair has no tile (streamed and resident weights,
    # a 96-column block whose halves are 48 weight rows per CTA, four column blocks)
    ("3x3_odd_tiles", 3, 16, 48, 128, 128, 3, 1, 128, 0, 128, 0, True, True),
    ("3x3_odd_resident", 1, 48, 16, 64, 64, 3, 1, 64, 0, 64, 0, False, False),
    ("3x3_odd_n96", 1, 40, 56, 64, 96, 3, 1, 64, 0, 96, 0, True, False),
    ("3x3_odd_4blocks", 1, 16, 16, 256, 1024, 3, 1, 256, 0, 1024, 0, False, False),
    # 128 -> 64: resident weights in the CTA-pair kernel (72 KB per CTA), two 64-channel slabs per tile
    ("3x3_pair_resident", 2, 32, 48, 128, 64, 3, 1, 128, 0, 64, 0, True, True),
    # generic kernel, staged epilogue: weights streamed (operand > 64 KB) with bias and addend; 32-column GEMM
    ("1x1_wide_k", 2, 32, 32, 512, 256, 1, 1, 512, 0, 256, 0, True, True),
    ("1x1_n32_slice", 3, 24, 40, 64, 32, 1, 1, 128, 32, 96, 64, True, False),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_conv_forward(case):
    import rbunet
    from rbunet import ops
    name, N, H, W, Cin, Cout, ksz, dil, x_ld, x_off, y_ld, y_off, use_bias, use_add = case
    dev = torch.device("cuda:0")
    x = _rand((N, Cin, H, W), 1)
    w = _rand((Cout, Cin, ksz, ksz), 2, scale=(1.0 / (Cin * ksz * ksz)) ** 0.5)
    bias = _rand((Cout,), 3) if use_bias else None
    add = _rand((N, Cout, H, W), 4) if use_add else None
    xb = x.to(torch.bfloat16).float()
    wb = w.to(torch.bfloat16).float()
    ref = F.conv2d(xb, wb, bias, padding=dil * (ksz // 2), dilation=dil)
    if add is not None:
        ref = ref + add.to(torch.bfloat16).float()

    xbuf = _nhwc_buffer(x, x_ld, x_off, dev)
    ybuf = torch.full((N, H, W, y_ld), 55.0, dtype=torch.bfloat16, device=dev)
    wp = ops.pack_weight(w.to(dev).contiguous(), 0)
    addv = ops.View(_nhwc_buffer(add, Cout, 0, dev)) if add is not None else None
    ops.conv_gemm(N, H, W, [(ops.View(xbuf, x_off, Cin), wp, ksz * ksz, dil, False)], Cout,
                  ops.View(ybuf, y_off, Cout), bias=bias.to(dev) if bias is not None else None, addend=addv)
    torch.cuda.synchronize()
    out = ybuf[..., y_off:y_off + Cout].float().cpu().permute(0, 3, 1, 2)
    err = _rel_l2(out, ref)
    assert err < 4e-3, f"{name}: rel-L2 {err}"
    # untouched channels of the output buffer keep the sentinel
    if y_ld != Cout:
        rest = torch.cat([ybuf[..., :y_off], ybuf[..., y_off + Cout:]], dim=-1).float()
        assert (rest == 55.0).all(), f"{name}: wrote outside the output slice"
    # the SIMT device reference agrees too (it is used at sizes the CPU oracle cannot reach)
    ref_dev = ops.conv_direct_ref(ops.View(xbuf, x_off, Cin), N, H, W, w.to(dev), bias.to(dev) if use_bias else None,
                                  ksz, dil)
    ref_dev = ref_dev.cpu().permute(0, 3, 1, 2)
    if add is not None:
        ref_dev = ref_dev + add.to(torch.bfloat16).float()
    assert _rel_l2(ref_dev, ref) < 1e-5


def test_conv_dgrad_matches_autograd():
    from rbunet import ops
    dev = torch.device("cuda:0")
    N, H, W, Cin, Cout = 2, 16, 16, 64, 128
    for dil in (1, 2):
        w = _rand((Cout, Cin, 3, 3), 5, scale=0.05)
        dy = _rand((N, Cout, H, W), 6)
        x = torch.zeros((N, Cin, H, W), requires_grad=True)
        y = F.conv2d(x, w.to(torch.bfloat16).float(), padding=dil, dilation=dil)
        y.backward(dy.to(torch.bfloat16).float())
        wp = ops.pack_weight(w.to(dev).contiguous(), 1)   # [Cin][9][Cout], rotated taps
        dybuf = _nhwc_buffer(dy, Cout, 0, dev)
        dx = torch.empty((N, H, W, Cin), dtype=torch.bfloat16, device=dev)
        ops.conv_gemm(N, H, W, [(ops.View(dybuf), wp, 9, dil, False)], Cin, ops.View(dx))
        torch.cuda.synchronize()
        err = _rel_l2(dx.float().cpu().permute(0, 3, 1, 2), x.grad)
        assert err < 4e-3, f"dgrad dil={dil}: rel-L2 {err}"


def test_conv_transpose_forward_and_dgrad():
    from rbunet import ops
    dev = torch.device("cuda:0")
    N, H, W, Cin, Cout = 2, 8, 8, 128, 64
    x = _rand((N, Cin, H, W), 7)
    w = _rand((Cin, Cout, 2, 2), 8, scale=0.08)
    b = _rand((Cout,), 9)
    xb = x.to(torch.bfloat16).float().requires_grad_(True)
    ref = F.conv_transpose2d(xb, w.to(torch.bfloat16).float(), b, stride=2)
    # forward: scatter into the second half of a concat buffer [N,2H,2W,2*Cout]
    cat = torch.full((N, 2 * H, 2 * W, 2 * Cout), 33.0, dtype=torch.bfloat16, device=dev)
    wp = ops.pack_weight(w.to(dev).contiguous(), 2)
    ops.conv_gemm(N, H, W, [(ops.View(_nhwc_buffer(x, Cin, 0, dev)), wp, 1, 0, False)], 4 * Cout,
                  ops.View(cat, Cout, Cout), scatter=True, Cout=Cout, bias=b.to(dev))
    torch.cuda.synchronize()
    out = cat[..., Cout:].float().cpu().permute(0, 3, 1, 2)
    assert _rel_l2(out, ref.detach()) < 4e-3
    assert (cat[..., :Cout].float() == 33.0).all()
    # data gradient: gather the four stride-2 quadrants of dout
    dout = _rand((N, Cout, 2 * H, 2 * W), 10)
    ref.backward(dout.to(torch.bfloat16).float())
    dcat = torch.full((N, 2 * H, 2 * W, 2 * Cout), 1e4, dtype=torch.bfloat16, device=dev)
    dcat[..., Cout:] = dout.permute(0, 2, 3, 1).to(torch.bfloat16).to(dev)
    wpd = ops.pack_weight(w.to(dev).contiguous(), 3)
    dx = torch.empty((N, H, W, Cin), dtype=torch.bfloat16, device=dev)
    ops.conv_gemm(N, H, W, [(ops.View(dcat, Cout, Cout), wpd, 4, 0, True)], Cin, ops.View(dx))
    torch.cuda.synchronize()
    err = _rel_l2(dx.float().cpu().permute(0, 3, 1, 2), xb.grad)
    assert err < 4e-3, f"convT dgrad rel-L2 {err}"


def test_two_segment_accumulation():
    """conv1-dgrad (3x3) + shortcut-dgrad (1x1) accumulated in one TMEM accumulator."""
    from rbunet import ops
    dev = torch.device("cuda:0")
    N, H, W, Cin, Cout = 2, 16, 16, 64, 128
    w1 = _rand((Cout, Cin, 3, 3), 11, scale=0.05)
    ws = _rand((Cout, Cin, 1, 1), 12, scale=0.1)
    dy1 = _rand((N, Cout, H, W), 13)
    dys = _rand((N, Cout, H, W), 14)
    x = torch.zeros((N, Cin, H, W), requires_grad=True)
    (F.conv2d(x, w1.to(torch.bfloat16).float(), padding=1) * dy1.to(torch.bfloat16).float()).sum().backward()
    (F.conv2d(x, ws.to(torch.bfloat16).float()) * dys.to(torch.bfloat16).float()).sum().backward()
    dx = torch.empty((N, H, W, Cin), dtype=torch.bfloat16, device=dev)
    ops.conv_gemm(N, H, W,
                  [(ops.View(_nhwc_buffer(dy1, Cout, 0, dev)), ops.pack_weight(w1.to(dev), 1), 9, 1, False),
                   (ops.View(_nhwc_buffer(dys, Cout, 0, dev)), ops.pack_weight(ws.to(dev), 1), 1, 0, False)],
                  Cin, ops.View(dx))
    torch.cuda.synchronize()
    assert _rel_l2(dx.float().cpu().permute(0, 3, 1, 2), x.grad) < 4e-3


def test_invalid_arguments_raise():
    from rbunet import ops
    dev = torch.device("cuda:0")
    x = torch.zeros((1, 4, 4, 64), dtype=torch.bfloat16, device=dev)
    y = torch.zeros((1, 4, 4, 64), dtype=torch.bfloat16, device=dev)
    w = torch.zeros((64, 1, 64), dtype=torch.bfloat16, device=dev)
    with pytest.raises(RuntimeError):
        ops.conv_gemm(1, 4, 4, [(ops.View(x), w, 5, 1, False)], 64, ops.View(y))   # taps must be 1 or 9
    with pytest.raises(RuntimeError):
        ops.conv_gemm(1, 4, 4, [(ops.View(x), w, 1, 1, False)], 60, ops.View(y))   # Ncols % 8


@pytest.mark.parametrize("shape", [
    # N, H, W, Cin, Ncols, bias
    (3, 32, 32, 64, 64, False),      # shortcut-like
    (2, 24, 40, 32, 128, False),     # ragged tile edges (W, H not multiples of the 16 x 8 pixel tile), stem-like 128 columns
    (5, 8, 8, 128, 32, True),        # tiny images: a tile spans two images; one 32-column job
    (2, 16, 16, 256, 512, True),     # two column blocks of 256
    (70, 4, 4, 64, 96, False),       # 16-pixel images, 8 per tile, odd number of 32-column chunks
])
def test_conv_epilogue_statistics(shape):
    """rbu_conv_gemm(stats=...) of the generic kernel (staged epilogue: statistics read off the staged outputs): the rows of
    per-(CTA, warp) partial sums add up to the column sums / sums of squares of the stored bf16 output."""
    from rbunet import _lib, ops
    N, H, W, Cin, Ncols, use_bias = shape
    dev = torch.device("cuda:0")
    x = _rand((N, Cin, H, W), 21)
    w = _rand((Ncols, Cin, 1, 1), 22, scale=(1.0 / Cin) ** 0.5)
    bias = _rand((Ncols,), 23).to(dev) if use_bias else None
    xbuf = _nhwc_buffer(x, Cin, 0, dev)
    y = torch.zeros((N, H, W, Ncols), dtype=torch.bfloat16, device=dev)
    st = torch.full((_lib.lib().rbu_conv_stats_floats(Ncols),), 7.0, dtype=torch.float32, device=dev)
    ops.conv_gemm(N, H, W, [(ops.View(xbuf), ops.pack_weight(w.to(dev).contiguous(), 0), 1, 0, False)], Ncols, ops.View(y),
                  bias=bias, stats=st)
    torch.cuda.synchronize()
    got = st.view(-1, 2, Ncols).double().sum(0).cpu()
    yf = y.double().reshape(-1, Ncols)
    ref = torch.stack([yf.sum(0), (yf * yf).sum(0)]).cpu()
    assert _rel_l2(got[0], ref[0]) < 1e-5 and _rel_l2(got[1], ref[1]) < 1e-5, (_rel_l2(got[0], ref[0]), _rel_l2(got[1], ref[1]))
    yref = F.conv2d(x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float(), bias.cpu() if use_bias else None)
    assert _rel_l2(y.float().cpu().permute(0, 3, 1, 2), yref) < 4e-3


@pytest.mark.parametrize("shape", [
    # N, H, W, Cin, Ncols
    (2, 32, 48, 64, 128),      # CTA pairs, one column block, 12 tiles
    (3, 16, 48, 128, 256),     # two column blocks, odd number of spatial tiles (idle CTA in the last pair)
    (1, 40, 56, 64, 96),       # ragged tile edges, 96 columns (trailing 32-column job)
    (2, 16, 16, 256, 1024),    # one-tile images, 256-column blocks, four column blocks
    (2, 32, 32, 64, 64),       # single-CTA kernel (resident 64 -> 64)
    (2, 32, 32, 128, 512),     # four column blocks of 128
])
def test_halo_epilogue_statistics(shape):
    """rbu_conv_gemm(stats=...) on the 3x3 halo kernels (staged epilogue, single CTA and CTA pairs): the one-row-per-CTA partial
    sums add up to the column sums / sums of squares of the stored bf16 output."""
    from rbunet import _lib, ops
    N, H, W, Cin, Ncols = shape
    dev = torch.device("cuda:0")
    x = _rand((N, Cin, H, W), 31)
    w = _rand((Ncols, Cin, 3, 3), 32, scale=(1.0 / (9 * Cin)) ** 0.5)
    xbuf = _nhwc_buffer(x, Cin, 0, dev)
    y = torch.zeros((N, H, W, Ncols), dtype=torch.bfloat16, device=dev)
    st = torch.full((_lib.lib().rbu_conv_stats_floats(Ncols),), 7.0, dtype=torch.float32, device=dev)
    ops.conv_gemm(N, H, W, [(ops.View(xbuf), ops.pack_weight(w.to(dev).contiguous(), 0), 9, 1, False)], Ncols, ops.View(y),
                  stats=st)
    torch.cuda.synchronize()
    got = st.view(-1, 2, Ncols).double().sum(0).cpu()
    yf = y.double().reshape(-1, Ncols)
    ref = torch.stack([yf.sum(0), (yf * yf).sum(0)]).cpu()
    assert _rel_l2(got[0], ref[0]) < 1e-5 and _rel_l2(got[1], ref[1]) < 1e-5, (_rel_l2(got[0], ref[0]), _rel_l2(got[1], ref[1]))
    yref = F.conv2d(x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float(), padding=1)
    assert _rel_l2(y.float().cpu().permute(0, 3, 1, 2), yref) < 4e-3
