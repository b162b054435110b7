"""Bit-exact tests of every convolution and weight-gradient kernel variant (conv_gemm.cu, conv_halo.cu, wgrad_gemm.cu,
wgrad_halo.cu), one row per variant.

The operands are small integers and every accumulator stays below 2^22 in absolute sum (tests/conv_exact_ref.py), so
each output has exactly one correct value whatever the tiling, split-K, CTA pairing or accumulation order: the bf16
outputs must equal the exact fp64 result rounded fp64 -> fp32 -> bf16, bit for bit, and the fp32 weight gradients the
exact result in fp32.  A single wrong element anywhere fails, which the relative-L2 tests cannot promise.

Each row names the selection rule it reaches and the kernels it must launch; the call runs under torch.profiler and the
set of launched kernel names is asserted, so a row that drifts to another variant fails instead of silently testing
something else.  Sub-variants that the kernel name does not show (resident weights, staging buffers, block_n) are argued
in the row's comment from the selection code.  The wgrad rows that pick a reduction kernel depend on the split-K factor
and therefore on the SM count; the comments assume the 148 SMs of a B200.

Every call reads channel slices (ld > C, offset > 0) whose neighbouring channels, and one extra image after the last,
hold a large finite sentinel (2^15), and writes a slice of a buffer with sentinel channels on both sides and a sentinel
image after the last one; all sentinels must survive.  Weight gradients land inside a larger fp32 buffer whose guard
regions must survive, and the split-K workspace starts out filled with the sentinel.

The exactness of the tensor cores' fp32 accumulation below 2^22 is an argument from the number format (every partial
sum is an integer fp32 holds), confirmed by these rows passing on a B200, not a documented guarantee.
"""
import ctypes
import json
import os
import tempfile

import pytest
import torch

import conv_exact_ref as R

pytestmark = pytest.mark.gpu

SENT = 2.0 ** 15
PAD = 8
HALO, PAIR, GEN = "conv_halo_kernel", "conv_halo_pair_kernel", "conv_gemm_kernel"
W1, W2, WP, WG = "wgrad_halo_kernel", "wgrad_halo2_kernel", "wgrad_pair_kernel", "wgrad_gemm_kernel"
R64, R32, R16 = "wgrad_reduce_kernel<64>", "wgrad_reduce_kernel<32>", "wgrad_reduce_kernel<16>"


def _dev():
    return torch.device("cuda:0")


def _kernel_name(s):
    s = s.replace("(anonymous namespace)::", "")
    if s.startswith("void "):
        s = s[5:]
    return s.split("(")[0].strip()


def _launch(fn):
    """Run fn() under torch.profiler and return the set of kernel names it launched (memsets and copies excluded)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    return {_kernel_name(e["name"]) for e in events if e.get("cat") == "kernel"}


def _act(t, off=PAD, pad_hi=PAD):
    """fp64 NCHW (CPU) -> View of channels [off, off + C) of a sentinel-filled NHWC bf16 buffer with one extra image."""
    from rbunet import View
    n, c, h, w = t.shape
    buf = torch.full((n + 1, h, w, off + c + pad_hi), SENT, dtype=torch.bfloat16)
    buf[:n, ..., off:off + c] = t.permute(0, 2, 3, 1).to(torch.bfloat16)
    return View(buf.to(_dev()), off, c)


def _out(n, h, w, c, off=PAD, pad_hi=PAD):
    from rbunet import View
    return View(torch.full((n + 1, h, w, off + c + pad_hi), SENT, dtype=torch.bfloat16, device=_dev()), off, c)


def _read(v, n):
    """The first n images of an output View as NCHW bf16 (CPU), after checking every other element kept the sentinel."""
    base = v.base.cpu()
    inside = torch.zeros(base.shape, dtype=torch.bool)
    inside[:n, ..., v.off:v.off + v.C] = True
    outside = base[~inside]
    bad = int((outside != SENT).sum())
    assert bad == 0, f"{bad} elements outside the output view were overwritten"
    return base[:n, ..., v.off:v.off + v.C].permute(0, 3, 1, 2).contiguous()


def _row(id, op, N, H, W, cin, cout, kernels, k=3, dil=1, **epi):
    return pytest.param(dict(id=id, op=op, N=N, H=H, W=W, cin=cin, cout=cout, k=k, dil=dil, kernels=frozenset(kernels),
                             **epi), id=id)


# Forward and data-gradient rows.  op: fwd (pack mode 0), dgrad (mode 1), dgrad2 (3x3 dgrad + 1x1 shortcut dgrad in one
# accumulator), convT (ConvTranspose2d forward, scatter into the second half of a concat buffer), convT_dgrad (gather).
# Halo selection: conv_halo.cu:705-720 (rbu_conv_halo_supported: 3x3 dil 1 / 1x1 segments, H, W >= 16, no scatter /
# gather); block_n conv_halo.cu:734-735; single-CTA resident vs pair conv_halo.cu:754-758 (single CTA only when the whole
# operand is resident: one 3x3 segment, one column block, C % 64 == 0, C/64 * block_n <= 96); staging buffers
# conv_halo.cu:764-775 (streamed) and :777-792 (resident: 2 / 1 / 0 buffers by the room left).
# Generic: conv_gemm.cu:617-622 (everything the halo kernel refuses), :628-642 (tiles), :644 (block_n), :665-673 (TMA
# stores), :679-686 (resident weights).
CONV_ROWS = [
    # --- single-CTA halo kernel, resident weights (conv_halo.cu:754-756, :781-791)
    _row("halo1_64to64_res_1buf", "fwd", 2, 32, 32, 64, 64, [HALO], bias=True),          # 72 KB weights: 1 buffer
    _row("halo1_64to32_res_2buf", "fwd", 3, 16, 16, 64, 32, [HALO], bias=True),          # 36 KB weights: 2 buffers
    _row("halo1_64to96_res_direct", "fwd", 2, 32, 16, 64, 96, [HALO], bias=True),       # 96: no room, per-thread
    _row("halo1_128to32_res", "fwd", 2, 16, 48, 128, 32, [HALO], addend=True),           # 2 slabs x 32 columns
    _row("halo1_192to32_res_direct", "fwd", 1, 48, 16, 192, 32, [HALO]),                 # 3 slabs: 96, per-thread stores
    # --- CTA-pair halo kernel
    _row("pair_128to64_res", "fwd", 2, 32, 48, 128, 64, [PAIR], bias=True),              # 128 > 96: pair, resident
    _row("pair_128to256_streamed", "fwd", 2, 32, 48, 128, 256, [PAIR], bias=True),       # block_n 128, 2 blocks
    _row("pair_128to128_odd_tiles", "fwd", 3, 16, 48, 128, 128, [PAIR], addend=True),    # 9 spatial tiles: idle 2nd CTA
    _row("pair_1024to1024_one_tile", "fwd", 2, 16, 16, 1024, 1024, [PAIR]),              # one tile: block_n 256
    _row("pair_256to1024_one_tile_odd", "fwd", 3, 16, 16, 256, 1024, [PAIR], bias=True), # 3 tiles: idle CTA, 256 columns
    _row("pair_dgrad_128to64", "dgrad", 2, 32, 32, 64, 128, [PAIR]),                     # pack mode 1, 2 slabs -> 64 columns
    # --- per-thread stores (Ncols % 32 != 0: conv_halo.cu:764)
    _row("halo1_n40_ragged", "fwd", 2, 24, 20, 64, 40, [HALO], bias=True),               # block_n 64, resident
    _row("halo1_n72", "fwd", 2, 16, 16, 64, 72, [HALO], addend=True),                    # block_n 96: resident
    _row("pair_n40", "fwd", 2, 16, 32, 128, 40, [PAIR], bias=True),                      # 2 slabs: pair, resident
    _row("pair_n72_streamed", "fwd", 1, 32, 32, 256, 72, [PAIR], addend=True),           # 4 slabs x 96: streamed
    # --- two segments (conv1 3x3 dgrad + shortcut 1x1 dgrad): not resident -> pair, block_n 64, 2 staging buffers
    _row("pair_two_segments_ragged", "dgrad2", 2, 20, 36, 64, 128, [PAIR]),
    # --- halo epilogue: single CTA (64 -> 64 resident) and pair (128 -> 128 streamed)
    _row("epi_bias_single", "fwd", 2, 32, 32, 64, 64, [HALO], bias=True),
    _row("epi_bias_pair", "fwd", 2, 32, 32, 128, 128, [PAIR], bias=True),
    _row("epi_addend_single", "fwd", 2, 32, 32, 64, 64, [HALO], addend=True),
    _row("epi_addend_pair", "fwd", 2, 32, 32, 128, 128, [PAIR], addend=True),
    _row("epi_scale_relu_single", "fwd", 2, 32, 32, 64, 64, [HALO], scale=True, bias=True, relu="all"),
    _row("epi_scale_relu_pair", "fwd", 2, 32, 32, 128, 128, [PAIR], scale=True, bias=True, relu="all"),
    _row("epi_relu24_single", "fwd", 2, 32, 32, 64, 64, [HALO], bias=True, relu=24),
    _row("epi_relu40_pair", "fwd", 2, 32, 32, 128, 128, [PAIR], bias=True, relu=40),
    _row("epi_all_relu72_pair", "fwd", 2, 32, 32, 128, 128, [PAIR], scale=True, bias=True, addend=True, relu=72),
    _row("epi_scale_relu_direct", "fwd", 2, 32, 16, 64, 96, [HALO], scale=True, bias=True, relu=48),
    # --- halo epilogue, per-CTA statistics (one row per CTA).  The single-CTA kernel only ever has one column block
    # (single_resident needs n_blocks == 1), so "several column blocks" exists for the pair kernel only.
    _row("stats_single_staged", "fwd", 2, 32, 32, 64, 64, [HALO], stats=True, sparse=True),
    _row("stats_single_direct", "fwd", 2, 32, 16, 64, 96, [HALO], stats=True, sparse=True),
    _row("stats_pair_one_block", "fwd", 2, 32, 32, 128, 128, [PAIR], stats=True, sparse=True),
    _row("stats_pair_four_blocks", "fwd", 2, 32, 32, 128, 512, [PAIR], stats=True, sparse=True),
    # --- halo epilogue, per-image tile statistics on ragged 40 x 24 images
    _row("tile_stats_single_staged", "fwd", 2, 40, 24, 64, 64, [HALO], tile_stats=True, sparse=True),
    _row("tile_stats_single_direct", "fwd", 2, 40, 24, 64, 96, [HALO], tile_stats=True, sparse=True),
    _row("tile_stats_pair", "fwd", 1, 40, 24, 128, 128, [PAIR], tile_stats=True, sparse=True),
    # --- generic kernel (conv_gemm.cu): everything the halo kernel does not take
    _row("gen_1x1_resident", "fwd", 2, 32, 32, 64, 64, [GEN], k=1, bias=True),           # 8 KB operand: resident
    _row("gen_1x1_streamed", "fwd", 2, 32, 32, 512, 256, [GEN], k=1, bias=True, addend=True),   # 256 KB: streamed
    _row("gen_3x3_dil2_streamed", "fwd", 2, 16, 16, 64, 64, [GEN], dil=2, bias=True),    # 9 k-blocks x 64: 72 KB streamed
    _row("gen_3x3_dil4_resident", "fwd", 2, 32, 32, 32, 32, [GEN], dil=4),               # 9 x 32 columns: 36 KB resident
    _row("gen_dgrad_dil2", "dgrad", 2, 16, 16, 64, 128, [GEN], dil=2),
    _row("gen_3x3_8x8_tn2", "fwd", 3, 8, 8, 128, 64, [GEN], bias=True),                  # TW = TH = 8, TN = 2, N odd
    _row("gen_3x3_4x4_tn8", "fwd", 5, 4, 4, 64, 64, [GEN], addend=True),                 # TN = 8 images per tile
    _row("gen_3x3_1x1_130_images", "fwd", 130, 1, 1, 64, 64, [GEN]),                     # TN = 128: two tiles
    _row("gen_1x1_1024to512_two_blocks", "fwd", 2, 16, 16, 1024, 512, [GEN], k=1),       # block_n 256, 2 column blocks
    _row("gen_1x1_n40_direct", "fwd", 2, 16, 24, 64, 40, [GEN], k=1, bias=True),         # Ncols % 32 != 0: per-thread stores
    _row("gen_two_segments_8x8", "dgrad2", 2, 8, 8, 64, 128, [GEN]),
    _row("gen_scale_relu_prefix", "fwd", 2, 16, 16, 128, 64, [GEN], k=1, scale=True, bias=True, relu=16),
    _row("gen_stats_staged", "fwd", 3, 24, 40, 64, 128, [GEN], k=1, stats=True, sparse=True),
    _row("gen_stats_direct_n40", "fwd", 3, 24, 40, 64, 40, [GEN], k=1, stats=True, sparse=True),
    # --- ConvTranspose2d(2, s=2) (conv_gemm.cu:670-671: TMA stores need Cout % 64 == 0)
    _row("convT_scatter_c64_tma", "convT", 2, 8, 8, 128, 64, [GEN], bias=True),
    _row("convT_scatter_c32_direct", "convT", 2, 8, 8, 64, 32, [GEN], bias=True),
    _row("convT_dgrad_gather", "convT_dgrad", 2, 8, 8, 128, 64, [GEN]),
]


def _operands(c):
    """Seeded integer operands of a row (fp64, CPU).  Statistics rows use sparse {-1, 0, 1} operands so that the column
    sums of the stored outputs stay exact in fp32."""
    N, H, W, cin, cout, k = c["N"], c["H"], c["W"], c["cin"], c["cout"], c["k"]
    kw = dict(vmax=1, zero_frac=0.8) if c.get("sparse") else {}
    op = c["op"]
    if op == "fwd":
        return dict(x=R.int_operand((N, cin, H, W), 1, **kw), w=R.int_operand((cout, cin, k, k), 2, **kw))
    if op == "dgrad":
        return dict(dy=R.int_operand((N, cout, H, W), 3, **kw), w=R.int_operand((cout, cin, k, k), 4, **kw))
    if op == "dgrad2":
        return dict(dy1=R.int_operand((N, cout, H, W), 5), w1=R.int_operand((cout, cin, 3, 3), 6),
                    dys=R.int_operand((N, cout, H, W), 7), ws=R.int_operand((cout, cin, 1, 1), 8))
    if op == "convT":
        return dict(x=R.int_operand((N, cin, H, W), 9), w=R.int_operand((cin, cout, 2, 2), 10))
    if op == "convT_dgrad":
        return dict(dout=R.int_operand((N, cout, 2 * H, 2 * W), 11), w=R.int_operand((cin, cout, 2, 2), 12))
    raise ValueError(op)


@pytest.mark.parametrize("c", CONV_ROWS)
def test_conv_variant_bit_exact(c):
    from rbunet import _lib, ops
    dev = _dev()
    op, N, H, W, cin, cout = c["op"], c["N"], c["H"], c["W"], c["cin"], c["cout"]
    k, dil = c["k"], c["dil"]
    o = _operands(c)
    g = {name: t.to(dev) for name, t in o.items()}
    oh, ow, scatter, Cout = H, W, False, 0
    if op == "fwd":
        acc, smax = R.exact(lambda x, w: R.conv_fwd(x, w, dil), g["x"], g["w"])
        segs = [(_act(o["x"]), ops.pack_weight(g["w"].float().contiguous(), 0), k * k, dil, False)]
        Ncols = C = cout
    elif op == "dgrad":
        acc, smax = R.exact(lambda dy, w: R.conv_dgrad(dy, w, dil), g["dy"], g["w"])
        segs = [(_act(o["dy"]), ops.pack_weight(g["w"].float().contiguous(), 1), k * k, dil, False)]
        Ncols = C = cin
    elif op == "dgrad2":
        acc, smax = R.exact(lambda a, b, d, e: R.conv_dgrad(a, b) + R.conv_dgrad(d, e), g["dy1"], g["w1"], g["dys"], g["ws"])
        segs = [(_act(o["dy1"]), ops.pack_weight(g["w1"].float().contiguous(), 1), 9, 1, False),
                (_act(o["dys"], pad_hi=24), ops.pack_weight(g["ws"].float().contiguous(), 1), 1, 0, False)]
        Ncols = C = cin
    elif op == "convT":
        acc, smax = R.exact(R.convT_fwd, g["x"], g["w"])
        segs = [(_act(o["x"]), ops.pack_weight(g["w"].float().contiguous(), 2), 1, 0, False)]
        Ncols, C, oh, ow, scatter, Cout = 4 * cout, cout, 2 * H, 2 * W, True, cout
    else:   # convT_dgrad: dout is the second half of a concat buffer
        acc, smax = R.exact(R.convT_dgrad, g["dout"], g["w"])
        segs = [(_act(o["dout"], off=cout), ops.pack_weight(g["w"].float().contiguous(), 3), 4, 0, True)]
        Ncols = C = cin

    scale = R.dyadic_scale(C, 20).to(dev) if c.get("scale") else None
    bias = (R.dyadic_bias(C, 21) if scale is not None else R.dyadic_bias(C, 21).round()).to(dev) if c.get("bias") else None
    add_t = R.int_operand((N, C, oh, ow), 22, vmax=100) if c.get("addend") else None
    relu = C if c.get("relu") == "all" else c.get("relu", 0)
    exact = R.epilogue(acc, scale, bias, add_t.to(dev) if add_t is not None else None, relu)
    want = R.expected_bf16(exact)

    y = _out(N, oh, ow, C, off=Cout if scatter else PAD)
    addv = _act(add_t) if add_t is not None else None
    stats = tstats = None
    if c.get("stats"):
        stats = torch.full((_lib.lib().rbu_conv_stats_floats(Ncols),), SENT, dtype=torch.float32, device=dev)
    if c.get("tile_stats"):
        chunks = _lib.lib().rbu_conv_tile_stats_chunks(H, W)
        tstats = torch.full((N * chunks * 4 * Ncols,), SENT, dtype=torch.float32, device=dev)
    bias32 = bias.float().contiguous() if bias is not None else None
    scale32 = scale.float().contiguous() if scale is not None else None
    seen = _launch(lambda: ops.conv_gemm(N, H, W, segs, Ncols, y, scatter=scatter, Cout=Cout, bias=bias32, addend=addv,
                                         stats=stats, scale=scale32, relu=relu, tile_stats=tstats))
    assert seen == c["kernels"], f"launched {sorted(seen)}, expected {sorted(c['kernels'])}"
    got = _read(y, N)
    compared = R.assert_bits_equal(got, want, "output")

    yq = want.double()                            # the stored values (equal to `got` from here on)
    if stats is not None:
        ref = torch.stack([yq.sum((0, 2, 3)), (yq * yq).sum((0, 2, 3))])
        bound = max(float(yq.abs().sum((0, 2, 3)).max()), float(ref[1].max()))
        assert bound < R.EXACT_STATS, f"statistics bound violated: {bound}"
        compared += R.assert_bits_equal(stats.view(-1, 2, Ncols).double().sum(0), ref, "stats", dims="QC")
    if tstats is not None:
        compared += R.assert_bits_equal(tstats.view(N, -1, 4, Ncols).cpu(), _tile_stats_ref(yq, H, W), "tile_stats",
                                        dims=("N", "chunk", "Q", "C"))
    print(f"\n[conv_exact] {c['id']:32s} kernels={sorted(seen)} max_S={smax:.0f} compared={compared}")


def _tile_stats_ref(y, H, W):
    """[N][chunks][4][C] reference of the halo epilogue's tile statistics: per image and 16 x 8-pixel half-tile (chunk =
    (tile_row * tiles_w + tile_col) * 2 + half) the sum, sum of squares, max and min of the stored values; a half-tile
    wholly outside the image holds (0, 0, -inf, +inf)."""
    N, C = y.shape[0], y.shape[1]
    tw, th = -(-W // 16), -(-H // 16)
    out = torch.empty((N, th * tw * 2, 4, C), dtype=torch.float64)
    for ty in range(th):
        for tx in range(tw):
            for half in range(2):
                ch = (ty * tw + tx) * 2 + half
                blk = y[:, :, ty * 16:ty * 16 + 16, tx * 16 + 8 * half:tx * 16 + 8 * half + 8].reshape(N, C, -1)
                if blk.shape[-1] == 0:
                    out[:, ch] = torch.tensor([0.0, 0.0, -float("inf"), float("inf")], dtype=torch.float64).view(1, 4, 1)
                    continue
                out[:, ch, 0], out[:, ch, 1] = blk.sum(-1), (blk * blk).sum(-1)
                out[:, ch, 2], out[:, ch, 3] = blk.amax(-1), blk.amin(-1)
    assert float(out[:, :, 1].max()) < R.EXACT_STATS and float(out[:, :, 0].abs().max()) < R.EXACT_STATS
    return out.float()


def test_gpu_reference_matches_cpu_reference():
    """The fp64 references run on the GPU for speed; with integer operands they must agree with the CPU exactly."""
    dev = _dev()
    x, w, dy = R.int_operand((2, 64, 9, 7), 30), R.int_operand((32, 64, 3, 3), 31), R.int_operand((2, 32, 9, 7), 32)
    wt, dout = R.int_operand((64, 32, 2, 2), 33), R.int_operand((2, 32, 18, 14), 34)
    for name, fn, args in [("conv_fwd d1", lambda a, b: R.conv_fwd(a, b, 1), (x, w)),
                           ("conv_fwd d2", lambda a, b: R.conv_fwd(a, b, 2), (x, w)),
                           ("conv_dgrad d4", lambda a, b: R.conv_dgrad(a, b, 4), (dy, w)),
                           ("convT_fwd", R.convT_fwd, (x, wt)),
                           ("convT_dgrad", R.convT_dgrad, (dout, wt)),
                           ("conv_wgrad d1", lambda a, b: R.conv_wgrad(a, b, 3, 1), (x, dy)),
                           ("conv_wgrad d2", lambda a, b: R.conv_wgrad(a, b, 3, 2), (x, dy)),
                           ("convT_wgrad", R.convT_wgrad, (x, dout))]:
        cpu = fn(*args)
        gpu = fn(*(a.to(dev) for a in args)).cpu()
        assert torch.equal(cpu, gpu), name


# Weight-gradient rows.  Halo kernels: wgrad_halo.cu:572-574 (3x3 dil 1, H >= 8, W >= 16), forms wgrad_halo.cu:533-543
# (form 2 when Cout % 128 == 0 and Cin % 32 == 0, the pair form when also Cout % 256 == 0, else form 1); split-K from the
# cost model wgrad_halo.cu:547-566.  Generic kernel: wgrad_gemm.cu:294-298 and :311-357 (ksplit = ceil(2 * SMs /
# items), capped by the pixel tiles).  Reduction kernel: wgrad_gemm.cu:371-381 (<64> for Cin >= 64 and ksplit <= 16, <32>
# for Cin >= 32 and ksplit <= 64, else <16>).  The ksplit values in the comments are for 148 SMs.
WGRAD_ROWS = [
    _row("w_form1_64x64", "wgrad", 2, 32, 32, 64, 64, [W1, R64]),                      # ksplit 2
    _row("w_form1_cin32_partial", "wgrad", 2, 16, 32, 32, 64, [W1, R32]),              # one 64-channel block, half used
    _row("w_form1_cin96_ragged", "wgrad", 2, 24, 40, 96, 64, [W1, R64]),               # second block partial, ragged
    _row("w_form1_cout192", "wgrad", 1, 16, 16, 64, 192, [W1, R64]),                   # 192 % 128 != 0: form 1, 3 blocks
    _row("w_form2_128x32", "wgrad", 2, 32, 32, 32, 128, [W2, R32]),
    _row("w_form2_384x64", "wgrad", 2, 16, 16, 64, 384, [W2, R64]),                    # 384 % 256 != 0: form 2
    _row("w_form2_min_tile", "wgrad", 3, 8, 16, 64, 128, [W2, R64]),                   # H = 8, W = 16: one tile per image
    _row("w_pair_256x64", "wgrad", 2, 32, 32, 64, 256, [WP, R64]),
    _row("w_pair_1024x256", "wgrad", 2, 16, 16, 256, 1024, [WP, R64]),
    _row("w_pair_256x128_ragged", "wgrad", 1, 20, 36, 128, 256, [WP, R64]),
    _row("w_gen_1x1", "wgrad", 2, 16, 16, 128, 64, [WG, R64], k=1),                    # ksplit 4
    _row("w_gen_dil2", "wgrad", 1, 16, 16, 64, 128, [WG, R64], dil=2),
    _row("w_gen_dil4", "wgrad", 2, 16, 16, 128, 64, [WG, R64], dil=4),
    _row("w_gen_small_map", "wgrad", 4, 4, 8, 64, 64, [WG, R64]),                      # H < 8: generic 3x3
    _row("w_gen_convT_gather", "wgradT", 2, 8, 8, 128, 64, [WG, R64]),
    _row("w_gen_reduce32_cin32", "wgrad", 2, 32, 32, 32, 64, [WG, R32], k=1),          # Cin 32, ksplit 16
    _row("w_gen_reduce32_long", "wgrad", 2, 64, 64, 64, 64, [WG, R32], k=1),           # ksplit 64 > 16
    _row("w_gen_reduce16_long", "wgrad", 4, 64, 64, 64, 64, [WG, R16], k=1),           # ksplit 128 > 64
    _row("w_gen_reduce16_cin16", "wgrad", 2, 16, 16, 16, 32, [WG, R16], k=1),          # Cin 16 < 32
    _row("w_accumulate_halo", "wgrad", 2, 16, 16, 64, 64, [W1, R64], accumulate=True),
    _row("w_accumulate_generic", "wgrad", 2, 16, 16, 64, 64, [WG, R64], k=1, accumulate=True),
]


@pytest.mark.parametrize("c", WGRAD_ROWS)
def test_wgrad_variant_bit_exact(c):
    from rbunet import _lib
    from rbunet._lib import WgradArgs, call, stream_ptr
    dev = _dev()
    op, N, H, W, cin, cout, k, dil = c["op"], c["N"], c["H"], c["W"], c["cin"], c["cout"], c["k"], c["dil"]
    x = R.int_operand((N, cin, H, W), 40)
    if op == "wgrad":
        dy = R.int_operand((N, cout, H, W), 41)
        ref, smax = R.exact(lambda a, b: R.conv_wgrad(a, b, k, dil), x.to(dev), dy.to(dev))
        a, b, taps, gather = _act(dy), _act(x), k * k, 0
    else:   # ConvTranspose weight gradient: A = x, B = dout gathered from the second half of a concat buffer
        dout = R.int_operand((N, cout, 2 * H, 2 * W), 42)
        ref, smax = R.exact(R.convT_wgrad, x.to(dev), dout.to(dev))
        a, b, taps, gather = _act(x), _act(dout, off=cout), 4, 1
    guard = 64
    buf = torch.full((ref.numel() + 2 * guard,), SENT, dtype=torch.float32, device=dev)
    out = buf[guard:guard + ref.numel()]
    if c.get("accumulate"):
        prefill = R.int_operand(tuple(ref.shape), 43, vmax=1000).to(dev)
        out.copy_(prefill.flatten())
        ref = prefill + ref
        assert float(ref.abs().max()) < 2 ** 24
    want = R.expected_fp32(ref)

    args = WgradArgs()
    args.N, args.H, args.W = N, H, W
    args.a, args.a_ld, args.Ca = a.ptr, a.ld, a.C
    args.b, args.b_ld, args.Cb = b.ptr, b.ld, b.C
    args.taps, args.dil, args.gather = taps, dil if taps == 9 else 0, gather
    args.out, args.accumulate = out.data_ptr(), int(bool(c.get("accumulate")))
    nbytes = int(_lib.lib().rbu_wgrad_workspace_bytes(ctypes.byref(args)))
    ws = torch.full((nbytes // 4 + 64,), SENT, dtype=torch.float32, device=dev)
    seen = _launch(lambda: call("rbu_wgrad_gemm", ctypes.byref(args), ctypes.c_void_p(ws.data_ptr()), ws.numel() * 4,
                                stream_ptr()))
    assert seen == c["kernels"], f"launched {sorted(seen)}, expected {sorted(c['kernels'])}"
    host = buf.cpu()
    assert bool((host[:guard] == SENT).all()) and bool((host[-guard:] == SENT).all()), "guard region overwritten"
    compared = R.assert_bits_equal(host[guard:guard + ref.numel()].view(ref.shape), want, "weight gradient",
                                   dims=("O", "I", "KH", "KW"))
    print(f"\n[conv_exact] {c['id']:32s} kernels={sorted(seen)} max_S={smax:.0f} compared={compared}")


def test_relu_must_name_whole_8_channel_groups():
    """relu = 12 would rectify channels 0-15 (the epilogue works on 8-channel groups): rbu_conv_gemm refuses it, and a
    relu beyond Ncols; relu = 16 rectifies exactly channels 0-15."""
    from rbunet import ops
    dev = _dev()
    N, H, W, C = 1, 16, 16, 64
    x, w = R.int_operand((N, C, H, W), 50), R.int_operand((C, C, 1, 1), 51)
    xv, wp = _act(x), ops.pack_weight(w.to(dev).float().contiguous(), 0)
    for bad in (12, 4, C + 8, -8):
        y = _out(N, H, W, C)
        with pytest.raises(RuntimeError, match="relu"):
            ops.conv_gemm(N, H, W, [(xv, wp, 1, 0, False)], C, y, relu=bad)
        torch.cuda.synchronize()
        _read(y, 0)                                          # nothing was written
    y = _out(N, H, W, C)
    ops.conv_gemm(N, H, W, [(xv, wp, 1, 0, False)], C, y, relu=16)
    acc = R.conv_fwd(x, w)
    assert bool((acc[:, :16] < 0).any()) and bool((acc[:, 16:] < 0).any())
    R.assert_bits_equal(_read(y, N), R.expected_bf16(R.epilogue(acc, relu=16)))
    # the scatter form bounds relu by Cout, not by the 4 * Cout GEMM columns
    xt, wt = R.int_operand((N, 64, 8, 8), 52), R.int_operand((64, 32, 2, 2), 53)
    yt = _out(N, 16, 16, 32)
    with pytest.raises(RuntimeError, match="relu"):
        ops.conv_gemm(N, 8, 8, [(_act(xt), ops.pack_weight(wt.to(dev).float().contiguous(), 2), 1, 0, False)], 128, yt,
                      scatter=True, Cout=32, relu=64)
