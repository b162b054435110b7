"""CPU checks of tests/conv_exact_ref.py: its fp64 references against brute-force loops, its operand bounds, and that its
comparator catches a one-ulp change and a single dropped tap."""
import itertools

import pytest
import torch

import conv_exact_ref as R


def _brute_conv(x, w, dil):
    N, Cin, H, W = x.shape
    Cout, _, k, _ = w.shape
    y = torch.zeros((N, Cout, H, W), dtype=torch.float64)
    for kh, kw, h, ww in itertools.product(range(k), range(k), range(H), range(W)):
        hi, wi = h + (kh - k // 2) * dil, ww + (kw - k // 2) * dil
        if 0 <= hi < H and 0 <= wi < W:
            y[:, :, h, ww] += x[:, :, hi, wi] @ w[:, :, kh, kw].T
    return y


def _brute_dgrad(dy, w, dil):
    """The adjoint of _brute_conv, scattered term by term."""
    N, Cout, H, W = dy.shape
    _, Cin, k, _ = w.shape
    dx = torch.zeros((N, Cin, H, W), dtype=torch.float64)
    for kh, kw, h, ww in itertools.product(range(k), range(k), range(H), range(W)):
        hi, wi = h + (kh - k // 2) * dil, ww + (kw - k // 2) * dil
        if 0 <= hi < H and 0 <= wi < W:
            dx[:, :, hi, wi] += dy[:, :, h, ww] @ w[:, :, kh, kw]
    return dx


def _brute_wgrad(x, dy, k, dil):
    N, Cin, H, W = x.shape
    dw = torch.zeros((dy.shape[1], Cin, k, k), dtype=torch.float64)
    for kh, kw, h, ww in itertools.product(range(k), range(k), range(H), range(W)):
        hi, wi = h + (kh - k // 2) * dil, ww + (kw - k // 2) * dil
        if 0 <= hi < H and 0 <= wi < W:
            dw[:, :, kh, kw] += dy[:, :, h, ww].T @ x[:, :, hi, wi]
    return dw


def _brute_convT(x, w):
    N, Cin, H, W = x.shape
    y = torch.zeros((N, w.shape[1], 2 * H, 2 * W), dtype=torch.float64)
    for i, j, h, ww in itertools.product(range(2), range(2), range(H), range(W)):
        y[:, :, 2 * h + i, 2 * ww + j] = x[:, :, h, ww] @ w[:, :, i, j]
    return y


def _brute_convT_dgrad(dout, w):
    N, Cout, H2, W2 = dout.shape
    dx = torch.zeros((N, w.shape[0], H2 // 2, W2 // 2), dtype=torch.float64)
    for i, j, h, ww in itertools.product(range(2), range(2), range(H2 // 2), range(W2 // 2)):
        dx[:, :, h, ww] += dout[:, :, 2 * h + i, 2 * ww + j] @ w[:, :, i, j].T
    return dx


def _brute_convT_wgrad(x, dout):
    N, Cin, H, W = x.shape
    dw = torch.zeros((Cin, dout.shape[1], 2, 2), dtype=torch.float64)
    for i, j, h, ww in itertools.product(range(2), range(2), range(H), range(W)):
        dw[:, :, i, j] += x[:, :, h, ww].T @ dout[:, :, 2 * h + i, 2 * ww + j]
    return dw


@pytest.mark.parametrize("k,dil", [(3, 1), (3, 2), (3, 4), (1, 1)])
def test_conv_references_match_brute_force(k, dil):
    x = R.int_operand((2, 5, 7, 6), 1)
    w = R.int_operand((4, 5, k, k), 2)
    dy = R.int_operand((2, 4, 7, 6), 3)
    assert torch.equal(R.conv_fwd(x, w, dil), _brute_conv(x, w, dil))
    assert torch.equal(R.conv_dgrad(dy, w, dil), _brute_dgrad(dy, w, dil))
    assert torch.equal(R.conv_wgrad(x, dy, k, dil), _brute_wgrad(x, dy, k, dil))
    # the data gradient reference is the adjoint of the forward one: <conv(x), dy> == <x, dgrad(dy)>
    assert torch.equal((R.conv_fwd(x, w, dil) * dy).sum(), (x * R.conv_dgrad(dy, w, dil)).sum())


def test_conv_transpose_references_match_brute_force():
    x = R.int_operand((2, 5, 3, 4), 4)
    w = R.int_operand((5, 3, 2, 2), 5)
    dout = R.int_operand((2, 3, 6, 8), 6)
    assert torch.equal(R.convT_fwd(x, w), _brute_convT(x, w))
    assert torch.equal(R.convT_dgrad(dout, w), _brute_convT_dgrad(dout, w))
    assert torch.equal(R.convT_wgrad(x, dout), _brute_convT_wgrad(x, dout))


def test_generator_bounds_and_exactness():
    v = R.int_operand((64, 64, 3, 3), 7)
    assert v.abs().max() <= 8 and bool((v == v.round()).all()) and (v == 0).float().mean() > 0.25
    assert torch.equal(v.float().to(torch.bfloat16).double(), v)             # bf16 holds the operands exactly
    assert R.int_operand((3, 5), 8).equal(R.int_operand((3, 5), 8))          # seeded
    s, b = R.dyadic_scale(1000, 9), R.dyadic_bias(1000, 10)
    assert torch.equal(s.float().double(), s) and torch.equal(b * 4, (b * 4).round())
    # the accumulation bound is asserted: a 1024-channel 3x3 convolution of [-8, 8] operands stays below 2^22 ...
    x, w = R.int_operand((1, 1024, 4, 4), 11), R.int_operand((8, 1024, 3, 3), 12)
    _, smax = R.exact(R.conv_fwd, x, w)
    assert 2 ** 16 < smax < R.EXACT_ACC
    # ... and one that crosses it is refused
    with pytest.raises(AssertionError, match="accumulation bound"):
        R.exact(R.conv_fwd, x * 64, w)
    # the epilogue refuses a step that fp32 would round
    with pytest.raises(AssertionError, match="not exact in fp32"):
        R.epilogue(torch.full((1, 1, 1, 1), 2.0 ** 23 + 1, dtype=torch.float64),
                   scale=torch.tensor([1.5], dtype=torch.float64))


def test_epilogue_is_exact_and_rounds_like_the_kernel():
    acc = R.int_operand((2, 16, 5, 5), 13, vmax=4000)
    scale, bias = R.dyadic_scale(16, 14), R.dyadic_bias(16, 15)
    add = R.int_operand((2, 16, 5, 5), 16)
    y = R.epilogue(acc, scale, bias, add, relu=8)
    ref = acc * scale.view(1, -1, 1, 1) + bias.view(1, -1, 1, 1) + add
    ref[:, :8] = ref[:, :8].clamp_min(0)
    assert torch.equal(y, ref)
    # fp32 arithmetic in the kernel's order gives the same fp32 values (no rounding before the bf16 store)
    f = acc.float() * scale.float().view(1, -1, 1, 1) + bias.float().view(1, -1, 1, 1) + add.float()
    f[:, :8] = f[:, :8].clamp_min(0)
    assert torch.equal(f.double(), y)
    e = R.expected_bf16(y)
    assert bool((y.abs() > 256).any()) and not torch.equal(e.double(), y)    # the bf16 rounding is exercised


def test_comparator_catches_one_ulp():
    x = R.int_operand((2, 64, 6, 5), 17)
    w = R.int_operand((32, 64, 3, 3), 18)
    want = R.expected_bf16(R.conv_fwd(x, w))
    assert R.assert_bits_equal(want.clone(), want) == want.numel()
    for idx in [(0, 0, 0, 0), (1, 31, 5, 4), (1, 7, 2, 3)]:
        got = want.clone()
        bits = got.view(torch.int16)
        bits[idx] += 1                                                       # one bf16 ulp
        with pytest.raises(AssertionError, match=r"1 of \d+ elements differ"):
            R.assert_bits_equal(got, want)
    # one ulp of an fp32 weight gradient
    g = R.expected_fp32(R.conv_wgrad(x, R.int_operand((2, 32, 6, 5), 19), 3))
    got = g.clone()
    got.view(torch.int32)[3, 5, 1, 2] += 1
    with pytest.raises(AssertionError, match=r"first at \(N=3, C=5, H=1, W=2\)"):
        R.assert_bits_equal(got, g)


def test_comparator_catches_a_dropped_tap():
    """The result with one tap of one border pixel left out (what a halo or ragged-edge bug looks like) must fail."""
    x = R.int_operand((2, 64, 6, 5), 20)
    w = R.int_operand((32, 64, 3, 3), 21)
    exact = R.conv_fwd(x, w)
    want = R.expected_bf16(exact)
    n, co, h, ww, kh, kw = 1, 9, 0, 4, 1, 0                                   # top-right border pixel, left tap
    contrib = float((x[n, :, h + kh - 1, ww + kw - 1] * w[co, :, kh, kw]).sum())
    assert contrib != 0
    wrong = exact.clone()
    wrong[n, co, h, ww] -= contrib
    got = R.expected_bf16(wrong)
    assert got[n, co, h, ww] != want[n, co, h, ww]                          # the change survives the bf16 rounding
    with pytest.raises(AssertionError, match=r"first at \(N=1, C=9, H=0, W=4\)"):
        R.assert_bits_equal(got, want)


def test_zero_sign_is_not_a_difference():
    a = torch.tensor([0.0, -0.0, 1.0]).to(torch.bfloat16)
    b = torch.tensor([-0.0, 0.0, 1.0]).to(torch.bfloat16)
    assert R.assert_bits_equal(a, b, dims="C") == 3
