"""Exact-arithmetic references for the convolution and weight-gradient kernels (conv_gemm.cu, conv_halo.cu,
wgrad_gemm.cu, wgrad_halo.cu).

The operands are small integers, which bf16 stores exactly, so every product is exact.  If, for every output element,
S = sum |a*b| over its whole reduction is below 2^22, every partial sum in any order is an integer of magnitude < 2^22:
fp32 holds it exactly and no alignment inside the tensor-core adder can drop an integer bit.  The kernel's fp32
accumulator then has exactly one correct value whatever the tiling, split-K, CTA pairing or accumulation order, and a
test can demand bit equality.  S is computed by running the same reference on the absolute values of the operands, and
the bound is asserted, not assumed.

The epilogue keeps this property: `scale` values have at most two significant bits and `bias` values are multiples of
1/4, and `epilogue()` asserts that scale*acc, + bias and + addend are each exactly representable in fp32 (so the result
is the same whether or not the compiler contracts the multiply-add into an FMA).  The only rounding left is the final
fp32 -> bf16 round-to-nearest-even, which `expected_bf16()` reproduces with torch's CPU conversion.

The references are torch float64 convolutions, on whatever device the operands live.  cuDNN is switched off for them:
its transform-based algorithms (FFT, Winograd) are not exact, while the im2col + GEMM fallbacks are, and every integer
result is additionally checked to be an integer.
"""
import contextlib

import torch
import torch.nn.functional as F

EXACT_ACC = 2 ** 22      # bound on S = sum |a*b| of one accumulator (fp32 accumulation stays exact below it)
EXACT_STATS = 2 ** 24    # bound on sum |y| and sum y^2 per statistics column (fp32 partial sums stay exact below it)

# scales with at most two significant bits: scale * integer keeps at most two more bits than the integer
SCALES = (1.0, -1.0, 2.0, -2.0, 0.5, -0.5, 0.75, -0.75, 1.5, -1.5, 0.25, 3.0)


def int_operand(shape, seed, vmax=8, zero_frac=0.25):
    """Seeded integers uniform in [-vmax, vmax] with an extra fraction `zero_frac` of zeros, as float64 on the CPU."""
    g = torch.Generator().manual_seed(seed)
    v = torch.randint(-vmax, vmax + 1, tuple(shape), generator=g, dtype=torch.int64)
    if zero_frac:
        v[torch.rand(tuple(shape), generator=g) < zero_frac] = 0
    return v.double()


def dyadic_scale(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.tensor(SCALES, dtype=torch.float64)[torch.randint(0, len(SCALES), (n,), generator=g)]


def dyadic_bias(n, seed, qmax=400):
    """Multiples of 1/4 in [-qmax/4, qmax/4]."""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(-qmax, qmax + 1, (n,), generator=g, dtype=torch.int64).double() / 4


@contextlib.contextmanager
def _exact_backend():
    with torch.backends.cudnn.flags(enabled=False):
        yield


def _integral(t):
    assert torch.equal(t, t.round()), "fp64 reference of integer operands is not integral: the reference is not exact"
    return t


# ------------------------------------------------------------------ fp64 references (NCHW, any device)
def conv_fwd(x, w, dil=1):
    """Conv2d forward, stride 1, padding = dil * (k // 2): x [N,Cin,H,W], w [Cout,Cin,k,k]."""
    with _exact_backend():
        return F.conv2d(x, w, padding=dil * (w.shape[-1] // 2), dilation=dil)


def rot_weight(w):
    """The data gradient as a forward convolution: [Cout,Cin,k,k] -> [Cin,Cout,k,k] with the taps rotated by 180
    degrees (what pack mode 1 builds)."""
    return w.transpose(0, 1).flip(2, 3)


def conv_dgrad(dy, w, dil=1):
    """Conv2d data gradient: dy [N,Cout,H,W], w [Cout,Cin,k,k] -> dx [N,Cin,H,W]."""
    return conv_fwd(dy, rot_weight(w), dil)


def convT_fwd(x, w):
    """ConvTranspose2d(2, stride 2) forward without bias: x [N,Cin,H,W], w [Cin,Cout,2,2] -> [N,Cout,2H,2W]."""
    with _exact_backend():
        return F.conv_transpose2d(x, w, stride=2)


def convT_dgrad(dout, w):
    """ConvTranspose2d(2, stride 2) data gradient: dout [N,Cout,2H,2W], w [Cin,Cout,2,2] -> [N,Cin,H,W]."""
    with _exact_backend():
        return F.conv2d(dout, w, stride=2)


def conv_wgrad(x, dy, ksz, dil=1):
    """Conv2d weight gradient: x [N,Cin,H,W], dy [N,Cout,H,W] -> [Cout,Cin,k,k]."""
    with _exact_backend():
        return torch.nn.grad.conv2d_weight(x, (dy.shape[1], x.shape[1], ksz, ksz), dy, padding=dil * (ksz // 2),
                                           dilation=dil)


def convT_wgrad(x, dout):
    """ConvTranspose2d(2, stride 2) weight gradient: x [N,Cin,H,W], dout [N,Cout,2H,2W] -> [Cin,Cout,2,2]."""
    n, co, h2, w2 = dout.shape
    return torch.einsum("nchw,ndhiwj->cdij", x, dout.reshape(n, co, h2 // 2, 2, w2 // 2, 2))


def exact(fn, *operands, bound=EXACT_ACC):
    """(fn(*operands), S) for a reference `fn` that is linear in each operand: S = fn on the absolute values is the
    sum of |products| of every output element.  Asserts that the result is integral and max S < bound."""
    ref = _integral(fn(*operands))
    s = fn(*(o.abs() for o in operands))
    smax = float(s.max())
    assert smax < bound, f"accumulation bound violated: max sum |a*b| = {smax:.0f} >= {bound}"
    return ref, smax


# ------------------------------------------------------------------ epilogue and expected bits
def _fp32_exact(t, what):
    bad = t.float().double() != t
    assert not bool(bad.any()), f"epilogue step '{what}' is not exact in fp32 (first value {t[bad][0].item()!r})"
    return t


def epilogue(acc, scale=None, bias=None, addend=None, relu=0):
    """acc [N,C,...] fp64 -> relu_prefix(scale*acc + bias + addend) exactly, asserting that every step the kernel rounds
    to fp32 is exact; `relu` rectifies channels [0, relu)."""
    shape = (1, -1) + (1,) * (acc.dim() - 2)
    y = _fp32_exact(acc, "accumulator")
    if scale is not None:
        y = _fp32_exact(y * scale.view(shape), "scale")
    if bias is not None:
        y = _fp32_exact(y + bias.view(shape), "bias")
    if addend is not None:
        y = _fp32_exact(y + addend, "addend")
    if relu:
        y = y.clone()
        y[:, :relu] = y[:, :relu].clamp_min(0)
    return y


def expected_bf16(t):
    """Exact fp64 -> the bf16 the kernel stores: fp32 (exact here) then round-to-nearest-even (torch's CPU cast)."""
    return t.cpu().float().to(torch.bfloat16)


def expected_fp32(t):
    return t.cpu().float()


def _canonical(t):
    # the sign of an exact zero depends on the summation order (x + -x = +0, -0 + -0 = -0): not a property of the result
    t = t.detach().cpu().contiguous()
    return torch.where(t == 0, torch.zeros_like(t), t)


def assert_bits_equal(got, want, what="output", dims="NCHW"):
    """Bitwise equality (zeros of either sign are equal).  On failure, reports how many elements differ and the first
    one by its coordinates in `dims`."""
    got, want = _canonical(got), _canonical(want)
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, want.dtype, got.shape, want.shape)
    itype = {torch.bfloat16: torch.int16, torch.float32: torch.int32, torch.float64: torch.int64}[got.dtype]
    diff = got.view(itype) != want.view(itype)
    n = int(diff.sum())
    if n:
        first = tuple(int(i) for i in diff.nonzero()[0])
        coords = ", ".join(f"{d}={i}" for d, i in zip(dims, first))
        raise AssertionError(f"{what}: {n} of {got.numel()} elements differ; first at ({coords}): "
                             f"got {got[first].item()!r}, want {want[first].item()!r}")
    return got.numel()
