"""Numerics of the tensor-core split (csrc/tc_common.cuh), modelled in numpy with the kernels' roundings and summed in fp64.

Per 8 k the kernels compute  x.w ~= x_hi.w_hi + bf16(x_hi).bf16(w_lo) + bf16(x_lo).bf16(w_hi), with hi = v rounded to nearest
TF32 (cvt.rna.tf32.f32) and lo = v - hi.  Per product the error is below 1.04 * 2^-17 |x||w|: each cross term is at most
(1 + 2^-11) 2^-11 |x||w| and carries the rounding of both operands to bf16 (2^-8 each); the dropped lo.lo is below 2^-22.
The former split (hi = v & 0xffffe000, three tf32 products, lo truncated to TF32 by the MMA) is kept as a comparison."""
import numpy as np

K = 4609                                       # VGG16 conv5: 9 x 512 taps + bias
BOUND = (2.0 ** -7 + 2.0 ** -16) * (1 + 2.0 ** -11) * 2.0 ** -10 + 2.0 ** -22


def _bits(v):
    return np.ascontiguousarray(v, dtype=np.float32).view(np.uint32).astype(np.uint64)


def tf32_rna(v):
    """cvt.rna.tf32.f32 on finite values: round the 13 dropped bits half away from zero (sign-magnitude)."""
    return (((_bits(v) + 0x1000) & 0xFFFFE000).astype(np.uint32)).view(np.float32)


def tf32_trunc(v):
    return ((_bits(v) & 0xFFFFE000).astype(np.uint32)).view(np.float32)


def bf16_rn(v):
    """cvt.rn.bf16.f32 (round to nearest even), returned as the fp32 value it represents."""
    u = _bits(v)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return (r.astype(np.uint32)).view(np.float32)


def split(v):
    hi = tf32_rna(v)
    return hi, (v - hi).astype(np.float32)      # exact in fp32


def products_new(x, w):
    (xh, xl) = split(x)
    (wh, wl) = split(w)
    f = lambda a: bf16_rn(a).astype(np.float64)
    return xh.astype(np.float64) * wh + f(xh) * f(wl) + f(xl) * f(wh)


def products_old(x, w):
    xh, wh = tf32_trunc(x), tf32_trunc(w)
    xl, wl = (x - xh).astype(np.float32), (w - wh).astype(np.float32)
    d = lambda a: a.astype(np.float64)
    return d(xh) * d(wh) + d(tf32_trunc(xl)) * d(wh) + d(xh) * d(tf32_trunc(wl))


def products_fp16_corr(x, w):
    """The same split with the correction operands in FP16 instead of BF16."""
    (xh, xl) = split(x)
    (wh, wl) = split(w)
    with np.errstate(over='ignore', invalid='ignore'):
        f = lambda a: a.astype(np.float16).astype(np.float64)
        return xh.astype(np.float64) * wh + f(xh) * f(wl) + f(xl) * f(wh)


def _he(rs, n_dots):
    x = np.abs(rs.randn(n_dots, K)).astype(np.float32)                         # post-ReLU activations
    lim = np.sqrt(6.0 / K)
    w = rs.uniform(-lim, lim, (n_dots, K)).astype(np.float32)                  # He-uniform weights
    return x, w


def _wide(rs, n_dots):
    x = (10.0 ** rs.uniform(-30, 30, (n_dots, K)) * rs.choice([-1, 1], (n_dots, K))).astype(np.float32)
    w = (10.0 ** rs.uniform(-30, 30, (n_dots, K)) * rs.choice([-1, 1], (n_dots, K))).astype(np.float32)
    return x, w


def _rel_err(prod, x, w):
    exact = x.astype(np.float64) * w.astype(np.float64)
    return np.abs(prod - exact) / (np.abs(x.astype(np.float64)) * np.abs(w.astype(np.float64)))


def test_rounding_models_match_their_definitions():
    v = np.array([1.0, 1 + 2.0 ** -11, 1 + 3 * 2.0 ** -11, -(1 + 2.0 ** -11), 1 + 2.0 ** -8, 1 + 3 * 2.0 ** -8], dtype=np.float32)
    assert np.array_equal(tf32_rna(v), np.float32([1.0, 1 + 2.0 ** -10, 1 + 2 * 2.0 ** -10, -(1 + 2.0 ** -10), 1 + 2.0 ** -8, 1 + 3 * 2.0 ** -8]))
    assert np.array_equal(bf16_rn(v[[0, 4, 5]]), np.float32([1.0, 1.0, 1 + 2.0 ** -6]))       # ties to even
    (hi, lo) = split(v)
    assert np.all(hi.astype(np.float64) + lo == v.astype(np.float64))
    assert np.all(np.abs(lo) <= 2.0 ** -11 * np.abs(v))


def test_per_product_bound_he_scaled():
    rs = np.random.RandomState(0)
    (x, w) = _he(rs, 64)
    assert _rel_err(products_new(x, w), x, w).max() <= BOUND
    assert _rel_err(products_old(x, w), x, w).max() <= 3 * 2.0 ** -20


def test_per_product_bound_wide_range():
    rs = np.random.RandomState(1)
    (x, w) = _wide(rs, 64)
    assert _rel_err(products_new(x, w), x, w).max() <= BOUND


def test_dot_products_k4609_within_bound():
    """Dot products of VGG16 conv5 length: |sum(new) - x.w| <= BOUND * sum|x||w| (sums in fp64), He-scaled and wide range."""
    rs = np.random.RandomState(2)
    for (x, w) in (_he(rs, 500), _wide(rs, 200)):
        exact = np.sum(x.astype(np.float64) * w.astype(np.float64), axis=1)
        scale = np.sum(np.abs(x.astype(np.float64) * w.astype(np.float64)), axis=1)
        err = np.abs(products_new(x, w).sum(axis=1) - exact)
        assert np.all(err <= BOUND * scale)
    # He-scaled: the worst error over max|y| stays far below the parity bar (rtol 1e-4)
    (x, w) = _he(rs, 500)
    y = np.sum(x.astype(np.float64) * w.astype(np.float64), axis=1)
    assert np.abs(products_new(x, w).sum(axis=1) - y).max() / np.abs(y).max() < 1e-5


def test_fp16_corrections_fail_the_wide_range():
    """FP16 correction operands underflow (x_lo ~ 2^-11 x below FP16's normal range) or overflow (|x| > 65504)."""
    rs = np.random.RandomState(3)
    (x, w) = _wide(rs, 16)
    with np.errstate(invalid='ignore'):
        err = _rel_err(products_fp16_corr(x, w), x, w)
    assert not np.all(err <= BOUND)
    assert np.mean(~(err <= BOUND)) > 0.5
