"""The TF32 + BF16 split of the tensor-core kernels on the GPU: kn_pg_tc_split's planes bit for bit against the numpy model of
tests/test_split_numerics.py, and the two tcgen05 kernels (pg_tc at G = 256, pg_tile_tc at G = 64) and the split-K fc path on
inputs spanning 1e-20 .. 1e20 against an fp64 product of the compiled matrix: within the split's bound plus fp32 accumulation,
no inf or NaN."""
import numpy as np
import pytest
import torch

from tests.test_split_numerics import BOUND, bf16_rn, tf32_rna

pytestmark = pytest.mark.gpu


def _model_planes(v):
    hi = tf32_rna(v)
    lo = (v - hi).astype(np.float32)
    b = lambda a: (bf16_rn(a).view(np.uint32) >> 16).reshape(-1, 4, 2)
    pair = lambda a: b(a)[:, :, 0] | (b(a)[:, :, 1] << 16)                     # lower half: the lower k
    corr = np.concatenate([pair(lo), pair(hi)], axis=1).reshape(-1)             # per 8 k: w_lo pairs, then w_hi pairs
    return hi.view(np.uint32), corr.astype(np.uint32)


def test_split_planes_bit_equal_to_model():
    from keynet_b200 import _native
    from keynet_b200._native import check, ptr, stream_ptr
    rs = np.random.RandomState(0)
    n = 1 << 16
    v = np.concatenate([rs.uniform(-0.05, 0.05, n // 2),
                        10.0 ** rs.uniform(-30, 30, n // 2) * rs.choice([-1, 1], n // 2)]).astype(np.float32)
    v[:8] = np.float32([1 + 2.0 ** -11, -(1 + 2.0 ** -11), 1 + 2.0 ** -8 + 2.0 ** -11, 0.0, -0.0, 1.0, 2.0 ** -126, 3e38])
    vd = torch.from_numpy(v).cuda()
    (hi, corr) = (torch.empty_like(vd), torch.empty_like(vd))
    check(_native.lib().kn_pg_tc_split(ptr(vd), n, ptr(hi), ptr(corr), stream_ptr()))
    torch.cuda.synchronize()
    (hi_m, corr_m) = _model_planes(v)
    assert np.array_equal(hi.cpu().numpy().view(np.uint32), hi_m)
    assert np.array_equal(corr.cpu().numpy().view(np.uint32), corr_m)


def _wide_inputs(rs, K, N):
    X = (10.0 ** rs.uniform(-20, 20, (K, N)) * rs.choice([-1, 1], (K, N))).astype(np.float32)
    X[-1] = 1                                                                   # homogeneous coordinate (bias)
    return X


def _check_rows(W, X, y, n_rows, rs):
    """Sampled rows of y against the fp64 product of W's CSR: |y - y64| <= (BOUND + 2 (k / 8 + 1) 2^-23) sum|w||x| per row --
    the split's bound per product plus one fp32 rounding per MMA accumulation (one tf32 and one bf16 MMA per 8 k)."""
    assert np.all(np.isfinite(y))
    (ip, ix, dt) = W.csr_arrays()
    worst = 0.0
    for r in rs.choice(len(ip) - 1, n_rows, replace=False):
        (idx, w) = (ix[ip[r]:ip[r + 1]], dt[ip[r]:ip[r + 1]].astype(np.float64))
        xs = X[idx].astype(np.float64)
        y64 = w @ xs
        scale = np.abs(w) @ np.abs(xs)
        tol = (BOUND + 2 * (len(idx) / 8 + 1) * 2.0 ** -23) * scale
        err = np.abs(y[r] - y64)
        assert np.all(err <= tol), (r, float((err / scale).max()))
        worst = max(worst, float((err / scale).max()))
    return worst


@pytest.mark.parametrize('shape', [(256, 256, 8), (64, 64, 16)])
def test_conv_layers_wide_range_within_bound(shape):
    """conv3_2-shaped (256 -> 256 channels, K = 2305: pg_tc) and conv1_2-shaped (64 -> 64, pg_tile_tc) 3x3 layers."""
    from keynet_b200 import sparse
    from keynet_b200.sparse import MonomialKey
    (C, M, U) = shape
    rs = np.random.RandomState(C)
    lim = np.sqrt(6.0 / (9 * C))
    f = rs.uniform(-lim, lim, (M, C, 3, 3)).astype(np.float32)
    b = rs.uniform(-0.1, 0.1, M).astype(np.float32)
    K = C * U * U + 1
    perm = np.concatenate([rs.permutation(K - 1), [K - 1]])
    W = sparse.keyed_toeplitz_conv2d((C, U, U), f, b, 1, None, MonomialKey(perm))
    cls = W._pg.classes
    if M == 256:
        assert any(c['tc'] is not None and c.get('tile') is None for c in cls)
    else:
        assert any(c.get('tile') is not None for c in cls) and sparse.tiles_enabled()
    X = _wide_inputs(rs, K, 256)
    y = sparse.spmm(W, torch.from_numpy(X).cuda()).cpu().numpy()
    _check_rows(W, X, y, 256, rs)


def test_fc_split_k_wide_range_within_bound():
    """A dense 4096 -> 512 layer: one group holding every row, run as K slices plus the split-K reduction."""
    from keynet_b200 import sparse
    from keynet_b200.sparse import MonomialKey
    rs = np.random.RandomState(7)
    (n_in, n_out) = (4096, 512)
    lim = np.sqrt(6.0 / n_in)
    w = rs.uniform(-lim, lim, (n_out, n_in)).astype(np.float32)
    b = rs.uniform(-0.1, 0.1, n_out).astype(np.float32)
    perm = np.concatenate([rs.permutation(n_in), [n_in]])
    W = sparse.keyed_linear(w, b, None, MonomialKey(perm))
    assert W._pg is not None and any(c.get('splitk') is not None for c in W._pg.classes)
    X = _wide_inputs(rs, n_in + 1, 256)
    y = sparse.spmm(W, torch.from_numpy(X).cuda()).cpu().numpy()
    _check_rows(W, X, y, 128, rs)
