"""Sparse algebra of the keyed-layer path on B200: device-resident CSR matrices, key matrices,
Toeplitz construction and key compile.  Mirrors the public names of the reference's
keynet/sparse.py; every heavy operation is a hand-written sm_100a kernel behind the C ABI
(include/keynet_b200.h).  No scipy / torch.sparse / CPU fallback on the product path.

Representation choices (B200-first, not a port):
  * key matrices are never materialised as sparse matrices on the host: a permutation and/or
    diagonal-gain key is a `MonomialKey` = (perm, scale) with A[r, perm[r]] = scale[r]; composing
    keys is O(n) integer indexing + one fp32 multiply per row, done with the reference's fp32
    rounding so results match its scipy SpGEMM chain bit-for-bit (system.py:467-468).
  * layer matrices live on the GPU as CSR (int64 indptr, int32 indices, fp32 data) and are built
    there: Toeplitz rows are written in closed form (csrc/toeplitz.cu), keys are folded in by
    csrc/keycompile.cu.
"""
import ctypes
import os
import warnings

import numpy as np
import torch

from . import _native
from ._native import kn_conv2d_desc, ptr, stream_ptr, check
from .util import blockview


# =============================================================================================
# Key matrices
# =============================================================================================
class MonomialKey(object):
    """n x n matrix with exactly one stored entry per row: A[r, perm[r]] = scale[r].

    Covers the reference's identity / permutation / hierarchical block permutation / memory-order
    / diagonal gain keys and all their products (keynet/sparse.py:53-84,272-285,318-321)."""

    def __init__(self, perm, scale=None, bias=None):
        """bias (optional, homogeneous keys only): extra entries A[r, n-1] = bias[r] for r < n-1 -- the affine
        photometric keys [[D, b],[0, 1]] (keynet/sparse.py:99-119).  Keys with a bias column are closed under
        products, so the whole photometric key family stays O(n) on the host."""
        self._perm = np.ascontiguousarray(perm, dtype=np.int64)
        n = len(self._perm)
        self._scale = None if scale is None else np.ascontiguousarray(scale, dtype=np.float32)       # None: all ones (materialised on demand)
        assert self._scale is None or self._scale.shape == (n,)
        self.bias = None
        if bias is not None:
            b = np.ascontiguousarray(bias, dtype=np.float32).reshape(-1)
            assert b.shape == (n,) and b[-1] == 0 and self._perm[-1] == n - 1, 'bias needs a homogeneous key (last row e_last)'
            self.bias = b
        self._n = n
        self._unpermuted = None          # structure tests are evaluated once: keys are immutable once built
        self._unscaled = True if scale is None else None
        self.shape = (n, n)
        self.dtype = np.float32
        self.ndim = 2

    @classmethod
    def identity(cls, n):
        """The n x n identity without its index / value arrays (built on first use): most factors of keygen's
        A = C^-1 . p . g . P . G . C are identities, and for VGG16 every one of them used to cost two 3.2 M element arrays."""
        K = cls.__new__(cls)
        (K._perm, K._scale, K.bias, K._n, K._unpermuted, K._unscaled) = (None, None, None, int(n), True, True)
        (K.shape, K.dtype, K.ndim) = ((int(n), int(n)), np.float32, 2)
        return K

    @property
    def perm(self):
        if self._perm is None:
            self._perm = np.arange(self._n, dtype=np.int64)
        return self._perm

    @property
    def scale(self):
        if self._scale is None:
            self._scale = np.ones(self._n, dtype=np.float32)
        return self._scale

    def has_bias(self):
        return self.bias is not None

    def __repr__(self):
        return '<keynet_b200.MonomialKey: n=%d, permuted=%s, scaled=%s>' % (self.shape[0], not self.is_unpermuted(), not self.is_unscaled())

    # -- structure tests
    def is_unpermuted(self):
        if self._unpermuted is None:
            self._unpermuted = bool(np.array_equal(self._perm, np.arange(self._n)))
        return self._unpermuted

    def is_unscaled(self):
        if self._unscaled is None:
            self._unscaled = bool(np.all(self._scale == np.float32(1.0)))
        return self._unscaled

    def is_identity(self):
        return self.is_unpermuted() and self.is_unscaled() and self.bias is None

    _identity = is_identity

    @property
    def nnz(self):
        return self._n

    # -- algebra (fp32 products rounded once, like scipy's csr_matmat on single-entry rows)
    def dot(self, other):
        """self . other.  other: MonomialKey -> MonomialKey; SparseMatrix -> SparseMatrix (row gather + scale)."""
        if isinstance(other, MonomialKey):
            assert self.shape[1] == other.shape[0], 'non-conformal keys %s, %s' % (str(self.shape), str(other.shape))
            # products with the identity are exact in fp32 (1*x = x): most factors of keygen's A = C^-1.p.g.P.G.C are identities
            if self.bias is None and other.bias is None:
                if other._identity():
                    return self
                if self._identity():
                    return other
            bias = None
            if self.bias is not None or other.bias is not None:
                # row r of the product: scale_a[r] * (row perm_a[r] of B) + bias_a[r] * e_last; scipy accumulates the
                # last column as fl(fl(scale_a * bias_b[perm_a]) + bias_a)
                bb = np.zeros(len(self.perm), dtype=np.float32) if other.bias is None else (self.scale * other.bias[self.perm]).astype(np.float32)
                bias = bb if self.bias is None else (bb + self.bias).astype(np.float32)
                bias[-1] = 0
            if self.is_unscaled() and other.is_unscaled():
                scale = None                                   # 1 * 1: no value array
            elif other.is_unscaled():
                scale = self.scale
            else:
                scale = (self.scale * other.scale[self.perm]).astype(np.float32)
            perm = other.perm if self.is_unpermuted() else (self.perm if other.is_unpermuted() else other.perm[self.perm])
            return MonomialKey(perm, scale, bias)
        if isinstance(other, SparseMatrix):
            return other._left_monomial(self)
        if isinstance(other, SparseKey):
            return SparseKey.from_monomial(self).dot(other)
        raise TypeError('cannot multiply MonomialKey with %s' % str(type(other)))

    def apply(self, X):
        """self . X for a dense host array X [n, m] (image-side plumbing: mat2gray keys, keynet/system.py:176-197)."""
        X = np.asarray(X)
        Y = self.scale.reshape(-1, 1).astype(X.dtype) * X[self.perm]
        if self.bias is not None:
            Y = Y + self.bias.reshape(-1, 1).astype(X.dtype) * X[-1:, :]
        return Y

    def transpose(self):
        assert self.bias is None, 'a key with a bias column has no monomial transpose (use the inverse from the generator)'
        n = self._n
        if self.is_unpermuted():
            return self                                        # diagonal: its own transpose
        perm = np.empty(n, dtype=np.int64)
        perm[self.perm] = np.arange(n)
        if self.is_unscaled():
            return MonomialKey(perm)
        scale = np.empty(n, dtype=np.float32)
        scale[self.perm] = self.scale
        return MonomialKey(perm, scale)

    @property
    def T(self):
        return self.transpose()

    def astype(self, dtype):
        assert np.dtype(dtype) == np.float32
        return self

    def diagonal(self):
        d = np.zeros(len(self.perm), dtype=np.float32)
        on = self.perm == np.arange(len(self.perm))
        d[on] = self.scale[on]
        return d

    # -- interop (tests, visualisation); not used by the product path
    def todense(self):
        D = np.zeros(self.shape, dtype=np.float32)
        D[np.arange(len(self.perm)), self.perm] = self.scale
        if self.bias is not None:
            D[:-1, -1] += self.bias[:-1]
        return D

    def toscipy(self, format='csr'):
        import scipy.sparse
        n = len(self.perm)
        A = scipy.sparse.csr_matrix((self.scale, self.perm.astype(np.int32), np.arange(n + 1)), shape=self.shape)
        if self.bias is not None:
            nz = np.nonzero(self.bias)[0]
            A = A + scipy.sparse.csr_matrix((self.bias[nz], (nz, np.full(len(nz), n - 1))), shape=self.shape)
        return A.asformat(format)


class SparseKey(object):
    """General sparse key on the host: CSR with ascending columns (numpy).  The reference's key families with several
    entries per row -- Givens-rotation orthogonal blocks, doubly stochastic blocks and their dense inverses, and any
    product of those with monomial / affine keys (keynet/sparse.py:238-353, keynet/system.py:382-410,467-468).
    Key algebra stays on the host like the reference's (keys have O(n) .. O(n * blocksize) entries); the compile of a
    layer matrix with such a key is the GPU SpGEMM of csrc/spgemm.cu."""

    def __init__(self, indptr, indices, data, shape):
        self.indptr = np.ascontiguousarray(indptr, dtype=np.int64)
        self.indices = np.ascontiguousarray(indices, dtype=np.int64)
        self.data = np.ascontiguousarray(data)
        assert self.data.dtype in (np.float32, np.float64)
        self.shape = (int(shape[0]), int(shape[1]))
        assert len(self.indptr) == self.shape[0] + 1 and len(self.indices) == len(self.data) == self.indptr[-1]
        self.ndim = 2
        self.bias = None          # a bias column is an ordinary column here

    dtype = property(lambda self: self.data.dtype)
    nnz = property(lambda self: int(len(self.data)))

    def __repr__(self):
        return '<keynet_b200.SparseKey: shape=%s, nnz=%d, dtype=%s>' % (str(self.shape), self.nnz, str(self.data.dtype))

    def has_bias(self):
        return False

    def is_identity(self):
        n = self.shape[0]
        return self.shape[0] == self.shape[1] and self.nnz == n and bool(np.array_equal(self.indices, np.arange(n))) and bool(np.all(self.data == 1))

    # -- constructors
    @staticmethod
    def from_coo(rows, cols, vals, shape, sum_duplicates=True, drop_zeros=True):
        """Canonical CSR from triplets: duplicates added in the given order, exact zeros dropped (scipy csr_matmat / tocsr)."""
        rows = np.asarray(rows, dtype=np.int64); cols = np.asarray(cols, dtype=np.int64); vals = np.asarray(vals)
        order = np.lexsort((cols, rows))                     # stable: equal (row, col) keep their input order
        (rows, cols, vals) = (rows[order], cols[order], vals[order])
        if len(rows) and sum_duplicates:
            head = np.ones(len(rows), dtype=bool)
            head[1:] = (rows[1:] != rows[:-1]) | (cols[1:] != cols[:-1])
            starts = np.nonzero(head)[0]
            if len(starts) != len(rows):
                vals = np.add.reduceat(vals, starts)
                (rows, cols) = (rows[starts], cols[starts])
        if drop_zeros and len(vals):
            keep = vals != 0
            (rows, cols, vals) = (rows[keep], cols[keep], vals[keep])
        indptr = np.zeros(shape[0] + 1, dtype=np.int64)
        np.add.at(indptr, rows + 1, 1)
        return SparseKey(np.cumsum(indptr), cols, vals, shape)

    @staticmethod
    def from_monomial(K):
        n = K.shape[0]
        if K.bias is None:
            return SparseKey(np.arange(n + 1), K.perm, K.scale, K.shape)
        nz = np.nonzero(K.bias)[0]
        return SparseKey.from_coo(np.concatenate([np.arange(n), nz]), np.concatenate([K.perm, np.full(len(nz), n - 1)]),
                                  np.concatenate([K.scale, K.bias[nz]]), K.shape, sum_duplicates=True, drop_zeros=False)

    @staticmethod
    def from_dense(D):
        (r, c) = np.nonzero(D)
        return SparseKey.from_coo(r, c, np.asarray(D)[r, c], D.shape, sum_duplicates=False)

    @staticmethod
    def coerce(K):
        return K if isinstance(K, SparseKey) else SparseKey.from_monomial(K)

    # -- algebra
    def rows(self):
        return np.repeat(np.arange(self.shape[0]), np.diff(self.indptr))

    def dot(self, other):
        """self . other: SparseKey / MonomialKey -> SparseKey (host, expand-sort-compress like csr_matmat: products in the
        common dtype, duplicates added in expansion order, exact zeros dropped); SparseMatrix -> SparseMatrix (GPU SpGEMM)."""
        if isinstance(other, SparseMatrix):
            return other._left_general(self)
        b = SparseKey.coerce(other)
        assert self.shape[1] == b.shape[0], 'non-conformal keys %s, %s' % (str(self.shape), str(b.shape))
        dt = np.result_type(self.data.dtype, b.data.dtype)
        blen = np.diff(b.indptr)[self.indices]                           # products per entry of self
        tot = int(blen.sum())
        off = np.concatenate([[0], np.cumsum(blen)])[:-1]
        idx = np.arange(tot, dtype=np.int64) - np.repeat(off, blen) + np.repeat(b.indptr[self.indices], blen)
        vals = np.repeat(self.data.astype(dt), blen) * b.data.astype(dt)[idx]
        return SparseKey.from_coo(np.repeat(self.rows(), blen), b.indices[idx], vals, (self.shape[0], b.shape[1]))

    def apply(self, X):
        """self . X for a dense host array X [n, m]."""
        X = np.asarray(X)
        Y = np.zeros((self.shape[0], X.shape[1]), dtype=np.result_type(self.data.dtype, X.dtype))
        np.add.at(Y, self.rows(), self.data.reshape(-1, 1) * X[self.indices])
        return Y

    def transpose(self):
        return SparseKey.from_coo(self.indices, self.rows(), self.data, (self.shape[1], self.shape[0]), sum_duplicates=False, drop_zeros=False)

    T = property(lambda self: self.transpose())

    def astype(self, dtype):
        return SparseKey(self.indptr, self.indices, self.data.astype(dtype), self.shape)

    def diagonal(self):
        d = np.zeros(min(self.shape), dtype=self.data.dtype)
        r = self.rows()
        on = (r == self.indices) & (r < len(d))
        d[r[on]] = self.data[on]
        return d

    def block(self, r0, r1, c0, c1):
        """Sub-matrix [r0:r1, c0:c1] (scipy slicing)."""
        r = self.rows()
        keep = (r >= r0) & (r < r1) & (self.indices >= c0) & (self.indices < c1)
        return SparseKey.from_coo(r[keep] - r0, self.indices[keep] - c0, self.data[keep], (r1 - r0, c1 - c0), sum_duplicates=False, drop_zeros=False)

    # -- interop (tests, visualisation); not used by the product path
    def todense(self):
        D = np.zeros(self.shape, dtype=self.data.dtype)
        D[self.rows(), self.indices] = self.data
        return D

    def toscipy(self, format='csr'):
        import scipy.sparse
        return scipy.sparse.csr_matrix((self.data, self.indices.astype(np.int32), self.indptr), shape=self.shape).asformat(format)


def is_key(A):
    return isinstance(A, (MonomialKey, SparseKey))



def sparse_identity_matrix(n, dtype=np.float32):
    return MonomialKey.identity(n)


def sparse_identity_matrix_like(A):
    return MonomialKey.identity(A.shape[0])


def sparse_permutation_matrix(n, dtype=np.float32, withinverse=False):
    """P[r, perm[r]] = 1 with perm drawn from numpy's global legacy RNG, consuming exactly the stream
    the reference consumes (np.random.permutation over range(n), keynet/sparse.py:280-285)."""
    P = MonomialKey(np.random.permutation(int(n)))
    return (P, P.transpose()) if withinverse else P


def sparse_uniform_random_diagonal_matrix(n, scale=1, bias=0, eps=1E-6, dtype=np.float32, withinverse=False):
    """diag(scale*U[0,1) + eps + bias); the inverse is 1/d evaluated in float64 and then rounded to
    float32, as the reference does (keynet/sparse.py:318-321)."""
    d = np.array(scale * np.random.rand(int(n)) + eps + bias)      # float64
    D = MonomialKey(np.arange(int(n)), d.astype(np.float32))
    return (D, MonomialKey(np.arange(int(n)), (1.0 / d).astype(np.float32))) if withinverse else D


def sparse_gaussian_random_diagonal_matrix(n, mu=1, sigma=1, eps=1E-6, withinverse=False, dtype=np.float32):
    d = np.maximum(eps, np.array(sigma * np.random.randn(int(n)) + mu))
    D = MonomialKey(np.arange(int(n)), d.astype(np.float32))
    return (D, MonomialKey(np.arange(int(n)), (1.0 / d).astype(np.float32))) if withinverse else D


def sparse_channelorder_to_pixelorder_matrix(shape, withinverse=False):
    """Permutation taking a CxHxW (channel order) flattening to HxWxC (pixel order), keynet/sparse.py:53-62."""
    img = np.arange(int(np.prod(shape))).reshape(shape)
    P = MonomialKey(np.moveaxis(img, 0, 2).flatten())
    return P if not withinverse else (P, P.transpose())


def sparse_channelorder_to_blockorder_matrix(shape, blocksize, withinverse=True):
    """Permutation taking CxHxW to Cx(H//B)x(W//B)xBxB block order, keynet/sparse.py:65-84."""
    assert isinstance(shape, tuple) and len(shape) == 3, "Shape must be (C,H,W) tuple"
    (C, H, W) = shape
    if (H * W) % blocksize != 0:
        warnings.warn('[keynet_b200.sparse.sparse_channelorder_to_blockorder]:  Ragged blockorder for blocksize=%d and shape=%s' % (blocksize, str(shape)))
    (H_pad, W_pad) = (int(blocksize * np.ceil(H / float(blocksize))), int(blocksize * np.ceil(W / float(blocksize))))
    order = blockview(np.arange(H_pad * W_pad).reshape(H_pad, W_pad), blocksize).flatten()[0:H * W]
    if (H_pad != H or W_pad != W) and not np.array_equal(np.sort(order), np.arange(H * W)):
        # (the reference truncates the padded block order; for Cx1x1 activations that is the identity, otherwise not a permutation)
        raise ValueError('ragged block order (blocksize=%d, shape=%s) is not a permutation' % (blocksize, str(shape)))
    perm = np.concatenate([order + c * H * W for c in range(C)])
    A = MonomialKey(perm)
    return A if not withinverse else (A, A.transpose())


def sparse_affine_to_linear(A, bias=None, dtype=np.float32):
    """[A 0; 0 1]: homogeneous augmentation of a key (keynet/sparse.py:87-96).  Keys with a bias
    column are not monomial and belong to the general-key path (SURVEY.md 8f-2)."""
    if isinstance(A, SparseKey):
        n = A.shape[0]
        (rows, cols, vals) = (A.rows(), A.indices, A.data)
        if bias is not None:
            bias = np.asarray(bias).reshape(-1)
            nz = np.nonzero(bias)[0]
            (rows, cols, vals) = (np.concatenate([rows, nz]), np.concatenate([cols, np.full(len(nz), n)]), np.concatenate([vals, bias[nz].astype(vals.dtype)]))
        (rows, cols, vals) = (np.concatenate([rows, [n]]), np.concatenate([cols, [n]]), np.concatenate([vals, np.ones(1, dtype=vals.dtype)]))
        return SparseKey.from_coo(rows, cols, vals, (n + 1, n + 1), sum_duplicates=False, drop_zeros=False)
    assert isinstance(A, MonomialKey), 'sparse_affine_to_linear expects a key matrix'
    n = A.shape[0]
    b = None
    if bias is not None:
        bias = np.asarray(bias).reshape(-1)
        assert bias.shape[0] == n
        b = np.concatenate([bias.astype(np.float32), np.zeros(1, dtype=np.float32)])
    if b is None and A.is_identity():
        return MonomialKey.identity(n + 1)
    perm = np.empty(n + 1, dtype=np.int64)
    perm[:n] = A.perm
    perm[n] = n
    scale = None
    if not A.is_unscaled():
        scale = np.empty(n + 1, dtype=np.float32)
        scale[:n] = A.scale
        scale[n] = 1.0
    return MonomialKey(perm, scale, b)


def diagonal_affine_to_linear(A, bias=None, withinverse=False, dtype=np.float32):
    """[[D, b],[0, 1]] for a diagonal key D and its inverse [[D^-1, -D^-1 b],[0, 1]] (keynet/sparse.py:99-119).
    The reference evaluates the inverse with a rank-one (Woodbury) update in float64 and rounds to float32 at the end:
    diagonal f32(1/d), last column f32(-((1/d)*b)) with d = f64(f32 diagonal), b = the float64 bias."""
    assert isinstance(A, MonomialKey) and A.is_unpermuted() and A.bias is None, 'diagonal_affine_to_linear expects a diagonal key'
    n = A.shape[0]
    L = sparse_affine_to_linear(A, bias)
    if not withinverse:
        return L
    d = A.scale.astype(np.float64)
    inv = 1.0 / d
    if bias is None:
        return (L, MonomialKey(np.arange(n + 1), np.concatenate([inv, [1.0]]).astype(np.float32)))
    b = np.asarray(bias, dtype=np.float64).reshape(-1)
    binv = 0.0 - (inv * b * 2.0) / 2.0          # (Ainv u)(v Ainv) / (1 + v Ainv u): the factors of two are exact
    return (L, MonomialKey(np.arange(n + 1), np.concatenate([inv, [1.0]]).astype(np.float32), np.concatenate([binv, [0.0]]).astype(np.float32)))


def mat2gray(x, dtype=np.float32):
    """Affine key pair mapping the values of x onto [0, 1]: xh = x / (max - min) - min / (max - min) (keynet/sparse.py:25-33)."""
    x = np.asarray(x)
    (xmin, xmax) = (np.min(x), np.max(x))
    gain = 1.0 / (xmax - xmin)
    bias = -xmin / (xmax - xmin)
    n = int(np.max(x.shape))
    return diagonal_affine_to_linear(MonomialKey(np.arange(n), np.full(n, gain, dtype=np.float64).astype(np.float32)), np.ones((n, 1)) * bias, withinverse=True, dtype=dtype)


def _jet(v):
    """v in [0, 1] -> uint8 RGB with the classic jet ramp."""
    v = np.clip(v, 0.0, 1.0)
    rgb = np.stack([np.clip(1.5 - np.abs(4 * v - 3), 0, 1), np.clip(1.5 - np.abs(4 * v - 2), 0, 1), np.clip(1.5 - np.abs(4 * v - 1), 0, 1)], axis=-1)
    return (255 * rgb).astype(np.uint8)


def spy(A, mindim=256, showdim=1024, range=None, eps=None):
    """Picture of the sparsity / values of A (a key, a SparseMatrix or anything with tocoo()): the block
    A[range[0]:range[1], range[0]:range[1]] binned to about mindim x mindim cells (cell = mean of its stored values), min-max
    normalised, jet-coloured and enlarged to showdim with nearest-neighbour interpolation (keynet/sparse.py:382-415).
    Returns a PIL image (the reference returns a vipy image)."""
    from PIL import Image
    if isinstance(A, MonomialKey):
        A = SparseKey.from_monomial(A)
    if isinstance(A, SparseKey):
        (shape, row, col, val) = (A.shape, A.rows(), A.indices, A.data.astype(np.float32))
    else:
        C = A.tocoo()
        (shape, row, col, val) = (tuple(C.shape), np.asarray(C.row, dtype=np.int64), np.asarray(C.col, dtype=np.int64), np.asarray(C.data, dtype=np.float32))
    if range is not None:
        assert isinstance(range, tuple) and len(range) == 2, "Range must be tuple (start_dim, end_dim)"
        (i, j) = range
        keep = (row >= i) & (row < j) & (col >= i) & (col < j)
        (row, col, val, shape) = (row[keep] - i, col[keep] - i, val[keep], (j - i, j - i))
    if eps is not None:
        keep = np.abs(val) > eps
        (row, col, val) = (row[keep], col[keep], val[keep])
    scale = float(mindim) / min(shape)
    n = 1.0 if scale >= 1 else 1.0 / scale
    (H, W) = (int(np.ceil(shape[0] / n)) + (0 if scale >= 1 else 1), int(np.ceil(shape[1] / n)) + (0 if scale >= 1 else 1))
    (bi, bj) = ((row // n).astype(np.int64), (col // n).astype(np.int64))
    (acc, cnt) = (np.zeros(H * W, dtype=np.float64), np.zeros(H * W, dtype=np.float64))
    np.add.at(acc, bi * W + bj, val)
    np.add.at(cnt, bi * W + bj, 1.0)
    img = (acc / np.maximum(cnt, 1.0)).reshape(H, W).astype(np.float32)
    (lo, hi) = (float(img.min()), float(img.max()))
    img = (img - lo) / (hi - lo) if hi > lo else np.zeros_like(img)
    im = Image.fromarray(_jet(img), 'RGB')
    f = float(showdim) / max(im.size)
    return im.resize((max(1, int(round(im.size[0] * f))), max(1, int(round(im.size[1] * f)))), Image.NEAREST)


def sparse_orthogonal_matrix(n, k_iter, balanced=True, withinverse=False, dtype=np.float32):
    """Product of k_iter random Givens rotations S = G_k ... G_1 (keynet/sparse.py:288-309), same numpy RNG draws as the
    reference: one rand() for the angle per rotation, one permutation(n) whenever the index pool runs low.  Rows are
    kept sparse in float64 (a rotation rewrites two rows), rounded to `dtype` at the end; the inverse is the transpose."""
    assert n >= 2
    assert balanced, 'only the balanced construction is used by keygen (keynet/system.py:385,406)'
    rows = {}                                    # row -> {col: float64}; rows never touched are identity rows
    G_index = []
    for k in range(0, int(k_iter)):
        theta = np.random.rand() * 2 * np.pi
        G_index = np.random.permutation(range(0, n)).tolist() + G_index if len(G_index) <= 1 else G_index
        (i, j) = (G_index.pop(), G_index.pop())
        (c, sn) = (np.cos(theta), np.sin(theta))
        (Si, Sj) = (rows.get(i, {i: 1.0}), rows.get(j, {j: 1.0}))
        (ni, nj) = ({}, {})
        for col in set(Si) | set(Sj):
            (a, b) = (Si.get(col), Sj.get(col))
            # row i of G = (c at i, -sin at j), row j = (sin at i, c at j); csr_matmat adds the products of a row in column
            # order of G -- two terms, so the order does not matter -- and never stores an exact zero
            vi = (c * a if a is not None else 0.0) + (-sn * b if b is not None else 0.0) if (a is not None and b is not None) else (c * a if a is not None else -sn * b)
            vj = (sn * a if a is not None else 0.0) + (c * b if b is not None else 0.0) if (a is not None and b is not None) else (sn * a if a is not None else c * b)
            if vi != 0:
                ni[col] = vi
            if vj != 0:
                nj[col] = vj
        (rows[i], rows[j]) = (ni, nj)
    (r, cidx, v) = ([], [], [])
    for (row, d) in rows.items():
        for (col, val) in d.items():
            r.append(row); cidx.append(col); v.append(val)
    untouched = np.setdiff1d(np.arange(n), np.fromiter(rows.keys(), dtype=np.int64, count=len(rows)))
    S = SparseKey.from_coo(np.concatenate([np.asarray(r, dtype=np.int64), untouched]), np.concatenate([np.asarray(cidx, dtype=np.int64), untouched]),
                           np.concatenate([np.asarray(v, dtype=np.float64), np.ones(len(untouched))]), (n, n), sum_duplicates=False, drop_zeros=False).astype(dtype)
    return S if not withinverse else (S, S.transpose())


def sparse_random_diagonally_dominant_doubly_stochastic_matrix(n, k, n_iter=100, withinverse=False):
    """Doubly stochastic band matrix with k diagonals made diagonally dominant, Sinkhorn-normalised and conjugated by two
    random permutations; inverse by dense inversion (keynet/sparse.py:335-353).  Same RNG draws as the reference
    (rand(k, n), then the left and the right permutation).  Evaluated densely in float64 -- the block is at most
    blocksize^2 x blocksize^2 -- and returned as float64 SparseKeys like the reference's."""
    n_iter = 10 if k <= 3 else n_iter
    d = np.random.rand(k, n)
    d[0, :] = np.maximum(d[0, :], np.sum(d[1:, :], axis=0) + 0.1)
    d = d / np.sum(d, axis=0).reshape(1, n)
    k_range = list(range(-((k - 1) // 2), 1 + ((k - 1) // 2)) if k % 2 == 1 else list(range(-(k // 2), k // 2)))
    k_range.remove(0)
    k_range = [0] + k_range
    A = np.zeros((n, n), dtype=np.float64)
    for (row, off) in enumerate(k_range):                       # scipy.sparse.spdiags: data[row, j] sits at A[j - off, j]
        j = np.arange(max(0, off), min(n, n + off))
        A[j - off, j] = d[row, j]
    for it in range(0, n_iter):
        nrm = np.abs(A).sum(axis=0); nrm[nrm == 0] = 1.0
        A = A / nrm.reshape(1, n)                               # sklearn normalize(norm='l1', axis=0)
        nrm = np.abs(A).sum(axis=1); nrm[nrm == 0] = 1.0
        A = A / nrm.reshape(n, 1)
    P1 = sparse_permutation_matrix(n)
    P2 = sparse_permutation_matrix(n)
    B = np.zeros_like(A)
    B[:, P2.perm] = A[P1.perm, :]                               # P1 . A . P2
    if not withinverse:
        return SparseKey.from_dense(B)
    return (SparseKey.from_dense(B), SparseKey.from_dense(np.linalg.inv(B)))


def sparse_block_diagonal_repeat(B, shape):
    """Key B repeated down the diagonal of an (N,N) matrix, truncated at N (the monomial case of the
    reference's DiagonalTiledMatrix / sparse_block_diagonal, keynet/sparse.py:215-235,657-687)."""
    assert shape[0] == shape[1]
    if isinstance(B, SparseKey):
        (n, h) = (int(shape[0]), B.shape[0])
        if h > n:
            B = B.block(0, n, 0, n)                       # keynet/sparse.py:662-663
            h = n
        reps = n // h
        (r, c, v) = (B.rows(), B.indices, B.data)
        rows = (np.tile(r, reps) + np.repeat(np.arange(reps) * h, len(r)))
        cols = (np.tile(c, reps) + np.repeat(np.arange(reps) * h, len(r)))
        vals = np.tile(v, reps)
        tail = np.arange(reps * h, n)                     # ragged tail tile is the identity (sparse.py:680-681)
        return SparseKey.from_coo(np.concatenate([rows, tail]), np.concatenate([cols, tail]), np.concatenate([vals, np.ones(len(tail), dtype=v.dtype)]),
                                  (n, n), sum_duplicates=False, drop_zeros=False)
    assert isinstance(B, MonomialKey)
    (n, h) = (int(shape[0]), B.shape[0])
    reps = int(np.ceil(n / float(h)))
    perm = (np.tile(B.perm, reps) + np.repeat(np.arange(reps) * h, h))[0:n]
    scale = np.tile(B.scale, reps)[0:n]
    if n % h != 0:
        tail = np.arange(n - (n % h), n)          # ragged tail tile is the identity (sparse.py:680-681)
        perm[tail] = tail
        scale[tail] = 1.0
    assert perm.max() < n
    return MonomialKey(perm, scale)


# =============================================================================================
# Device CSR matrix
# =============================================================================================
def _device():
    _native.require_cuda()
    return torch.device('cuda', torch.cuda.current_device())


def _scan_counts_inplace(indptr):
    """indptr[1:] holds per-row counts on entry; on exit indptr is the exclusive prefix sum."""
    n = indptr.numel() - 1
    check(_native.lib().kn_exclusive_scan_i64(ptr(indptr[1:]) if n > 0 else None, ptr(indptr), n, stream_ptr()))


def _two_phase(n_rows, count, fill, device):
    """count(row_nnz) -> scan -> allocate -> fill(indptr, indices, data).  One host sync (the nnz readback)."""
    indptr = torch.empty(n_rows + 1, dtype=torch.int64, device=device)
    if n_rows > 0:
        count(indptr[1:])
    _scan_counts_inplace(indptr)
    nnz = int(indptr[-1].item())
    indices = torch.empty(nnz, dtype=torch.int32, device=device)
    data = torch.empty(nnz, dtype=torch.float32, device=device)
    if n_rows > 0 and nnz > 0:
        fill(indptr, indices, data)
    return (indptr, indices, data)


def _spgemm_device(a, n_rows, b):
    """C = A . B on the GPU (csrc/spgemm.cu).  a, b: (indptr int64, indices int32, data f32) CUDA tensors (indptr may be a
    row-slice view with a non-zero base).  Returns canonical CSR (ascending columns, exact zeros dropped)."""
    L = _native.lib()
    (a_ip, a_ix, a_dt) = a
    (b_ip, b_ix, b_dt) = b
    dev = a_dt.device
    tmp_ptr = torch.empty(n_rows + 1, dtype=torch.int64, device=dev)
    if n_rows > 0:
        check(L.kn_spgemm_bound(ptr(a_ip), ptr(a_ix), n_rows, ptr(b_ip), ptr(tmp_ptr[1:]), stream_ptr()))
    _scan_counts_inplace(tmp_ptr)
    total = int(tmp_ptr[-1].item())
    tmp_ix = torch.empty(total, dtype=torch.int32, device=dev)
    tmp_dt = torch.empty(total, dtype=torch.float32, device=dev)
    out_ip = torch.empty(n_rows + 1, dtype=torch.int64, device=dev)
    if n_rows > 0:
        check(L.kn_spgemm_rows(ptr(a_ip), ptr(a_ix), ptr(a_dt), n_rows, ptr(b_ip), ptr(b_ix), ptr(b_dt), ptr(tmp_ptr), ptr(tmp_ix), ptr(tmp_dt), ptr(out_ip[1:]), stream_ptr()))
    _scan_counts_inplace(out_ip)
    nnz = int(out_ip[-1].item())
    out_ix = torch.empty(nnz, dtype=torch.int32, device=dev)
    out_dt = torch.empty(nnz, dtype=torch.float32, device=dev)
    if n_rows > 0 and nnz > 0:
        check(L.kn_csr_compact(ptr(tmp_ptr), ptr(tmp_ix), ptr(tmp_dt), n_rows, ptr(out_ip), ptr(out_ix), ptr(out_dt), stream_ptr()))
    return (out_ip, out_ix, out_dt)


class SparseMatrix(object):
    """Device-resident CSR matrix implementing the reference's SparseMatrix operator protocol
    (keynet/sparse.py:419-514): torchdot / dot / matmul / nnz / transpose / tocoo / tocsr /
    from_scipy_sparse / from_torch_dense / from_torch_conv2d."""

    def __init__(self, A=None, device=None):
        self.ndim = 2
        self.dtype = np.float32
        self._pg = None          # optional pattern-grouped execution format (PatternGroups)
        if A is None:
            (self.shape, self._indptr, self._indices, self._data) = ((0, 0), None, None, None)
            return
        dev = device if device is not None else _device()
        if isinstance(A, SparseMatrix):
            (self.shape, self._indptr, self._indices, self._data) = (A.shape, A._indptr, A._indices, A._data)
        elif isinstance(A, MonomialKey) and A.bias is None:
            n = A.shape[0]
            self.shape = A.shape
            self._indptr = torch.arange(n + 1, dtype=torch.int64, device=dev)
            self._indices = torch.from_numpy(A.perm.astype(np.int32)).to(dev)
            self._data = torch.from_numpy(A.scale).to(dev)
        elif isinstance(A, MonomialKey):
            # key with a bias column: one or two entries per row, canonical order (the permuted column is < n-1)
            n = A.shape[0]
            has = A.bias != 0
            counts = 1 + has.astype(np.int64)
            indptr = np.concatenate([[0], np.cumsum(counts)])
            indices = np.empty(indptr[-1], dtype=np.int32); data = np.empty(indptr[-1], dtype=np.float32)
            indices[indptr[:-1]] = A.perm; data[indptr[:-1]] = A.scale
            indices[indptr[:-1][has] + 1] = n - 1; data[indptr[:-1][has] + 1] = A.bias[has]
            self.shape = A.shape
            self._indptr = torch.from_numpy(indptr.astype(np.int64)).to(dev)
            self._indices = torch.from_numpy(indices).to(dev)
            self._data = torch.from_numpy(data).to(dev)
        elif isinstance(A, SparseKey):
            self.shape = A.shape
            self._indptr = torch.from_numpy(A.indptr).to(dev)
            self._indices = torch.from_numpy(A.indices.astype(np.int32)).to(dev)
            self._data = torch.from_numpy(A.data.astype(np.float32)).to(dev)
        elif isinstance(A, tuple) and len(A) == 4:
            (shape, indptr, indices, data) = A
            self.shape = (int(shape[0]), int(shape[1]))
            self._indptr = torch.as_tensor(np.asarray(indptr) if not torch.is_tensor(indptr) else indptr).to(device=dev, dtype=torch.int64).contiguous()
            self._indices = torch.as_tensor(np.asarray(indices) if not torch.is_tensor(indices) else indices).to(device=dev, dtype=torch.int32).contiguous()
            self._data = torch.as_tensor(np.asarray(data) if not torch.is_tensor(data) else data).to(device=dev, dtype=torch.float32).contiguous()
            assert self._indptr.numel() == self.shape[0] + 1 and self._indices.numel() == self._data.numel()
        elif isinstance(A, np.ndarray):
            M = self.from_torch_dense(torch.from_numpy(np.ascontiguousarray(A, dtype=np.float32)))
            (self.shape, self._indptr, self._indices, self._data) = (M.shape, M._indptr, M._indices, M._data)
        elif hasattr(A, 'tocsr'):     # scipy sparse (interop only)
            M = self.from_scipy_sparse(A)
            (self.shape, self._indptr, self._indices, self._data) = (M.shape, M._indptr, M._indices, M._data)
        else:
            raise AssertionError('Invalid input - %s' % str(type(A)))

    def __repr__(self):
        return '<keynet_b200.SparseMatrix: H=%d, W=%d, nnz=%d, backend=b200-csr>' % (self.shape[0], self.shape[1], self.nnz())

    # ---- protocol --------------------------------------------------------------------------
    def new(self):
        return SparseMatrix()

    def clone(self):
        return SparseMatrix((self.shape, self._indptr.clone(), self._indices.clone(), self._data.clone()), device=self._data.device)

    def nnz(self):
        if self._data is None:
            return int(getattr(self, '_nnz', 0))
        return int(self._data.numel())

    def drop_csr(self):
        """Free the canonical CSR and keep only the pattern-grouped execution format (VGG16-scale layers: 120 GB of
        CSR vs < 1 GB of unique value blocks + gather lists).  The matrix can no longer be exported or row-sliced."""
        assert self._pg is not None, 'drop_csr() needs the pattern-grouped format'
        if self._data is None:
            return self                       # built without a CSR in the first place (direct pattern groups)
        self._nnz = self.nnz()
        self._device = self._data.device
        (self._indptr, self._indices, self._data) = (None, None, None)
        return self

    def from_torch_dense(self, A):
        """Non-zero entries of a dense matrix, row-major (scipy coo_matrix(dense) semantics)."""
        assert torch.is_tensor(A) and A.ndim == 2
        dev = _device()
        W = A.detach().to(device=dev, dtype=torch.float32).contiguous()
        (R, C) = W.shape
        # [[W],[.]] without the homogeneous row: reuse the linear builder with n_rows = R and no bias
        L = _native.lib()
        (indptr, indices, data) = _two_phase(
            R,
            lambda row_nnz: check(L.kn_linear_count(ptr(W), None, R, C, None, R, ptr(row_nnz), stream_ptr())),
            lambda ip, ix, dt: check(L.kn_linear_fill(ptr(W), None, R, C, None, R, ptr(ip), ptr(ix), ptr(dt), stream_ptr())),
            dev)
        return SparseMatrix(((R, C), indptr, indices, data), device=dev)

    def from_scipy_sparse(self, A):
        A = A.tocsr().astype(np.float32)
        A.sum_duplicates()
        A.sort_indices()
        return SparseMatrix((A.shape, A.indptr.astype(np.int64), A.indices.astype(np.int32), A.data), device=_device())

    def from_torch_conv2d(self, inshape, w, b, stride):
        return sparse_toeplitz_conv2d(inshape, w.detach(), bias=b.detach() if b is not None else None, stride=stride)

    def torchdot(self, x_torch, relu=False):
        """SpMM W . x for x of shape (C, N); returns (R, N) float32 on x's device.

        Replaces keynet/sparse.py:488-492.  A transposed view of a feature-major activation (what
        KeyedLayer.forward passes) is consumed without a copy; CPU tensors are staged through the GPU."""
        assert x_torch.ndim == 2 and x_torch.shape[0] == self.shape[1], "Non-conformal shape for W=%s, x=%s" % (str(self.shape), str(tuple(x_torch.shape)))
        dev = self._data.device if self._data is not None else self._device
        on_host = not x_torch.is_cuda
        x = x_torch.detach()
        if x.dtype != torch.float32:
            x = x.to(torch.float32)
        x = x.to(dev, non_blocking=True) if on_host else x
        if not x.is_contiguous():
            x = x.contiguous()
        N = x.shape[1]
        if self._data is not None and (self._pg is None or N < 32 or N % 4 != 0) and (getattr(self, '_exec', None) is None or N < 32):
            # plain CSR product: the dispatcher-visible op (keynet_b200/ops.py -> kn_spmm_csr_f32)
            from . import ops as _ops       # registers the torch.library ops on first use
            y = torch.ops.keynet_b200.spmm_csr(self._indptr, self._indices, self._data, self.shape[1], x, bool(relu))    # row pointers are absolute: views work
        else:
            y = spmm(self, x, relu=relu)
        return y.cpu() if on_host else y


    def dot(self, x_numpy):
        if isinstance(x_numpy, MonomialKey):
            return self.clone().matmul(x_numpy)
        assert isinstance(x_numpy, np.ndarray)
        x = torch.from_numpy(np.ascontiguousarray(x_numpy, dtype=np.float32))
        return self.torchdot(x.reshape(self.shape[1], -1)).numpy()

    def matmul(self, A):
        """In-place self <- self . A for a monomial key A (column reindex + scale + zero drop + sort),
        the right-hand SpGEMM of keynet/layer.py:35 / keynet/sparse.py:472-480."""
        if isinstance(A, (SparseKey, SparseMatrix)):
            # general right factor: GPU SpGEMM (csrc/spgemm.cu)
            B = A if isinstance(A, SparseMatrix) else SparseMatrix(A, device=self._data.device)
            assert self.shape[1] == B.shape[0]
            (self._indptr, self._indices, self._data) = _spgemm_device((self._indptr, self._indices, self._data), self.shape[0], (B._indptr, B._indices, B._data))
            self.shape = (self.shape[0], B.shape[1])
            self._pg = None
            return self
        if not isinstance(A, MonomialKey):
            raise TypeError('matmul expects a key or a SparseMatrix, got %s' % str(type(A)))
        assert self.shape[1] == A.shape[0]
        (self._indptr, self._indices, self._data) = _keycompile((self._indptr, self._indices, self._data), self.shape[0], self.shape[1],
                                                                None, A, self._data.device)
        self.shape = (self.shape[0], A.shape[1])
        self._pg = None                    # the grouped execution form described the old matrix
        self._exec = None
        return self

    def _left_general(self, A):
        """A . self for a general sparse key A (GPU SpGEMM): the left product of keynet/layer.py:35."""
        assert A.shape[1] == self.shape[0]
        dev = self._data.device
        K = SparseMatrix(A, device=dev)
        csr = _spgemm_device((K._indptr, K._indices, K._data), A.shape[0], (self._indptr, self._indices, self._data))
        return SparseMatrix(((A.shape[0], self.shape[1]), *csr), device=dev)

    def _left_monomial(self, A):
        """A . self for a monomial key A: row gather + row scale + zero drop."""
        assert A.shape[1] == self.shape[0]
        dev = self._data.device
        L = _native.lib()
        n = A.shape[0]
        rows = torch.from_numpy(A.perm).to(dev)
        (indptr, indices, data) = _two_phase(
            n,
            lambda row_nnz: check(L.kn_csr_gather_rows_count(ptr(self._indptr), ptr(rows), n, ptr(row_nnz), stream_ptr())),
            lambda ip, ix, dt: check(L.kn_csr_gather_rows_fill(ptr(self._indptr), ptr(self._indices), ptr(self._data), ptr(rows), n, ptr(ip), ptr(ix), ptr(dt), stream_ptr())),
            dev)
        (indptr, indices, data) = _keycompile((indptr, indices, data), n, self.shape[1], A, None, dev)
        return SparseMatrix(((n, self.shape[1]), indptr, indices, data), device=dev)

    def transpose(self):
        """In-place transpose (plumbing, not on the forward path): stable sort of the COO form by column."""
        (R, C) = self.shape
        rows = torch.repeat_interleave(torch.arange(R, device=self._data.device, dtype=torch.int64), self._indptr[1:] - self._indptr[:-1])
        key = self._indices.to(torch.int64) * R + rows
        order = torch.argsort(key)
        counts = torch.bincount(self._indices.to(torch.int64), minlength=C)
        indptr = torch.zeros(C + 1, dtype=torch.int64, device=self._data.device)
        indptr[1:] = torch.cumsum(counts, 0)
        (self._indptr, self._indices, self._data) = (indptr, rows[order].to(torch.int32).contiguous(), self._data[order].contiguous())
        self.shape = (C, R)
        self._pg = None
        self._exec = None
        return self

    def tocsr(self):
        return self

    def tocsc(self):
        raise NotImplementedError('CSC storage is not used on the B200 path')

    def csr_arrays(self):
        """(indptr int64, indices int32, data float32) as numpy arrays on the host (canonical: sorted columns)."""
        return (self._indptr.cpu().numpy(), self._indices.cpu().numpy(), self._data.cpu().numpy())

    def spy(self, mindim=256, showdim=1024, range=None, eps=None):
        """PIL picture of the matrix (keynet/sparse.py:460-462)."""
        return spy(self, mindim, showdim, range, eps)

    def tocoo(self):
        import scipy.sparse
        (ip, ix, dt) = self.csr_arrays()
        return scipy.sparse.csr_matrix((dt, ix, ip), shape=self.shape).tocoo()

    def todense(self):
        (ip, ix, dt) = self.csr_arrays()
        D = np.zeros(self.shape, dtype=np.float32)
        D[np.repeat(np.arange(self.shape[0]), np.diff(ip)), ix] = dt
        return D

    def used_columns(self):
        """bool CUDA tensor [n_cols]: columns some stored entry (or padded slot of the grouped format) reads."""
        if self._pg is not None:
            lists = [c['cols'] for c in self._pg.classes] + ([self._pg.rest['indices']] if self._pg.rest is not None else [])
        else:
            lists = [self._indices[int(self._indptr[0]):int(self._indptr[-1])]]
        used = torch.zeros(self.shape[1], dtype=torch.bool, device=lists[0].device)
        for ix in lists:
            used[ix.to(torch.int64)] = True
        return used

    def optimize(self, min_group=4, min_nnz=4096):
        """Build the pattern-grouped execution format (csrc/pgroup.cu) next to the canonical CSR.  The CSR stays
        the source of truth (parity, export, small batches); batches of >= 32 images run on the groups."""
        if self._pg is None and self.nnz() >= min_nnz:
            self._pg = PatternGroups.build(self, min_group=min_group)
        return self

    def row_slice(self, r0, r1):
        """Rows [r0, r1) as a view-like SparseMatrix sharing indices/data (indptr offsets stay absolute)."""
        M = SparseMatrix()
        (M.shape, M._indptr, M._indices, M._data) = ((r1 - r0, self.shape[1]), self._indptr[r0:r1 + 1], self._indices, self._data)
        return M


# =============================================================================================
# Pattern-grouped execution format
# =============================================================================================
_TC = {'enabled': os.environ.get('KEYNET_B200_TENSOR_CORES', '1') != '0'}


def tensor_cores_enabled(flag=None):
    """Switch for the tcgen05 path of pattern groups (default on; KEYNET_B200_TENSOR_CORES=0 or
    tensor_cores_enabled(False) keeps everything on the fp32 FMA kernels)."""
    if flag is not None:
        _TC['enabled'] = bool(flag)
    return _TC['enabled']


_CLUSTERS = [True]
_DIRECT = [os.environ.get('KEYNET_B200_DIRECT_COMPILE', '1') != '0']
_TILES = [os.environ.get('KEYNET_B200_TILES', '1') != '0']


def tiles_enabled(flag=None):
    """Switch for the spatially tiled tensor-core kernel of conv layers with G <= 128 (csrc/pgtile_tc.cu); off = one output
    pixel per CTA (csrc/pgroup_tc.cu).  A/B measurements and tests."""
    if flag is not None:
        _TILES[0] = bool(flag)
    return _TILES[0]



def direct_compile_enabled(flag=None):
    """Switch for the fused key compile of conv / linear layers (csrc/keyedconv.cu); off = Toeplitz CSR + per-row key compile +
    pattern hashing (the two-kernel path, kept for keys with bias columns and for A/B tests)."""
    if flag is not None:
        _DIRECT[0] = bool(flag)
    return _DIRECT[0]



def clusters_enabled(flag=None):
    """Switch the clustered small-group kernel on / off (A/B measurements and tests); returns the current setting."""
    if flag is not None:
        _CLUSTERS[0] = bool(flag)
    return _CLUSTERS[0]


def _dedup_value_blocks(cols, vals, group_k, ng, G, K_pad, chunk_bytes=1 << 30):
    """Store identical value blocks once (the reference's unique tiles, keynet/sparse.py:553-568,690-779).

    Two groups hold the same block only up to the order of their columns (each group lists its columns by ascending
    permuted index), so every group's columns are first put in a canonical order -- sorted by a 64-bit signature of
    the column's G values, padding last -- with `cols` permuted alongside; blocks are then hashed, grouped with
    torch.unique and VERIFIED element-wise against their representative.  Returns (cols, vals_unique, block_of) or the
    inputs unchanged with block_of=None when nothing is shared.  Build-time plumbing on torch device ops."""
    dev = vals.device
    v3 = vals.view(ng, G, K_pad)
    c2 = cols.view(ng, K_pad)
    rw = (torch.arange(G, device=dev, dtype=torch.int64) * 0x9E3779B1 + 0x7F4A7C15) | 1          # odd per-row weights
    kw = (torch.arange(K_pad, device=dev, dtype=torch.int64) * 0x85EBCA77 + 0x165667B1) | 1      # odd per-column weights
    step = max(1, int(chunk_bytes // (G * K_pad * 8)))
    blk_hash = torch.empty(ng, dtype=torch.int64, device=dev)
    big = torch.iinfo(torch.int64).max
    karange = torch.arange(K_pad, device=dev).view(1, K_pad)
    for g0 in range(0, ng, step):
        g1 = min(ng, g0 + step)
        vi = v3[g0:g1].view(torch.int32).to(torch.int64)                                          # bit patterns
        sig = (vi * rw.view(1, G, 1)).sum(dim=1)                                                   # [n, K_pad] column signatures
        sig = torch.where(karange < group_k[g0:g1].view(-1, 1), sig, torch.full_like(sig, big))   # padding columns last
        order = torch.argsort(sig, dim=1, stable=True)
        c2[g0:g1] = torch.gather(c2[g0:g1], 1, order)
        v3[g0:g1] = torch.gather(v3[g0:g1], 2, order.view(-1, 1, K_pad).expand(-1, G, -1))
        vi = v3[g0:g1].view(torch.int32).to(torch.int64)
        blk_hash[g0:g1] = ((vi * rw.view(1, G, 1)).sum(dim=1) * kw.view(1, K_pad)).sum(dim=1) + group_k[g0:g1].to(torch.int64) * 0x27D4EB2F
        del vi, sig, order
    (uniq, inverse) = torch.unique(blk_hash, return_inverse=True)
    nu = int(uniq.numel())
    if nu == ng:
        return (cols, vals, None)
    # representative = first group of every hash value; verify every group against its representative
    first = torch.full((nu,), ng, dtype=torch.int64, device=dev)
    first.scatter_reduce_(0, inverse, torch.arange(ng, device=dev), reduce='amin')
    rep = first[inverse]
    ok = True
    for g0 in range(0, ng, step):
        g1 = min(ng, g0 + step)
        if not bool(torch.equal(v3[g0:g1].view(torch.int32), v3[rep[g0:g1]].view(torch.int32))):
            ok = False
            break
    if not ok:
        nbad = int(sum(int((v3[g0:min(ng, g0 + step)].view(torch.int32) != v3[rep[g0:min(ng, g0 + step)]].view(torch.int32)).flatten(1).any(dim=1).sum()) for g0 in range(0, ng, step)))
        warnings.warn('value-block hash collision: blocks of this class are stored per group (G=%d K_pad=%d groups=%d unique hashes=%d mismatching groups=%d)' % (G, K_pad, ng, nu, nbad))
        return (cols, vals, None)
    vals_u = v3[first].contiguous().view(-1)
    return (cols, vals_u, inverse.to(torch.int32).contiguous())


class PatternGroups(object):
    """Rows with an identical column set, packed as dense value blocks (see csrc/pgroup.cu).

    classes: list of dict(G, K_pad, n_groups, rows int32[n_groups*G], cols int32[n_groups*K_pad], vals f32[n_groups*G*K_pad])
    rest:    rows not covered by a group, as a compact CSR + out_rows int32 (None if every row is grouped)
    Grouping / sorting uses torch device ops (build-time plumbing); hashing, verification, packing and the
    product itself are kernels of libkeynet_b200."""

    TC_MIN_G = 32          # groups at least this tall are "true small GEMMs": tcgen05 path
    TC_MIN_BATCH = 128
    TC_MAX_K = 32768       # the group's column list is staged in shared memory next to the weight ring
    TC_MIN_K = 128         # shorter reductions do not amortise the per-CTA TMEM / barrier set-up: fp32 FMA kernel

    def __init__(self):
        self.classes = []
        self.rest = None
        self.shape = None
        self.grouped_rows = 0
        self.padded_values = 0

    @staticmethod
    def build(W, min_group=4, max_pad_waste=0.25, dedup=True, hint=None):
        """max_pad_waste: a class is split when a group's K falls below this fraction of the class maximum.
        hint: optional int64 CUDA tensor [n_rows], a spatial cluster id per row (rows of neighbouring output pixels share
        an id, < 0 = none): classes of small groups (G <= 16) are then also stored clustered (csrc/pgcluster.cu)."""
        L = _native.lib()
        dev = W._data.device
        (R, C) = W.shape
        pg = PatternGroups()
        pg.shape = W.shape
        (indptr, indices, data) = (W._indptr, W._indices, W._data)
        if indptr[0].item() != 0:                      # row-slice view: rebase offsets
            (indices, data) = (indices[indptr[0]:indptr[-1]], data[indptr[0]:indptr[-1]])
            indptr = indptr - indptr[0]
        h = torch.empty(R, dtype=torch.int64, device=dev)
        check(L.kn_csr_row_pattern_hash(ptr(indptr), ptr(indices), R, ptr(h), stream_ptr()))
        (hs, order) = torch.sort(h)
        new = torch.ones(R, dtype=torch.bool, device=dev)
        new[1:] = hs[1:] != hs[:-1]
        gid = torch.cumsum(new.to(torch.int64), 0) - 1
        start = torch.nonzero(new).reshape(-1)                       # first position of every group in `order`
        gsize = torch.diff(torch.cat([start, torch.tensor([R], device=dev)]))
        leader = order[start]
        # a 64-bit hash collision would merge different patterns: verify every row against its group leader
        mismatch = torch.empty(R, dtype=torch.int32, device=dev)
        check(L.kn_pg_verify(ptr(indptr), ptr(indices), ptr(order), ptr(leader[gid].contiguous()), R, ptr(mismatch), stream_ptr()))
        if bool(mismatch.any()):
            warnings.warn('pattern hash collision: matrix stays on the CSR kernel')
            return None
        nnz_row = indptr[1:] - indptr[:-1]
        K = nnz_row[leader]
        first_col = torch.where(K > 0, indices[indptr[leader].clamp(max=max(indices.numel() - 1, 0))].to(torch.int64), torch.full_like(K, C))
        sel = (gsize >= min_group) & (K > 0)
        in_group = torch.zeros(R, dtype=torch.bool, device=dev)
        for G in torch.unique(gsize[sel]).tolist():
            gi = torch.nonzero(sel & (gsize == G)).reshape(-1)
            # one class per group height: groups share K_pad (storage) and carry their own K, so border pixels with
            # fewer taps cost neither extra launches nor padded arithmetic.  Only a very ragged class is split.
            Ks = K[gi]
            (Ks_sorted, o) = torch.sort(Ks, descending=True)
            gi = gi[o]
            bounds = [0]
            Kl = Ks_sorted.tolist()
            for (j, k) in enumerate(Kl):
                if k < max_pad_waste * Kl[bounds[-1]]:
                    bounds.append(j)
            bounds.append(len(Kl))
            for (b0, b1) in zip(bounds[:-1], bounds[1:]):
                g_sub = gi[b0:b1]
                g_sub = g_sub[torch.argsort(first_col[g_sub])]       # neighbouring CTAs gather neighbouring X rows
                cid = None
                if hint is not None and int(G) <= PatternGroups.CG_MAX_G:
                    cid = hint[leader[g_sub]]
                    if bool((cid >= 0).all()):
                        o2 = torch.argsort(cid, stable=True)         # groups stored cluster by cluster
                        (g_sub, cid) = (g_sub[o2], cid[o2])
                    else:
                        cid = None
                K_pad = int((Kl[b0] + 31) // 32 * 32)
                ng = int(g_sub.numel())
                pos = (start[g_sub].reshape(-1, 1) + torch.arange(G, device=dev).reshape(1, -1)).reshape(-1)
                rows64 = order[pos].contiguous()
                # ascending row ids inside a group: deterministic output layout
                rows64 = torch.sort(rows64.reshape(ng, G), dim=1)[0].reshape(-1).contiguous()
                cols = torch.empty(ng * K_pad, dtype=torch.int32, device=dev)
                vals = torch.empty(ng * G * K_pad, dtype=torch.float32, device=dev)
                check(L.kn_pg_pack(ptr(indptr), ptr(indices), ptr(data), ptr(rows64), ng, int(G), K_pad, ptr(cols), ptr(vals), stream_ptr()))
                group_k = K[g_sub].to(torch.int32).contiguous()
                block_of = None
                if dedup and ng > 1:
                    (cols, vals, block_of) = _dedup_value_blocks(cols, vals, group_k, ng, int(G), K_pad)
                cls = dict(G=int(G), K_pad=K_pad, n_groups=ng, rows=rows64.to(torch.int32), cols=cols, vals=vals, tc=None,
                           group_k=group_k, block_of=block_of, n_blocks=ng if block_of is None else int(vals.numel() // (int(G) * K_pad)))
                PatternGroups._finish_class(cls, int(Kl[b0]), cid, C)
                pg.classes.append(cls)
                in_group[rows64] = True
                pg.grouped_rows += ng * int(G)
                pg.padded_values += cls['n_blocks'] * int(G) * K_pad
        rest_rows = torch.nonzero(~in_group).reshape(-1)
        if rest_rows.numel() > 0:
            n = int(rest_rows.numel())
            csr = _two_phase(
                n,
                lambda row_nnz: check(L.kn_csr_gather_rows_count(ptr(indptr), ptr(rest_rows), n, ptr(row_nnz), stream_ptr())),
                lambda ip, ix, dt: check(L.kn_csr_gather_rows_fill(ptr(indptr), ptr(indices), ptr(data), ptr(rest_rows), n, ptr(ip), ptr(ix), ptr(dt), stream_ptr())),
                dev)
            pg.rest = dict(n=n, indptr=csr[0], indices=csr[1], data=csr[2], out_rows=rest_rows.to(torch.int32))
        if len(pg.classes) == 0:
            return None
        return pg

    @staticmethod
    def _finish_class(cls, K_max, cid, n_cols):
        """Execution extras of one class: TF32 hi/lo planes + TMA descriptors for the tensor-core kernel, K slices for a
        single tall group (dense fc layers), the clustered form for short reductions (cid: cluster id per group, sorted)."""
        (G, K_pad, ng, vals) = (cls['G'], cls['K_pad'], cls['n_groups'], cls['vals'])
        if G >= PatternGroups.TC_MIN_G and PatternGroups.TC_MIN_K <= K_pad <= PatternGroups.TC_MAX_K and tensor_cores_enabled():
            cls['tc'] = _tc_planes(vals, cls['n_blocks'] * G, G, K_pad)
        if cls['tc'] is not None and ng == 1 and K_max >= PatternGroups.SPLITK_MIN_K:
            cls['splitk'] = PatternGroups._split_k(cls, int(K_max))
        if cid is not None and K_pad <= PatternGroups.CG_KERNEL_MAX_K:
            cls['cg'] = PatternGroups._cluster(cls, cid, n_cols)
        return cls

    SPLITK_MAX_BATCH = 1024  # wider batches already give every SM a batch tile
    SPLITK_MIN_K = 2048      # a single group with a reduction at least this long is cut into K slices (dense fc layers)

    @staticmethod
    def _split_k(cls, K):
        """A class that is ONE group (all rows of a dense layer share the column set): S groups over K slices writing partial
        rows, so that row chunks x S >= the SM count.  Returns the inner class dict (own TF32 planes and TMA descriptors)."""
        (G, K_pad) = (cls['G'], cls['K_pad'])
        dev = cls['vals'].device
        chunks = -(-G // 256) if G > 256 else 1                        # row chunks of the tensor-core kernel
        S = max(2, min(-(-148 // chunks), K // 512))
        Kp = (-(-K // S) + 31) // 32 * 32
        S = -(-K // Kp)
        cols = cls['cols'][:K].to(torch.int64)
        vals = cls['vals'].reshape(G, K_pad)[:, :K]
        pad = S * Kp - K
        cols_s = torch.cat([cols, cols[-1:].expand(pad)]).reshape(S, Kp).to(torch.int32).contiguous()
        vals_s = torch.cat([vals, torch.zeros((G, pad), dtype=torch.float32, device=dev)], dim=1).reshape(G, S, Kp).permute(1, 0, 2).contiguous().reshape(-1)
        group_k = torch.tensor([min(Kp, K - s * Kp) for s in range(S)], dtype=torch.int32, device=dev)
        return dict(S=S, G=G, K_pad=Kp, rows=torch.arange(S * G, dtype=torch.int32, device=dev), cols=cols_s.reshape(-1), group_k=group_k,
                    tc=_tc_planes(vals_s, S * G, G, Kp), part={})

    CG_MAX_G = 128           # groups up to this height are ordered by their spatial hint (L1 / L2 locality of the gathers)
    CG_KERNEL_MAX_K = 32     # ... and run on the clustered kernel when the reduction is short (K_pad <= 32: first conv layers,
                             # 1 or 3 input channels): there the product is bound by L2 -> SM gather traffic and per-CTA latency
                             # (measured: LeNet conv1 0.48 -> 0.34 ms); LeNet conv2 (G=16, K=55) is FMA-bound: pg_small
    CG_MAX_UNION = 224       # KN_CG_MAX_UNION: rows of the staged tile (224 x 512 B = 112 KB, two CTAs per SM)
    CG_MAX_BYTES = 256 << 20

    @staticmethod
    def _cluster(cls, cid, n_cols):
        """Clustered form of a class of small groups (kn_spmm_cg_f32): union column list per cluster, per-group byte
        offsets into the staged tile, k-major value blocks.  cid: sorted int64 cluster id of every group."""
        (G, K_pad, ng) = (cls['G'], cls['K_pad'], cls['n_groups'])
        dev = cid.device
        GM = (G + 1) // 2 * 2 if G <= 16 else (G + 15) // 16 * 16
        n_blocks = cls['n_blocks']
        if (n_blocks * K_pad * GM + ng * K_pad) * 4 > PatternGroups.CG_MAX_BYTES:
            return None
        (ucid, cl_of_group) = torch.unique_consecutive(cid, return_inverse=True)
        n_cl = int(ucid.numel())
        cols = cls['cols'].reshape(ng, K_pad).to(torch.int64)
        key = cl_of_group.reshape(-1, 1) * int(n_cols) + cols                       # (cluster, column), row-major
        (uniq, inv) = torch.unique(key.reshape(-1), sorted=True, return_inverse=True)
        ucl = uniq // int(n_cols)
        cl_uptr = torch.zeros(n_cl + 1, dtype=torch.int64, device=dev)
        cl_uptr[1:] = torch.cumsum(torch.bincount(ucl, minlength=n_cl), 0)
        u_max = int((cl_uptr[1:] - cl_uptr[:-1]).max())
        cl_gcount = torch.bincount(cl_of_group, minlength=n_cl)
        g_max = int(cl_gcount.max())
        if u_max * 512 + g_max * K_pad * 4 > PatternGroups.CG_MAX_UNION * 512:
            return None
        lidx = ((inv.reshape(ng, K_pad) - cl_uptr[cl_of_group].reshape(-1, 1)) * 512).to(torch.int32).contiguous()
        cl_gptr = torch.zeros(n_cl + 1, dtype=torch.int64, device=dev)
        cl_gptr[1:] = torch.cumsum(cl_gcount, 0)
        vT = torch.zeros((n_blocks, K_pad, GM), dtype=torch.float32, device=dev)
        vT[:, :, :G] = cls['vals'].reshape(n_blocks, G, K_pad).permute(0, 2, 1)
        return dict(n_clusters=n_cl, u_max=u_max, g_max=g_max, cl_gptr=cl_gptr.to(torch.int32), cl_uptr=cl_uptr.to(torch.int32), ucols=(uniq % int(n_cols)).to(torch.int32),
                    lidx=lidx, valsT=vT.contiguous())

    def spmm(self, x, y, relu, peers=None):
        """peers: _native.Peers (the output slot on every rank + need mask, dist.py) or None for plain stores to y."""
        L = _native.lib()
        N = x.shape[1]
        flags = _native.KN_SPMM_RELU if relu else 0
        pp = _native.peers_arg(peers)
        for c in self.classes:
            cg = c.get('cg')
            if cg is not None and clusters_enabled():
                check(L.kn_spmm_cg_f32(ptr(cg['cl_gptr']), ptr(cg['cl_uptr']), ptr(cg['ucols']), ptr(c['rows']), ptr(cg['lidx']), ptr(cg['valsT']), ptr(c['group_k']), ptr(c['block_of']),
                                       cg['n_clusters'], c['G'], c['K_pad'], cg['u_max'], cg['g_max'], ptr(x), N, ptr(y), N, N, flags, pp, stream_ptr()))
            elif c.get('splitk') is not None and N >= PatternGroups.TC_MIN_BATCH and N <= PatternGroups.SPLITK_MAX_BATCH and tensor_cores_enabled():
                k = c['splitk']
                part = k['part'].get(N)
                if part is None:
                    part = k['part'][N] = torch.empty((k['S'] * k['G'], N), dtype=torch.float32, device=x.device)
                check(L.kn_spmm_pg_tc_f32(k['tc']['maps'], ptr(k['rows']), ptr(k['cols']), ptr(k['group_k']), None, k['S'], k['G'], k['K_pad'],
                                          ptr(x), N, ptr(part), N, N, 0, None, stream_ptr()))       # the partial rows are local scratch
                check(L.kn_splitk_reduce_f32(ptr(part), k['S'], k['G'], ptr(c['rows']), ptr(y), N, N, flags, pp, stream_ptr()))
            elif c.get('tile') is not None and N >= PatternGroups.TC_MIN_BATCH and tensor_cores_enabled() and tiles_enabled():
                t = c['tile']
                check(L.kn_spmm_tile_tc_f32(t['maps'], ptr(t['cols']), ptr(t['rows']), t['bias_col'], t['n_tiles'], t['C'], t['G'], t['th'], t['tw'], t['stride'], t['P'], t['Q'],
                                            ptr(x), N, ptr(y), N, N, flags, pp, stream_ptr()))
            elif c['tc'] is not None and N >= PatternGroups.TC_MIN_BATCH and tensor_cores_enabled():
                check(L.kn_spmm_pg_tc_f32(c['tc']['maps'], ptr(c['rows']), ptr(c['cols']), ptr(c['group_k']), ptr(c['block_of']), c['n_groups'], c['G'], c['K_pad'],
                                          ptr(x), N, ptr(y), N, N, flags, pp, stream_ptr()))
            else:
                check(L.kn_spmm_pg_f32(ptr(c['rows']), ptr(c['cols']), ptr(c['vals']), ptr(c['group_k']), ptr(c['block_of']), c['n_groups'], c['G'], c['K_pad'],
                                       ptr(x), N, ptr(y), N, N, flags, pp, stream_ptr()))
        r = self.rest
        if r is not None:
            check(L.kn_spmm_csr_rows_f32(ptr(r['indptr']), ptr(r['indices']), ptr(r['data']), r['n'], self.shape[1], ptr(r['out_rows']),
                                         ptr(x), N, ptr(y), N, N, flags, pp, stream_ptr()))

    NARROW_TILE = 128        # batch-column slots of pg_simt's tile: a run of the narrow path holds up to 128 / NB groups

    @staticmethod
    def _run_table(cls, P):
        """The class's groups ordered by (value block, group_k) and cut into runs of at most P groups that share both:
        dict(groups int32 [n_groups] run by run, start int32 [n_runs + 1], n_runs)."""
        ng = cls['n_groups']
        dev = cls['cols'].device
        blk = cls['block_of'].to(torch.int64) if cls['block_of'] is not None else torch.arange(ng, dtype=torch.int64, device=dev)
        key = blk * (cls['K_pad'] + 1) + cls['group_k'].to(torch.int64)
        (ks, order) = torch.sort(key, stable=True)
        new = torch.ones(ng, dtype=torch.bool, device=dev)
        new[1:] = ks[1:] != ks[:-1]
        seg_start = torch.nonzero(new).reshape(-1)
        pos = torch.arange(ng, device=dev) - seg_start[torch.cumsum(new.to(torch.int64), 0) - 1]     # position inside its block
        start = torch.nonzero(pos % P == 0).reshape(-1)
        start = torch.cat([start, torch.tensor([ng], device=dev)]).to(torch.int32).contiguous()
        return dict(groups=order.to(torch.int32).contiguous(), start=start, n_runs=int(start.numel()) - 1)

    @staticmethod
    def _narrow_plan(cls, N):
        """How the class runs at 1 <= N < 32 batch columns (cached per NB on the class: built by the first call, so a CUDA
        graph captured after a warm-up run allocates nothing).  Row form (row_form = 1: one warp per row, lanes over K) when
        NB <= 8 and the shared-block tile would be less than a quarter full (mean run length x NB < 32 of its 128 columns);
        shared-block form otherwise.  Dense fc layers (one group) and gain-keyed layers (a block per group) take the row form
        up to N = 8; convolutions under permutation keys take the shared form except where few pixels share a block (VGG16
        conv5 at N = 1: 196 pixels, ~20 per run)."""
        NB = 1 << max(0, (int(N) - 1).bit_length())
        plans = cls.setdefault('narrow', {})
        p = plans.get(NB)
        if p is None:
            p = PatternGroups._run_table(cls, PatternGroups.NARROW_TILE // NB)
            p.update(NB=NB, row_form=int(NB <= 8 and cls['n_groups'] * NB < 32 * p['n_runs']))
            plans[NB] = p
        return p

    def spmm_narrow(self, x, y, relu):
        """Y = W . X for 1 <= N < 32 batch columns, no output peers (kn_spmm_pg_narrow_f32): no padding of the batch."""
        L = _native.lib()
        N = x.shape[1]
        assert 1 <= N < 32
        flags = _native.KN_SPMM_RELU if relu else 0
        for c in self.classes:
            p = PatternGroups._narrow_plan(c, N)
            check(L.kn_spmm_pg_narrow_f32(ptr(c['rows']), ptr(c['cols']), ptr(c['vals']), ptr(c['group_k']), ptr(c['block_of']), c['n_groups'], c['G'], c['K_pad'],
                                          ptr(p['groups']), ptr(p['start']), p['n_runs'], p['row_form'],
                                          ptr(x), N, ptr(y), N, N, flags, None, stream_ptr()))
        r = self.rest
        if r is not None:
            check(L.kn_spmm_csr_rows_f32(ptr(r['indptr']), ptr(r['indices']), ptr(r['data']), r['n'], self.shape[1], ptr(r['out_rows']),
                                         ptr(x), N, ptr(y), N, N, flags, None, stream_ptr()))

    def launches_narrow(self):
        """Kernel launches of spmm_narrow: one per class and one for `rest`."""
        return len(self.classes) + (1 if self.rest is not None else 0)

    def launches(self):
        return sum(2 if c.get('splitk') is not None else 1 for c in self.classes) + (1 if self.rest is not None else 0)

    def summary(self):
        return dict(classes=[(c['G'], c['K_pad'], c['n_groups']) for c in self.classes], unique_blocks=[c['n_blocks'] for c in self.classes], tensor_core=[c['tc'] is not None for c in self.classes], grouped_rows=self.grouped_rows,
                    rest_rows=0 if self.rest is None else self.rest['n'], padded_values=self.padded_values)


# =============================================================================================
# SpMM
# =============================================================================================
def spmm(W, x, relu=False, out=None, peers=None):
    """y[R, N] = W . x[C, N] (+ReLU) on the current CUDA stream.  x: contiguous float32 CUDA tensor.
    peers (_native.Peers): store every output row into the same slot of several ranks' buffers instead (fused all-gather)."""
    assert x.is_cuda and x.dtype == torch.float32 and x.ndim == 2 and x.is_contiguous()
    assert x.shape[0] == W.shape[1], "Non-conformal shape for W=%s, x=%s" % (str(W.shape), str(tuple(x.shape)))
    (R, N) = (W.shape[0], x.shape[1])
    y = out if out is not None else torch.empty((R, N), dtype=torch.float32, device=x.device)
    assert y.shape == (R, N) and y.is_contiguous()
    if W._pg is not None and N >= 32 and N % 4 == 0:
        W._pg.spmm(x, y, relu, peers)
        return y
    if W._data is None:
        # the grouped kernels would store into the peers' buffers with leading dimension Np: the fused row-sharded path
        # must pad its batch itself (dist.ShardedKeyedModel does)
        assert peers is None, 'ragged batch on a dropped-CSR matrix with output peers: the fused row-sharded path pads its batch itself'
        if 0 < N < 32:
            W._pg.spmm_narrow(x, y, relu)
            return y
        # CSR was dropped (drop_csr): ragged batches are padded to the grouped kernels' granularity
        Np = max(32, (N + 3) // 4 * 4)
        xp = torch.zeros((x.shape[0], Np), dtype=torch.float32, device=x.device)
        xp[:, :N] = x
        yp = torch.empty((R, Np), dtype=torch.float32, device=x.device)
        W._pg.spmm(xp, yp, relu)
        y.copy_(yp[:, :N])
        return y
    ex = getattr(W, '_exec', None)
    if ex is not None and peers is None and N >= 32:
        check(_native.lib().kn_spmm_csr_rows_f32(ptr(ex['indptr']), ptr(ex['indices']), ptr(ex['data']), ex['n'], W.shape[1], ptr(ex['out_rows']),
                                                 ptr(x), N, ptr(y), N, N, _native.KN_SPMM_RELU if relu else 0, None, stream_ptr()))
        return y
    check(_native.lib().kn_spmm_csr_f32(ptr(W._indptr), ptr(W._indices), ptr(W._data), R, W.shape[1],
                                        ptr(x), N, ptr(y), N, N, _native.KN_SPMM_RELU if relu else 0, _native.peers_arg(peers), stream_ptr()))
    return y


# =============================================================================================
# Toeplitz construction + key compile
# =============================================================================================
def _offset_round(values, emitted_min):
    """fl32(fl32(w + off) - off) with off = fl32(|min|+1): the reference's sparsity-preserving offset
    (keynet/sparse.py:184-187,193-196) leaves every stored value rounded this way."""
    off = np.float32(np.abs(np.float32(emitted_min)) + np.float32(1.0))
    v = (np.asarray(values, dtype=np.float32) + off).astype(np.float32)
    return (v - off).astype(np.float32)


def _emitted_taps(U, k, stride):
    """Which of the k taps along one axis are ever in bounds for some strided output position."""
    h = (k - 1) // 2
    u = np.arange(0, U, stride)
    return np.array([np.any((u + p >= 0) & (u + p < U)) for p in range(-h, h + 1)])


def _keycompile(csr, n_rows, n_cols, A, Ainv, dev, row_scale_slice=None, keep_zeros=False):
    """Apply column map/scales of Ainv and row scales of A to an already row-gathered CSR."""
    (indptr, indices, data) = csr
    L = _native.lib()
    row_scale = None
    if A is not None and not A.is_unscaled():
        rs = A.scale if row_scale_slice is None else A.scale[row_scale_slice]
        row_scale = torch.from_numpy(np.ascontiguousarray(rs)).to(dev)
    (col_map, col_scale, row_bias, col_bias) = (None, None, None, None)
    if A is not None and A.bias is not None:
        rb = A.bias if row_scale_slice is None else A.bias[row_scale_slice]
        row_bias = torch.from_numpy(np.ascontiguousarray(rb)).to(dev)
    if Ainv is not None and Ainv.bias is not None:
        col_bias = torch.from_numpy(Ainv.bias).to(dev)
    n_cols_out = n_cols if Ainv is None else int(Ainv.shape[1])      # physical column space of the compiled matrix
    if Ainv is not None:
        assert Ainv.shape[0] == n_cols
        if Ainv.shape[0] != Ainv.shape[1] or not Ainv.is_unpermuted():
            col_map = torch.from_numpy(Ainv.perm.astype(np.int32)).to(dev)
        if not Ainv.is_unscaled():
            col_scale = torch.from_numpy(Ainv.scale).to(dev)
    return _two_phase(
        n_rows,
        lambda row_nnz: check(L.kn_keycompile_count(ptr(indptr), ptr(indices), ptr(data), n_rows, ptr(row_scale), ptr(col_scale), ptr(row_bias), ptr(col_bias), n_cols, int(keep_zeros), ptr(row_nnz), stream_ptr())),
        lambda ip, ix, dt: check(L.kn_keycompile_fill(ptr(indptr), ptr(indices), ptr(data), n_rows, n_cols_out, ptr(col_map), ptr(row_scale), ptr(col_scale), ptr(row_bias), ptr(col_bias), n_cols, int(keep_zeros),
                                                      ptr(ip), ptr(ix), ptr(dt), stream_ptr())),
        dev)


def _row_ids(A, n_total_rows, rows, dev):
    """Source row of every output row.  rows = None (all), (r0, r1) (a contiguous shard of W_hat's rows) or an int64
    array of W_hat row indices in the order the shard stores them (row-sharding by whole pattern groups, dist.py).
    Returns (device row ids | None, selection) where selection indexes A.scale (slice or array)."""
    if rows is not None and not isinstance(rows, tuple):
        sel = np.ascontiguousarray(rows, dtype=np.int64)
        assert sel.ndim == 1 and (len(sel) == 0 or (sel.min() >= 0 and sel.max() < n_total_rows))
        src = sel if (A is None) else A.perm[sel]
        return (torch.from_numpy(np.ascontiguousarray(src)).to(dev), sel)
    (r0, r1) = (0, n_total_rows) if rows is None else (int(rows[0]), int(rows[1]))
    assert 0 <= r0 <= r1 <= n_total_rows
    if A is None or A.is_unpermuted():
        ids = None if (r0 == 0 and r1 == n_total_rows) else torch.arange(r0, r1, dtype=torch.int64, device=dev)
    else:
        ids = torch.from_numpy(np.ascontiguousarray(A.perm[r0:r1])).to(dev)
    return (ids, slice(r0, r1))


def _n_selected(sel, n_total):
    return len(sel) if not isinstance(sel, slice) else (sel.stop - sel.start)


def _remapped(Ainv, col_remap, n_cols_phys):
    """Fold a physical column layout into the input key: column c of the canonical matrix lives at position
    col_remap[c] of an activation buffer with n_cols_phys rows (the all-gathered, shard-major layout of dist.py)."""
    if col_remap is None:
        return (Ainv, Ainv.shape[0])
    col_remap = np.ascontiguousarray(col_remap, dtype=np.int64)
    assert len(col_remap) == Ainv.shape[0] and n_cols_phys > int(col_remap.max())
    K = MonomialKey(Ainv.perm, Ainv.scale, Ainv.bias)          # the bias column rides along: position[R] is the last physical row
    assert Ainv.bias is None or int(col_remap[-1]) == int(n_cols_phys) - 1, 'homogeneous coordinate must stay the last gathered row'
    K._perm = col_remap[Ainv.perm]           # no longer square: only used as (col_map, col_scale, col_bias) by _keycompile
    K._unpermuted = False
    K.shape = (Ainv.shape[0], int(n_cols_phys))
    return (K, int(n_cols_phys))


def _toeplitz_rows(desc, weight, bias, ids, n_rows, dev):
    L = _native.lib()
    w = torch.from_numpy(np.ascontiguousarray(weight, dtype=np.float32)).to(dev)
    b = torch.from_numpy(np.ascontiguousarray(bias, dtype=np.float32)).to(dev) if bias is not None else None
    return _two_phase(
        n_rows,
        lambda row_nnz: check(L.kn_toeplitz_conv2d_count(desc, ptr(ids), n_rows, ptr(row_nnz), stream_ptr())),
        lambda ip, ix, dt: check(L.kn_toeplitz_conv2d_fill(desc, ptr(w), ptr(b), ptr(ids), n_rows, ptr(ip), ptr(ix), ptr(dt), stream_ptr())),
        dev)


def _conv_weights_rounded(inshape, f, bias, stride):
    (C, U, V) = [int(s) for s in inshape]
    f = np.ascontiguousarray(f, dtype=np.float32)
    (M, C2, P, Q) = f.shape
    assert len(inshape) == 3 and f.ndim == 4
    assert C2 == C, 'filter in-channels %d != input channels %d' % (C2, C)
    assert P == Q and P % 2 == 1, 'filter must be square and odd'
    assert U % stride == 0 and V % stride == 0, 'image size must be divisible by the stride'
    mask = np.outer(_emitted_taps(U, P, stride), _emitted_taps(V, Q, stride))
    fq = _offset_round(f, np.min(f[:, :, mask]))
    bq = None
    if bias is not None:
        bias = np.ascontiguousarray(bias, dtype=np.float32)
        assert bias.shape == (M,)
        bq = _offset_round(bias, np.min(bias))
    return (fq, bq, (C, U, V, M, P, Q))


def _axis_class(U, k, stride):
    """Per output position along one axis: (first in-bounds tap offset + h) * (k+1) + number of in-bounds taps."""
    h = (k - 1) // 2
    u = np.arange(0, U, stride)
    lo = np.maximum(-h, -u)
    hi = np.minimum(h, U - 1 - u)
    return ((lo + h) * (k + 1) + np.maximum(0, hi - lo + 1)).astype(np.int64)


def _keyed_conv_direct(geom, wq, bq, A, Ainv, rows, col_remap, n_cols_phys, want_csr, build_groups, dev, clustered=False):
    """Fused compile of a conv / linear layer under monomial keys (csrc/keyedconv.cu): canonical CSR written in one pass
    with one column sort per output pixel (want_csr) and / or the pattern-group execution format straight from the
    geometry (build_groups).  Returns a SparseMatrix, or None when the keys / the shard do not fit this route (bias
    columns, a shard that cuts through a pixel's channel rows): the caller then takes the two-kernel path."""
    (C, U, V, M, P, Q, stride, has_bias) = geom
    L = _native.lib()
    if (A is not None and A.bias is not None) or Ainv.bias is not None:
        return None
    (Uo, Vo) = (U // stride, V // stride)
    UoVo = Uo * Vo
    R_src = M * UoVo + 1
    K_src = C * U * V + 1
    desc = kn_conv2d_desc(C, U, V, M, P, Q, int(stride), 0, 1 if has_bias else 0)
    # ---- which compiled row holds which Toeplitz row
    if rows is None:
        (n, sel) = (R_src, slice(0, R_src))
        src = None if (A is None or A.is_unpermuted()) else A.perm
    elif isinstance(rows, tuple):
        sel = slice(int(rows[0]), int(rows[1]))
        n = sel.stop - sel.start
        src = (np.arange(sel.start, sel.stop, dtype=np.int64) if A is None else A.perm[sel])
    else:
        sel = np.ascontiguousarray(rows, dtype=np.int64)
        n = len(sel)
        src = sel if A is None else A.perm[sel]
    if n == 0:
        return None
    if src is None:
        (row_of_src, pix, pix_np, n_groups) = (None, None, np.arange(UoVo, dtype=np.int64), UoVo)
    else:
        inv = np.full(R_src, -1, dtype=np.int32)
        inv[src] = np.arange(n, dtype=np.int32)
        main = src[src < R_src - 1]
        pix_np = np.unique(main % UoVo) if rows is not None else np.arange(UoVo, dtype=np.int64)
        if len(main) != M * len(pix_np):
            return None                                  # the shard cuts through a pixel's channel rows
        row_of_src = torch.from_numpy(inv).to(dev)
        n_groups = len(pix_np)
        pix = None if n_groups == UoVo else torch.from_numpy(pix_np.astype(np.int32)).to(dev)
    # ---- keys as vectors
    (AinvP, Kp) = _remapped(Ainv, col_remap, n_cols_phys)
    assert Ainv.shape[0] == K_src
    col_map = None
    if AinvP.shape[0] != AinvP.shape[1] or not AinvP.is_unpermuted():
        col_map = torch.from_numpy(AinvP.perm.astype(np.int32)).to(dev)
    col_scale = None if Ainv.is_unscaled() else torch.from_numpy(Ainv.scale).to(dev)
    row_scale = None
    if A is not None and not A.is_unscaled():
        row_scale = torch.from_numpy(np.ascontiguousarray(A.scale[sel])).to(dev)
    as_dev = lambda t: t.detach().to(device=dev, dtype=torch.float32).contiguous() if torch.is_tensor(t) else torch.from_numpy(np.ascontiguousarray(t, dtype=np.float32)).to(dev)
    w = as_dev(wq)                                       # (a device tensor is used as is: no host round trip for a 411 MB fc6)
    b = as_dev(bq) if has_bias else None
    # ---- canonical CSR (or only its row counts: nnz() of a layer that never holds a CSR)
    indptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    check(L.kn_keyed_conv2d_count(desc, ptr(w), ptr(b), ptr(pix), n_groups, ptr(row_of_src), ptr(row_scale), ptr(col_scale), 0, ptr(indptr[1:]), stream_ptr()))
    _scan_counts_inplace(indptr)
    nnz = int(indptr[-1].item())
    W = SparseMatrix()
    W.shape = (n, Kp)
    if want_csr:
        indices = torch.empty(nnz, dtype=torch.int32, device=dev)
        data = torch.empty(nnz, dtype=torch.float32, device=dev)
        if nnz > 0:
            rc = L.kn_keyed_conv2d_fill(desc, ptr(w), ptr(b), ptr(pix), n_groups, ptr(row_of_src), ptr(col_map), ptr(row_scale), ptr(col_scale), 0,
                                        ptr(indptr), ptr(indices), ptr(data), stream_ptr())
            if rc == _native.KN_ERR_UNSUPPORTED:
                return None                              # more taps per pixel than the shared-memory sort holds
            check(rc)
        (W._indptr, W._indices, W._data) = (indptr, indices, data)
    else:
        (W._nnz, W._device) = (nnz, dev)
        del indptr
    if not (build_groups and M >= 4 and nnz >= 4096 and n_groups > 0):
        return W if want_csr else None
    # ---- pattern groups: one per output pixel, one class per layer
    K_pad = (C * P * Q + (1 if has_bias else 0) + 31) // 32 * 32
    cid = None
    if clustered and M <= PatternGroups.CG_MAX_G and K_pad <= PatternGroups.CG_KERNEL_MAX_K:
        # groups stored tile by tile for the clustered kernel (csrc/pgcluster.cu): t x t output pixels whose union of taps
        # fits its staging buffer
        staged = lambda t: (((t - 1) * stride + P) ** 2 * C + 1) * 512 + t * t * K_pad * 4
        t = 0
        while t < max(Uo, Vo) and staged(t + 1) <= PatternGroups.CG_MAX_UNION * 512:
            t += 1
        if t > 0:
            for dd in range(t, max(1, t // 2), -1):
                if Uo % dd == 0 and Vo % dd == 0:
                    t = dd
                    break
            tile = (pix_np // Vo // t) * (-(-Vo // t)) + (pix_np % Vo) // t
            o = np.argsort(tile, kind='stable')
            (pix_np, tile) = (pix_np[o], tile[o])
            pix = torch.from_numpy(pix_np.astype(np.int32)).to(dev)
            cid = torch.from_numpy(tile.astype(np.int64)).to(dev)
    ng = n_groups
    rows_t = torch.empty(ng * M, dtype=torch.int32, device=dev)
    cols = torch.empty(ng * K_pad, dtype=torch.int32, device=dev)
    group_k = torch.empty(ng, dtype=torch.int32, device=dev)
    check(L.kn_conv2d_groups_index(desc, ptr(pix), ng, ptr(row_of_src), ptr(col_map), K_pad, ptr(rows_t), ptr(cols), ptr(group_k), stream_ptr()))
    scaled = row_scale is not None or col_scale is not None
    block_of = None
    if scaled or ng == 1:
        block_pix = pix if pix is not None else torch.arange(ng, dtype=torch.int32, device=dev)
        n_blocks = ng
    else:
        # permutation-only keys: the value block depends only on which taps are in bounds
        key = _axis_class(U, P, stride)[pix_np // Vo] * ((P + 1) * (P + 1) + 1) + _axis_class(V, Q, stride)[pix_np % Vo]
        (_, first, inverse) = np.unique(key, return_index=True, return_inverse=True)
        n_blocks = len(first)
        block_pix = torch.from_numpy(pix_np[first].astype(np.int32)).to(dev)
        block_of = torch.from_numpy(inverse.astype(np.int32)).to(dev)
    vals = torch.empty(n_blocks * M * K_pad, dtype=torch.float32, device=dev)
    check(L.kn_conv2d_groups_values(desc, ptr(w), ptr(b), ptr(block_pix), n_blocks, ptr(row_of_src), ptr(row_scale), ptr(col_scale), K_pad, ptr(vals), stream_ptr()))
    pg = PatternGroups()
    pg.shape = W.shape
    cls = dict(G=M, K_pad=K_pad, n_groups=ng, rows=rows_t, cols=cols, vals=vals, tc=None, group_k=group_k, block_of=block_of, n_blocks=n_blocks)
    PatternGroups._finish_class(cls, C * P * Q + (1 if has_bias else 0), cid, Kp)
    if cls['tc'] is not None and not scaled and has_bias and UoVo > 1:
        cls['tile'] = _conv_tiles(desc, (C, U, V, M, P, Q, int(stride)), wq, bq, pix_np, row_of_src, col_map, int(AinvP.perm[K_src - 1]), dev)
    pg.classes.append(cls)
    pg.grouped_rows = ng * M
    pg.padded_values = n_blocks * M * K_pad
    # the homogeneous row e_last (one entry) is the only row outside the groups
    r_h = (R_src - 1) if src is None else int(inv[R_src - 1])
    if r_h >= 0:
        v = np.float32(1.0)
        if A is not None and not A.is_unscaled():
            v = np.float32(A.scale[sel][r_h] * v)
        if not Ainv.is_unscaled():
            v = np.float32(v * Ainv.scale[K_src - 1])
        if v != 0:
            c_h = int(AinvP.perm[K_src - 1])
            pg.rest = dict(n=1, indptr=torch.tensor([0, 1], dtype=torch.int64, device=dev), indices=torch.tensor([c_h], dtype=torch.int32, device=dev),
                           data=torch.tensor([float(v)], dtype=torch.float32, device=dev), out_rows=torch.tensor([r_h], dtype=torch.int32, device=dev))
    W._pg = pg
    return W



def _tc_planes(vals, n_rows, G, K_pad):
    """Operands of the tensor-core kernels (csrc/pgroup_tc.cu, csrc/pgtile_tc.cu) for row-major value rows [n_rows][K_pad]
    read in boxes of G rows: the TF32 hi / bf16 corr planes and their TMA descriptors (4 x 128 bytes, host memory)."""
    L = _native.lib()
    (hi, corr) = (torch.empty_like(vals), torch.empty_like(vals))
    check(L.kn_pg_tc_split(ptr(vals), vals.numel(), ptr(hi), ptr(corr), stream_ptr()))
    maps = ctypes.create_string_buffer(4 * 128)
    check(L.kn_pg_tc_tensormaps(ptr(hi), ptr(corr), n_rows, G, K_pad, maps))
    return dict(hi=hi, corr=corr, maps=maps)


def _conv_tiles(desc, geom, wq, bq, pix_np, row_of_src, col_map, bias_col, dev):
    """Tile format of a conv layer for the spatially tiled tensor-core kernel (csrc/pgtile_tc.cu), or None when the layer
    does not qualify: G <= 128 output channels (taller groups are tensor-bound on the per-pixel kernel already), C a
    multiple of 16, the image divisible into th x tw tiles and the pixel set a union of whole tiles."""
    (C, U, V, M, P, Q, stride) = geom
    L = _native.lib()
    Gp = (M + 15) // 16 * 16
    if not (32 <= Gp <= 128 and C % 16 == 0 and C >= 16):
        return None
    (th, tw) = (2, 2) if Gp <= 96 else (1, 2)
    (Uo, Vo) = (U // stride, V // stride)
    (uh, uw) = ((th - 1) * stride + P, (tw - 1) * stride + Q)
    if Uo % th != 0 or Vo % tw != 0 or uh * uw > 32 or th * tw * Gp + 4 * 32 > 512:
        return None
    slab = 2 * Gp * 64
    if (226 * 1024 - (uh * uw * C * 4 + 8192) - (P * Q + 1) * slab) // 8192 < 3:
        return None                                   # weight slabs of a channel chunk + a raw gather ring must fit shared memory
    (py, px) = (pix_np // Vo, pix_np % Vo)
    origin = (py // th * th) * Vo + (px // tw * tw)
    (tiles, counts) = np.unique(origin, return_counts=True)
    if not np.all(counts == th * tw):
        return None                                   # the shard cuts through a tile
    n_tiles = len(tiles)
    n_taps = P * Q
    K_pad = n_taps * C + 16
    Wt = np.zeros((M, K_pad), dtype=np.float32)
    Wt[:, :n_taps * C] = np.ascontiguousarray(wq, dtype=np.float32).reshape(M, C, n_taps).transpose(0, 2, 1).reshape(M, n_taps * C)      # k = tap * C + c
    Wt[:, n_taps * C] = bq
    w = torch.from_numpy(Wt).to(dev).reshape(-1)
    t_origin = torch.from_numpy(tiles.astype(np.int32)).to(dev)
    tile_cols = torch.empty(n_tiles * uh * uw * C, dtype=torch.int32, device=dev)
    tile_rows = torch.empty(n_tiles * th * tw * M, dtype=torch.int32, device=dev)
    check(L.kn_conv2d_tiles_index(desc, ptr(t_origin), n_tiles, th, tw, ptr(row_of_src), ptr(col_map), ptr(tile_cols), ptr(tile_rows), stream_ptr()))
    return dict(_tc_planes(w, M, M, K_pad), cols=tile_cols, rows=tile_rows, bias_col=bias_col, n_tiles=n_tiles, C=C, G=M, th=th, tw=tw, stride=stride, P=P, Q=Q)


def _recipe(kind, geom, A, Ainv, rows, col_remap, **extra):
    """How a keyed layer was built (geometry, coefficients, key permutations): lets the batched engine fuse a conv (+ReLU)
    with the average pooling that follows it (csrc/convpool.cu).  None when the layer is sharded or its keys are not plain
    permutations -- those layers are never fused."""
    if rows is not None or col_remap is not None:
        return None
    for K in (A, Ainv):
        if K is not None and not (isinstance(K, MonomialKey) and K.bias is None and K.is_unscaled()):
            return None
    return dict(kind=kind, geom=geom, out_perm=None if (A is None or A.is_unpermuted()) else A.perm, in_perm=None if Ainv.is_unpermuted() else Ainv.perm, **extra)


def keyed_toeplitz_conv2d(inshape, f, bias, stride, A, Ainv, rows=None, build_groups=True, col_remap=None, n_cols_phys=None, want_csr=True):
    """W_hat = A . toeplitz(conv2d) . Ainv built on the GPU for monomial keys (keynet/layer.py:32-35).

    rows=(r0, r1) builds only that row range of W_hat (row shard); indptr then has r1-r0+1 entries.
    want_csr=False (with build_groups): only the pattern-group execution format is built -- the layer never exists as a
    CSR (VGG16: 120 GB); nnz() still reports the reference's stored-entry count."""
    dev = _device()
    (fq, bq, (C, U, V, M, P, Q)) = _conv_weights_rounded(inshape, f, bias, stride)
    if _DIRECT[0] and (A is None or isinstance(A, MonomialKey)) and isinstance(Ainv, MonomialKey):
        clustered = M <= PatternGroups.CG_MAX_G and (C * P * Q + 1 + 31) // 32 * 32 <= PatternGroups.CG_KERNEL_MAX_K
        W = _keyed_conv_direct((C, U, V, M, P, Q, int(stride), True), fq, bq, A, Ainv, rows, col_remap, n_cols_phys, want_csr, build_groups, dev, clustered=clustered)
        if W is not None:
            W._recipe = _recipe('conv', (C, U, V, M, P, Q, int(stride)), A, Ainv, rows, col_remap, fq=fq, bq=bq)
            return W
    R = M * (U // stride) * (V // stride) + 1
    K = C * U * V + 1
    desc = kn_conv2d_desc(C, U, V, M, P, Q, int(stride), 0, 1)
    (ids, sel) = _row_ids(A, R, rows, dev)
    n = _n_selected(sel, R)
    (Ainv, Kp) = _remapped(Ainv, col_remap, n_cols_phys)
    csr0 = _toeplitz_rows(desc, fq, bq, ids, n, dev)
    csr = _keycompile(csr0, n, K, A, Ainv, dev, row_scale_slice=sel)
    W = SparseMatrix(((n, Kp), *csr), device=dev)
    if build_groups and W.nnz() >= 4096:
        # pattern groups come from the STRUCTURAL matrix (exact zeros kept): every output pixel keeps its full
        # M-row group even where the reference's offset rounding turned a tiny weight into a dropped zero
        S = SparseMatrix(((n, Kp), *_keycompile(csr0, n, K, A, Ainv, dev, row_scale_slice=sel, keep_zeros=True)), device=dev)
        # spatial clusters only where the clustered kernel applies: short reductions (first conv layer: 1 or 3 input channels)
        clustered = M <= PatternGroups.CG_MAX_G and (C * P * Q + 1 + 31) // 32 * 32 <= PatternGroups.CG_KERNEL_MAX_K
        hint = _pixel_tile_hint(ids, n, (M, U // stride, V // stride), C, P, stride, False, dev) if clustered else None
        W._pg = PatternGroups.build(S, hint=hint)
    return W


def _pixel_tile_hint(ids, n, outshape, C, k, stride, depthwise, dev):
    """Spatial cluster id of every compiled row: rows whose underlying Toeplitz row lies in the same t x t tile of output
    pixels (and, for pooling, the same channel) share an id.  t is the largest tile whose union of taps fits the staging
    buffer of the clustered kernel; None if not even one pixel does.  ids: Toeplitz row of every compiled row (None = identity)."""
    (M, Uo, Vo) = outshape
    K_pad = ((k * k * (1 if depthwise else C) + 1) + 31) // 32 * 32
    # staged bytes of a t x t tile: union rows x 512 B + one lidx row (K_pad ints) per group
    staged = lambda t: (((t - 1) * stride + k) ** 2 * (1 if depthwise else C) + 1) * 512 + t * t * K_pad * 4
    t = 0
    while t < max(Uo, Vo) and staged(t + 1) <= PatternGroups.CG_MAX_UNION * 512:
        t += 1
    if t == 0:
        return None
    t = min(t, max(Uo, Vo))
    for d in range(t, max(1, t // 2), -1):          # prefer a tile that divides the image (equal clusters)
        if Uo % d == 0 and Vo % d == 0:
            t = d
            break
    (th, tw) = (t, t)
    src = ids if ids is not None else torch.arange(n, dtype=torch.int64, device=dev)
    px = src % (Uo * Vo)
    ch = src // (Uo * Vo)
    (py, pxx) = (px // Vo, px % Vo)
    nt = -(-Vo // tw)
    hint = (py // th) * nt + (pxx // tw)
    if depthwise:
        hint = ch * (nt * -(-Uo // th)) + hint
    n_ids = (M if depthwise else 1) * nt * -(-Uo // th)
    return torch.where(src < M * Uo * Vo, hint, torch.full_like(hint, n_ids))        # homogeneous row: a cluster of its own


def shard_compiled(W, rows, col_remap, n_cols_phys):
    """Rows `rows` ((r0, r1) or an index array, in that order) of an already compiled W_hat, with column c moved to position
    col_remap[c] of a buffer with n_cols_phys rows (dist.py).  Used for general-key layers; monomial keys shard at build time."""
    dev = W._data.device
    L = _native.lib()
    (R, K) = W.shape
    if rows is None:
        ids = torch.arange(R, dtype=torch.int64, device=dev)
    elif isinstance(rows, tuple):
        ids = torch.arange(int(rows[0]), int(rows[1]), dtype=torch.int64, device=dev)
    else:
        ids = torch.from_numpy(np.ascontiguousarray(rows, dtype=np.int64)).to(dev)
    n = int(ids.numel())
    csr = _two_phase(
        n,
        lambda row_nnz: check(L.kn_csr_gather_rows_count(ptr(W._indptr), ptr(ids), n, ptr(row_nnz), stream_ptr())),
        lambda ip, ix, dt: check(L.kn_csr_gather_rows_fill(ptr(W._indptr), ptr(W._indices), ptr(W._data), ptr(ids), n, ptr(ip), ptr(ix), ptr(dt), stream_ptr())),
        dev)
    Kp = K
    if col_remap is not None:
        (Kmap, Kp) = _remapped(MonomialKey(np.arange(K)), col_remap, n_cols_phys)
        csr = _keycompile(csr, n, K, None, Kmap, dev)
    return SparseMatrix(((n, Kp), *csr), device=dev)


def keyed_toeplitz_avgpool2d(inshape, kernel_size, stride, A, Ainv, rows=None, col_remap=None, n_cols_phys=None):
    """W_hat = A . toeplitz(avgpool) . Ainv (keynet/layer.py:56-59).  The reference builds C*C channel
    pairs and lets the SpGEMM drop the zero ones; here only the channel diagonal is generated."""
    dev = _device()
    (C, U, V) = [int(s) for s in inshape]
    k = int(kernel_size)
    assert k % 2 == 1 and U % stride == 0 and V % stride == 0
    w = np.float32(1.0 / (k * k))
    # emitted-value minimum of the reference's dense-channel filter: 0 if any off-diagonal channel pair exists
    emitted_min = np.float32(0.0) if C > 1 else w
    wq = _offset_round(np.full((C, k, k), w, dtype=np.float32), emitted_min)
    R = C * (U // stride) * (V // stride) + 1
    K = C * U * V + 1
    desc = kn_conv2d_desc(C, U, V, C, k, k, int(stride), 1, 0)     # zero bias column is dropped by the compile
    (ids, sel) = _row_ids(A, R, rows, dev)
    n = _n_selected(sel, R)
    (Ainv, Kp) = _remapped(Ainv, col_remap, n_cols_phys)
    csr = _toeplitz_rows(desc, wq, None, ids, n, dev)
    csr = _keycompile(csr, n, K, A, Ainv, dev, row_scale_slice=sel)
    W = SparseMatrix(((n, Kp), *csr), device=dev)
    W._recipe = _recipe('pool', (C, U, V, C, k, k, int(stride)), A, Ainv, rows, col_remap, pool_w=float(wq.reshape(-1)[0]))
    if rows is None and ids is not None and n > 4096:
        # EXECUTION ORDER of a pooling layer with a permuted output key: the rows of the canonical matrix follow the keyed row
        # numbering, i.e. consecutive rows pool windows from random places of the image, and every window row is fetched from
        # DRAM again (VGG16 pool1: 8.2 GB of traffic for 4.1 GB of data, 85 % of the HBM peak spent on re-reads).  Processing the
        # rows in the order of the underlying pooled pixel makes neighbouring windows neighbours in time, so the shared window
        # rows hit in L2; each result still goes to its keyed row (kn_spmm_csr_rows_f32 scatters by out_rows).
        L = _native.lib()
        order = torch.argsort(ids).contiguous()
        ex = _two_phase(
            n,
            lambda row_nnz: check(L.kn_csr_gather_rows_count(ptr(W._indptr), ptr(order), n, ptr(row_nnz), stream_ptr())),
            lambda ip, ix, dt: check(L.kn_csr_gather_rows_fill(ptr(W._indptr), ptr(W._indices), ptr(W._data), ptr(order), n, ptr(ip), ptr(ix), ptr(dt), stream_ptr())),
            dev)
        W._exec = dict(n=n, indptr=ex[0], indices=ex[1], data=ex[2], out_rows=order.to(torch.int32).contiguous())
    return W


def keyed_linear(weight, bias, A, Ainv, rows=None, col_remap=None, n_cols_phys=None, build_groups=True, want_csr=True):
    """W_hat = A . [[W, b],[0, 1]] . Ainv (keynet/layer.py:69-70)."""
    dev = _device()
    L = _native.lib()
    W = torch.as_tensor(weight).detach().to(device=dev, dtype=torch.float32).contiguous()
    (n_out, n_in) = W.shape
    if _DIRECT[0] and (A is None or isinstance(A, MonomialKey)) and isinstance(Ainv, MonomialKey) and Ainv.bias is None and (A is None or A.bias is None):
        # a linear layer is a 1x1 convolution on a 1x1 image: one output "pixel", one pattern group holding every row
        wn = W                                                  # stays on the device
        bn = None if bias is None else torch.as_tensor(bias).detach().to(device=dev, dtype=torch.float32).contiguous()
        (A_, rows_, n_out_) = (A, rows, int(n_out))
        if rows is not None:
            # a row shard of a linear layer is a smaller linear layer: its weight rows in the shard's own order, the output
            # key reduced to the gains of those rows (one group must hold EVERY row it is given -- residual dense rows on
            # the CSR kernel cost a warp 25 k sequential taps each)
            sel_ = np.arange(int(rows[0]), int(rows[1]), dtype=np.int64) if isinstance(rows, tuple) else np.ascontiguousarray(rows, dtype=np.int64)
            src_ = sel_ if A is None else A.perm[sel_]
            main_ = src_ < n_out
            n_out_ = int(main_.sum())
            take = torch.from_numpy(np.ascontiguousarray(src_[main_])).to(dev)
            wn = W[take].contiguous()
            bn = None if bn is None else bn[take].contiguous()
            rows_ = np.where(main_, np.cumsum(main_) - 1, n_out_).astype(np.int64)          # local row -> row of the reduced layer
            scale_ = np.ones(n_out_ + 1, dtype=np.float32)
            if A is not None:
                scale_[rows_] = A.scale[sel_]
            A_ = MonomialKey(np.arange(n_out_ + 1), scale_)
        M_ = None
        if n_out_ > 0:
            M_ = _keyed_conv_direct((int(n_in), 1, 1, n_out_, 1, 1, 1, bn is not None), wn, bn, A_, Ainv, rows_, col_remap, n_cols_phys, want_csr, build_groups, dev)
        if M_ is not None:
            return M_
        pg = None
    else:
        pg = None
    b = torch.as_tensor(bias).detach().to(device=dev, dtype=torch.float32).contiguous() if bias is not None else None
    (ids, sel) = _row_ids(A, n_out + 1, rows, dev)
    n = _n_selected(sel, n_out + 1)
    (Ainv, Kp) = _remapped(Ainv, col_remap, n_cols_phys)
    csr = _two_phase(
        n,
        lambda row_nnz: check(L.kn_linear_count(ptr(W), ptr(b), n_out, n_in, ptr(ids), n, ptr(row_nnz), stream_ptr())),
        lambda ip, ix, dt: check(L.kn_linear_fill(ptr(W), ptr(b), n_out, n_in, ptr(ids), n, ptr(ip), ptr(ix), ptr(dt), stream_ptr())),
        dev)
    csr = _keycompile(csr, n, n_in + 1, A, Ainv, dev, row_scale_slice=sel)
    M_ = SparseMatrix(((n, Kp), *csr), device=dev)
    M_._pg = pg
    return M_


def sparse_toeplitz_conv2d(inshape, f, bias=None, as_correlation=True, stride=1, format='csr'):
    """Un-keyed sparse Toeplitz matrix of conv2d (explicit zeros kept), canonical CSR on the GPU.
    Same contract as the reference's keynet/sparse.py:163-203:  conv2d(img, f) == W . img.flatten()."""
    assert as_correlation, 'only cross-correlation (torch conv2d) is supported'
    assert format == 'csr'
    dev = _device()
    f = f.detach().cpu().numpy() if torch.is_tensor(f) else f
    bias = bias.detach().cpu().numpy() if torch.is_tensor(bias) else bias
    (fq, bq, (C, U, V, M, P, Q)) = _conv_weights_rounded(inshape, f, bias, stride)
    R = M * (U // stride) * (V // stride)
    desc = kn_conv2d_desc(C, U, V, M, P, Q, int(stride), 0, 1 if bias is not None else 0)
    n_rows = R + 1 if bias is not None else R
    csr = _toeplitz_rows(desc, fq, bq, None, n_rows, dev)
    return SparseMatrix(((n_rows, C * U * V + (1 if bias is not None else 0)), *csr), device=dev)


def sparse_toeplitz_avgpool2d(inshape, filtershape, stride):
    """Un-keyed Toeplitz matrix of avgpool2d exactly as the reference stores it (dense channel pairs with
    explicit zeros, zero bias column; keynet/sparse.py:206-212)."""
    (outchannel, inchannel, filtersize, filtersize2) = filtershape
    F = np.zeros(filtershape, dtype=np.float32)
    for k in range(0, outchannel):
        F[k, k, :, :] = 1.0 / (filtersize * filtersize)
    return sparse_toeplitz_conv2d(inshape, F, bias=np.zeros(outchannel, dtype=np.float32), stride=stride)


def is_scipy_sparse(A):
    try:
        import scipy.sparse
        return scipy.sparse.issparse(A)
    except ImportError:
        return False
