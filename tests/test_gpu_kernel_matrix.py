"""Every SpMM kernel instantiation of tests/kernel_ledger.py, run under its own name and checked against an exact reference.

Run this module WHOLE (`python -m pytest tests/test_gpu_kernel_matrix.py -m gpu`): its last test fails unless every entry
of SPMM_KERNELS was launched by at least one passing case of the same run, and prints which case verified which kernel.

Each case is one layer built with the product's own builders (keyed_toeplitz_conv2d, keyed_linear, SparseMatrix,
PatternGroups.build), one batch width N, and the instantiation it must reach.  Every call runs under torch.profiler: the
expected kernels must have been launched and no other SpMM-family kernel (nothing falls back silently).

Reference: the compiled matrix itself (W.csr_arrays()) as a dense float64 matrix, W64 @ X64 by cuBLAS DGEMM.
  * exact family: integer weights in [-4, 4] (some zero), integer biases, integer X in [-8, 8] (X[-1] = 1), power-of-two
    gains of at most 2^+-2 where the path allows them (not the tile kernel).  sum|w||x| stays below 2^20 quanta (asserted),
    so every product and partial sum is an exact fp32 -- and exact in TF32 with lo = 0 -- whatever the summation order or
    the tensor pipe's adder width: every kernel must equal the fp64 product BIT FOR BIT, ReLU included.  Wrong columns,
    taps, rows, stages, tiles or biases land here.
  * wide family: activations over 1e-20 .. 1e20 with random signs and weights scaled per output channel by 2^-10 .. 2^10,
    so a row's size says nothing about its error.  Per element |y - y64| <= bound * sum|w||x| (fp64 |W| @ |X|), no atol:
    tensor-core paths (BOUND + (2 (K/8 + 1) + S) 2^-23) with BOUND the split's per-product bound (test_split_numerics.py),
    fp32 FMA / CSR paths gamma(K + S + 1) = n u / (1 - n u), u = 2^-24.  K is the row's reduction length (rounded up to a
    stage, plus the bias stage), S the split-K slice count.  No inf or NaN.  Precision errors (a lost correction) land here.

Modes (exact family):
  * plain: sparse.spmm into a NaN-filled output; every element must be written.
  * abi:   the same classes launched through their kn_* entry points with the loosest layout each header allows: X a view
           of a wider buffer whose extra columns hold NaN (odd ldx for the CSR kernels), Y a view with an odd ldy, offset by
           one float, for the CSR and tensor-core entry points (the tile kernel's per-lane epilogue) and padded rows of
           NaN with a fixed payload otherwise.  The padding must be bit-for-bit unchanged and the result equal plain's bit
           for bit: no kernel does arithmetic that depends on the strides.
  * abi4:  the same at n_vecs = 4 (16-byte output rows: the smallest bulk-copy row of the tile epilogue), against plain's
           first four columns, bit for bit.
  * peers: the fused all-gather into two local destinations under a random need mask: needed rows equal plain bit for
           bit, other rows and the layer's own Y stay NaN.
"""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

from tests import kernel_ledger as kl
from tests.test_split_numerics import BOUND

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAYLOAD = 0x7FC0DEAD                    # quiet NaN with a payload: Y padding must keep exactly these bits
RESULTS = {}                            # kernel -> [(case, modes, worst |err| / sum|w||x| of the wide family)]
SAMPLE_NAME = []                        # one kernel name as the profiler spells it
_B = ('false', 'true')


# ---------------------------------------------------------------------------------------------------------------------
# layers
# ---------------------------------------------------------------------------------------------------------------------
def _key(rs, n, permute=True, gains=False):
    from keynet_b200.sparse import MonomialKey
    perm = np.concatenate([rs.permutation(n - 1) if permute else np.arange(n - 1), [n - 1]])
    if not gains:
        return MonomialKey(perm)
    scale = (2.0 ** rs.randint(-2, 3, n) * rs.choice([-1.0, 1.0], n)).astype(np.float32)
    scale[-1] = 1.0                                                  # the homogeneous coordinate stays 1
    return MonomialKey(perm, scale)


def _values(rs, family, shape, n_out, nonzero=False):
    """Weights [n_out, ...] and biases [n_out] of one family."""
    if family == 'exact':
        w = rs.randint(-4, 5, shape).astype(np.float32)
        b = rs.randint(-4, 5, n_out).astype(np.float32)
        if nonzero:
            (w[w == 0], b[b == 0]) = (1.0, 1.0)
        return (w, b)
    scale = 2.0 ** rs.randint(-10, 11, n_out)
    w = (rs.uniform(-1, 1, shape) * scale.reshape((-1,) + (1,) * (len(shape) - 1))).astype(np.float32)
    return (w, (rs.uniform(-1, 1, n_out) * scale).astype(np.float32))


def _conv(family, rs, C, U, M, V=None, k=3, stride=1, gains=False, out_key=True):
    from keynet_b200 import sparse
    V = U if V is None else V
    (f, b) = _values(rs, family, (M, C, k, k), M)
    (R, K) = (M * (U // stride) * (V // stride) + 1, C * U * V + 1)
    A = _key(rs, R, gains=gains) if out_key else None
    return sparse.keyed_toeplitz_conv2d((C, U, V), f, b, stride, A, _key(rs, K, gains=gains))


def _conv_g2(family, rs, N_unused=None):
    """M = 2 output channels: below the fused compile's group minimum, grouped by PatternGroups.build(min_group=1) with a
    spatial hint (clustered kernel, GM = 2).  Non-zero weights keep every pixel's two rows on one column pattern."""
    from keynet_b200 import sparse
    (C, U, M) = (3, 16, 2)
    (f, b) = _values(rs, family, (M, C, 3, 3), M, nonzero=True)
    W = sparse.keyed_toeplitz_conv2d((C, U, U), f, b, 1, None, _key(rs, C * U * U + 1), build_groups=False)
    hint = sparse._pixel_tile_hint(None, W.shape[0], (M, U, U), C, 3, 1, False, W._indptr.device)
    W._pg = sparse.PatternGroups.build(W, min_group=1, hint=hint)
    assert W._pg is not None and all(c.get('cg') is not None for c in W._pg.classes)
    return W


def _linear(family, rs, n_in, n_out):
    from keynet_b200 import sparse
    (w, b) = _values(rs, family, (n_out, n_in), n_out)
    return sparse.keyed_linear(w, b, None, _key(rs, n_in + 1))


def _csr(family, rs, R=300, K=500):
    """Random CSR (sorted columns) with empty rows and rows of more than 64 entries; no pattern groups."""
    from keynet_b200 import sparse
    nnz = rs.randint(0, 20, R)
    nnz[[5, 77, 299]] = 0
    nnz[[10, 11]] = (100, 70)
    cols = [np.sort(rs.choice(K - 1, n, replace=False)) for n in nnz]
    if family == 'exact':
        vals = [rs.choice([-4, -3, -2, -1, 1, 2, 3, 4], n).astype(np.float32) for n in nnz]
    else:
        vals = [(rs.uniform(-1, 1, n) * 2.0 ** rs.randint(-10, 11)).astype(np.float32) for n in nnz]
    indptr = np.concatenate([[0], np.cumsum(nnz)]).astype(np.int64)
    W = sparse.SparseMatrix(((R, K), indptr, np.concatenate(cols).astype(np.int32), np.concatenate(vals)))
    assert W._pg is None
    return W


# ---------------------------------------------------------------------------------------------------------------------
# cases: id -> (builder(family, rs), {N: expected main kernels}, quantum of the exact family)
# Expected names use {r} for ReLU and {p} for the fused all-gather (PEERS) template argument.  The CSR kernel that runs the
# layer's leftover rows (the homogeneous row) is added from W._pg.rest.
# ---------------------------------------------------------------------------------------------------------------------
def _csr_kernel(N, relu):
    """spmm.cu's choice for contiguous, 16-byte aligned X and Y with ld = N."""
    r = _B[relu]
    if N <= 8:
        return 'spmm_lanes_nnz_kernel<%d,%s>' % ({1: 1, 2: 2}.get(N, 4 if N <= 4 else 8), r)
    if N % 4 == 0 and N >= 2048:
        return 'spmm_rowwarp_wide_kernel<%d,%s>' % (int(os.environ.get('KN_CSR_WIDE', '2')), r)
    if N % 4 == 0 and N >= 128:
        return 'spmm_rowwarp_kernel<4,%s>' % r
    if N % 2 == 0 and N >= 64:
        return 'spmm_rowwarp_kernel<2,%s>' % r
    return 'spmm_rowwarp_kernel<1,%s>' % r


CSR_NS = (1, 2, 3, 7, 33, 66, 132, 2052)
CASES = {
    'csr': (lambda fam, rs: _csr(fam, rs), {n: [] for n in CSR_NS}, 1.0),
}
for (M, GM) in ((6, 8), (12, 16)):             # C = 4: K_pad 64, too long for the clustered kernel, short for pg_simt
    CASES['small_M%d' % M] = (lambda fam, rs, M=M: _conv(fam, rs, 4, 8, M, gains=True), {64: ['pg_small_kernel<%d,{r}>' % GM]}, 2.0 ** -4)
for (M, RW, Ns) in ((8, 1, (64, 200)), (16, 2, (64, 200)), (24, 4, (64, 200)), (48, 8, (64,)), (96, 12, (64,)), (100, 16, (64,))):
    # C = 16 (K_pad 160); M >= 32 would take the tensor cores from N = 128 on
    CASES['simt_M%d' % M] = (lambda fam, rs, M=M: _conv(fam, rs, 16, 8, M, gains=True), {n: ['pg_simt_kernel<%d,{r}>' % RW] for n in Ns}, 2.0 ** -4)
for (M, GM) in ((4, 4), (6, 6), (8, 8), (10, 10), (12, 12), (14, 14), (16, 16), (40, 16)):
    # first-layer geometry: C = 3, K_pad 32, groups clustered by output-pixel tile; M = 40 runs in chunks of 16 rows
    CASES['cluster_M%d' % M] = (lambda fam, rs, M=M: _conv(fam, rs, 3, 16, M, gains=True), {200: ['pg_cluster_kernel<%d,{r}>' % GM]}, 2.0 ** -4)
CASES['cluster_M2'] = (_conv_g2, {200: ['pg_cluster_kernel<2,{r}>']}, 1.0)
CASES['splitk_fc'] = (lambda fam, rs: _linear(fam, rs, 4096, 300),
                      {256: ['pg_tc_kernel<1,false,2,false>', 'splitk_reduce_kernel<{r}>']}, 1.0)
# pg_tc<NB, RELU, CS, PEERS>: NB = 2 when two Gp-wide accumulators + a 2-deep ring fit TMEM, CS = 2 for an even number of
# CTA batch tiles.  Super-tile kSuperTiles / NB: N = 1280 leaves a remainder (G = 256: 8 + 2 tiles, G = 160: 4 + 1, and
# N = 1536 at G = 160: 4 + 2).
CASES['tc_G256'] = (lambda fam, rs: _conv(fam, rs, 16, 8, 256, gains=True),
                    {384: ['pg_tc_kernel<1,{r},1,{p}>'], 256: ['pg_tc_kernel<1,{r},2,{p}>'], 1280: ['pg_tc_kernel<1,{r},2,{p}>']}, 2.0 ** -4)
CASES['tc_G300'] = (lambda fam, rs: _conv(fam, rs, 16, 8, 300), {384: ['pg_tc_kernel<1,{r},1,{p}>']}, 1.0)      # 256 + 44 rows
CASES['tc_G160_perm'] = (lambda fam, rs: _conv(fam, rs, 16, 8, 160),           # 9 shared border-class blocks, ragged group_k
                         {768: ['pg_tc_kernel<2,{r},1,{p}>'], 1280: ['pg_tc_kernel<2,{r},1,{p}>'],
                          512: ['pg_tc_kernel<2,{r},2,{p}>'], 1536: ['pg_tc_kernel<2,{r},2,{p}>']}, 1.0)
CASES['tc_G160_gain'] = (lambda fam, rs: _conv(fam, rs, 16, 8, 160, gains=True),   # one block per pixel
                         {768: ['pg_tc_kernel<2,{r},1,{p}>'], 512: ['pg_tc_kernel<2,{r},2,{p}>']}, 2.0 ** -4)
# pg_tile_tc<RELU, PEERS, TH, TW, GP>: the interior-tile issuers for 3x3 / stride 1 at Gp = 64, 96 (2x2 tiles) and 128 (1x2)
for (M, spec) in ((64, '2,2,64'), (96, '2,2,96'), (128, '1,2,128')):
    CASES['tile_M%d' % M] = (lambda fam, rs, M=M: _conv(fam, rs, 16, 8, M), {200: ['pg_tile_tc_kernel<{r},{p},%s>' % spec],
                                                                           1280: ['pg_tile_tc_kernel<{r},{p},%s>' % spec]}, 1.0)
# 128 rows of 512 channels per pixel (64 KB) do not fit the 6-stage gather ring (48 KB): per-lane epilogue (epi_pixels = 0)
CASES['tile_M128_C512_4x6'] = (lambda fam, rs: _conv(fam, rs, 512, 4, 128, V=6), {200: ['pg_tile_tc_kernel<{r},{p},1,2,128>']}, 1.0)
GENERIC = {
    'tile_M40': lambda fam, rs: _conv(fam, rs, 16, 8, 40),                    # Gp 48 != G, merged 2x2
    'tile_M80': lambda fam, rs: _conv(fam, rs, 16, 8, 80),
    'tile_M112': lambda fam, rs: _conv(fam, rs, 16, 8, 112),                  # merged 1x2
    'tile_M64_s2': lambda fam, rs: _conv(fam, rs, 16, 8, 64, stride=2),       # one issuer per pixel, 2x2
    'tile_M128_s2': lambda fam, rs: _conv(fam, rs, 16, 8, 128, stride=2),     # one issuer per pixel, 1x2
    'tile_1x1_C128': lambda fam, rs: _conv(fam, rs, 128, 8, 64, k=1),
    'tile_M40_6x10': lambda fam, rs: _conv(fam, rs, 16, 6, 40, V=10),
}
for (name, fn) in GENERIC.items():
    CASES[name] = (fn, {200: ['pg_tile_tc_kernel<{r},{p},0,0,0>'], **({1280: ['pg_tile_tc_kernel<{r},{p},0,0,0>']} if name == 'tile_M40' else {})}, 1.0)


def _layout(W, path_N):
    """'csr' (no constraint), 'tc' (X: ldx % 4, 16-byte aligned; Y: anything) or 'fma' (X and Y: ld % 4, 16-byte aligned)."""
    from keynet_b200.sparse import PatternGroups
    if W._pg is None:
        return 'csr'
    for c in W._pg.classes:
        if c.get('cg') is not None or path_N < PatternGroups.TC_MIN_BATCH or (c.get('splitk') is None and c.get('tile') is None and c['tc'] is None):
            return 'fma'
        if c.get('splitk') is not None:
            return 'fma'                                             # kn_splitk_reduce_f32 stores float4 rows
    return 'tc'


def _abi_spmm(W, path_N, x_addr, ldx, y_addr, ldy, n, relu):
    """PatternGroups.spmm / sparse.spmm with explicit leading dimensions and addresses: every class through the entry point
    the plain run at batch width path_N takes, over n_vecs = n columns."""
    import ctypes
    from keynet_b200 import _native, sparse
    from keynet_b200._native import check, ptr, stream_ptr
    from keynet_b200.sparse import PatternGroups
    L = _native.lib()
    (xp, yp, s) = (ctypes.c_void_p(x_addr), ctypes.c_void_p(y_addr), stream_ptr())
    flags = _native.KN_SPMM_RELU if relu else 0
    pg = W._pg
    if pg is None:
        check(L.kn_spmm_csr_f32(ptr(W._indptr), ptr(W._indices), ptr(W._data), W.shape[0], W.shape[1], xp, ldx, yp, ldy, n, flags, None, s))
        return
    for c in pg.classes:
        (cg, t, k) = (c.get('cg'), c.get('tile'), c.get('splitk'))
        tc_ok = path_N >= PatternGroups.TC_MIN_BATCH
        if cg is not None and sparse.clusters_enabled():
            check(L.kn_spmm_cg_f32(ptr(cg['cl_gptr']), ptr(cg['cl_uptr']), ptr(cg['ucols']), ptr(c['rows']), ptr(cg['lidx']), ptr(cg['valsT']), ptr(c['group_k']), ptr(c['block_of']),
                                   cg['n_clusters'], c['G'], c['K_pad'], cg['u_max'], cg['g_max'], xp, ldx, yp, ldy, n, flags, None, s))
        elif k is not None and tc_ok and path_N <= PatternGroups.SPLITK_MAX_BATCH:
            part = torch.empty((k['S'] * k['G'], n), dtype=torch.float32, device='cuda')
            check(L.kn_spmm_pg_tc_f32(k['tc']['maps'], ptr(k['rows']), ptr(k['cols']), ptr(k['group_k']), None, k['S'], k['G'], k['K_pad'], xp, ldx, ptr(part), n, n, 0, None, s))
            check(L.kn_splitk_reduce_f32(ptr(part), k['S'], k['G'], ptr(c['rows']), yp, ldy, n, flags, None, s))
        elif t is not None and tc_ok:
            check(L.kn_spmm_tile_tc_f32(t['maps'], ptr(t['cols']), ptr(t['rows']), t['bias_col'], t['n_tiles'], t['C'], t['G'], t['th'], t['tw'], t['stride'], t['P'], t['Q'],
                                        xp, ldx, yp, ldy, n, flags, None, s))
        elif c['tc'] is not None and tc_ok:
            check(L.kn_spmm_pg_tc_f32(c['tc']['maps'], ptr(c['rows']), ptr(c['cols']), ptr(c['group_k']), ptr(c['block_of']), c['n_groups'], c['G'], c['K_pad'],
                                      xp, ldx, yp, ldy, n, flags, None, s))
        else:
            check(L.kn_spmm_pg_f32(ptr(c['rows']), ptr(c['cols']), ptr(c['vals']), ptr(c['group_k']), ptr(c['block_of']), c['n_groups'], c['G'], c['K_pad'],
                                   xp, ldx, yp, ldy, n, flags, None, s))
    r = pg.rest
    if r is not None:
        check(L.kn_spmm_csr_rows_f32(ptr(r['indptr']), ptr(r['indices']), ptr(r['data']), r['n'], pg.shape[1], ptr(r['out_rows']), xp, ldx, yp, ldy, n, flags, None, s))


# ---------------------------------------------------------------------------------------------------------------------
# running and checking
# ---------------------------------------------------------------------------------------------------------------------
def _profiled(fn):
    """Run fn (and wait for it); the SpMM-family kernels it launched, normalised."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        n = kl.normalise(e.name)
        if kl.family(n) in kl.SPMM_FAMILIES:
            names.add(n)
            if not SAMPLE_NAME:
                SAMPLE_NAME.append(e.name)
    return names


def _dense(W):
    (ip, ix, dt) = W.csr_arrays()
    (R, K) = W.shape
    rows = torch.from_numpy(np.repeat(np.arange(R), np.diff(ip))).cuda()
    W64 = torch.zeros((R, K), dtype=torch.float64, device='cuda')
    W64[rows, torch.from_numpy(ix.astype(np.int64)).cuda()] = torch.from_numpy(dt.astype(np.float64)).cuda()
    return W64


def _inputs(family, rs, K, N):
    if family == 'exact':
        X = rs.randint(-8, 9, (K, N)).astype(np.float32)
    else:
        X = (10.0 ** rs.uniform(-20, 20, (K, N)) * rs.choice([-1, 1], (K, N))).astype(np.float32)
    X[-1] = 1.0                                                      # homogeneous coordinate (bias)
    return torch.from_numpy(X).cuda()


def _bits(t):
    return t.contiguous().view(torch.int32)


def _strided_x(X, ldx):
    Xb = torch.full((X.shape[0], ldx), float('nan'), device='cuda')
    Xb[:, :X.shape[1]] = X
    return Xb


def _run_abi(W, path_N, X, n, relu, layout):
    """One ABI-mode launch over the first n columns of X; returns Y (bits checked for the padding here)."""
    (R, K) = W.shape
    odd = lambda v: v + 1 + (v % 2)
    ldx = odd(n) if layout == 'csr' else n + 4
    if layout == 'fma' or (layout == 'tc' and n == 4):
        (ldy, off) = (n + 4, 0)                                       # n = 4 on the tile kernel: bulk rows of 16 bytes
    else:
        (ldy, off) = (odd(n), 1)
    Xb = _strided_x(X[:, :n], ldx)
    Yb = torch.full((off + R * ldy + 4,), PAYLOAD, dtype=torch.int32, device='cuda')
    _abi_spmm(W, path_N, Xb.data_ptr(), ldx, Yb.data_ptr() + 4 * off, ldy, n, relu)
    torch.cuda.synchronize()
    body = Yb[off:off + R * ldy].view(R, ldy)
    pad_ok = bool((Yb[:off] == PAYLOAD).all()) and bool((Yb[off + R * ldy:] == PAYLOAD).all()) and bool((body[:, n:] == PAYLOAD).all())
    assert pad_ok, 'Y padding (offset, columns [n_vecs, ldy), tail) was written (ldx=%d ldy=%d off=%d n=%d)' % (ldx, ldy, off, n)
    assert torch.equal(Xb[:, n:].isnan(), torch.ones_like(Xb[:, n:], dtype=torch.bool))
    return body[:, :n].contiguous().view(torch.float32)


def _rel_bound(W, case_kernels, S, nnz_row):
    """Per-row error coefficient of the wide family (see the module docstring)."""
    tc = any(kl.family(k) in ('pg_tc_kernel', 'pg_tile_tc_kernel') for k in case_kernels)
    Kr = nnz_row.astype(np.float64)
    if tc:
        Kr = np.ceil(Kr / 16.0) * 16.0 + 16.0
        return BOUND + (2.0 * (Kr / 8.0 + 1.0) + S) * 2.0 ** -23
    n = Kr + S + 1.0
    u = 2.0 ** -24
    return n * u / (1.0 - n * u)


def _record(kernels, case, modes, worst):
    for k in kernels:
        RESULTS.setdefault(k, []).append((case, modes, worst))


def _run_case(case_id, N, relu):
    """Builds the case's layer twice (exact and wide family), runs every mode, records what it verified."""
    from keynet_b200 import _native, sparse
    (builder, Ns, quantum) = CASES[case_id]
    r = _B[relu]
    rs = np.random.RandomState(zlib.crc32(('%s/%d/%d' % (case_id, N, relu)).encode()))
    # ---------------- exact family
    W = builder('exact', rs)
    (R, K) = W.shape
    rest = (W._pg is not None and W._pg.rest is not None)
    expect = set(k.format(r=r, p='false') for k in Ns[N]) | ({_csr_kernel(N, relu)} if (W._pg is None or rest) else set())
    expect_peers = set(k.format(r=r, p='true') for k in Ns[N]) | ({_csr_kernel(N, relu)} if (W._pg is None or rest) else set())
    if any(kl.family(k) == 'pg_tile_tc_kernel' and not k.endswith(',0,0,0>') for k in expect):
        t = W._pg.classes[0]['tile']
        cols = t['cols'].view(t['n_tiles'], -1)
        assert bool((cols >= 0).all(dim=1).any()), 'no interior tile: the specialised issuers would not run'
    W64 = _dense(W)
    X = _inputs('exact', rs, K, N)
    X64 = X.double()
    S = W64.abs() @ X64.abs()
    assert float(S.max()) < 2.0 ** 20 * quantum, 'exact family: sum|w||x| = %g reaches 2^20 quanta (%g)' % (float(S.max()), quantum)
    y64 = W64 @ X64
    ref = (y64.clamp(min=0) if relu else y64).float()
    del S

    out = torch.full((R, N), float('nan'), device='cuda')
    got = _profiled(lambda: sparse.spmm(W, X, relu=relu, out=out))
    assert got == expect, '%s N=%d relu=%s plain: launched %s, expected %s' % (case_id, N, relu, sorted(got), sorted(expect))
    bad = ~(out == ref)
    assert not bool(bad.any()), '%s N=%d relu=%s plain: %d of %d elements differ from the exact product, first at %s: %r vs %r' % (
        case_id, N, relu, int(bad.sum()), bad.numel(), tuple(bad.nonzero()[0].tolist()), float(out[bad][0]), float(ref[bad][0]))
    modes = ['plain']

    layout = _layout(W, N)
    for n in ((N, 4) if N > 4 else (N,)):
        y = _run_abi(W, N, X, n, relu, layout)
        bad = _bits(y) != _bits(out[:, :n])
        assert not bool(bad.any()), '%s N=%d relu=%s abi n_vecs=%d (layout %s): %d elements differ from plain bit for bit, first at %s' % (
            case_id, N, relu, n, layout, int(bad.sum()), tuple(bad.nonzero()[0].tolist()))
        modes.append('abi' if n == N else 'abi4')

    g = torch.Generator(device='cuda').manual_seed(R + N)
    mask = torch.randint(0, 4, (R,), generator=g, device='cuda', dtype=torch.uint8)
    (yo, d0, d1) = (torch.full((R, N), float('nan'), device='cuda') for _ in range(3))
    peers = _native.Peers([d0.data_ptr(), d1.data_ptr()], mask)
    got_p = _profiled(lambda: sparse.spmm(W, X, relu=relu, out=yo, peers=peers))
    assert got_p == expect_peers, '%s N=%d relu=%s peers: launched %s, expected %s' % (case_id, N, relu, sorted(got_p), sorted(expect_peers))
    assert bool(yo.isnan().all()), 'the layer wrote its own Y although peers were given'
    for (p, d) in enumerate((d0, d1)):
        need = ((mask >> p) & 1).bool()
        assert bool((_bits(d[need]) == _bits(out[need])).all()), '%s N=%d relu=%s peers: needed rows of rank %d differ from plain' % (case_id, N, relu, p)
        assert bool(d[~need].isnan().all()), '%s N=%d relu=%s peers: rows rank %d does not need were written' % (case_id, N, relu, p)
    modes.append('peers')
    del W64, X64, y64, ref, out, yo, d0, d1

    # ---------------- wide family (plain)
    W = builder('wide', rs)
    W64 = _dense(W)
    X = _inputs('wide', rs, K, N)
    y = torch.full((R, N), float('nan'), device='cuda')
    got_w = _profiled(lambda: sparse.spmm(W, X, relu=relu, out=y))
    assert got_w == expect, '%s N=%d relu=%s wide: launched %s, expected %s' % (case_id, N, relu, sorted(got_w), sorted(expect))
    assert bool(torch.isfinite(y).all()), '%s N=%d relu=%s wide: inf or NaN in the output' % (case_id, N, relu)
    X64 = X.double()
    S = W64.abs() @ X64.abs()
    y64 = W64 @ X64
    if relu:
        y64 = y64.clamp(min=0)
    err = (y.double() - y64).abs()
    (ip, _, _) = W.csr_arrays()
    n_split = max([c['splitk']['S'] for c in (W._pg.classes if W._pg is not None else []) if c.get('splitk') is not None] or [0])
    coef = torch.from_numpy(_rel_bound(W, expect, n_split, np.diff(ip))).cuda().view(-1, 1)
    over = err > coef * S
    ratio = torch.where(S > 0, err / S, torch.zeros_like(err))
    worst = float(ratio.max())
    assert not bool(over.any()), '%s N=%d relu=%s wide: %d elements over the bound, worst |err|/sum|w||x| = %.3g at %s' % (
        case_id, N, relu, int(over.sum()), worst, tuple(over.nonzero()[0].tolist()))
    modes.append('wide')
    _record(got | got_p, '%s N=%d' % (case_id, N), '+'.join(modes), worst)


PARAMS = [(c, n) for (c, (_, Ns, _)) in CASES.items() for n in Ns]


@pytest.mark.parametrize('relu', [False, True])
@pytest.mark.parametrize('case_id,N', PARAMS, ids=['%s-N%d' % p for p in PARAMS])
def test_instantiation(case_id, N, relu):
    from keynet_b200 import sparse
    assert sparse.tensor_cores_enabled() and sparse.tiles_enabled() and sparse.clusters_enabled()
    _run_case(case_id, N, relu)


def _child_wide4():
    """Runs in a process started with KN_CSR_WIDE=4 (read once per process by spmm.cu)."""
    for relu in (False, True):
        _run_case('csr', 2052, relu)
    return RESULTS


def test_csr_rowwarp_wide4():
    """spmm_rowwarp_wide<4>: the CSR case at N = 2052 in a process of its own with KN_CSR_WIDE=4."""
    env = dict(os.environ, KN_CSR_WIDE='4')
    code = ('import json, sys; sys.path.insert(0, %r); from tests import test_gpu_kernel_matrix as m; '
            'print("RESULTS=" + json.dumps(m._child_wide4()))' % ROOT)
    p = subprocess.run([sys.executable, '-c', code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    line = [s for s in p.stdout.splitlines() if s.startswith('RESULTS=')][-1]
    res = json.loads(line[len('RESULTS='):])
    assert any(k.startswith('spmm_rowwarp_wide_kernel<4,') for k in res), sorted(res)
    for (k, v) in res.items():
        RESULTS.setdefault(k, []).extend(tuple(e) for e in v)


def test_zz_every_instantiation_verified():
    """Run last (module order): every SPMM_KERNELS entry has at least one passing case in this run."""
    print('\nprofiler spelling of a kernel name: %s' % (SAMPLE_NAME[0] if SAMPLE_NAME else '(none seen)'))
    print('%-42s %-30s %-32s %s' % ('instantiation', 'case', 'modes', 'worst |err|/sum|w||x| (wide)'))
    for k in kl.SPMM_KERNELS:
        for (case, modes, worst) in RESULTS.get(k, [])[:1] or [('-', '-', float('nan'))]:
            print('%-42s %-30s %-32s %.3g' % (k, case, modes, worst))
    missing = [k for k in kl.SPMM_KERNELS if k not in RESULTS]
    print('%d / %d instantiations launched and verified' % (len(kl.SPMM_KERNELS) - len(missing), len(kl.SPMM_KERNELS)))
    assert not missing, 'not launched by any passing case: %s' % missing
