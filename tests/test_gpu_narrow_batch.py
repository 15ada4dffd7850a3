"""Narrow batches (1..31 columns) on layers whose CSR was dropped: PatternGroups.spmm_narrow (kn_spmm_pg_narrow_f32).

Layer cases are built with the product's own builders (as in test_gpu_kernel_matrix.py), then W.drop_csr().  For every
case, N in NS and ReLU on / off:
  * exact family (small integers, power-of-two gains): equal to the fp64 product of W.csr_arrays() (taken before the drop)
    bit for bit;
  * wide family (activations 1e-20..1e20, channels scaled 2^-10..2^10): |y - y64| <= gamma(K + S + 1) sum|w||x| per
    element, no atol (K = the row's stored entries, S = 0);
  * old route: where every class runs the shared-block form and the padded route ran pg_simt, the result equals the padded
    route (X zero-padded to 32 columns through W._pg.spmm) bit for bit, in the wide family (G16 / G48 / G100 at every N,
    G160_perm and G300 where they take the shared form);
  * kernel names (torch.profiler, in a process of its own): pg_simt (shared-block form) or the CSR kernel's lanes_nnz
    (row form) as the class plans name them and, for leftover rows, the CSR kernel -- nothing else (no padded route: neither
    pg_small nor pg_cluster, no copy to 32 columns);
  * ABI layout: X a view whose extra columns hold NaN (odd ldx), Y offset by one float with an odd ldy and NaN padding: the
    padding keeps its bits and the result equals the plain call bit for bit.
"""
import ctypes
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

from tests import kernel_ledger as kl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAYLOAD = 0x7FC0DEAD
NS = (1, 2, 3, 4, 5, 7, 8, 15, 16, 17, 31)
_B = ('false', 'true')


@pytest.fixture(scope='module')
def built():
    import __graft_entry__ as g
    g.build()
    from keynet_b200 import _native
    return _native


# ---------------------------------------------------------------------------------------------------------------------
# CPU: argument validation and the run table
# ---------------------------------------------------------------------------------------------------------------------
def test_narrow_argument_validation_without_gpu(built):
    """kn_spmm_pg_narrow_f32 rejects bad arguments with an error code and a message before any CUDA work."""
    L = built.lib()
    one = (ctypes.c_int32 * 2)(0, 1)
    p = ctypes.cast(one, ctypes.c_void_p)

    def call(n_vecs=1, ldx=1, ldy=1, n_groups=1, n_runs=1, run=p, peers=None, row_form=0):
        return L.kn_spmm_pg_narrow_f32(p, p, p, None, None, n_groups, 4, 32, run, run, n_runs, row_form,
                                       p, ldx, p, ldy, n_vecs, 0, peers, None)
    assert call(n_vecs=0, ldx=1, ldy=1) == -1 and b'n_vecs' in L.kn_last_error()
    assert call(n_vecs=33, ldx=33, ldy=33) == -1 and b'n_vecs' in L.kn_last_error()
    assert call(n_vecs=3, ldx=2, ldy=3) == -1 and b'leading dimension' in L.kn_last_error()
    assert call(n_vecs=3, ldx=3, ldy=2) == -1 and b'leading dimension' in L.kn_last_error()
    pe = built.kn_peers(); pe.n = 1
    assert call(peers=ctypes.byref(pe)) == -1 and b'peers' in L.kn_last_error()
    assert call(n_runs=0) == -1 and b'run table' in L.kn_last_error()
    assert call(run=None) == -1 and b'run table' in L.kn_last_error()
    assert call(n_vecs=9, ldx=9, ldy=9, row_form=1) == -1 and b'row form' in L.kn_last_error()
    assert call(row_form=2) == -1 and b'row form' in L.kn_last_error()
    assert call(n_groups=0, n_runs=0, run=None) == 0                         # nothing to do: no CUDA work either


@pytest.mark.parametrize('P', [1, 4, 32, 128])
def test_run_table_covers_every_group_once_and_runs_share_block_and_k(P):
    from keynet_b200.sparse import PatternGroups
    rs = np.random.RandomState(P)
    ng = 1000
    block_of = torch.from_numpy(rs.randint(0, 9, ng).astype(np.int32))
    group_k = torch.from_numpy(rs.choice([40, 60, 90], ng).astype(np.int32))
    for bo in (block_of, None):
        cls = dict(n_groups=ng, K_pad=96, cols=torch.zeros(ng * 96, dtype=torch.int32), block_of=bo, group_k=group_k)
        t = PatternGroups._run_table(cls, P)
        (groups, start) = (t['groups'].numpy(), t['start'].numpy())
        assert np.array_equal(np.sort(groups), np.arange(ng))
        assert start[0] == 0 and start[-1] == ng and t['n_runs'] == len(start) - 1
        blk = np.arange(ng) if bo is None else bo.numpy()
        for (a, b) in zip(start[:-1], start[1:]):
            assert 0 < b - a <= P
            g = groups[a:b]
            assert len(set(blk[g])) == 1 and len(set(group_k.numpy()[g])) == 1
        # runs are only cut where the block / group_k changes or P groups are full
        n_keys = len(set(zip(blk.tolist(), group_k.numpy().tolist())))
        assert t['n_runs'] <= n_keys + ng // P


# ---------------------------------------------------------------------------------------------------------------------
# GPU: layers (test_gpu_kernel_matrix.py style)
# ---------------------------------------------------------------------------------------------------------------------
def _key(rs, n, permute=True, gains=False):
    from keynet_b200.sparse import MonomialKey
    perm = np.concatenate([rs.permutation(n - 1) if permute else np.arange(n - 1), [n - 1]])
    if not gains:
        return MonomialKey(perm)
    scale = (2.0 ** rs.randint(-2, 3, n) * rs.choice([-1.0, 1.0], n)).astype(np.float32)
    scale[-1] = 1.0
    return MonomialKey(perm, scale)


def _values(rs, family, shape, n_out):
    if family == 'exact':
        return (rs.randint(-4, 5, shape).astype(np.float32), rs.randint(-4, 5, n_out).astype(np.float32))
    scale = 2.0 ** rs.randint(-10, 11, n_out)
    w = (rs.uniform(-1, 1, shape) * scale.reshape((-1,) + (1,) * (len(shape) - 1))).astype(np.float32)
    return (w, (rs.uniform(-1, 1, n_out) * scale).astype(np.float32))


def _conv(family, rs, C, U, M, gains=False):
    from keynet_b200 import sparse
    (f, b) = _values(rs, family, (M, C, 3, 3), M)
    (R, K) = (M * U * U + 1, C * U * U + 1)
    return sparse.keyed_toeplitz_conv2d((C, U, U), f, b, 1, _key(rs, R, gains=gains), _key(rs, K, gains=gains))


def _linear(family, rs, n_in, n_out):
    from keynet_b200 import sparse
    (w, b) = _values(rs, family, (n_out, n_in), n_out)
    return sparse.keyed_linear(w, b, None, _key(rs, n_in + 1))


# id -> (builder(family, rs), quantum of the exact family)
CASES = {
    'G6': (lambda fam, rs: _conv(fam, rs, 4, 8, 6, gains=True), 2.0 ** -4),        # padded route: pg_small
    'G12': (lambda fam, rs: _conv(fam, rs, 4, 8, 12, gains=True), 2.0 ** -4),
    'G16': (lambda fam, rs: _conv(fam, rs, 16, 24, 16), 1.0),                       # padded route: pg_simt; shared form at every N
    'G48': (lambda fam, rs: _conv(fam, rs, 16, 24, 48), 1.0),
    'G100': (lambda fam, rs: _conv(fam, rs, 16, 24, 100), 1.0),
    'C3_first': (lambda fam, rs: _conv(fam, rs, 3, 16, 16), 1.0),                   # padded route: pg_cluster
    'G160_perm': (lambda fam, rs: _conv(fam, rs, 16, 8, 160), 1.0),                 # 9 shared blocks, ragged group_k; 64 pixels:
                                                                                    # row form at N <= 4, shared form above
    'G160_gain': (lambda fam, rs: _conv(fam, rs, 16, 8, 160, gains=True), 2.0 ** -4),   # one block per pixel: row form
    'G300': (lambda fam, rs: _conv(fam, rs, 16, 8, 300), 1.0),                      # row tiles
    'fc_4096_300': (lambda fam, rs: _linear(fam, rs, 4096, 300), 1.0),              # one group: row form up to N = 8
}


def _plans(W, N):
    from keynet_b200.sparse import PatternGroups
    return [PatternGroups._narrow_plan(c, N) for c in W._pg.classes]


def _lanes_nb(N):
    return {1: 1, 2: 2}.get(N, 4 if N <= 4 else 8)


def _expected(W, N, relu):
    """Kernels one sparse.spmm call must launch: per class pg_simt<RW> (shared-block form: RW = 1 / 2 / 4 for G <= 8 / 16 /
    more) or spmm_lanes_nnz<NB> (row form), and the CSR kernel of leftover rows (N <= 8: lanes_nnz, else rowwarp<1>)."""
    r = _B[relu]
    exp = set()
    for (c, p) in zip(W._pg.classes, _plans(W, N)):
        if p['row_form']:
            exp.add('spmm_lanes_nnz_kernel<%d,%s>' % (_lanes_nb(N), r))
        else:
            exp.add('pg_simt_kernel<%d,%s>' % (1 if c['G'] <= 8 else 2 if c['G'] <= 16 else 4, r))
    if W._pg.rest is not None:
        exp.add('spmm_lanes_nnz_kernel<%d,%s>' % (_lanes_nb(N), r) if N <= 8 else 'spmm_rowwarp_kernel<1,%s>' % r)
    return exp


def _profiled(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        n = kl.normalise(e.name)
        if kl.family(n) in kl.SPMM_FAMILIES:
            names.add(n)
    return names


def _dense(arrays, shape):
    (ip, ix, dt) = arrays
    (R, K) = shape
    rows = torch.from_numpy(np.repeat(np.arange(R), np.diff(ip))).cuda()
    W64 = torch.zeros((R, K), dtype=torch.float64, device='cuda')
    W64[rows, torch.from_numpy(ix.astype(np.int64)).cuda()] = torch.from_numpy(dt.astype(np.float64)).cuda()
    return W64


def _inputs(family, rs, K, N):
    if family == 'exact':
        X = rs.randint(-8, 9, (K, N)).astype(np.float32)
    else:
        X = (10.0 ** rs.uniform(-20, 20, (K, N)) * rs.choice([-1, 1], (K, N))).astype(np.float32)
    X[-1] = 1.0
    return torch.from_numpy(X).cuda()


def _bits(t):
    return t.contiguous().view(torch.int32)


def _old_route(W, X, relu):
    """What sparse.spmm did for N < 32 on a dropped-CSR layer before the narrow path: pad X to 32 columns, run the grouped
    kernels, keep the first N columns."""
    (K, N) = X.shape
    xp = torch.zeros((K, 32), dtype=torch.float32, device='cuda')
    xp[:, :N] = X
    yp = torch.empty((W.shape[0], 32), dtype=torch.float32, device='cuda')
    W._pg.spmm(xp, yp, relu)
    return yp[:, :N].contiguous()


def _old_route_ran_simt(W):
    return all(c.get('cg') is None and not (c['G'] <= 16 and c['K_pad'] <= 128) for c in W._pg.classes)


def _abi_narrow(W, X, n, relu):
    """Every class through kn_spmm_pg_narrow_f32 (and `rest` through the CSR rows kernel) with X a NaN-padded view of odd ldx
    and Y offset by one float with an odd ldy; returns Y's body after checking that the padding kept its bits."""
    from keynet_b200 import _native
    from keynet_b200._native import check, ptr, stream_ptr
    L = _native.lib()
    (R, K) = W.shape
    odd = lambda v: v + 1 + (v % 2)
    (ldx, ldy, off) = (odd(n), odd(n), 1)
    Xb = torch.full((K, ldx), float('nan'), device='cuda')
    Xb[:, :n] = X[:, :n]
    Yb = torch.full((off + R * ldy + 4,), PAYLOAD, dtype=torch.int32, device='cuda')
    (xp, yp, s) = (ctypes.c_void_p(Xb.data_ptr()), ctypes.c_void_p(Yb.data_ptr() + 4 * off), stream_ptr())
    flags = _native.KN_SPMM_RELU if relu else 0
    for (c, p) in zip(W._pg.classes, _plans(W, n)):
        check(L.kn_spmm_pg_narrow_f32(ptr(c['rows']), ptr(c['cols']), ptr(c['vals']), ptr(c['group_k']), ptr(c['block_of']), c['n_groups'], c['G'], c['K_pad'],
                                      ptr(p['groups']), ptr(p['start']), p['n_runs'], p['row_form'], xp, ldx, yp, ldy, n, flags, None, s))
    r = W._pg.rest
    if r is not None:
        check(L.kn_spmm_csr_rows_f32(ptr(r['indptr']), ptr(r['indices']), ptr(r['data']), r['n'], W.shape[1], ptr(r['out_rows']), xp, ldx, yp, ldy, n, flags, None, s))
    torch.cuda.synchronize()
    body = Yb[off:off + R * ldy].view(R, ldy)
    assert bool((Yb[:off] == PAYLOAD).all()) and bool((Yb[off + R * ldy:] == PAYLOAD).all()) and bool((body[:, n:] == PAYLOAD).all()), \
        'Y padding was written (ldx=%d ldy=%d n=%d)' % (ldx, ldy, n)
    assert bool(Xb[:, n:].isnan().all())
    return body[:, :n].contiguous().view(torch.float32)


def _run_case(case_id, N, relu):
    from keynet_b200 import sparse
    (builder, quantum) = CASES[case_id]
    rs = np.random.RandomState(zlib.crc32(('narrow/%s/%d/%d' % (case_id, N, relu)).encode()))
    tag = '%s N=%d relu=%s' % (case_id, N, relu)
    # ---------------- exact family
    W = builder('exact', rs)
    (R, K) = W.shape
    W64 = _dense(W.csr_arrays(), W.shape)
    W.drop_csr()
    X = _inputs('exact', rs, K, N)
    X64 = X.double()
    S = W64.abs() @ X64.abs()
    assert float(S.max()) < 2.0 ** 20 * quantum
    y64 = W64 @ X64
    ref = (y64.clamp(min=0) if relu else y64).float()
    out = torch.full((R, N), float('nan'), device='cuda')
    sparse.spmm(W, X, relu=relu, out=out)
    bad = ~(out == ref)
    assert not bool(bad.any()), '%s exact: %d of %d elements differ from the fp64 product, first at %s: %r vs %r' % (
        tag, int(bad.sum()), bad.numel(), tuple(bad.nonzero()[0].tolist()), float(out[bad][0]), float(ref[bad][0]))
    y = _abi_narrow(W, X, N, relu)
    assert torch.equal(_bits(y), _bits(out)), '%s abi: differs from the plain call' % tag
    del W64, X64, y64, ref, S

    # ---------------- wide family
    W = builder('wide', rs)
    arrays = W.csr_arrays()
    W64 = _dense(arrays, W.shape)
    W.drop_csr()
    X = _inputs('wide', rs, K, N)
    y = torch.full((R, N), float('nan'), device='cuda')
    sparse.spmm(W, X, relu=relu, out=y)
    assert bool(torch.isfinite(y).all()), '%s wide: inf or NaN' % tag
    X64 = X.double()
    S = W64.abs() @ X64.abs()
    y64 = W64 @ X64
    if relu:
        y64 = y64.clamp(min=0)
    n = torch.from_numpy(np.diff(arrays[0]).astype(np.float64) + 1.0).cuda().view(-1, 1)
    u = 2.0 ** -24
    over = (y.double() - y64).abs() > (n * u / (1.0 - n * u)) * S
    assert not bool(over.any()), '%s wide: %d elements over gamma(K+S+1) sum|w||x|' % (tag, int(over.sum()))
    if _old_route_ran_simt(W) and not any(p['row_form'] for p in _plans(W, N)):
        old = _old_route(W, X, relu)
        assert torch.equal(_bits(y), _bits(old)), '%s: differs from the padded pg_simt route bit for bit (%d elements)' % (
            tag, int((_bits(y) != _bits(old)).sum()))


PARAMS = [(c, n) for c in CASES for n in NS]


def _names_case(case_id, N, relu):
    """(message or '', expected narrow kernels): '' if exactly those (and the CSR kernel iff the layer has leftover rows) ran."""
    from keynet_b200 import sparse
    rs = np.random.RandomState(zlib.crc32(('names/%s/%d/%d' % (case_id, N, relu)).encode()))
    W = CASES[case_id][0]('exact', rs)
    W.drop_csr()
    X = _inputs('exact', rs, W.shape[1], N)
    expect = _expected(W, N, relu)
    got = _profiled(lambda: sparse.spmm(W, X, relu=relu))
    if got != expect:
        return ('%s N=%d relu=%s: launched %s, expected %s' % (case_id, N, relu, sorted(got), sorted(expect)), expect)
    return ('', expect)


def _child_names():
    """Runs in a process of its own: every (case, N, ReLU) under torch.profiler."""
    (bad, seen) = ([], set())
    for (case_id, N) in PARAMS:
        for relu in (False, True):
            (msg, expect) = _names_case(case_id, N, relu)
            if msg:
                bad.append(msg)
            else:
                seen |= expect
    return dict(bad=bad, seen=sorted(seen))


@pytest.mark.gpu
def test_kernel_names():
    """Which kernels every layer case launches, under torch.profiler in a process of its own (a fresh profiler: this
    module's numerics run in the suite's process after hundreds of other profiled calls): exactly the narrow kernels the
    class plans name, plus the CSR kernel when the layer has leftover rows.  Together the cases launch both forms at every
    row tile and batch width they use."""
    code = ('import json, sys; sys.path.insert(0, %r); from tests import test_gpu_narrow_batch as m; '
            'print("NAMES=" + json.dumps(m._child_names()))' % ROOT)
    p = subprocess.run([sys.executable, '-c', code], cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    res = json.loads([l for l in p.stdout.splitlines() if l.startswith('NAMES=')][-1][len('NAMES='):])
    assert not res['bad'], '\n'.join(res['bad'][:20])
    want = set('pg_simt_kernel<%d,%s>' % (rw, r) for rw in (1, 2, 4) for r in _B) | set('spmm_lanes_nnz_kernel<%d,%s>' % (nb, r) for nb in (1, 2, 4, 8) for r in _B)
    assert want <= set(res['seen']), 'not launched by any case: %s' % sorted(want - set(res['seen']))


@pytest.mark.gpu
@pytest.mark.parametrize('case_id,N', PARAMS, ids=['%s-N%d' % p for p in PARAMS])
def test_narrow_layer(case_id, N):
    for relu in (False, True):
        _run_case(case_id, N, relu)


@pytest.mark.gpu
def test_forms_chosen_per_class():
    """Row form where the shared-block tile would be less than a quarter full at NB <= 8, shared form otherwise."""
    rs = np.random.RandomState(0)
    expect = {'G48': {1: 'shared', 8: 'shared', 31: 'shared'}, 'G160_perm': {1: 'rows', 8: 'shared', 31: 'shared'},
              'G160_gain': {1: 'rows', 8: 'rows', 31: 'shared'}, 'fc_4096_300': {1: 'rows', 8: 'rows', 9: 'shared', 31: 'shared'}}
    for (case_id, forms) in expect.items():
        W = CASES[case_id][0]('exact', rs)
        for (N, form) in forms.items():
            rf = [p['row_form'] for p in _plans(W, N)]
            assert all(bool(f) == (form == 'rows') for f in rf), (case_id, N, rf)


# ---------------------------------------------------------------------------------------------------------------------
# end to end
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def acn_dropped():
    import bench
    from keynet_b200 import system
    wl = bench.workload('acn')
    np.random.seed(0)
    (sensor, knet) = system.Keynet(wl['inshape'], wl['net'], keep_csr=False, **wl['keys'])
    return (wl, sensor, knet)


@pytest.mark.gpu
@pytest.mark.parametrize('N', [1, 3])
def test_allconvnet_dropped_csr_narrow_batch_matches_plain_net(acn_dropped, N):
    import bench
    (wl, sensor, knet) = acn_dropped
    x = torch.randn((N,) + wl['inshape'], generator=torch.Generator().manual_seed(N))
    y = knet.forward(sensor.fromtensor(x.cuda()).encrypt().astensor()).reshape(N, -1).cpu().numpy()
    plain = bench.keyed_pooling(wl['net'])
    with torch.no_grad():
        yp = plain(x).numpy()
    scale = float(np.abs(yp).max())
    assert np.allclose(y, yp, atol=1e-4 * max(1.0, scale)), (np.abs(y - yp).max(), scale)
    assert np.array_equal(y.argmax(1), yp.argmax(1))
    NB = 1 << (N - 1).bit_length()
    grouped = [L.W._pg for (_, L) in knet.keyedlayers() if L.W._pg is not None and L.W._data is None]
    assert grouped and all(NB in c.get('narrow', {}) for pg in grouped for c in pg.classes)     # every class went narrow


@pytest.mark.gpu
def test_forwardplan_batch1_graph_equals_eager(acn_dropped):
    from keynet_b200 import engine
    (wl, sensor, knet) = acn_dropped
    images = torch.randn((1,) + wl['inshape'], device='cuda', generator=torch.Generator(device='cuda').manual_seed(7))
    eager = engine.ForwardPlan(sensor, knet, 1, use_graph=False)
    y_e = eager.run_device(images).clone()
    graph = engine.ForwardPlan(sensor, knet, 1, use_graph=True)
    assert graph.graph is not None
    y_g = graph.run_device(images).clone()
    y_g2 = graph.run_device(images).clone()
    torch.cuda.synchronize()
    assert torch.equal(_bits(y_e), _bits(y_g)) and torch.equal(_bits(y_g), _bits(y_g2))
    n_narrow = sum(W._pg.launches_narrow() for (_, W, _) in graph.layers[1:] if W._pg is not None and W._data is None)
    assert n_narrow > 0 and graph.launches_per_run >= n_narrow


@pytest.mark.gpu
@pytest.mark.slow
def test_vgg16_dropped_csr_narrow_batch_matches_plain_net():
    import bench
    from keynet_b200 import system
    if torch.cuda.mem_get_info()[0] < 120e9:
        pytest.skip('needs ~120 GB of free HBM for the per-layer compile transients')
    wl = bench.workload('vgg16')
    np.random.seed(0)
    (sensor, knet) = system.Keynet(wl['inshape'], wl['net'], keep_csr=False, **wl['keys'])
    plain = bench.keyed_pooling(wl['net']).cuda()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    for N in (1, 3):
        x = torch.randn((N,) + wl['inshape'], generator=torch.Generator().manual_seed(10 + N))
        y = knet.forward(sensor.fromtensor(x.cuda()).encrypt().astensor()).reshape(N, -1).cpu().numpy()
        with torch.no_grad():
            yp = plain(x.cuda()).cpu().numpy()
        scale = float(np.abs(yp).max())
        assert np.allclose(y, yp, atol=1e-3 * max(1.0, scale)), (N, np.abs(y - yp).max(), scale)
        assert np.array_equal(y.argmax(1), yp.argmax(1))
