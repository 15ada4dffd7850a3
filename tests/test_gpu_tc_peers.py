"""The fused all-gather (PEERS) instantiations of the tensor-core kernels on one GPU: every layer stores into two local
buffers standing in for two ranks' output slots, under a random need mask.  Rows a rank needs must equal a plain run of the
same layer; rows it does not need, and the layer's own output buffer, must stay untouched.

Layers (permutation input keys) and the paths they take:
  * G = 64 conv:                pg_tile_tc (tile class)
  * G = 256 conv at N = 384:    pg_tc, one batch tile per CTA, 3 batch tiles: no cluster
  * G = 256 conv at N = 512:    pg_tc, one batch tile per CTA, 4 batch tiles: 2-CTA multicast clusters
  * G = 192 conv at N = 512:    pg_tc, two batch tiles per CTA
  * 4096 -> 512 linear:         pg_tc over K slices into local partial rows, then kn_splitk_reduce_f32 stores to the peers
"""
import functools

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

LAYERS = {  # name: (kind, C, M, U) -- linear: C inputs, M outputs
    'tile64': ('conv', 64, 64, 16),
    'tc256': ('conv', 256, 256, 8),
    'tc192': ('conv', 64, 192, 8),
    'splitk': ('linear', 4096, 512, None),
}


@functools.lru_cache(maxsize=None)
def _layer(name):
    from keynet_b200 import sparse
    from keynet_b200.sparse import MonomialKey
    (kind, C, M, U) = LAYERS[name]
    rs = np.random.RandomState(C + M)
    if kind == 'conv':
        lim = np.sqrt(6.0 / (9 * C))
        f = rs.uniform(-lim, lim, (M, C, 3, 3)).astype(np.float32)
        b = rs.uniform(-0.1, 0.1, M).astype(np.float32)
        K = C * U * U + 1
        W = sparse.keyed_toeplitz_conv2d((C, U, U), f, b, 1, None, MonomialKey(np.concatenate([rs.permutation(K - 1), [K - 1]])))
    else:
        lim = np.sqrt(6.0 / C)
        w = rs.uniform(-lim, lim, (M, C)).astype(np.float32)
        b = rs.uniform(-0.1, 0.1, M).astype(np.float32)
        W = sparse.keyed_linear(w, b, None, MonomialKey(np.concatenate([rs.permutation(C), [C]])))
    cls = W._pg.classes
    if name == 'tile64':
        assert any(c.get('tile') is not None for c in cls) and sparse.tiles_enabled()
    elif name == 'splitk':
        assert any(c.get('splitk') is not None for c in cls)
    else:
        assert any(c['tc'] is not None and c.get('tile') is None and c.get('splitk') is None for c in cls)
    assert sparse.tensor_cores_enabled()
    return W


@pytest.mark.parametrize('relu', [False, True])
@pytest.mark.parametrize('name,N', [('tile64', 256), ('tc256', 384), ('tc256', 512), ('tc192', 512), ('splitk', 256)])
def test_peers_stores_match_plain(name, N, relu):
    from keynet_b200 import _native, sparse
    W = _layer(name)
    (R, K) = W.shape
    g = torch.Generator(device='cuda').manual_seed(N + K)
    x = torch.randn((K, N), generator=g, device='cuda')
    x[-1] = 1.0                                                          # homogeneous coordinate (bias)
    ref = sparse.spmm(W, x, relu=relu)
    row_mask = torch.randint(0, 4, (R,), generator=g, device='cuda', dtype=torch.uint8)
    (y, d0, d1) = (torch.full((R, N), float('nan'), device='cuda') for _ in range(3))
    sparse.spmm(W, x, relu=relu, out=y, peers=_native.Peers([d0.data_ptr(), d1.data_ptr()], row_mask))
    torch.cuda.synchronize()
    assert torch.isnan(y).all(), 'the layer wrote its own output buffer although peers were given'
    ref = ref.cpu().numpy()
    tol = 1e-4 * np.abs(ref) + 1e-5 * np.abs(ref).max()
    mask = row_mask.cpu().numpy()
    for (p, d) in enumerate((d0.cpu().numpy(), d1.cpu().numpy())):
        need = ((mask >> p) & 1).astype(bool)
        assert need.any() and (~need).any()
        assert np.all(np.abs(d[need] - ref[need]) <= tol[need]), (p, float(np.nanmax(np.abs(d[need] - ref[need]))))
        assert np.isnan(d[~need]).all(), 'rows rank %d does not need were written' % p
