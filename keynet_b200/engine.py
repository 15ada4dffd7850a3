"""Batched forward engine: the keyed layer chain for a fixed batch size with pre-allocated, feature-major
activation buffers, launched either eagerly or as one CUDA graph (the chain is launch-latency bound for
LeNet-sized nets).  B200-side replacement for looping `KeyedLayer.forward` (keynet/system.py:130-133)."""
import os

import numpy as np
import torch

from . import _native
from . import layer as _layer
from .sparse import spmm


_FUSE = [os.environ.get('KEYNET_B200_FUSE', '0') != '0']


def fusion_enabled(flag=None):
    """Switch for the fused conv (+ReLU) -> average-pooling kernel (csrc/convpool.cu); off (default) = one launch per keyed
    layer.  Measured on B200, LeNet batch 65 536: the fused pairs take 1.16 + 1.85 ms against 0.66 + 0.81 ms unfused -- the
    intermediate stays in shared memory (HBM traffic 5.8x lower) but with 4 batch columns per CTA the direct convolution runs at
    15 % of the fp32 FMA peak; it needs register tiling over pixels before it pays.  KEYNET_B200_FUSE=1 enables it."""
    if flag is not None:
        _FUSE[0] = bool(flag)
    return _FUSE[0]


def _fusable(Wc, relu_c, Wp, N):
    """Tables of the fused conv -> ReLU -> avgpool kernel for two consecutive layers, or None: permutation-only keys, the
    conv's output key cancelling against the pool's input key, and the whole image (input + conv output) of 4 batch columns
    fitting shared memory."""
    (rc, rp) = (getattr(Wc, '_recipe', None), getattr(Wp, '_recipe', None))
    if rc is None or rp is None or rc['kind'] != 'conv' or rp['kind'] != 'pool' or not relu_c or N % 4 != 0:
        return None
    (C, U, V, M, P, Q, stride) = rc['geom']
    (Cp, Up_in, Vp_in, _, k, _, pstride) = rp['geom']
    (Uo, Vo) = (U // stride, V // stride)
    if (Cp, Up_in, Vp_in) != (M, Uo, Vo) or Uo % pstride != 0 or Vo % pstride != 0:
        return None
    if ((C * U * V + M * Uo * Vo) * 4 + (M + 5) * (C * P * Q + 1)) * 4 > 220 * 1024:
        return None
    n_mid = M * Uo * Vo + 1
    (po, pi) = (rc['out_perm'], rp['in_perm'])
    if (po is None) != (pi is None):
        return None
    if po is not None and not np.array_equal(np.asarray(pi)[np.asarray(po)], np.arange(n_mid)):
        return None                                       # the pool does not read the conv's rows where the conv writes them
    dev = torch.device('cuda', torch.cuda.current_device())
    n_in = C * U * V + 1
    xrow = np.arange(n_in, dtype=np.int32) if rc['in_perm'] is None else np.asarray(rc['in_perm'], dtype=np.int32)
    n_out = M * (Uo // pstride) * (Vo // pstride) + 1
    if rp['out_perm'] is None:
        yrow = np.arange(n_out, dtype=np.int32)
    else:
        yrow = np.empty(n_out, dtype=np.int32)
        yrow[np.asarray(rp['out_perm'])] = np.arange(n_out, dtype=np.int32)
    return dict(desc=_native.kn_conv2d_desc(C, U, V, M, P, Q, int(stride), 0, 1), w=torch.from_numpy(np.ascontiguousarray(rc['fq'], dtype=np.float32)).to(dev),
                b=torch.from_numpy(np.ascontiguousarray(rc['bq'], dtype=np.float32)).to(dev), xrow=torch.from_numpy(xrow).to(dev), yrow=torch.from_numpy(yrow).to(dev),
                k=int(k), pstride=int(pstride), pool_w=float(rp['pool_w']))


class ForwardPlan(object):
    """sensor.encrypt() + knet.forward() for batches of exactly N images.

    run_device(images[N,C,H,W] cuda) -> logits[N,K] cuda     (everything stays in HBM)
    run_host(images pinned host)     -> logits host tensor    (H2D + chain + D2H, checks the homogeneous coordinate)
    """

    def __init__(self, sensor, knet, batch, use_graph=True, time_layers=False, event_sets=1):
        _native.require_cuda()
        self.dev = torch.device('cuda', torch.cuda.current_device())
        self.N = int(batch)
        self.sensor = sensor
        self.knet = knet
        self.layers = [('sensor', sensor.W, False)] + [(k, L.W, L._fused_relu or 'ReLU' in L._layertype) for (k, L) in knet.keyedlayers()]
        self.D = int(np.prod(sensor._inshape))
        assert sensor.W.shape[1] == self.D + 1
        self.K = self.layers[-1][1].shape[0] - 1
        N = self.N
        self.images = torch.empty((N, self.D), dtype=torch.float32, device=self.dev)
        self.acts = [torch.empty((W.shape[0], N), dtype=torch.float32, device=self.dev) for (_, W, _) in self.layers]
        self.logits = torch.empty((N, self.K), dtype=torch.float32, device=self.dev)
        self.bad = torch.zeros(1, dtype=torch.int32, device=self.dev)
        from .sparse import MonomialKey
        self.fused_encrypt = isinstance(sensor.keypair()[0], MonomialKey)          # image key applied inside the transpose kernel
        # conv (+ReLU) -> avgpool pairs whose intermediate fits shared memory run as ONE launch (csrc/convpool.cu)
        self.fused = {}
        if fusion_enabled():
            i = 1
            while i + 1 < len(self.layers):
                f = _fusable(self.layers[i][1], self.layers[i][2], self.layers[i + 1][1], N) if not self.layers[i + 1][2] else None
                if f is not None:
                    self.fused[i] = f
                    i += 2
                else:
                    i += 1
        skip = set(i + 1 for i in self.fused)
        def spmm_launches(W):
            if W._pg is not None and N >= 32 and N % 4 == 0:
                return W._pg.launches()
            if W._pg is not None and W._data is None and N < 32:
                return W._pg.launches_narrow()
            return 1
        self.launches_per_run = (1 if self.fused_encrypt else 3) + sum(0 if i in skip else (1 if i in self.fused else spmm_launches(W))
                                                                        for (i, (_, W, _)) in enumerate(self.layers) if i >= 1)
        self.time_layers = time_layers
        # per-layer CUDA events on the launch stream, one set per timed step (read back after the timed region)
        self.layer_events = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in self.layers]
                             for _ in range(max(1, event_sets))] if time_layers else None
        self.event_set = 0
        self.graph = None
        if use_graph and not time_layers:
            self._capture()

    # ---- the chain: encrypt kernel + one SpMM per keyed layer + 1 layout kernel
    def _chain(self):
        L = _native.lib()
        s = _native.stream_ptr()
        x = None
        skip = -1
        for (i, (name, W, relu)) in enumerate(self.layers):
            if self.time_layers:
                self.layer_events[self.event_set][i][0].record()
            if i == 0:
                self.sensor.encrypt_into(self.images, self.acts[0])     # homogenise + transpose + image key (one kernel for monomial keys)
            elif i == skip:
                pass                                                    # produced by the fused launch of the previous layer
            elif i in self.fused:
                f = self.fused[i]
                _native.check(L.kn_convpool_f32(f['desc'], _native.ptr(f['w']), _native.ptr(f['b']), _native.ptr(f['xrow']), f['k'], f['pstride'], f['pool_w'], _native.ptr(f['yrow']),
                                                _native.ptr(x), self.N, _native.ptr(self.acts[i + 1]), self.N, self.N, s))
                skip = i + 1
            else:
                spmm(W, x, relu=relu, out=self.acts[i])
            if self.time_layers:
                self.layer_events[self.event_set][i][1].record()
            if i not in self.fused:
                x = self.acts[i]
        _native.check(L.kn_linear_to_affine_t(_native.ptr(x), self.N, self.N, self.K, _native.ptr(self.logits), 1e-3, _native.ptr(self.bad), s))

    def _capture(self):
        self._chain()                      # warm-up outside capture (lazy module load, smem attributes)
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                self._chain()
        torch.cuda.current_stream().wait_stream(side)
        self.graph = g

    def _launch(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self._chain()

    def run_device(self, images=None):
        """images: [N,C,H,W] (or [N,D]) float32 on this device, or None to reuse the staged batch."""
        if images is not None:
            self.images.copy_(images.reshape(self.N, self.D), non_blocking=True)
        self._launch()
        return self.logits

    def run_host(self, images_host, out_host=None):
        """End-to-end call with HOST buffers: H2D of the images, the whole chain, D2H of the logits."""
        self.bad.zero_()
        self.images.copy_(images_host.reshape(self.N, self.D), non_blocking=True)
        self._launch()
        out = out_host if out_host is not None else torch.empty((self.N, self.K), dtype=torch.float32, pin_memory=True)
        out.copy_(self.logits, non_blocking=True)
        bad = self.bad.cpu()               # synchronises the stream
        if int(bad.item()) != 0:
            raise ValueError('invalid affine vector: %d outputs lost the homogeneous coordinate' % int(bad.item()))
        return out

    def run_host_many(self, batches, outs):
        """End-to-end over a sequence of HOST batches (pinned), software-pipelined: the H2D copy of batch k+1 runs on a copy
        stream while the chain of batch k runs on the compute stream (two device staging buffers); every batch still pays
        its own H2D of the images and D2H of the logits.  outs: pinned host tensors [N, K], one per batch (may repeat).
        Synchronises once at the end and checks the homogeneous coordinate of every batch."""
        assert len(batches) == len(outs)
        if not hasattr(self, '_stage'):
            self._stage = [torch.empty_like(self.images) for _ in range(2)]
            self._copy_stream = torch.cuda.Stream()
            self._h2d_done = [torch.cuda.Event() for _ in range(2)]
            self._stage_free = [torch.cuda.Event() for _ in range(2)]
        main = torch.cuda.current_stream()
        self.bad.zero_()
        for b in range(2):
            self._stage_free[b].record(main)
        def h2d(k):
            b = k % 2
            with torch.cuda.stream(self._copy_stream):
                self._copy_stream.wait_event(self._stage_free[b])          # the chain has consumed what was staged here
                self._stage[b].copy_(batches[k].reshape(self.N, self.D), non_blocking=True)
                self._h2d_done[b].record(self._copy_stream)
        if len(batches) > 0:
            h2d(0)
        for k in range(len(batches)):
            b = k % 2
            if k + 1 < len(batches):
                h2d(k + 1)
            main.wait_event(self._h2d_done[b])
            self.images.copy_(self._stage[b], non_blocking=True)           # device-to-device, then the staging buffer is free again
            self._stage_free[b].record(main)
            self._launch()
            outs[k].copy_(self.logits, non_blocking=True)
        bad = self.bad.cpu()               # synchronises the stream
        if int(bad.item()) != 0:
            raise ValueError('invalid affine vector: %d outputs lost the homogeneous coordinate' % int(bad.item()))
        return outs

    def layer_times_ms_mean(self, n_sets):
        """Mean launch duration of every layer's SpMM over the first n_sets recorded steps."""
        assert self.layer_events is not None
        torch.cuda.synchronize()
        out = []
        for (i, (name, _, _)) in enumerate(self.layers):
            ts = [self.layer_events[k][i][0].elapsed_time(self.layer_events[k][i][1]) for k in range(n_sets)]
            out.append((name, float(np.mean(ts))))
        return out

    def algorithmic_bytes(self):
        """SURVEY.md 8(d): per layer nnz*8 + (R+1)*4 + (C+R)*N*4."""
        out = []
        for (name, W, _) in self.layers:
            (R, C) = W.shape
            out.append((name, W.nnz() * 8 + (R + 1) * 4 + (C + R) * self.N * 4))
        return out
