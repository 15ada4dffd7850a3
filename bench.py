#!/usr/bin/env python
"""bench.py -- encrypted images/s of the keyed-layer forward path on B200 (BASELINE.json metric:
"encrypted imgs/sec keyed VGG16-224 & LeNet at 1/2/4/8 B200; SpMM HBM GB/s").

Default run = the metric's own workloads, in ONE JSON line (rank 0):
  headline   VGG16 3x224x224 `PermutationKeynet` (15.0 G stored non-zeros = 120 GB as CSR), global batch 256:
             --gpus 1   one GPU holds the whole keyed network as pattern groups with unique value blocks;
             --gpus N>1 every keyed layer ROW-SHARDED over the N GPUs, SpMM epilogues store straight into the peers'
                        activation buffers over NVLink (fused all-gather, keynet_b200/dist.py) -- strong scaling.
  extra.lenet  LeNet_AvgPool 1x28x28 PermutationKeynet (BASELINE configs[0]), 65 536 images per GPU, replicas.
  extra.acn    AllConvNet 3x32x32 hierarchical block-permutation keys (configs[1]), 4096 images in total, replicas.
One step = sensor.encrypt() + knet.forward() over one batch.

  python bench.py [--gpus N] [--steps K] [--warmup W]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --net lenet|acn|vgg16 [--batch B] [--parallel dp|rows|rows-fused]      (one workload only)
  python bench.py --mode keycompile                 (BASELINE configs[4]: key-compile sweep over the VGG16 layers)
  python bench.py --impl reference ...              (CPU arm: the oracle port of the reference's scipy path, all host threads)
  python bench.py ... --dump-outputs DIR            (also write the logits of the last timed step of every workload as DIR/<net>_logits.npy)

`value` = whole-job images/s with inputs resident in HBM; `e2e` = the same through the host-buffer API (pinned H2D of
the images and D2H of the logits inside the timed region); `roofline` = the dominant launch against the measured peaks
(MEASURED_PEAKS.json) plus the whole network against the HBM roofline; `cpu_baseline` = the oracle port on the host
cores on a bounded sample; `check` = parity of the very buffers that were timed (oracle / plain network), computed
after the timed region.
"""
import argparse
import glob
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

HBM_FALLBACK_GBS = 6650.0     # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
VGG_BATCH = 256
LENET_BATCH = 65536
ACN_BATCH = 4096
DUMP_BYTES = 64 * 10**6       # --dump-outputs: at most this much in all


# =================================================================================================
# workloads
def numpy_weights(net, seed):
    """Deterministic kaiming-uniform-like init from numpy's legacy RNG (same as tests/golden/make_golden.py)."""
    import torch
    rs = np.random.RandomState(seed)
    with torch.no_grad():
        for (name, p) in net.named_parameters():
            fan_in = int(np.prod(p.shape[1:])) if p.ndim > 1 else int(p.shape[0])
            bound = 1.0 / np.sqrt(max(1, fan_in))
            p.copy_(torch.from_numpy(rs.uniform(-bound, bound, size=tuple(p.shape)).astype(np.float32)))
    return net


def he_weights(net, seed):
    """He-uniform weights (bound sqrt(6/fan_in)), small biases: the activation scale survives 16 ReLU layers, so the VGG16
    logits depend on the input and an argmax comparison means something (SURVEY.md 7 / cfg 4)."""
    import torch
    rg = np.random.Generator(np.random.PCG64(seed))
    with torch.no_grad():
        for (name, p) in net.named_parameters():
            bound = np.float32(np.sqrt(6.0 / int(np.prod(p.shape[1:]))) if p.ndim > 1 else 0.1)
            p.copy_(torch.from_numpy((rg.random(size=tuple(p.shape), dtype=np.float32) * (2 * bound) - bound).astype(np.float32)))
    return net


class _no_default_init(object):
    """Skip torch's own parameter initialisation while a net is constructed (138 M parameters that he_weights overwrites)."""

    def __enter__(self):
        import torch
        self.saved = (torch.nn.Linear.reset_parameters, torch.nn.modules.conv._ConvNd.reset_parameters)
        torch.nn.Linear.reset_parameters = lambda m: None
        torch.nn.modules.conv._ConvNd.reset_parameters = lambda m: None

    def __exit__(self, *a):
        import torch
        (torch.nn.Linear.reset_parameters, torch.nn.modules.conv._ConvNd.reset_parameters) = self.saved


def workload(name):
    from keynet_b200 import nets
    if name == 'acn':
        return dict(name='acn', net=numpy_weights(nets.AllConvNet(batchnorm=False), 0).eval(), inshape=(3, 32, 32),
                    keys=dict(global_geometric='hierarchical_permutation', hierarchical_blockshape=(2, 2), hierarchical_permute_at_level=(0, 1)),
                    label='AllConvNet 3x32x32, hierarchical block-permutation keys (BASELINE configs[1])')
    if name == 'lenet':
        return dict(name='lenet', net=numpy_weights(nets.LeNet_AvgPool(), 0).eval(), inshape=(1, 28, 28), keys=dict(global_geometric='permutation'),
                    label='LeNet_AvgPool 1x28x28, PermutationKeynet (BASELINE configs[0])')
    if name == 'vgg16':
        with _no_default_init():
            net = nets.VGG16()
        return dict(name='vgg16', net=he_weights(net, 0).eval(), inshape=(3, 224, 224), keys=dict(global_geometric='permutation'),
                    label='VGG16 3x224x224, PermutationKeynet (BASELINE metric / configs[3]: 15.0 G stored non-zeros = 120 GB as CSR)')
    raise ValueError(name)


def keyed_pooling(net):
    """Copy of `net` with the pooling the reference actually keys: centred k x k windows, divisor k*k
    (keynet/layer.py:48-56 ignores padding / ceil_mode)."""
    import copy
    import torch
    plain = copy.deepcopy(net)
    for (k, mod) in list(plain.named_children()):
        if isinstance(mod, torch.nn.AvgPool2d):
            ks = mod.kernel_size if isinstance(mod.kernel_size, int) else mod.kernel_size[0]
            st = mod.stride if isinstance(mod.stride, int) else mod.stride[0]
            setattr(plain, k, torch.nn.AvgPool2d(ks, st, ks // 2, ceil_mode=False, count_include_pad=True))
    return plain


# =================================================================================================
# peaks, traffic, clocks
def _peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return {}


def hbm_peak():
    d = _peaks()
    if 'hbm_gbs' in d:
        return (float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)')
    return (HBM_FALLBACK_GBS, 'fallback (B200_PROFILING.md)')


def tensor_peak():
    """Dense bf16 tensor throughput measured on this pool's B200s (sustained figure: the kernel is timed inside a long step)."""
    d = _peaks()
    if 'bf16_tflops_sustained' in d:
        return (float(d['bf16_tflops_sustained']), 'measured bf16 sustained (MEASURED_PEAKS.json)')
    return (1400.0, 'fallback (B200_PROFILING.md, sustained)')


def lib_sha16():
    """Identity of the kernel code the library is built from: sha256 over keynet_b200/csrc/* and include/*.h, in name order.
    (Not the hash of the .so: a rebuild on another box embeds other source paths in its line tables and would read as stale.)"""
    h = hashlib.sha256()
    try:
        files = sorted(glob.glob(os.path.join(ROOT, 'keynet_b200', 'csrc', '*')) + glob.glob(os.path.join(ROOT, 'include', '*.h')))
        for f in files:
            h.update(os.path.basename(f).encode())
            with open(f, 'rb') as fh:
                h.update(fh.read())
        return h.hexdigest()[:16] if files else None
    except Exception:
        return None


def profiled_traffic(net, batch, layer):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed `ncu --set full`
    capture (profiles/traffic.json).  An entry is only valid for the kernel code it was captured from: entries carry the
    sha256 of the library's sources (lib_sha16) and are dropped (None) when the kernel code has changed since."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            t = json.load(f)
        e = t.get('%s:%d:%s' % (net, batch, layer))
        if isinstance(e, dict):
            return (e.get('bytes'), None) if e.get('lib_sha16') == lib_sha16() else (None, 'capture %s is from other kernel sources (stale)' % e.get('capture'))
        return (None, None if e is None else 'capture without a build hash (stale)')
    except Exception:
        return (None, None)


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled every 50 ms.  The sampler is started BEFORE the warm-up (nvidia-smi needs
    up to a second to produce its first line) and every line is time-stamped on arrival; stop() summarises the lines that
    arrived between mark_begin() and mark_end().  A timed region shorter than a few sampling periods is followed by
    hold(): the same step keeps running (untimed) until at least `min_samples` readings were taken under that load."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index
        (self.t0, self.t1) = (None, None)

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu_index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def in_region(self):
        (t0, t1) = (self.t0 if self.t0 is not None else 0.0, self.t1 if self.t1 is not None else float('inf'))
        return [r for (t, r) in list(self.rows) if t0 <= t <= t1]

    def hold(self, step, sync, min_samples=3, max_s=2.5):
        """Keep the GPU under the same load until the region holds min_samples readings (the end mark moves with it)."""
        if self.proc is None:
            return 0
        (extra, t_start) = (0, time.perf_counter())
        while len(self.in_region()) < min_samples and time.perf_counter() - t_start < max_s:
            step(); sync()
            extra += 1
            self.t1 = time.perf_counter()
        return extra

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable'], 'samples': 0}
        rows = self.in_region()
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        (sm, smax, reasons) = ([], [], set())
        for r in rows:
            f = [t.strip() for t in r.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1]))
            except ValueError:
                continue
            for (name, v) in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(smax) if smax else None, 'reasons': sorted(reasons), 'samples': len(sm)}


def host_threads():
    """Host cores this process may use.  (torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm runs on rank 0 alone
    and is meant to use all the host threads it can, so the OpenMP default is not what we want there.)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# =================================================================================================
# CPU legs (oracle port of the reference's scipy path).  Only this section touches oracle/.
def oracle_layers_from_gpu(sensor, knet):
    """Copy the (bit-exact, verified) compiled matrices to the host for the CPU baseline."""
    from oracle import keynet_oracle as ko
    layers = []
    (ip, ix, dt) = sensor.W.csr_arrays()
    layers.append((ko.csr(sensor.W.shape, ip, ix, dt), False))
    for (k, L) in knet.keyedlayers():
        (ip, ix, dt) = L.W.csr_arrays()
        layers.append((ko.csr(L.W.shape, ip - ip[0], ix, dt), bool(L._fused_relu)))
    return layers


def _walk_keyed_layers(wl, f_build):
    """Drive the host-side key chaining (keynet_b200.system.KeyedModel: keys only, no GPU) and call
    f_build(module, inshape, outshape, A, Ainv) -> (W_hat, extra) for every keyed layer, in order.
    Returns (image key A, [record with .W .relu .extra])."""
    from keynet_b200 import system
    from torch import nn
    recorded = []

    def f_layergen(module, inshape, outshape, A, Ainv):
        (What, extra) = f_build(module, inshape, outshape, A, Ainv)

        class Rec(nn.Module):       # stands in for a KeyedLayer inside KeyedModel's Sequential
            def fuse_relu(self, flag=True):
                self.relu = bool(flag)
                return self
        r = Rec(); r.W = What; r.relu = False; r.extra = extra
        recorded.append(r)
        return r
    np.random.seed(0)
    f_keypair = system.keypair_policy(**wl['keys'])
    (A, Ainv) = f_keypair('input', wl['inshape'])
    system.KeyedModel(wl['net'], wl['inshape'], Ainv, f_keypair, f_layergen)
    return (A, recorded)


def _pool_params(module):
    ks = module.kernel_size if isinstance(module.kernel_size, int) else module.kernel_size[0]
    st = module.stride if isinstance(module.stride, int) else module.stride[0]
    return (int(ks), int(st))


def oracle_layers_on_cpu(wl):
    """Reference arm, small networks: key the whole network on the CPU with the oracle (Toeplitz + two SpGEMMs per layer)."""
    from oracle import keynet_oracle as ko
    from torch import nn

    def f_build(module, inshape, outshape, A, Ainv):
        k = lambda K: None if K is None else ko.monomial_key(K.perm, K.scale)
        if isinstance(module, nn.Conv2d):
            W = ko.toeplitz_conv2d(inshape, module.weight.detach().numpy(), module.bias.detach().numpy(), module.stride[0])
        elif isinstance(module, nn.AvgPool2d):
            W = ko.toeplitz_avgpool2d(inshape, *_pool_params(module))
        elif isinstance(module, nn.Linear):
            W = ko.linear_matrix(module.weight.detach().numpy(), module.bias.detach().numpy())
        else:
            raise ValueError(str(type(module)))
        return (ko.key_compile(k(A), W, k(Ainv)), None)
    (A, rec) = _walk_keyed_layers(wl, f_build)
    return [(ko.monomial_key(A.perm, A.scale), False)] + [(r.W, r.relu) for r in rec]


def _axis_taps(U, k, stride):
    h = (k - 1) // 2
    return sum(sum(1 for p in range(-h, h + 1) if 0 <= u + p < U) for u in range(0, U, stride))


def oracle_bands_on_cpu(wl, frac):
    """VGG16-scale networks: the reference cannot key them on a host (~30 min, > 64 GB; BASELINE.md 2), so every layer
    is keyed on a ROW BAND -- the rows of an evenly spaced set of output pixels (all channels), about `frac` of the layer --
    with the oracle's Toeplitz emission and the same two csr_matmat products (oracle.key_compile_rows).  The bands are bit-
    equal to those rows of the full compile (tests/test_oracle_bands.py).  Returns a list of dicts (W band CSR, rows = the
    W_hat rows it holds, relu, nnz_full = stored entries of the full layer in closed form, name)."""
    from oracle import keynet_oracle as ko
    from torch import nn

    def f_build(module, inshape, outshape, A, Ainv):
        k = lambda K: None if K is None else ko.monomial_key(K.perm, K.scale)
        if isinstance(module, (nn.Conv2d, nn.AvgPool2d)):
            (C, U, V) = [int(s) for s in inshape]
            if isinstance(module, nn.Conv2d):
                (M, ks, st) = (module.out_channels, module.kernel_size[0], module.stride[0])
                (per_pix_build, per_pix) = (M * C * ks * ks, M * C * ks * ks)
            else:
                (ks, st) = _pool_params(module)
                (M, per_pix_build, per_pix) = (C, C * C * ks * ks, C * ks * ks)       # the reference emits C*C channel pairs per pixel
            (Uo, Vo) = (U // st, V // st)
            nnz_full = (M * C if isinstance(module, nn.Conv2d) else C) * _axis_taps(U, ks, st) * _axis_taps(V, ks, st) + (M * Uo * Vo if isinstance(module, nn.Conv2d) else 0) + 1
            n_pix = int(min(Uo * Vo, max(1, round(frac * nnz_full / per_pix)), max(1, 6000000 // per_pix_build)))
            pix = np.unique(np.linspace(0, Uo * Vo - 1, n_pix).astype(np.int64))
            if isinstance(module, nn.Conv2d):
                W = ko.toeplitz_conv2d_pixels(inshape, module.weight.detach().numpy(), module.bias.detach().numpy(), st, pix)
            else:
                W = ko.toeplitz_avgpool2d_pixels(inshape, ks, st, pix)
            src = (np.arange(M, dtype=np.int64).reshape(-1, 1) * (Uo * Vo) + pix.reshape(1, -1)).reshape(-1)
            R = M * Uo * Vo + 1
        elif isinstance(module, nn.Linear):
            (out, inn) = [int(s) for s in module.weight.shape]
            nnz_full = out * inn + out + 1
            src = np.unique(np.linspace(0, out - 1, int(min(out, max(256, round(frac * out))))).astype(np.int64))
            W = ko.linear_matrix_rows(module.weight.detach().numpy(), module.bias.detach().numpy(), src)
            R = out + 1
        else:
            raise ValueError(str(type(module)))
        if A is None:
            rows = np.sort(src)
        else:
            inv = np.empty(R, dtype=np.int64)
            inv[A.perm] = np.arange(R)
            rows = np.sort(inv[src])                       # rows of W_hat = A.W.Ainv whose Toeplitz row lies in the band
        return (ko.key_compile_rows(k(A), rows, W, k(Ainv)), dict(rows=rows, nnz_full=int(nnz_full)))
    (A, rec) = _walk_keyed_layers(wl, f_build)
    return [dict(W=r.W, rows=r.extra['rows'], nnz_full=r.extra['nnz_full'], relu=r.relu) for r in rec]


def time_bands(bands, n_images, threads, repeats=2, X=None):
    """Seconds the full network would take on n_images: per layer, csr_matvecs on the band (best of `repeats`) scaled by
    nnz_full / nnz_band.  Returns (scaled seconds, measured seconds, X list for reuse)."""
    from oracle import keynet_oracle as ko
    rs = np.random.RandomState(0)
    if X is None:
        X = [rs.rand(b['W'].shape[1], n_images).astype(np.float32) for b in bands]
    (scaled, measured) = (0.0, 0.0)
    for (b, x) in zip(bands, X):
        best = None
        for _ in range(repeats):
            t0 = time.perf_counter()
            ko.spmm(b['W'], x, relu=b['relu'], threads=threads)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        measured += best
        scaled += best * b['nnz_full'] / max(1, len(b['W'].data))
    return (scaled, measured, X)


def time_oracle(layers, inshape, n_images, threads, repeats=1):
    from oracle import keynet_oracle as ko
    rs = np.random.RandomState(0)
    x = ko.affine_to_linear(rs.randn(n_images, *inshape).astype(np.float32))
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        y = ko.keyed_forward(layers, x, threads=threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    ko.linear_to_affine(y)
    return best


def cpu_baseline(layers, inshape, budget_s=15.0):
    threads = host_threads()
    t_probe = time_oracle(layers, inshape, 32, threads)
    n = int(max(32, min(262144, (budget_s / max(t_probe / 32.0, 1e-6)))))
    dt = time_oracle(layers, inshape, n, threads)
    return {'value': n / dt, 'unit': 'images/s', 'cores': threads, 'kind': 'port',
            'sample': '%d images through the same compiled layer stack, oracle csr_matvecs port (OpenMP over rows), %.1f s' % (n, dt)}


BAND_FRAC = 1.0 / 300.0
BAND_IMAGES = 32


def cpu_baseline_bands(bands, n_images=BAND_IMAGES, rounds=3):
    threads = host_threads()
    (best, X, meas) = (None, None, 0.0)
    for _ in range(rounds):
        (scaled, measured, X) = time_bands(bands, n_images, threads, X=X)
        if best is None or scaled < best:
            (best, meas) = (scaled, measured)
    nb = sum(len(b['W'].data) for b in bands)
    nf = sum(b['nnz_full'] for b in bands)
    return {'value': n_images / best, 'unit': 'images/s', 'cores': threads, 'kind': 'port',
            'sample': ('%d images; per layer the oracle csr_matvecs port (OpenMP over rows) on a row band keyed by the oracle (evenly spaced output pixels, all channels: '
                       '%.1f M of %.2f G stored entries in total), time scaled by nnz_layer / nnz_band and summed over the %d keyed layers; %.2f s measured -> %.1f s scaled'
                       % (n_images, nb / 1e6, nf / 1e9, len(bands), meas, best))}


def run_reference(args, rank, world):
    """CPU arm: rank 0 only; the oracle port keys and runs the same workload on the host cores."""
    if rank != 0:
        return
    net = args.net or 'vgg16'
    wl = workload(net)
    threads = host_threads()
    t0 = time.perf_counter()
    if net == 'vgg16':
        bands = oracle_bands_on_cpu(wl, BAND_FRAC)
        n = BAND_IMAGES
        X = None
        for _ in range(max(1, min(args.warmup, 1))):
            (_, _, X) = time_bands(bands, n, threads, repeats=1, X=X)
        t_key = time.perf_counter() - t0
        (scaled, measured) = (0.0, 0.0)
        for _ in range(args.steps):
            (s, m, X) = time_bands(bands, n, threads, repeats=1, X=X)
            scaled += s; measured += m
        dt = scaled                                                # seconds the full layers would take, summed over the steps
        nb = sum(len(b['W'].data) for b in bands)
        sample = ('%d images per step, %d steps; every layer runs on a row band keyed by the oracle (%.1f M of %.2f G stored entries in total) and its time is '
                  'scaled by nnz_layer / nnz_band: %.2f s measured -> %.1f s scaled' % (n, args.steps, nb / 1e6, sum(b['nnz_full'] for b in bands) / 1e9, measured, scaled))
    else:
        layers = oracle_layers_on_cpu(wl)
        t_key = time.perf_counter() - t0
        t_probe = time_oracle(layers, wl['inshape'], 2, threads)
        n = int(max(1, min(64, 4.0 / max(t_probe / 2.0, 1e-6))))       # ~4 s of CPU work per step
        for _ in range(max(1, min(args.warmup, 1))):
            time_oracle(layers, wl['inshape'], n, threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            time_oracle(layers, wl['inshape'], n, threads)
        dt = time.perf_counter() - t0
        sample = '%d images per step, %d steps, whole network keyed by the oracle' % (n, args.steps)
    v = n * args.steps / dt
    out = {'impl': 'reference', 'metric': 'encrypted_images_per_sec', 'value': v, 'unit': 'images/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
           'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'strong' if net == 'vgg16' else 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
           'config': {'workload': wl['label'], 'images_per_step': n, 'key_compile_s': round(t_key, 2),
                      'note': 'CPU arm: oracle port of the reference scipy path (csr_matmat key compile, csr_matvecs forward); each step is a bounded sample of the workload'},
           'cpu_baseline': {'value': v, 'unit': 'images/s', 'cores': threads, 'kind': 'port', 'sample': sample},
           'e2e': {'value': v, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(out))


# =================================================================================================
# parity of the timed buffers (after the timed region)
def _close_frac(y, ref, rtol=1e-4):
    """Fraction of entries outside |y - ref| <= rtol*|ref| + 1e-5*max|ref| and the largest error relative to max|ref|."""
    (y, ref) = (np.asarray(y, dtype=np.float64), np.asarray(ref, dtype=np.float64))
    scale = float(np.abs(ref).max()) if ref.size else 1.0
    bad = np.abs(y - ref) > rtol * np.abs(ref) + 1e-5 * scale
    return (float(bad.mean()) if bad.size else 0.0, float(np.abs(y - ref).max() / max(scale, 1e-30)) if ref.size else 0.0)


def check_against_plain_net(wl, images, logits, n=4):
    import torch
    torch.set_num_threads(host_threads())          # torchrun pins OMP_NUM_THREADS=1; this is the checker, outside every timed region
    plain = keyed_pooling(wl['net'])
    with torch.no_grad():
        yp = plain(images[:n].detach().cpu().reshape((n,) + wl['inshape'])).numpy().reshape(n, -1)
    yk = logits[:n].detach().cpu().numpy().reshape(n, -1)
    scale = float(np.abs(yp).max())
    return {'images': n, 'max_abs_err_vs_plain_net': float(np.abs(yk - yp).max()), 'max_abs_logit': scale, 'logit_std_over_images': float(np.std(yp, axis=0).max()),
            'allclose_atol_1e-3_scale': bool(np.abs(yk - yp).max() <= 1e-3 * max(1.0, scale)), 'argmax_equal': bool(np.array_equal(yk.argmax(1), yp.argmax(1)))}


def check_plan_against_oracle(plan, layers, n=64):
    """Small networks: the first n images of the timed batch through the oracle's csr_matvecs chain on the same compiled CSR."""
    from oracle import keynet_oracle as ko
    n = min(n, plan.N)
    x = ko.affine_to_linear(plan.images[:n].detach().cpu().numpy().reshape((n,) + tuple(plan.sensor._inshape[1:])))
    ref = ko.linear_to_affine(ko.keyed_forward(layers, x, threads=host_threads()))
    got = plan.logits[:n].detach().cpu().numpy()
    (frac_bad, rel) = _close_frac(got, ref)
    return {'images': n, 'vs': 'oracle keyed_forward on the compiled CSR', 'rtol': 1e-4, 'atol': '1e-5*max|y|', 'fraction_outside': frac_bad, 'max_err_over_max_abs': rel, 'ok': frac_bad == 0.0}


def check_plan_against_bands(plan, bands, n=4):
    """VGG16: every keyed layer's timed output rows [band rows, first n images] against the oracle band times the layer's timed
    INPUT activations (csr_matvecs, fp32) -- a full-size, per-layer oracle check of exactly the buffers the bench produced."""
    from oracle import keynet_oracle as ko
    import torch
    worst = {'fraction_outside': 0.0, 'max_err_over_max_abs': 0.0, 'layer': None}
    ok = True
    for (i, b) in enumerate(bands):
        (name, W, relu) = plan.layers[i + 1]
        x = plan.acts[i][:, :n].detach().cpu().numpy()
        rows = torch.from_numpy(b['rows']).to(plan.acts[i + 1].device)
        got = plan.acts[i + 1][rows][:, :n].detach().cpu().numpy()
        ref = ko.spmm(b['W'], x, relu=relu, threads=host_threads())
        (frac_bad, rel) = _close_frac(got, ref)
        ok = ok and frac_bad == 0.0
        if rel >= worst['max_err_over_max_abs']:
            worst = {'fraction_outside': frac_bad, 'max_err_over_max_abs': rel, 'layer': name}
    return {'images': n, 'vs': 'oracle row bands (csr_matmat key compile + csr_matvecs) on every keyed layer, inputs = the timed activations', 'rtol': 1e-4, 'atol': '1e-5*max|y|',
            'layers': len(bands), 'band_rows': int(sum(len(b['rows']) for b in bands)), 'worst': worst, 'ok': bool(ok)}


# =================================================================================================
# GPU legs
def _barrier(world):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _reduce_max(vals, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor(vals, device='cuda', dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def bench_replicas(name, batch, K, warmup, rank, world, local_rank, want_cpu=True, cpu_budget_s=15.0, scaling='weak', outputs=None):
    """One GPU holds the whole keyed network; N > 1 = data-parallel replicas, no collective on the data path.
    `batch` = images per GPU per step.  Returns the record on rank 0 (None elsewhere); `outputs` (a dict) receives the
    logits of the last timed step as '<name>_logits'."""
    import torch
    from keynet_b200 import system, engine
    wl = workload(name)
    N = int(batch)
    big = name == 'vgg16'
    t0 = time.perf_counter()
    np.random.seed(0)
    (sensor, knet) = system.Keynet(wl['inshape'], wl['net'], keep_csr=not big, **wl['keys'])
    torch.cuda.synchronize()
    t_compile = time.perf_counter() - t0

    plan = engine.ForwardPlan(sensor, knet, N, use_graph=False, time_layers=True, event_sets=K)
    g = torch.Generator(device='cuda').manual_seed(rank)
    images = torch.randn((N,) + wl['inshape'], device='cuda', generator=g)      # synthetic, resident in HBM
    plan.images.copy_(images.reshape(N, -1))
    sampler = ClockSampler(local_rank).start() if rank == 0 else None

    # ---- device-resident throughput ---------------------------------------------------------
    for _ in range(warmup):
        plan.run_device()
    _barrier(world)
    if sampler is not None:
        sampler.mark_begin()
    (e0, e1) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    e0.record()
    for k in range(K):
        plan.event_set = k
        plan.run_device()
    e1.record()
    _barrier(world)
    ms = e0.elapsed_time(e1)
    if outputs is not None:
        outputs[name + '_logits'] = plan.logits.cpu().numpy()
    launches = plan.launches_per_run * K
    per_layer = plan.layer_times_ms_mean(K)
    plan.time_layers = False

    # ---- end to end with host buffers -------------------------------------------------------
    # K batches through the public host-buffer API: every step copies its own images from pinned host memory and reads its
    # logits back; the copy of step k+1 overlaps the chain of step k (ForwardPlan.run_host_many)
    host_in = [torch.randn((N,) + wl['inshape']).pin_memory() for _ in range(2)]
    host_out = [torch.empty((N, plan.K), dtype=torch.float32).pin_memory() for _ in range(2)]
    plan.run_host_many([host_in[k % 2] for k in range(2)], [host_out[k % 2] for k in range(2)])
    _barrier(world)
    e0.record()
    plan.run_host_many([host_in[k % 2] for k in range(K)], [host_out[k % 2] for k in range(K)])
    e1.record()
    _barrier(world)
    ms_e2e = e0.elapsed_time(e1)
    clocks = None
    if sampler is not None:
        sampler.mark_end()
        held = sampler.hold(plan.run_device, torch.cuda.synchronize)
        clocks = sampler.stop()
        if held:
            clocks['note'] = 'timed region shorter than the sampling period: %d more identical (untimed) steps were run until 3 readings were taken under the same load' % held
    (ms, ms_e2e) = _reduce_max([ms, ms_e2e], world)
    if rank != 0:
        return None

    (peak, peak_src) = hbm_peak()
    (tpeak, tpeak_src) = tensor_peak()
    alg = dict(plan.algorithmic_bytes())
    flops = {nm: 2.0 * W.nnz() * N for (nm, W, _) in plan.layers}
    (dom, dom_ms) = max(per_layer, key=lambda kv: kv[1])
    names = [nm for (nm, _, _) in plan.layers]
    dom_i = names.index(dom)
    domW = plan.layers[dom_i][1]
    fused_pair = dom_i in getattr(plan, 'fused', {})
    if fused_pair:                                   # one launch computes this layer AND the pooling layer that follows
        partner = names[dom_i + 1]
        alg[dom] += alg[partner]
        flops[dom] += flops[partner]
    grouped = domW._pg is not None and N >= 32 and N % 4 == 0 and not fused_pair
    on_tc = grouped and any(c['tc'] is not None for c in domW._pg.classes) and N >= 128
    tiled = on_tc and any(c.get('tile') is not None for c in domW._pg.classes)
    clustered = grouped and any(c.get('cg') is not None for c in domW._pg.classes)
    any_tc = any(W._pg is not None and any(c['tc'] is not None for c in W._pg.classes) for (_, W, _) in plan.layers) and N >= 128
    if fused_pair:
        kname = 'convpool_kernel (fused conv + ReLU + average pooling of layers %s + %s, intermediate in shared memory, fp32 FMA)' % (dom, partner)
    elif grouped:
        kname = ('pg_tile_tc_kernel (tcgen05 3xTF32, spatial tiles)' if tiled else 'pg_tc_kernel (tcgen05 3xTF32)') if on_tc else ('pg_cluster_kernel (fp32 FMA, staged gathers)' if clustered else 'pg_simt_kernel / pg_small_kernel (fp32 FMA)')
        kname += ', pattern groups (G, K_pad, n_groups)=%s' % str(domW._pg.summary()['classes'])
    else:
        kname = 'spmm_rowwarp_kernel'
    hbm_achieved = alg[dom] / (dom_ms * 1e-3) / 1e9
    total_alg = sum(alg.values())
    (traffic, traffic_note) = profiled_traffic(name, N, dom)
    if on_tc:
        # this launch is bound by the tensor pipe, not HBM: arithmetic intensity 2*nnz*N / bytes is far above the machine
        # balance at this batch.  achieved = ALGORITHMIC flops (2*nnz*N) / launch time; peak = measured dense bf16 (the only
        # measured tensor number).  kind::tf32 runs at half the bf16 rate and the 3xTF32 split issues 3 MMAs per product,
        # so the ceiling for this arithmetic is peak/6.
        achieved = flops[dom] / (dom_ms * 1e-3) / 1e12
        roofline = {'bound': 'tensor', 'kernel': '%s on layer %s' % (kname, dom), 'achieved': achieved, 'peak': tpeak, 'unit': 'TFLOP/s', 'frac': achieved / tpeak,
                    'traffic': traffic, 'peak_source': tpeak_src, 'ceiling_3xtf32': tpeak / 6.0, 'frac_of_3xtf32_ceiling': achieved / (tpeak / 6.0),
                    'hbm': {'achieved': hbm_achieved, 'peak': peak, 'unit': 'GB/s', 'frac': hbm_achieved / peak, 'peak_source': peak_src}}
    else:
        roofline = {'bound': 'hbm', 'kernel': '%s on layer %s' % (kname, dom), 'achieved': hbm_achieved, 'peak': peak, 'unit': 'GB/s', 'frac': hbm_achieved / peak,
                    'traffic': traffic, 'peak_source': peak_src}
    if traffic_note:
        roofline['traffic_note'] = traffic_note
    step_s = ms / K * 1e-3
    roofline.update({'launch_ms': dom_ms, 'algorithmic_bytes_per_launch': alg[dom], 'algorithmic_flops_per_launch': flops[dom], 'share_of_step': dom_ms / (ms / K),
                     'network': {'algorithmic_bytes_per_step': total_alg, 'hbm_achieved_gbs': total_alg / step_s / 1e9, 'hbm_frac': total_alg / step_s / 1e9 / peak,
                                 'algorithmic_tflops': sum(flops.values()) / step_s / 1e12,
                                 'note': 'CSR-equivalent algorithmic bytes (8 B per stored entry + row pointers + activations, SURVEY 8d) / step time / measured HBM peak'},
                     'layers_ms': {k: round(v, 4) for (k, v) in per_layer},
                     'fused_pairs': ['%s+%s' % (names[i], names[i + 1]) for i in sorted(getattr(plan, 'fused', {}))]})
    nnz = int(sum(L[1].nnz() for L in plan.layers))
    rec = {'metric': 'encrypted_images_per_sec', 'value': world * N * K / (ms * 1e-3), 'unit': 'images/s', 'n_gpus': world, 'steps': K, 'warmup': warmup,
           'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None, 'dtype': '3xtf32 (f32 accumulate)' if any_tc else 'f32', 'data': 'synthetic',
           'config': {'workload': wl['label'], 'batch_per_gpu': N, 'global_batch': N * world, 'parallelism': 'one GPU' if world == 1 else 'dp%d replicas, no collective' % world,
                      'l2': 'inputs larger than L2: %.2f GB of CSR-equivalent matrix + %.2f GB of activations per step' % (nnz * 8 / 1e9, sum((L[1].shape[0] + L[1].shape[1]) * N * 4 for L in plan.layers) / 1e9),
                      'nnz': nnz, 'key_compile_s': round(t_compile, 3), 'hbm_allocated_gb': round(torch.cuda.max_memory_allocated() / 1e9, 2)},
           'e2e': {'value': world * N * K / (ms_e2e * 1e-3), 'unit': 'images/s', 'h2d_bytes_per_step': int(host_in[0].numel() * 4), 'd2h_bytes_per_step': int(host_out[0].numel() * 4),
                   'note': 'ForwardPlan.run_host_many: pinned H2D of step k+1 overlaps the chain of step k; one homogeneous-coordinate check (4 B D2H) per call',
                   'ms_per_step': ms_e2e / K},
           'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline}
    # ---- parity of the timed buffers + CPU baseline (after the timed region) ----------------------------------------
    plan.images.copy_(images.reshape(N, -1))
    plan.run_device()
    torch.cuda.synchronize()
    check = {'plain_net': check_against_plain_net(wl, images, plan.logits, n=4 if big else 64)}
    if want_cpu:
        if big:
            bands = oracle_bands_on_cpu(wl, BAND_FRAC)
            check['oracle'] = check_plan_against_bands(plan, bands)
            rec['cpu_baseline'] = cpu_baseline_bands(bands)
        else:
            layers = oracle_layers_from_gpu(sensor, knet)
            check['oracle'] = check_plan_against_oracle(plan, layers)
            rec['cpu_baseline'] = cpu_baseline(layers, wl['inshape'], budget_s=cpu_budget_s)
    rec['config']['check'] = check
    return rec


def bench_rows(name, batch, K, warmup, rank, world, local_rank, fused=True, want_cpu=True, outputs=None):
    """Strong scaling: ONE batch, every keyed layer's rows cut into `world` shards (keynet_b200/dist.py), activations
    all-gathered per layer over NVLink (NCCL, or fused into the SpMM epilogue: NVLink peer stores).  `outputs` (a dict)
    receives the logits of the last timed step as '<name>_logits'."""
    import torch
    import torch.distributed as dist
    from keynet_b200 import dist as kdist
    wl = workload(name)
    N = int(batch)
    t0 = time.perf_counter()
    np.random.seed(0)
    m = kdist.ShardedKeyedModel(wl['inshape'], wl['net'], rank=rank, world=world, fused=fused, keep_csr=False, **wl['keys'])
    torch.cuda.synchronize()
    t_compile = time.perf_counter() - t0
    x = torch.randn((N,) + wl['inshape'], generator=torch.Generator().manual_seed(1)).cuda()      # same batch on every rank
    D = int(np.prod(wl['inshape']))
    Xenc = torch.empty((D + 1, N), dtype=torch.float32, device='cuda')

    def step():
        m.sensor.encrypt_into(x.reshape(N, D), Xenc)
        return m.forward_linear(Xenc.t())

    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    for _ in range(2):
        y = step()
    graphed = False
    if fused and m.selective and m.flag_sync and world > 1 and N >= 32 and N % 4 == 0 and os.environ.get('KEYNET_B200_SHARD_GRAPH', '1') != '0':
        # the whole sharded chain (SpMM launches, peer stores, neighbourhood syncs) as CUDA graphs: at 8 GPUs a layer is shorter
        # than the host work that launches it
        m.capture(N)
        graphed = True

        def step():
            m.sensor.encrypt_into(x.reshape(N, D), m._gx)
            return m.forward_graph(m._gx)
    for _ in range(warmup):
        y = step()
    _barrier(world)
    if sampler is not None:
        sampler.mark_begin()
    (e0, e1) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    e0.record()
    for _ in range(K):
        y = step()
    e1.record()
    _barrier(world)
    ms = e0.elapsed_time(e1)
    y = y.clone()
    if outputs is not None:
        outputs[name + '_logits'] = y[:, :-1].cpu().numpy()      # drop the homogeneous coordinate, as forward() does
    # ---- end to end: pinned host batch in, logits out, on every rank (the batch is replicated: every rank encrypts it)
    host_in = [torch.randn((N,) + wl['inshape']).pin_memory() for _ in range(2)]
    Kout = int(y.shape[1]) - 1
    host_out = [torch.empty((N, Kout), dtype=torch.float32).pin_memory() for _ in range(2)]
    m.forward_host_many([host_in[k % 2] for k in range(2)], [host_out[k % 2] for k in range(2)])
    _barrier(world)
    e0.record()
    m.forward_host_many([host_in[k % 2] for k in range(K)], [host_out[k % 2] for k in range(K)])
    e1.record()
    _barrier(world)
    ms_e2e = e0.elapsed_time(e1)
    clocks = None
    if sampler is not None:
        sampler.mark_end()
    # short timed regions: keep every rank under the same load until rank 0 has its clock readings (all ranks take part in
    # the collective steps, so the number of extra steps is agreed first)
    extra = torch.zeros(1, device='cuda', dtype=torch.int64)
    if sampler is not None:
        extra[0] = 0 if len(sampler.in_region()) >= 3 else max(3, int(0.4 / max(ms / K * 1e-3, 1e-4)))
    if world > 1:
        dist.broadcast(extra, 0)
    for _ in range(int(extra.item())):
        step()
    torch.cuda.synchronize()
    if sampler is not None:
        if int(extra.item()):
            sampler.mark_end()
        clocks = sampler.stop()
        if int(extra.item()):
            clocks['note'] = 'timed region shorter than the sampling period: %d more identical (untimed) steps were run while sampling' % int(extra.item())
    # one extra (untimed) forward with per-layer events
    m.time_layers = True
    m.sensor.encrypt_into(x.reshape(N, D), Xenc)
    y = m.forward_linear(Xenc.t())                      # eager: per-layer events cannot be recorded inside a graph replay
    layer_ms = [(k, round(a, 3), round(b, 3)) for (k, a, b) in m.layer_times_ms()]
    m.time_layers = False
    check = None
    if rank == 0:
        check = {'plain_net': check_against_plain_net(wl, x, y[:, :-1], n=4)}
    nnz_local = m.num_parameters_local()
    (ms, ms_e2e, nnz_max, mem_max) = _reduce_max([ms, ms_e2e, float(nnz_local), torch.cuda.max_memory_allocated() / 1e9], world)
    s = torch.tensor([float(nnz_local), float(m.h2d_bytes(tuple(host_in[0].shape)))], device='cuda', dtype=torch.float64)
    if world > 1:
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
    if rank != 0:
        return None
    (peak, peak_src) = hbm_peak()
    (tpeak, tpeak_src) = tensor_peak()
    nnz = float(s[0])
    act = sum((L._shard.n_rows + L.W.shape[1]) * N * 4 for L in m.layers)          # every rank reads X_full; rows written once
    alg = nnz * 8 + act
    gather = sum((L._shard.n_phys - 1) * N * 4 for L in m.layers)
    step_s = ms / K * 1e-3
    hbm = alg / step_s / 1e9
    tflops = 2.0 * nnz * N / step_s / 1e12
    names = [k for (k, L) in m._model.keyedlayers()]
    rec = {'metric': 'encrypted_images_per_sec', 'value': N * K / (ms * 1e-3), 'unit': 'images/s', 'n_gpus': world, 'steps': K, 'warmup': warmup,
           'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': '3xtf32 (f32 accumulate)' if N >= 128 else 'f32', 'data': 'synthetic',
           'config': {'workload': wl['label'], 'global_batch': N, 'parallelism': 'rows x%d, %s' % (world, 'fused SpMM+all-gather (NVLink peer stores, need-masked)' if m.fused else 'NCCL all-gather per layer'),
                      'nnz': int(nnz), 'nnz_max_rank': int(nnz_max), 'key_compile_s': round(t_compile, 3), 'hbm_allocated_gb_max_rank': round(mem_max, 2),
                      'all_gather_bytes_per_step': int(gather), 'peer_store_fraction': m.peer_store_fraction() if m.fused else None,
                      'rank0_layer_ms_spmm_barrier': [(names[k], a, b) for (k, a, b) in layer_ms], 'rank0_barrier_ms_per_step': round(sum(b for (_, _, b) in layer_ms), 3),
                      'layer_sync': ('neighbourhood flags (kn_peer_sync): a rank waits only for the ranks it reads from / will store to' if (m.fused and m.selective and m.flag_sync) else 'barrier over all ranks') if m.fused else 'NCCL all-gather',
                      'sync_timed_out': bool(m.sync_timed_out()) if m.fused else None, 'cuda_graph': graphed,
                      'check': check, 'l2': 'inputs larger than L2'},
           'e2e': {'value': N * K / (ms_e2e * 1e-3), 'unit': 'images/s', 'h2d_bytes_per_step': int(float(s[1])), 'd2h_bytes_per_step': int(host_out[0].numel() * 4) * world,
                   'note': 'ShardedKeyedModel.forward_host_many on every rank: pinned H2D of the image rows the rank\'s first layer reads (its band + halo; all ranks together: h2d_bytes_per_step), sensor encryption, sharded chain, D2H of the logits on every rank; the H2D of step k+1 overlaps step k',
                   'ms_per_step': ms_e2e / K},
           'gpu_launches': (sum(L.W._pg.launches() if L.W._pg is not None else 1 for L in m.layers) + 2 * len(m.layers) + 2) * K, 'clocks': clocks,
           'roofline': {'bound': 'tensor', 'kernel': 'whole sharded network (pg_tc_kernel tcgen05 3xTF32 is > 90 % of the step)', 'achieved': tflops, 'peak': tpeak * world, 'unit': 'TFLOP/s',
                        'frac': tflops / (tpeak * world), 'traffic': None, 'peak_source': tpeak_src + ' x n_gpus', 'ceiling_3xtf32': tpeak * world / 6.0, 'frac_of_3xtf32_ceiling': tflops / (tpeak * world / 6.0),
                        'network': {'algorithmic_bytes_per_step': alg, 'hbm_achieved_gbs': hbm, 'hbm_frac': hbm / (peak * world), 'hbm_peak': peak * world, 'peak_source': peak_src + ' x n_gpus',
                                    'note': 'CSR-equivalent algorithmic bytes (8 B per stored entry + activations) / step time / aggregate measured HBM peak'}}}
    return rec


def bench_keycompile(args, rank, local_rank):
    """BASELINE configs[4]: key-compile sweep A.W.A^-1 over every VGG16 keyed layer on the GPU (canonical CSR out), with the
    oracle's csr_matmat compile of a row band of the same layer timed beside it and compared bit for bit."""
    import torch
    from keynet_b200 import system, layer as klayer
    from oracle import keynet_oracle as ko
    wl = workload('vgg16')
    bands = oracle_bands_on_cpu(wl, BAND_FRAC / 4)
    (peak, peak_src) = hbm_peak()
    rows = []
    state = {'i': 0}

    def f_layergen(module, inshape, outshape, A, Ainv):
        b = bands[state['i']]; state['i'] += 1
        torch.cuda.synchronize()
        best = None
        for rep in range(2):                                            # second pass: the caching allocator holds the blocks of the first
            torch.cuda.synchronize()
            (e0, e1) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            e0.record()
            L = klayer.KeyedLayer(module, inshape, outshape, A, Ainv, build_groups=False)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
            if rep == 0:
                del L
        W = L.W
        nnz = W.nnz()
        # bit-exact check of the band rows: canonical (sorted) oracle rows against the GPU rows
        r = torch.from_numpy(b['rows']).cuda()
        ip = W._indptr
        (beg, end) = (ip[r], ip[r + 1])
        ref = ko.sort_indices(b['W'])
        ok = bool(torch.equal((end - beg).cpu(), torch.from_numpy(np.diff(ref.indptr))))
        if ok:
            lens = (end - beg)
            take = torch.repeat_interleave(beg, lens) + (torch.arange(int(lens.sum()), device='cuda') - torch.repeat_interleave(torch.cumsum(lens, 0) - lens, lens))
            ok = bool(np.array_equal(W._indices[take].cpu().numpy(), ref.indices)) and bool(np.array_equal(W._data[take].cpu().numpy().view(np.uint32), ref.data.view(np.uint32)))
        # digest of the whole layer computed on the device (120 GB of CSR do not go through the host): wrapping 64-bit sums of
        # the row pointers, the column indices and the value bit patterns
        digest = '%016x' % ((int(W._indptr.sum().item()) * 1000003 + int(W._indices.sum(dtype=torch.int64).item()) * 10007 + int(W._data.view(torch.int32).sum(dtype=torch.int64).item())) & 0xffffffffffffffff)
        bytes_alg = nnz * 8 + (W.shape[0] + 1) * 8 + (W.shape[0] + W.shape[1]) * 4      # write W_hat once (+ the key vectors); the Toeplitz source is generated, not read
        rows.append({'layer': L._repr, 'shape': list(W.shape), 'nnz': int(nnz), 'gpu_ms': round(best, 3), 'csr_bytes': int(bytes_alg), 'gbs': bytes_alg / (best * 1e-3) / 1e9,
                     'hbm_frac': bytes_alg / (best * 1e-3) / 1e9 / peak, 'band_rows': int(len(b['rows'])), 'band_bit_exact': ok, 'digest': digest})
        del W
        L.W = None
        torch.cuda.empty_cache()

        class Done(torch.nn.Module):
            def fuse_relu(self, flag=True):
                return self
        return Done()
    np.random.seed(0)
    f_keypair = system.keypair_policy(**wl['keys'])
    (A, Ainv) = f_keypair('input', wl['inshape'])
    t0 = time.perf_counter()
    system.KeyedModel(wl['net'], wl['inshape'], Ainv, f_keypair, f_layergen)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    gpu_ms = sum(r['gpu_ms'] for r in rows)
    tot_bytes = sum(r['csr_bytes'] for r in rows)
    # CPU: oracle compile time of the bands, scaled by nnz
    t0 = time.perf_counter()
    bands2 = oracle_bands_on_cpu(wl, BAND_FRAC / 4)
    t_cpu = time.perf_counter() - t0
    nb = sum(len(b['W'].data) for b in bands2); nf = sum(b['nnz_full'] for b in bands2)
    out = {'metric': 'key_compile_seconds_vgg16', 'value': gpu_ms * 1e-3, 'unit': 's', 'n_gpus': 1, 'higher_is_better': False, 'mode': 'keycompile',
           'config': {'workload': 'key-compile sweep: A.W.A^-1 of every VGG16-224 keyed layer to canonical CSR on one B200 (BASELINE configs[4])', 'wall_s_incl_host_keys_and_checks': round(wall, 2)},
           'total': {'nnz': int(sum(r['nnz'] for r in rows)), 'gpu_ms': gpu_ms, 'csr_bytes': int(tot_bytes), 'gbs': tot_bytes / (gpu_ms * 1e-3) / 1e9, 'hbm_frac': tot_bytes / (gpu_ms * 1e-3) / 1e9 / peak, 'peak': peak, 'peak_source': peak_src,
                     'all_bands_bit_exact': all(r['band_bit_exact'] for r in rows)},
           'cpu_baseline': {'value': t_cpu * nf / max(nb, 1), 'unit': 's', 'cores': 1, 'kind': 'port',
                            'sample': 'oracle Toeplitz emission + two csr_matmat on row bands (%.1f M of %.2f G entries), %.1f s measured, scaled by nnz' % (nb / 1e6, nf / 1e9, t_cpu)},
           'layers': rows}
    print(json.dumps(out))


# =================================================================================================
def dump_outputs(outdir, outputs):
    """Write each array of `outputs` ({name: [rows, cols]}) as outdir/<name>.npy in float32, within DUMP_BYTES in all.  An array
    larger than its share keeps a fixed, seeded sample of its rows (in order), the same rows on every run."""
    os.makedirs(outdir, exist_ok=True)
    share = DUMP_BYTES // max(1, len(outputs)) - 4096           # room for the .npy header
    for (name, a) in sorted(outputs.items()):
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.nbytes > share:
            keep = max(1, share // (a.shape[1] * a.itemsize))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(outdir, name + '.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batch', type=int, default=None, help='images per step (vgg16: global batch; lenet / acn: per GPU)')
    ap.add_argument('--net', default=None, choices=['acn', 'lenet', 'vgg16'], help='run ONE workload as the headline (default: vgg16 headline + lenet and acn sub-records)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--mode', default='forward', choices=['forward', 'keycompile'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the lenet / acn sub-records of the default run')
    ap.add_argument('--parallel', default=None, choices=['dp', 'rows', 'rows-fused'],
                    help='N > 1: dp = replicas; rows = every keyed layer row-sharded + NCCL all-gather; rows-fused = SpMM epilogue stores to NVLink peers (default for vgg16)')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='write the logits of the last timed step of every workload as DIR/<net>_logits.npy (float32; rank 0; a seeded row sample beyond 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.mode != 'forward'):
        ap.error('--dump-outputs applies to the GPU forward benchmark only')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    from keynet_b200 import _native
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    _native.lib()
    if args.mode == 'keycompile':
        if rank == 0:
            bench_keycompile(args, rank, local_rank)
        return
    head = args.net or 'vgg16'
    parallel = args.parallel or ('rows-fused' if (head == 'vgg16' and world > 1) else 'dp')
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    elif parallel != 'dp':                                    # single-rank run of the sharded code path (layout / epilogue A-B)
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1'); os.environ.setdefault('MASTER_PORT', '29533')
        dist.init_process_group('nccl', rank=0, world_size=1, device_id=torch.device('cuda', local_rank))
    want_cpu = (world == 1) and not args.no_cpu_baseline
    default_batch = {'vgg16': VGG_BATCH, 'lenet': LENET_BATCH, 'acn': ACN_BATCH}
    K = args.steps
    outputs = {} if (args.dump_outputs and rank == 0) else None

    if parallel == 'dp':
        b = args.batch or default_batch[head]
        if head == 'acn' and args.batch is None:
            b = max(128, ACN_BATCH // world)                  # SURVEY cfg 2: 4096 images in total, split over the GPUs
        rec = bench_replicas(head, b, K, args.warmup, rank, world, local_rank, want_cpu=want_cpu, scaling='strong' if head in ('acn', 'vgg16') else 'weak', outputs=outputs)
    else:
        rec = bench_rows(head, args.batch or default_batch[head], K, args.warmup, rank, world, local_rank, fused=(parallel == 'rows-fused'), want_cpu=want_cpu, outputs=outputs)
    if args.net is None and not args.no_extra:
        torch.cuda.empty_cache()
        extra = {}
        for (nm, b, sc) in (('lenet', LENET_BATCH, 'weak'), ('acn', max(128, ACN_BATCH // world), 'strong')):
            try:
                r = bench_replicas(nm, b, K, args.warmup, rank, world, local_rank, want_cpu=want_cpu, cpu_budget_s=6.0, scaling=sc, outputs=outputs)
            except Exception as e:             # a failing sub-record must not take the headline line with it (all ranks fail alike)
                r = {'error': '%s: %s' % (type(e).__name__, str(e)[:300])}
            torch.cuda.empty_cache()
            if rank == 0:
                extra[nm] = r
        if rank == 0:
            rec['extra'] = extra
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0:
        print(json.dumps(rec))
    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
