#!/usr/bin/env python
"""bench_latency.py -- small-batch latency of the keyed forward on one GPU.

Per net (VGG16 and AllConvNet, both keep_csr=False, keys as in bench.workload) and per N, the time of one
ForwardPlan(N).run_device() replayed as a CUDA graph:
  route "narrow"       N in --ns: batches below 32 on the narrow grouped kernels (PatternGroups.spmm_narrow);
  route "padded_to_32" ForwardPlan(32): what a batch below 32 cost before the narrow path (it was padded to 32 columns);
  route "csr"          AllConvNet with its CSR kept at the same N (that net's default small-batch route: CSR kernels),
                       for information.
Every shape is warmed up, then timed with device events over windows of at least --window-s seconds of back-to-back replays;
the median of --windows windows is reported.  One JSON line per (net, N, route) with the GPU's name, power limit and the SM
clocks sampled during the timed windows, and whether the layers' stored values fit the 126 MB L2 (if they do not, replays are
not L2-resident).

  python bench_latency.py [--nets vgg16,acn] [--ns 1,2,4,8,16,31] [--window-s 1.0] [--windows 5]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

import bench

L2_BYTES = 126 * 2 ** 20


def _stored_bytes(knet):
    """Bytes a forward reads from its layers: value blocks + gather lists of pattern groups, CSR arrays of the rest."""
    total = 0
    for (_, L) in knet.keyedlayers():
        W = L.W
        if W._pg is not None and W._data is None:
            for c in W._pg.classes:
                total += c['vals'].numel() * 4 + c['cols'].numel() * 4 + c['rows'].numel() * 4
            if W._pg.rest is not None:
                total += W._pg.rest['data'].numel() * 8
        elif W._data is not None:
            total += W._data.numel() * 8 + W._indptr.numel() * 8
    return total


def _median_sm_mhz(sampler):
    """Median SM clock of the nvidia-smi readings taken between the sampler's marks (None without readings)."""
    sm = []
    for r in sampler.in_region():
        try:
            sm.append(float(r.split(',')[0]))
        except ValueError:
            pass
    return float(np.median(sm)) if sm else None


def _gpu_facts():
    import torch
    facts = {'gpu': torch.cuda.get_device_name(), 'power_limit_w': None, 'sm_max_mhz': None}
    try:
        out = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()), '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader,nounits'],
                             capture_output=True, text=True, timeout=20).stdout.strip().split(',')
        facts['power_limit_w'] = float(out[0])
        facts['sm_max_mhz'] = float(out[1])
    except Exception:
        pass
    return facts


def time_plan(plan, window_s, windows):
    """Median ms per replay of plan's CUDA graph over `windows` windows of >= window_s seconds each."""
    import torch
    (e0, e1) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    for _ in range(3):
        plan.run_device()
    torch.cuda.synchronize()
    reps = 1
    while True:                                            # warm-up that also sizes the window
        e0.record()
        for _ in range(reps):
            plan.run_device()
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= 200.0:
            break
        reps *= 2
    reps = max(1, int(np.ceil(reps * window_s * 1e3 / ms)))
    per = []
    for _ in range(windows):
        e0.record()
        for _ in range(reps):
            plan.run_device()
        e1.record()
        e1.synchronize()
        per.append(e0.elapsed_time(e1) / reps)
    return (float(np.median(per)), [round(p, 5) for p in per], reps)


def run_net(name, ns, window_s, windows, sampler, facts, routes):
    import torch
    from keynet_b200 import engine, system
    wl = bench.workload(name)
    lines = []
    for keep in ([False, True] if (name == 'acn' and 'csr' in routes) else [False]):
        np.random.seed(0)
        (sensor, knet) = system.Keynet(wl['inshape'], wl['net'], keep_csr=keep, **wl['keys'])
        nbytes = _stored_bytes(knet)
        todo = [(n, 'csr' if keep else 'narrow') for n in ns] + ([] if keep else [(32, 'padded_to_32')])
        for (N, route) in todo:
            if route not in routes:
                continue
            plan = engine.ForwardPlan(sensor, knet, N, use_graph=True)
            g = torch.Generator(device='cuda').manual_seed(N)
            plan.images.copy_(torch.randn((N,) + wl['inshape'], device='cuda', generator=g).reshape(N, -1))
            sampler.mark_begin()
            (ms, per, reps) = time_plan(plan, window_s, windows)
            sampler.mark_end()
            rec = dict(sm_mhz=_median_sm_mhz(sampler), metric='keyed forward latency', net=name, label=wl['label'], keep_csr=keep, route=route, N=N,
                       ms_per_forward=round(ms, 4), images_per_s=round(N * 1e3 / ms, 1), windows_ms=per, replays_per_window=reps,
                       launches_per_forward=plan.launches_per_run, stored_bytes=nbytes,
                       l2_resident=nbytes < L2_BYTES,
                       note=('layer values %.0f MB > 126 MB L2: replays are not L2-resident' % (nbytes / 1e6)) if nbytes >= L2_BYTES
                       else ('layer values %.0f MB fit the 126 MB L2: replays may run from L2' % (nbytes / 1e6)),
                       serves=('every N <= 32 before the narrow path' if route == 'padded_to_32' else None),
                       **facts)
            lines.append(rec)
            print(json.dumps(rec), flush=True)
            del plan
            torch.cuda.empty_cache()
        del sensor, knet
        torch.cuda.empty_cache()
    return lines


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    ap.add_argument('--nets', default='vgg16,acn')
    ap.add_argument('--ns', default='1,2,4,8,16,31')
    ap.add_argument('--routes', default='narrow,padded_to_32,csr')
    ap.add_argument('--window-s', type=float, default=1.0)
    ap.add_argument('--windows', type=int, default=5)
    args = ap.parse_args()
    import torch
    from keynet_b200 import _native
    _native.require_cuda()
    ns = [int(v) for v in args.ns.split(',')]
    assert all(1 <= n < 32 for n in ns), 'narrow batches are 1..31'
    facts = _gpu_facts()
    sampler = bench.ClockSampler(torch.cuda.current_device()).start()
    try:
        for name in args.nets.split(','):
            run_net(name, ns, args.window_s, args.windows, sampler, facts, set(args.routes.split(',')))
    finally:
        sampler.stop()                                     # ends the nvidia-smi child: nothing outlives the script


if __name__ == '__main__':
    main()
