#!/usr/bin/env python
"""The automatic scale of a robust loss (DESIGN K17) on one GPU: the residual pass and the median / MAD selection, and
refine(loss='huber', f_scale='auto') against refine(loss='huber', f_scale=c) at the known c, from the same swarm answers.

    python tools/auto_scale_probe.py [--reps 10] [--out profiles/auto_scale_probe.json]

For each workload the swarm runs once (fit_batch, device RNG).  Times are CUDA events on the call's stream, median of
--reps calls, L2 overwritten (256 MiB fill) before each, outside the event pair: Context.residual_scale (both kernels,
the copy of [B][2] and the synchronise), then utils.refine_with_loss with 'auto' and with c = 1.345 sigma (sigma = 1e-4,
the noise of synth.multiplet), alternated.  A separate torch.profiler run of residual_scale splits its device time into
the residual pass and the selection.  Workloads: BASELINE configs[2] (1,024 spectra x 16,384 points x 6 peaks, swarm
204 x 200), one spectrum of 65,536 points x 24 peaks (swarm 204 x 200) and one of 2,100,000 points x 1 peak (swarm
64 x 40)."""
import argparse
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from nmrfit_b200 import _cabi, core, utils    # noqa: E402
from uncertainty_probe import event_ms, gpu_identity   # noqa: E402
from test_gpu_refine import multiplet   # noqa: E402

WORKLOADS = [
    dict(name='c2_1024x16384x6', B=1024, N=16384, P=6, swarmsize=204, maxiter=200),
    dict(name='65536x24', B=1, N=65536, P=24, swarmsize=204, maxiter=200),
    dict(name='2100000x1', B=1, N=2100000, P=1, swarmsize=64, maxiter=40),
]
C = 1.345e-4


def kernel_split(fn):
    """Device time of one call by kernel, from torch.profiler (a run of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = dict(residuals_ms=0.0, median_mad_ms=0.0)
    for ev in prof.key_averages():
        t = getattr(ev, 'device_time_total', None)
        t = ev.cuda_time_total if t is None else t
        if 'residuals_kernel' in ev.key:
            split['residuals_ms'] += t / 1e3
        elif 'median_mad_kernel' in ev.key:
            split['median_mad_ms'] += t / 1e3
    return split


def probe(wl, reps, flush):
    import torch
    B, N, P = wl['B'], wl['N'], wl['P']
    datas, lows, ups = [], [], []
    for b in range(B):
        d, _ = multiplet(N, P, 100 + b)
        lo, up = d.generate_solution_bounds()
        datas.append(d); lows.append(lo); ups.append(up)
    opts = dict(swarmsize=wl['swarmsize'], maxiter=wl['maxiter'], rng='device', seed=1)
    fits = core.fit_batch(datas, lows, ups, options=opts)
    X = np.stack([f.params for f in fits])
    LB, UB = np.array(lows, dtype=np.float64), np.array(ups, dtype=np.float64)
    stream = torch.cuda.current_stream().cuda_stream
    shells = [types.SimpleNamespace(data=d, params=f.params.copy(), error=f.error) for d, f in zip(datas, fits)]
    with _cabi.Context(B, N, P) as ctx:
        ctx.set_spectra(*(np.stack([getattr(d, k) for d in datas]) for k in ('w', 'u', 'v')),
                        np.stack([f.weights for f in fits]))
        scale_ms, scale_min = event_ms(lambda: ctx.residual_scale(X, stream=stream), reps, flush)
        split = kernel_split(lambda: ctx.residual_scale(X, stream=stream))
        runs = {'auto': 'auto', 'known_c': C}
        times = {k: [] for k in runs}
        info = {}
        for k, fs in runs.items():                       # warm-up, and the outcome of each
            utils.refine_with_loss(ctx, shells, X, LB, UB, loss='huber', f_scale=fs)
            info[k] = [dict(s.refine_info) for s in shells]
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(reps):
            for k, fs in runs.items():                   # alternate the two
                flush.fill_(1)
                torch.cuda.synchronize()
                ev0.record()
                utils.refine_with_loss(ctx, shells, X, LB, UB, loss='huber', f_scale=fs)
                ev1.record()
                torch.cuda.synchronize()
                times[k].append(ev0.elapsed_time(ev1))
    sig = np.array([i['scale']['sigma'] for i in info['auto']])
    row = dict(workload=wl['name'], spectra=B, n_points=N, n_peaks=P, f_scale_known=C,
               swarm=dict(swarmsize=wl['swarmsize'], maxiter=wl['maxiter']),
               residual_scale_ms=scale_ms, residual_scale_ms_min=scale_min, profiler_split=split,
               sigma_over_1e4=dict(median=float(np.median(sig) / 1e-4), min=float(sig.min() / 1e-4),
                                   max=float(sig.max() / 1e-4)))
    for k in runs:
        row[k] = dict(refine_ms=float(np.median(times[k])), refine_ms_min=float(np.min(times[k])),
                      robust_passes_max=int(max(i['passes'] for i in info[k])),
                      robust_passes_median=float(np.median([i['passes'] for i in info[k]])))
    row['auto']['lsq_passes_max'] = int(max(i['scale']['lsq_passes'] for i in info['auto']))
    row['auto']['lsq_passes_median'] = float(np.median([i['scale']['lsq_passes'] for i in info['auto']]))
    print('%-16s residual_scale %.3f ms (residual pass %.3f ms, selection %.3f ms); refine huber auto %.2f ms '
          '(lsq passes max %d, robust max %d) vs known c %.2f ms (passes max %d); sigma/1e-4 median %.4f'
          % (wl['name'], scale_ms, split['residuals_ms'], split['median_mad_ms'], row['auto']['refine_ms'],
             row['auto']['lsq_passes_max'], row['auto']['robust_passes_max'], row['known_c']['refine_ms'],
             row['known_c']['robust_passes_max'], row['sigma_over_1e4']['median']), flush=True)
    return row


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'auto_scale_probe.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('auto_scale_probe needs a CUDA device')
    gpu = gpu_identity()
    print('%s, power limit %s' % (gpu['name'], gpu.get('power_limit')), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    rows = [probe(wl, args.reps, flush) for wl in WORKLOADS]
    out = dict(gpu=gpu, timing=dict(method='CUDA events on the call stream, median of %d calls, L2 overwritten before '
                                           'each; auto and known c alternated; kernel split from torch.profiler'
                                           % args.reps),
               workloads=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
