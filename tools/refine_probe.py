#!/usr/bin/env python
"""Timing of the refinement (csrc/refine.cu, DESIGN K13) on one GPU, next to the swarm fit it refines.

    python tools/refine_probe.py [--reps 10] [--out profiles/refine_probe.json]

For each workload it first runs the swarm (fit_batch, device RNG; its wall time is reported), then times
Context.refine from the swarm's answers with CUDA events on the call's stream, median of --reps calls, L2 overwritten
(256 MiB fill) before each, outside the event pair.  Every call starts from the same points, so every call runs the
same passes.  A separate torch.profiler run of one refinement splits the device time into the normal-equations
kernels (K12) and the step kernel (K13).  Workloads: BASELINE configs[2] (1,024 spectra x 16,384 points x 6 peaks,
swarm 204), configs[0] (one spectrum, 4,096 x 6, swarm 100 x 100) and one spectrum of 65,536 points x 24 peaks."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from nmrfit_b200 import _cabi, core, synth    # noqa: E402
from uncertainty_probe import event_ms, gpu_identity   # noqa: E402

WORKLOADS = [
    dict(name='c3_1024x16384x6', B=1024, N=16384, P=6, swarmsize=204, maxiter=200),
    dict(name='c1_4096x6', B=1, N=4096, P=6, swarmsize=100, maxiter=100),
    dict(name='65536x24', B=1, N=65536, P=24, swarmsize=204, maxiter=200),
]


def kernel_split(ctx, X, LB, UB, stream):
    """Device time of one refinement by kernel family, from torch.profiler (a run of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.refine(X, LB, UB, stream=stream)
        torch.cuda.synchronize()
    split = dict(normal_eq_ms=0.0, step_ms=0.0, other_ms=0.0)
    for ev in prof.key_averages():
        t = getattr(ev, 'device_time_total', None)
        if t is None:
            t = ev.cuda_time_total
        if 'normal_eq' in ev.key:
            split['normal_eq_ms'] += t / 1e3
        elif 'refine_step' in ev.key:
            split['step_ms'] += t / 1e3
        elif 'kernel' in ev.key.lower() or 'Memset' in ev.key or 'Memcpy' in ev.key:
            split['other_ms'] += t / 1e3
    return split


def probe(wl, reps, flush):
    import torch
    B, N, P = wl['B'], wl['N'], wl['P']
    datas, lows, ups = [], [], []
    for b in range(B):
        d, _ = synth.multiplet(N, P, seed=100 + b)
        lo, up = d.generate_solution_bounds()
        datas.append(d); lows.append(lo); ups.append(up)
    opts = dict(swarmsize=wl['swarmsize'], maxiter=wl['maxiter'], rng='device', seed=1)
    core.fit_batch(datas[:1], lows[:1], ups[:1], options=dict(opts, maxiter=2))      # warm the swarm path
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fits = core.fit_batch(datas, lows, ups, options=opts)
    swarm_s = time.perf_counter() - t0
    X = np.stack([f.params for f in fits])
    LB, UB = np.array(lows, dtype=np.float64), np.array(ups, dtype=np.float64)
    stream = torch.cuda.current_stream().cuda_stream
    with _cabi.Context(B, N, P) as ctx:
        ctx.set_spectra(*(np.stack([getattr(d, k) for d in datas]) for k in ('w', 'u', 'v')),
                        np.stack([f.weights for f in fits]))
        x, f, passes, accepted, status = ctx.refine(X, LB, UB, stream=stream)
        ms, ms_min = event_ms(lambda: ctx.refine(X, LB, UB, stream=stream), reps, flush)
        split = kernel_split(ctx, X, LB, UB, stream)
    start_err = np.array([fi.error for fi in fits])
    n_pass = int(passes.max())                           # the batch runs until its slowest member stops
    iters = -(-n_pass // 8) * 8 if n_pass % 8 else n_pass      # the host polls every 8 iterations
    row = dict(workload=wl['name'], spectra=B, n_points=N, n_peaks=P, D=4 + 3 * P,
               swarm=dict(swarmsize=wl['swarmsize'], maxiter=wl['maxiter'], wall_s=swarm_s),
               refine_ms=ms, refine_ms_min=ms_min, passes_max=n_pass, passes_median=float(np.median(passes)),
               iterations_run=min(iters, 50), ms_per_iteration=ms / min(iters, 50),
               status_counts={str(k): int(v) for k, v in zip(*np.unique(status, return_counts=True))},
               accepted_median=float(np.median(accepted)),
               error_ratio_swarm_over_refined_median=float(np.median(start_err / f)),
               profiler_split=split,
               step_share_of_device_time=split['step_ms'] / max(1e-12, split['step_ms'] + split['normal_eq_ms']),
               refine_over_swarm=ms * 1e-3 / swarm_s)
    print('%-16s refine %8.3f ms (%d passes max, %.1f median; %.3f ms per iteration; step kernel %.1f %% of the '
          'device time) | swarm %.3f s | status %s' % (wl['name'], ms, n_pass, row['passes_median'],
                                                      row['ms_per_iteration'], 100 * row['step_share_of_device_time'],
                                                      swarm_s, row['status_counts']), flush=True)
    return row


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'refine_probe.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('refine_probe needs a CUDA device')
    gpu = gpu_identity()
    print('%s, power limit %s' % (gpu['name'], gpu.get('power_limit')), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    rows = [probe(wl, args.reps, flush) for wl in WORKLOADS]
    out = dict(gpu=gpu, timing=dict(method='CUDA events around Context.refine on its stream, median of %d calls, L2 '
                                           'overwritten before each; swarm: host wall time of fit_batch' % args.reps),
               workloads=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
