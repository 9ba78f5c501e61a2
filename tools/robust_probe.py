#!/usr/bin/env python
"""A robust loss (Huber by default) against least-squares refinement (DESIGN K16) on one GPU, from the same swarm
answers.

    python tools/robust_probe.py [--reps 10] [--loss huber|soft_l1|cauchy] [--out profiles/robust_probe.json]

For each workload the swarm runs once (fit_batch, device RNG), then Context.refine is timed from its answers with the
linear loss (max_iter 50) and with the robust loss at c = 1.345 sigma (sigma = 1e-4, synth.multiplet's noise; max_iter
utils.ROBUST_MAX_ITER, the library's default for a robust loss), which also gives how many spectra would end MAX_ITER
at 50 passes (those that need more: the trajectory does not depend on max_iter): CUDA events on the call's
stream, median of --reps calls, L2 overwritten (256 MiB fill) before each, outside the event pair; the two are timed
alternately.  A separate torch.profiler run of each splits the device time into the normal-equations kernels (K12 or
its robust instantiation) and the step kernel, which gives the time of one pass.  Workloads: BASELINE configs[2]
(1,024 spectra x 16,384 points x 6 peaks, swarm 204 x 200) and one spectrum of 65,536 points x 24 peaks."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from nmrfit_b200 import _cabi, core, synth, utils    # noqa: E402
from ties_probe import kernel_split   # noqa: E402
from uncertainty_probe import gpu_identity   # noqa: E402

WORKLOADS = [
    dict(name='c3_1024x16384x6', B=1024, N=16384, P=6, swarmsize=204, maxiter=200),
    dict(name='65536x24', B=1, N=65536, P=24, swarmsize=204, maxiter=200),
]
C = 1.345e-4


def probe(wl, reps, flush, loss):
    import torch
    B, N, P = wl['B'], wl['N'], wl['P']
    datas, lows, ups = [], [], []
    for b in range(B):
        d, _ = synth.multiplet(N, P, seed=100 + b)
        lo, up = d.generate_solution_bounds()
        datas.append(d); lows.append(lo); ups.append(up)
    opts = dict(swarmsize=wl['swarmsize'], maxiter=wl['maxiter'], rng='device', seed=1)
    fits = core.fit_batch(datas, lows, ups, options=opts)
    X = np.stack([f.params for f in fits])
    LB, UB = np.array(lows, dtype=np.float64), np.array(ups, dtype=np.float64)
    stream = torch.cuda.current_stream().cuda_stream
    rows = {}
    with _cabi.Context(B, N, P) as ctx:
        ctx.set_spectra(*(np.stack([getattr(d, k) for d in datas]) for k in ('w', 'u', 'v')),
                        np.stack([f.weights for f in fits]))
        max_iter = {'linear': 50, loss: utils.ROBUST_MAX_ITER}
        runs = {'linear': lambda: ctx.refine(X, LB, UB, max_iter=max_iter['linear'], stream=stream),
                loss: lambda: ctx.refine(X, LB, UB, max_iter=max_iter[loss], stream=stream, loss=loss, f_scale=C)}
        results = {k: fn() for k, fn in runs.items()}
        times = {k: [] for k in runs}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(reps):
            for k, fn in runs.items():                   # alternate the two
                flush.fill_(1)
                ev0.record()
                fn()
                ev1.record()
                torch.cuda.synchronize()
                times[k].append(ev0.elapsed_time(ev1))
        for k in runs:
            split = kernel_split(runs[k])
            x, f, passes, accepted, status = results[k]
            n_pass = int(passes.max())
            iters = min(-(-n_pass // 8) * 8, max_iter[k])   # passes launched: the running count is read every 8
            ms = float(np.median(times[k]))
            rows[k] = dict(refine_ms=ms, refine_ms_min=float(np.min(times[k])), passes_max=n_pass,
                           passes_median=float(np.median(passes)), iterations_run=iters, max_iter=max_iter[k],
                           max_iter_at_50=int(np.sum(passes > 50)),
                           ms_per_iteration=ms / iters, normal_eq_ms_per_pass=split['normal_eq_ms'] / iters,
                           status_counts={str(a): int(c) for a, c in zip(*np.unique(status, return_counts=True))},
                           median_f=float(np.median(f)), profiler_split=split)
            print('%-16s %-6s refine %8.3f ms (%d passes max, %.1f median; %.3f ms per iteration; normal equations '
                  '%.3f ms per pass) status %s, %d past 50 passes' % (
                      wl['name'], k, ms, n_pass, rows[k]['passes_median'], rows[k]['ms_per_iteration'],
                      rows[k]['normal_eq_ms_per_pass'], rows[k]['status_counts'], rows[k]['max_iter_at_50']), flush=True)
    return dict(workload=wl['name'], spectra=B, n_points=N, n_peaks=P, D=4 + 3 * P, f_scale=C,
                swarm=dict(swarmsize=wl['swarmsize'], maxiter=wl['maxiter']),
                loss=loss, robust_pass_over_k12=rows[loss]['normal_eq_ms_per_pass'] /
                rows['linear']['normal_eq_ms_per_pass'],
                **rows)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--loss', default='huber', choices=('huber', 'soft_l1', 'cauchy'))
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'robust_probe.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('robust_probe needs a CUDA device')
    gpu = gpu_identity()
    print('%s, power limit %s' % (gpu['name'], gpu.get('power_limit')), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    rows = [probe(wl, args.reps, flush, args.loss) for wl in WORKLOADS]
    out = dict(gpu=gpu, timing=dict(method='CUDA events around Context.refine on its stream, median of %d calls, '
                                           '%s and linear alternated, L2 overwritten before each'
                                           % (args.reps, args.loss)),
               workloads=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
