#!/usr/bin/env python
"""Tied against untied refinement (DESIGN K15) on one GPU, from the same swarm answers.

    python tools/ties_probe.py [--reps 10] [--out profiles/ties_probe.json]

For each workload the swarm runs once (fit_batch, device RNG), then Context.refine is timed from its answers without
ties and with ``synth.satellite_ties``: CUDA events on the call's stream, median of --reps calls, L2 overwritten
(256 MiB fill) before each, outside the event pair; the two are timed alternately.  A separate torch.profiler run of
each splits the device time into the normal-equations kernels (K12) and the step kernel.  Workloads: BASELINE
configs[2] (1,024 spectra x 16,384 points x 6 peaks, swarm 204 x 200) and one spectrum of 65,536 points x 24 peaks,
both without jitter so that the satellite ties hold for the true vectors."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from nmrfit_b200 import _cabi, core, synth, utils    # noqa: E402
from uncertainty_probe import gpu_identity   # noqa: E402

WORKLOADS = [
    dict(name='c3_1024x16384x6', B=1024, N=16384, P=6, swarmsize=204, maxiter=200),
    dict(name='65536x24', B=1, N=65536, P=24, swarmsize=204, maxiter=200),
]


def kernel_split(fn):
    """Device time of one refinement by kernel family, from torch.profiler (a run of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = dict(normal_eq_ms=0.0, step_ms=0.0)
    for ev in prof.key_averages():
        t = getattr(ev, 'device_time_total', None)
        t = ev.cuda_time_total if t is None else t
        if 'normal_eq' in ev.key:
            split['normal_eq_ms'] += t / 1e3
        elif 'refine_step' in ev.key:
            split['step_ms'] += t / 1e3
    return split


def probe(wl, reps, flush):
    import torch
    B, N, P = wl['B'], wl['N'], wl['P']
    datas, lows, ups = [], [], []
    for b in range(B):
        d, _ = synth.multiplet(N, P, seed=100 + b, jitter=False)
        lo, up = d.generate_solution_bounds()
        datas.append(d); lows.append(lo); ups.append(up)
    opts = dict(swarmsize=wl['swarmsize'], maxiter=wl['maxiter'], rng='device', seed=1)
    fits = core.fit_batch(datas, lows, ups, options=opts)
    X = np.stack([f.params for f in fits])
    LB, UB = np.array(lows, dtype=np.float64), np.array(ups, dtype=np.float64)
    ties = utils.batch_ties(synth.satellite_ties(P), B, P)[1]
    stream = torch.cuda.current_stream().cuda_stream
    rows = {}
    with _cabi.Context(B, N, P) as ctx:
        ctx.set_spectra(*(np.stack([getattr(d, k) for d in datas]) for k in ('w', 'u', 'v')),
                        np.stack([f.weights for f in fits]))
        runs = dict(untied=lambda: ctx.refine(X, LB, UB, stream=stream),
                    tied=lambda: ctx.refine(X, LB, UB, stream=stream, ties=ties))
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
            iters = min(-(-n_pass // 8) * 8, 50)
            ms = float(np.median(times[k]))
            rows[k] = dict(refine_ms=ms, refine_ms_min=float(np.min(times[k])), passes_max=n_pass,
                           passes_median=float(np.median(passes)), iterations_run=iters,
                           ms_per_iteration=ms / iters,
                           status_counts={str(a): int(c) for a, c in zip(*np.unique(status, return_counts=True))},
                           median_f=float(np.median(f)), profiler_split=split,
                           step_share_of_device_time=split['step_ms'] / max(1e-12, split['step_ms'] +
                                                                           split['normal_eq_ms']))
            print('%-16s %-6s refine %8.3f ms (%d passes max, %.1f median; %.3f ms per iteration; step kernel %.1f %%)'
                  ' status %s' % (wl['name'], k, ms, n_pass, rows[k]['passes_median'], rows[k]['ms_per_iteration'],
                                  100 * rows[k]['step_share_of_device_time'], rows[k]['status_counts']), flush=True)
    return dict(workload=wl['name'], spectra=B, n_points=N, n_peaks=P, D=4 + 3 * P,
                free_parameters=int(synth.satellite_ties(P).free().size),
                swarm=dict(swarmsize=wl['swarmsize'], maxiter=wl['maxiter']), **rows)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'ties_probe.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('ties_probe needs a CUDA device')
    gpu = gpu_identity()
    print('%s, power limit %s' % (gpu['name'], gpu.get('power_limit')), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    rows = [probe(wl, args.reps, flush) for wl in WORKLOADS]
    out = dict(gpu=gpu, timing=dict(method='CUDA events around Context.refine on its stream, median of %d calls, '
                                           'tied and untied alternated, L2 overwritten before each' % args.reps),
               workloads=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
