#!/usr/bin/env python
"""Timing of the normal-equations pass (csrc/normal_eq.cu) on one GPU, next to one swarm evaluation of the same batch.

    python tools/uncertainty_probe.py [metric c1 c2 c3 c4] [--reps 20] [--out profiles/uncertainty_probe.json]

For each workload of bench.WORKLOADS (all 1,024 spectra at C3) it times the device pass at one parameter vector per
spectrum with CUDA events over --reps launches, L2 overwritten (256 MiB fill) before each, outside the event pair; in
the same run it times one objective evaluation of the workload's swarm the same way, and measures the sustained DFMA
rate (nmrfit_fp64_peak).  FLOP per pass = 2 B N (D(D+1) + D + 2): the upper triangles of H and M, g and the two sums
of squares.  Last, the wall time of FitUtility.compute_uncertainties() after a config-0 fit (6 peaks, 4,096 points)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                   # noqa: E402
from nmrfit_b200 import _cabi, synth, utils    # noqa: E402


def gpu_identity():
    import torch
    out = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out['power_limit'], out['max_sm_clock'] = [s.strip() for s in q.split(',')]
    except Exception as e:                     # the numbers are then reported without a power limit
        out['power_limit'] = 'unavailable: %s' % e
    return out


def event_ms(fn, reps, flush):
    import torch
    fn()
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.min(times))


def probe_workload(name, reps, flush, sustained):
    import torch
    wl = bench.WORKLOADS[name]
    P, N, S, B = wl['P'], wl['N'], wl['S'], wl.get('B', 1)
    D = 4 + 3 * P
    W, U, V, WT, X, XS = [], [], [], [], [], []
    for b in range(B):
        d, true = synth.multiplet(N, P, seed=wl['seed'] + b)
        W.append(d.w); U.append(d.u); V.append(d.v); WT.append(utils.compute_weights(d.w, d.peaks)); X.append(true)
        lo, up = d.generate_solution_bounds()
        XS.append(synth.particles(lo, up, S, seed=7 + b))
    ctx = _cabi.Context(B, N, P)
    ctx.set_spectra(np.array(W), np.array(U), np.array(V), np.array(WT))
    stream = torch.cuda.current_stream().cuda_stream
    x_dev = torch.from_numpy(np.array(X)).cuda()
    h_dev = torch.empty((B, D, D), dtype=torch.float64, device='cuda')

    def normal_pass():                         # both kernels; H copied device to device, the other outputs skipped
        _cabi.check(_cabi.lib().nmrfit_ctx_normal_equations(ctx._h, _cabi.ptr(x_dev), _cabi.ptr(h_dev), None, None,
                                                             None, _cabi.ptr(stream)))
    ne_ms, ne_min = event_ms(normal_pass, reps, flush)
    xs_dev = torch.from_numpy(np.array(XS)).cuda()
    f_dev = torch.empty((B, S), dtype=torch.float64, device='cuda')
    obj_ms, obj_min = event_ms(lambda: ctx.objective_device(xs_dev, S, f_dev, stream=stream), reps, flush)
    ctx.close()
    flop = 2.0 * B * N * (D * (D + 1) + D + 2)
    row = dict(workload=name, spectra=B, n_points=N, n_peaks=P, D=D, ms_per_pass=ne_ms, ms_per_pass_min=ne_min,
               flop_per_pass=flop, tflops=flop / (ne_ms * 1e-3) / 1e12,
               share_of_sustained_dfma=flop / (ne_ms * 1e-3) / 1e12 / sustained,
               swarm_eval_particles=S, swarm_eval_ms=obj_ms, pass_over_swarm_eval=ne_ms / obj_ms)
    print('%-6s B=%4d N=%6d D=%3d  pass %8.4f ms  %.3g FLOP  %6.2f TFLOP/s  %5.1f %% of DFMA  | swarm eval (S=%d) %8.4f ms'
          % (name, B, N, D, ne_ms, flop, row['tflops'], 100 * row['share_of_sustained_dfma'], S, obj_ms), flush=True)
    return row


def config0_wall(reps=20):
    data, _ = synth.multiplet(4096, 6, seed=1000)
    lo, up = data.generate_solution_bounds()
    f = utils.FitUtility(data, lo, up, summary=False, options=dict(swarmsize=100, maxiter=100, rng='device'))
    f.fit()
    t0 = time.perf_counter()
    f.compute_uncertainties()
    first = time.perf_counter() - t0
    walls = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f.compute_uncertainties()
        walls.append(time.perf_counter() - t0)
    return dict(first_call_ms=first * 1e3, warm_median_ms=float(np.median(walls)) * 1e3, warm_min_ms=min(walls) * 1e3,
                stderr=f.stderr.tolist(), area_fraction=float(f.calculate_area_fraction()),
                area_fraction_stderr=f.area_fraction_stderr())


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument('names', nargs='*', default=list(bench.WORKLOADS))
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'uncertainty_probe.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('uncertainty_probe needs a CUDA device')
    gpu = gpu_identity()
    burst, sustained = _cabi.fp64_peak()
    print('%s, power limit %s: DFMA %.1f TFLOP/s sustained (%.1f burst)' % (gpu['name'], gpu.get('power_limit'),
                                                                             sustained, burst), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    rows = [probe_workload(n, args.reps, flush, sustained) for n in args.names]
    c0 = config0_wall()
    print('config 0: compute_uncertainties() %.2f ms first call, %.2f ms warm (median of 20)'
          % (c0['first_call_ms'], c0['warm_median_ms']), flush=True)
    out = dict(gpu=gpu, dfma_tflops_sustained=sustained, dfma_tflops_burst=burst, timing=dict(
        method='CUDA events around the call on its stream, median of %d, L2 overwritten before each' % args.reps),
        workloads=rows, config0_compute_uncertainties=c0)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
