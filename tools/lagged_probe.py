#!/usr/bin/env python
"""Timing of the correlated-noise passes (csrc/lagged.cu, DESIGN K14) on one GPU, next to the normal-equations pass
(K12) in the same run.

    python tools/lagged_probe.py [--reps 10] [--out profiles/lagged_probe.json]

Workloads: BASELINE configs[2] (1,024 spectra x 16,384 points x 6 peaks) and one spectrum of 65,536 points x 24
peaks, at the true parameter vector of each spectrum, for L in {0, 32, the plan's cap}.  Each pass (partial kernel
plus reduce, device pointers in and out) is timed with CUDA events on the call's stream, median of --reps calls, L2
overwritten (256 MiB fill) before each, outside the event pair.  The card's name and power limit are read in the same
run.  FMA counts per point, as the passes are written: K12 16 nb(nb+1) for the two triangles of E = D + 1 columns
in 4x4 blocks; the M pass 16 nb(nb+1)/2 for its triangle plus (L+1) D for z; the residual pass L+1."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from nmrfit_b200 import _cabi, synth, utils       # noqa: E402
from uncertainty_probe import event_ms, gpu_identity   # noqa: E402

WORKLOADS = [dict(name='c3_1024x16384x6', B=1024, N=16384, P=6, seed=100),
             dict(name='65536x24', B=1, N=65536, P=24, seed=200)]


def probe(wl, reps, flush):
    import torch
    B, N, P = wl['B'], wl['N'], wl['P']
    D = 4 + 3 * P
    W, U, V, WT, X = [], [], [], [], []
    for b in range(B):
        d, true = synth.multiplet(N, P, seed=wl['seed'] + b)
        W.append(d.w); U.append(d.u); V.append(d.v); WT.append(utils.compute_weights(d.w, d.peaks)); X.append(true)
    stream = torch.cuda.current_stream().cuda_stream
    cap = _cabi.lagged_plan(N, P)['max_lag']
    rows = []
    with _cabi.Context(B, N, P) as ctx:
        ctx.set_spectra(np.array(W), np.array(U), np.array(V), np.array(WT))
        x_dev = torch.from_numpy(np.array(X)).cuda()
        m_dev = torch.empty((B, D, D), dtype=torch.float64, device='cuda')

        def k12():
            _cabi.check(_cabi.lib().nmrfit_ctx_normal_equations(ctx._h, _cabi.ptr(x_dev), None, _cabi.ptr(m_dev),
                                                                 None, None, _cabi.ptr(stream)))
        k12_ms, k12_min = event_ms(k12, reps, flush)
        print('%-16s K12 normal equations %8.3f ms' % (wl['name'], k12_ms), flush=True)
        for L in (0, 32, cap):
            plan = _cabi.lagged_plan(N, P, L)
            r_dev = torch.empty((B, L + 1), dtype=torch.float64, device='cuda')
            k = np.arange(L + 1)
            rho_dev = torch.from_numpy(np.repeat(utils.bartlett_taper(0.9 ** k)[None], B, axis=0)).cuda()

            def acf():
                _cabi.check(_cabi.lib().nmrfit_ctx_residual_acf(ctx._h, _cabi.ptr(x_dev), L, _cabi.ptr(r_dev),
                                                                _cabi.ptr(stream)))

            def mpass():
                _cabi.check(_cabi.lib().nmrfit_ctx_normal_m_lagged(ctx._h, _cabi.ptr(x_dev), _cabi.ptr(rho_dev), L,
                                                                   _cabi.ptr(m_dev), _cabi.ptr(stream)))
            acf_ms, acf_min = event_ms(acf, reps, flush)
            m_ms, m_min = event_ms(mpass, reps, flush)
            nb, nbe = -(-D // 4), -(-(D + 1) // 4)
            row = dict(workload=wl['name'], spectra=B, n_points=N, n_peaks=P, D=D, max_lag=L, cap=cap,
                       plan=plan, k12_ms=k12_ms, k12_ms_min=k12_min, acf_ms=acf_ms, acf_ms_min=acf_min,
                       m_ms=m_ms, m_ms_min=m_min, m_over_k12=m_ms / k12_ms,
                       fma_per_point=dict(k12=16 * nbe * (nbe + 1), m=8 * nb * (nb + 1) + (L + 1) * D, acf=L + 1),
                       halo_rows_per_tile_row=(plan['tile_points'] + 2 * L) / plan['tile_points'])
            print('%-16s L=%4d  residual acf %8.3f ms  M_rho %8.3f ms (%.2fx K12; tile %d, halo x%.2f)'
                  % (wl['name'], L, acf_ms, m_ms, m_ms / k12_ms, plan['tile_points'],
                     row['halo_rows_per_tile_row']), flush=True)
            rows.append(row)
    return rows


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'lagged_probe.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('lagged_probe needs a CUDA device')
    gpu = gpu_identity()
    print('%s, power limit %s' % (gpu['name'], gpu.get('power_limit')), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    rows = [r for wl in WORKLOADS for r in probe(wl, args.reps, flush)]
    out = dict(gpu=gpu, timing=dict(method='CUDA events around each call on its stream (partial kernel, reduce and '
                                           'the stream synchronise), device pointers in and out, median of %d calls, '
                                           'L2 overwritten before each' % args.reps), workloads=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
