#!/usr/bin/env python
"""Bit-for-bit comparison of nmrfit_ctx_refine between two builds of the library (DESIGN K15: the untied refinement
must not change when the tie map is added to the step kernel).

    NMRFIT_B200_LIB=<old .so> python tools/refine_bits_cmp.py dump old.npz
    python tools/refine_bits_cmp.py dump new.npz
    python tools/refine_bits_cmp.py compare old.npz new.npz [--out profiles/k15_refine_bits_cmp.txt]

``dump`` refines the inputs of tests/test_gpu_refine.py (the parity shapes from swarm answers and perturbed true
vectors, the bounded case, a 256-realisation noise batch) and tools/refine_probe.py's
configs[2] (1,024 x 16,384 x 6 from a 204 x 200 swarm) and configs[0] (4,096 x 6 from a 100 x 100 swarm) with
Context.refine and stores every output.  ``compare`` reports, per case and output, whether the bytes are equal."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from nmrfit_b200 import _cabi, core, synth, utils    # noqa: E402


def cases():
    import test_gpu_refine as tg
    for N, P, nonuniform, swarm, scale, max_iter in tg.SHAPES:
        seeds = (41, 42) if P <= 6 else (41,)
        ws, us, vs, wts, X0, LB, UB = tg.starts_for(N, P, seeds, nonuniform, swarm, scale)
        yield 'parity_%dx%d%s' % (N, P, '_nonuniform' if nonuniform else ''), (ws, us, vs, wts, X0, LB, UB), \
            dict(max_iter=max_iter)
    data, true = synth.multiplet(4096, 6, seed=43)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    up[12] = 0.9 * true[12]
    x0 = np.clip(true * (1 + 0.01 * np.random.default_rng(1).standard_normal(true.size)), lo, up)
    wts = utils.compute_weights(data.w, data.peaks)
    yield 'bounded_4096x6', (data.w[None], data.u[None], data.v[None], wts[None], x0[None], lo[None], up[None]), {}
    N, P, R, sigma = 4096, 6, 256, 1e-4
    base, true = synth.multiplet(N, P, seed=0, noise=0)
    wts = utils.compute_weights(base.w, base.peaks)
    lo, up = (np.array(a, dtype=np.float64) for a in base.generate_solution_bounds())
    rng = np.random.default_rng(1)
    us = base.u[None] + rng.normal(0, sigma, (R, N))
    vs = base.v[None] + rng.normal(0, sigma, (R, N))
    X0 = np.clip(true + 1e-3 * np.abs(true) * rng.choice([-1.0, 1.0], (R, true.size)), lo, up)
    yield 'calibration_256x4096x6', (np.repeat(base.w[None], R, 0), us, vs, np.repeat(wts[None], R, 0), X0,
                                     np.repeat(lo[None], R, 0), np.repeat(up[None], R, 0)), {}
    for name, B, N, P, ss, mi in (('configs2_1024x16384x6', 1024, 16384, 6, 204, 200),
                                  ('configs0_4096x6', 1, 4096, 6, 100, 100)):
        datas, lows, ups = [], [], []
        for b in range(B):
            d, _ = synth.multiplet(N, P, seed=100 + b)
            lo, up = d.generate_solution_bounds()
            datas.append(d); lows.append(lo); ups.append(up)
        fits = core.fit_batch(datas, lows, ups, options=dict(swarmsize=ss, maxiter=mi, rng='device', seed=1))
        yield name, (np.stack([d.w for d in datas]), np.stack([d.u for d in datas]), np.stack([d.v for d in datas]),
                     np.stack([f.weights for f in fits]), np.stack([f.params for f in fits]),
                     np.array(lows, dtype=np.float64), np.array(ups, dtype=np.float64)), {}


def dump(path):
    import ctypes
    handle = ctypes.CDLL(_cabi.LIB_PATH)
    for name in list(_cabi.SIGNATURES):                  # an older build lacks the symbols added since
        if not hasattr(handle, name):
            _cabi.SIGNATURES.pop(name)
    out = {}
    for name, (ws, us, vs, wts, X0, LB, UB), kw in cases():
        with _cabi.Context(len(X0), ws.shape[1], (X0.shape[1] - 4) // 3) as ctx:
            ctx.set_spectra(ws, us, vs, wts)
            res = ctx.refine(X0, LB, UB, **kw)
        out['%s/start' % name] = X0
        for key, v in zip(('x', 'f', 'passes', 'accepted', 'status'), res):
            out['%s/%s' % (name, key)] = v
        print(name, 'passes max %d' % res[2].max(), flush=True)
    np.savez(path, lib=os.path.abspath(_cabi.LIB_PATH), **out)


def compare(a, b, out):
    A, B = np.load(a), np.load(b)
    keys = sorted(k for k in A.files if k != 'lib')
    lines = ['nmrfit_ctx_refine outputs, old library %s against new library %s' % (A['lib'], B['lib'])]
    same = True
    for k in keys:
        eq = k in B.files and A[k].dtype == B[k].dtype and A[k].tobytes() == B[k].tobytes()
        same &= eq
        lines.append('%-40s %-10s %s' % (k, str(A[k].shape), 'identical' if eq else 'DIFFERENT'))
    lines.append('all identical' if same else 'DIFFERENCES FOUND')
    text = '\n'.join(lines) + '\n'
    print(text)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, 'w') as fh:
            fh.write(text)
    return same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('cmd', choices=('dump', 'compare'))
    ap.add_argument('files', nargs='+')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if args.cmd == 'dump':
        dump(args.files[0])
    else:
        sys.exit(0 if compare(args.files[0], args.files[1], args.out) else 1)


if __name__ == '__main__':
    main()
