#!/usr/bin/env python
"""Generate tests/golden/*.npz from the UNMODIFIED reference at /root/reference.

Run in the build container only (the reference does not travel to the GPU box):

    python tests/golden/make_golden.py

The reference has no tests or fixtures of its own (SURVEY.md section 4), so these files
are the pins: inputs are the deterministic synthetic spectra of
``nmrfit_b200.synth`` (stored in full, so later changes to the generator cannot
move them) and outputs come from the reference's own functions, imported with the
shim of SURVEY.md Appendix A:
  * numpy>=1.24 removed ``np.float`` / ``np.int`` (used at equations.py:242,
    utils.py:201-202) -> aliased before import;
  * matplotlib, peakutils, nmrglue are absent -> empty stub modules (never called);
  * pyswarm is absent -> ``pyswarm.pso`` is bound to oracle/pso_oracle.py (the
    restated algorithm; PARITY UNPINNED for that piece, see its header).
While generating, each output is also compared with oracle/nmrfit_oracle.py and the
worst disagreement is printed.
"""
import os
import sys
import types
import io
import contextlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import nmrfit_oracle as orc      # noqa: E402
from oracle import pso_oracle                # noqa: E402
from nmrfit_b200 import synth                # noqa: E402


def import_reference():
    np.float = float
    np.int = int
    for name in ('matplotlib', 'matplotlib.pyplot', 'matplotlib.gridspec', 'matplotlib.widgets',
                 'peakutils', 'nmrglue', 'pyswarm'):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules['matplotlib'].pyplot = sys.modules['matplotlib.pyplot']
    traces = []

    def pso(func, lb, ub, args=(), swarmsize=100, omega=0.5, phip=0.5, phig=0.5, maxiter=100,
            minstep=1e-8, minfunc=1e-8, processes=1, **kw):
        tr = []
        x, f, info = pso_oracle.pso(func, lb, ub, args=args, swarmsize=swarmsize, omega=omega, phip=phip,
                                    phig=phig, maxiter=maxiter, minstep=minstep, minfunc=minfunc, trace=tr,
                                    quiet=True)
        traces.append((tr, info))
        return x, f
    sys.modules['pyswarm'].pso = pso
    sys.path.insert(0, '/root/reference')
    import nmrfit
    return nmrfit, traces


def ref_data(ref, data):
    """reference Data/Peak objects carrying the same numbers as a synth Data"""
    d = ref.containers.Data(data.w.copy(), data.u.copy(), data.v.copy())
    d.p0, d.p1 = data.p0, data.p1
    peaks = ref.utils.Peaks()
    for p in data.peaks:
        q = ref.utils.Peak()
        q.loc, q.width, q.area, q.height, q.bounds = p.loc, p.width, p.area, p.height, list(p.bounds)
        peaks.append(q)
    d.peaks = peaks
    return d


worst = {}
# `python tests/golden/make_golden.py --only objective_c4` regenerates only the fixtures whose name starts with that
ONLY = sys.argv[sys.argv.index('--only') + 1] if '--only' in sys.argv else ''


def note(name, got, want):
    got, want = np.asarray(got, dtype=float), np.asarray(want, dtype=float)
    denom = np.maximum(np.abs(want), 1e-300)
    rel = float(np.max(np.abs(got - want) / denom)) if got.size else 0.0
    worst[name] = max(worst.get(name, 0.0), rel)


def main():
    ref, traces = import_reference()
    eq, pa = ref.equations, ref.proc_autophase
    out = {}

    # ---- objective on random particles inside the solution bounds ------------------------------
    cases = [('c1_4096x6', 4096, 6, 48, 0), ('ragged_1000x6', 1000, 6, 16, 3), ('p12_2048', 2048, 12, 16, 5),
             ('tiny_257x6', 257, 6, 8, 7), ('p24_1536', 1536, 24, 8, 9),
             # the full BASELINE shapes (synth seeds of bench.py's workloads): the reference itself pins the far-field
             # path at 64 / 128 / 256 regions of 256 points
             ('c3_16384x6', 16384, 6, 15, 3000), ('c2_32768x12', 32768, 12, 15, 2000), ('c4_65536x24', 65536, 24, 7, 4000)]
    for name, N, P, S, seed in cases:
        if ONLY and not ('objective_' + name).startswith(ONLY):
            continue
        data, true = synth.multiplet(N, P, seed=seed)
        rd = ref_data(ref, data)
        lo, up = rd.generate_solution_bounds()
        lo2, up2 = data.generate_solution_bounds()
        note('solution_bounds', np.r_[lo2, up2], np.r_[lo, up])
        note('solution_bounds_oracle', np.r_[orc.solution_bounds(data.peaks)], np.r_[lo, up])
        fu = ref.utils.FitUtility(rd, lo, up)
        wts = fu._compute_weights()
        note('weights', orc.compute_weights(data.w, data.peaks), wts)
        xs = synth.particles(lo, up, S, seed=7 + seed)
        xs = np.vstack([xs, true[None, :]])
        f = np.array([eq.objective(x, rd.w, rd.u, rd.v, wts, False) for x in xs])
        f_ones = np.array([eq.objective(x, rd.w, rd.u, rd.v, np.ones_like(wts), False) for x in xs[:4]])
        note('objective', orc.objective_swarm(xs, data.w, data.u, data.v, wts), f)
        # a 65,536-point axis stored whole would take the file over 1 MB: keep the np.linspace arguments instead
        # (tests/conftest.py load_golden rebuilds it)
        axis = dict(w=data.w)
        if N >= 65536:
            assert np.array_equal(np.linspace(synth.W_LO, synth.W_HI, N), data.w)
            axis = dict(w_linspace=np.array([synth.W_LO, synth.W_HI, N], dtype=float))
        out['objective_' + name] = dict(**axis, u=data.u, v=data.v, weights=wts, xs=xs, f=f, f_ones=f_ones,
                                        lower=np.array(lo), upper=np.array(up), true=true,
                                        peak_loc=[p.loc for p in data.peaks], peak_width=[p.width for p in data.peaks],
                                        peak_area=[p.area for p in data.peaks], peak_height=[p.height for p in data.peaks])

    # ---- fit_im=True objective with the reference's own quadrature (last peak only survives) ----
    data, true = synth.multiplet(96, 6, seed=11)
    rd = ref_data(ref, data)
    lo, up = rd.generate_solution_bounds()
    wts = ref.utils.FitUtility(rd, lo, up)._compute_weights()
    xs = np.vstack([synth.particles(lo, up, 3, seed=21), true[None, :]])
    f_im = np.array([eq.objective(x, rd.w, rd.u, rd.v, wts, True) for x in xs])
    note('objective_fit_im(closed vs quad)', [orc.objective(x, data.w, data.u, data.v, wts, True) for x in xs], f_im)
    out['objective_fit_im_96x6'] = dict(w=data.w, u=data.u, v=data.v, weights=wts, xs=xs, f=f_im)

    # ---- lineshape pieces ------------------------------------------------------------------------
    rng = np.random.default_rng(123)
    w = np.linspace(3.23, 3.60, 777)
    pars = [(0.55, 0.003, 0.0041, 3.41, 0.012), (0.0, -0.01, 0.002, 3.3, 1.5), (1.0, 0.01, 0.006, 3.59, 0.2),
            (0.3, 0.0, 0.0045, 3.9, 0.7)]
    out['voigt'] = dict(w=w, pars=np.array(pars), out=np.array([eq.voigt(w, *p) for p in pars]))
    note('voigt', [orc.voigt(w, *p) for p in pars], out['voigt']['out'])
    u = rng.normal(size=501)
    v = rng.normal(size=501)
    ph = [(0.25, 0.05), (-3.1, 3.1), (0.0, 0.0), (1e-3, -2.5)]
    fwd = np.array([np.stack(pa.ps2(u, v, p0, p1)) for p0, p1 in ph])
    inv = np.array([np.stack(pa.ps2(u, v, p0, p1, inv=True)) for p0, p1 in ph])
    note('ps2', [np.stack(orc.ps2(u, v, p0, p1)) for p0, p1 in ph], fwd)
    note('ps2_inv', [np.stack(orc.ps2(u, v, p0, p1, inv=True)) for p0, p1 in ph], inv)
    out['ps2'] = dict(u=u, v=v, phases=np.array(ph), fwd=fwd, inv=inv)

    # Kramers-Kronig by the reference's quad at scattered points (6.6 ms each)
    kw = np.sort(np.r_[rng.uniform(3.23, 3.60, 150), 3.40 + rng.normal(0, 0.004, 90), [3.40, 3.4005]])
    kpars = [(0.6, 0.0, 0.004, 3.40, 0.02), (0.0, 0.005, 0.003, 3.41, 0.5), (1.0, 0.0, 0.005, 3.39, 1.0)]
    kk = np.array([[eq.kk_relation(x, *p) for x in kw] for p in kpars])
    note('kk(closed vs quad, abs/peak)', [orc.kk_closed(kw, *p) / np.abs(kk[i]).max() for i, p in enumerate(kpars)],
         kk / np.abs(kk).max(axis=1, keepdims=True))
    out['kk'] = dict(w=kw, pars=np.array(kpars), out=kk)

    x = rng.uniform(0.5, 3.0, 300)
    out['laplace1d'] = dict(x=x.copy(), out=eq.laplace1d(x.copy()), out3=eq.laplace1d(x.copy(), n=3, omega=0.5))
    note('laplace1d', orc.laplace1d(x.copy()), out['laplace1d']['out'])

    # ---- generate_result through the reference FitUtility (quad KK: small grid) ---------------------
    data, true = synth.multiplet(40, 6, seed=13)
    rd = ref_data(ref, data)
    lo, up = rd.generate_solution_bounds()
    fu = ref.utils.FitUtility(rd, lo, up)
    fu.params = synth.particles(lo, up, 1, seed=31)[0]
    gr = {}
    for scale in (1, 1.5):
        fu.generate_result(scale=scale)
        o = orc.generate_result(fu.params, data.w, scale)
        note('generate_result V', o['V'], fu.V)
        note('generate_result u', o['u'], fu.u)
        note('generate_result real', o['real_contribs'], fu.real_contribs)
        gr['s%s' % str(scale).replace('.', '_')] = dict(
            w=fu.w, V=fu.V, I=fu.I, u=fu.u, v=fu.v, real=np.array(fu.real_contribs), imag=np.array(fu.imag_contribs),
            data_V=rd.V, data_I=rd.I)
    out['generate_result_40x6'] = dict(w=data.w, u=data.u, v=data.v, params=fu.params,
                                       **{k + '_' + kk_: vv for k, d in gr.items() for kk_, vv in d.items()})
    fu.params = true
    out['generate_result_40x6']['area_fraction_true'] = fu.calculate_area_fraction()
    out['generate_result_40x6']['areas_true'] = fu.get_areas()

    # ---- phase estimation before the fit: brute scan and ACME score / Nelder-Mead (reference Data.shift_phase) ----
    ph_cases = {}
    for tag, N, P, seed, p0t, p1t in (('a', 4096, 6, 41, 0.25, 0.05), ('b', 1500, 6, 42, -1.3, 0.0), ('c', 12000, 12, 43, 2.9, -0.2)):
        data, true = synth.multiplet(N, P, seed=seed)
        # move the spectrum's phase from synth's (0.25, 0.05) to (p0t, p1t)
        data.u, data.v = orc.ps2(data.u, data.v, p0t - true[0], p1t - true[1], inv=True)
        rd = ref.containers.Data(data.w.copy(), data.u.copy(), data.v.copy())
        p0b, p1b = rd._brute_phase()
        note('brute_phase', orc.brute_phase(data.u, data.v)[0], p0b)
        z = data.u + 1j * data.v
        phs = np.array([(0.0, 0.0), (p0t * 180 / np.pi, p1t * 180 / np.pi), (35.0, -10.0), (-120.0, 60.0), (179.0, 2.5)])
        sc = np.array([pa._ps_acme_score(ph_, z) for ph_ in phs])
        note('acme_score', [orc.acme_score(ph_, z) for ph_ in phs], sc)
        auto = pa.approximate_phase(z, 'acme')
        note('approximate_phase', orc.approximate_phase(z), auto)
        ph_cases.update({'u_' + tag: data.u, 'v_' + tag: data.v, 'brute_' + tag: np.array([p0b, p1b]),
                         'acme_ph_' + tag: phs, 'acme_score_' + tag: sc, 'auto_' + tag: np.array(auto),
                         'true_' + tag: np.array([p0t, p1t])})
    out['phase'] = ph_cases

    # ---- end-to-end fits through reference core.fit + restated pso, legacy RNG seeded -------------
    for name, N, P, S, maxiter, seed in (('fit_lite_1024x6', 1024, 6, 24, 12, 0), ('fit_c1_4096x6', 4096, 6, 100, 100, 0),
                                         ('fit_default_2048x6', 2048, 6, 204, 2000, 4)):
        data, true = synth.multiplet(N, P, seed=2)
        rd = ref_data(ref, data)
        lo, up = rd.generate_solution_bounds()
        np.random.seed(seed)
        del traces[:]
        with contextlib.redirect_stdout(io.StringIO()):
            fobj = ref.fit(rd, lo, up, options={'swarmsize': S, 'maxiter': maxiter}, summary=False)
        tr, info = traces[-1]
        nxt = np.random.rand()      # where the legacy stream stands after the fit
        out[name] = dict(w=data.w, u=data.u, v=data.v, lower=np.array(lo), upper=np.array(up), weights=fobj.weights,
                         params=np.array(fobj.params), error=fobj.error, seed=seed, swarmsize=S, maxiter=maxiter,
                         trace_it=np.array([t[0] for t in tr]), trace_fg=np.array([t[2] for t in tr]),
                         trace_g=np.array([t[1] for t in tr]), generations=info['it'], stop=info['stop'],
                         next_rand=nxt,
                         peak_loc=[p.loc for p in data.peaks], peak_width=[p.width for p in data.peaks],
                         peak_area=[p.area for p in data.peaks], peak_height=[p.height for p in data.peaks],
                         area_fraction=fobj.calculate_area_fraction())
        print(name, 'generations', info['it'], 'stop', info['stop'], 'error', fobj.error)

    # ---- auto peak selection (utils.py:670-783) through the reference's own AutoPeakSelector ---------------------
    # scipy.integrate.simps no longer exists (-> scipy.integrate.simpson, keyword x) and peakutils is absent
    # (-> oracle/peakutils_oracle.py, PARITY UNPINNED for that piece); the class itself is the reference's.
    if not ONLY or ONLY.startswith('peaks'):
        import scipy.integrate
        from oracle import peakutils_oracle
        scipy.integrate.simps = lambda y, x: scipy.integrate.simpson(y, x=x)
        sys.modules['peakutils'].baseline = peakutils_oracle.baseline
        sp_cases = [('peaks_1024x6', 1024, 6, 3, 0.0, 0.02, False), ('peaks_2500x12', 2500, 12, 5, 0.004, 0.01, False),
                    ('peaks_4096x6', 4096, 6, 1000, 0.002, 0.02, False), ('peaks_desc_1500x6', 1500, 6, 8, 0.0, 0.02, True)]
        if 'peaks_c3' in ONLY:                             # ~6 minutes: argrelmax with an 88,554-point window
            sp_cases = [('peaks_c3_16384x6', 16384, 6, 3000, 0.002, 0.02, False)]
        for name, N, P, seed, thresh, window, descending in sp_cases:
            if ONLY and not name.startswith(ONLY):
                continue
            data, true = synth.multiplet(N, P, seed=seed)
            V, I = pa.ps2(data.u, data.v, true[0], true[1])
            w = data.w[::-1].copy() if descending else data.w
            Vin = V[::-1].copy() if descending else V
            sel = ref.utils.AutoPeakSelector(w, Vin, thresh, window)
            sel.find_maxima()
            pre = [(p.i, p.loc, p.height) for p in sel.peaks]
            sel.find_width()
            M = sel.w.size
            probe = np.unique(np.r_[np.arange(0, 12), np.arange(M - 12, M), np.arange(0, M, 997), [p.i for p in sel.peaks]])
            out[name] = dict(w=w, V=Vin, thresh=thresh, window=window, baseline=sel.baseline, probe=probe,
                             wu_probe=sel.w[probe], uu_probe=sel.u[probe], us_probe=sel.u_smoothed[probe],
                             pre_i=[q[0] for q in pre], pre_loc=[q[1] for q in pre], pre_height=[q[2] for q in pre],
                             i=[p.i for p in sel.peaks], loc=[p.loc for p in sel.peaks], height=[p.height for p in sel.peaks],
                             width=[p.width for p in sel.peaks], area=[p.area for p in sel.peaks],
                             local_baseline=[p.baseline for p in sel.peaks],
                             bounds=[list(map(float, p.bounds)) for p in sel.peaks],
                             idx_lo=[int(p.idx[0][0]) for p in sel.peaks], idx_hi=[int(p.idx[0][-1]) for p in sel.peaks])
            print(name, 'maxima', len(pre), 'peaks', len(sel.peaks), 'baseline', sel.baseline)

    for name, d in out.items():
        if ONLY and not name.startswith(ONLY):
            continue
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **{k: np.asarray(v) for k, v in d.items()})
    print('worst relative disagreement oracle vs reference:')
    for k, v in worst.items():
        print('  %-40s %.3e' % (k, v))
    sizes = sum(os.path.getsize(os.path.join(HERE, f)) for f in os.listdir(HERE) if f.endswith('.npz'))
    print('wrote %d files, %.1f KB' % (len(out), sizes / 1024))


if __name__ == '__main__':
    main()
