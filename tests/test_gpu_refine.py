"""Refinement on the GPU (csrc/refine.cu, DESIGN K13) against the numpy restatement (refine_ref.refine) and an
independent bounded least-squares solver, its invariants and determinism, the calibration of the refined estimates,
and the ``refine`` paths of FitUtility, fit and fit_batch."""
import ctypes

import numpy as np
import pytest

from nmrfit_b200 import _cabi, core, synth, utils
import linearisation_ref as lin
import refine_ref as rr

pytestmark = pytest.mark.gpu


# Near the optimum a step of xtol noise scales changes s by about xtol^2 / (N - D) of itself, below FP64 rounding, so
# whether the last small step is accepted (CONVERGED) or every damped retry is rejected (STALLED) is decided by the
# last bits of s, which the device's FP64 sums and the reference's long-double sums round differently.  Both stop at
# the optimum; the objective and parameter tolerances below are what tell them apart.
AT_MINIMUM = (_cabi.REFINE_CONVERGED, _cabi.REFINE_STALLED)


def same_outcome(a, b):
    return a == b or (a in AT_MINIMUM and b in AT_MINIMUM)


def small_fit_options(**kw):
    opt = dict(swarmsize=64, maxiter=40)
    opt.update(kw)
    return opt


def stderr_at(x, w, u, v, wts, lo, up):
    H, M, g, ssr = lin.normal_equations(x, w, u, v, wts, accumulate=np.longdouble)
    C, info = utils.covariance_from_normal(H, M, g, ssr, w.size, x, lo, up)
    return np.sqrt(np.diag(C)), info


def device_refine(ws, us, vs, wts, X, LB, UB, precision=_cabi.FP64, **kw):
    B, N = ws.shape
    with _cabi.Context(B, N, (X.shape[1] - 4) // 3, precision=precision) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        return ctx.refine(X, LB, UB, **kw)


def multiplet(N, P, seed):
    """synth.multiplet for any P: a spectrum of 6 ceil(P/6) peaks (it builds groups of 6) with the peaks past P taken
    out of u and v again, so that the P-peak model fits it."""
    d, true = synth.multiplet(N, 6 * -(-P // 6), seed=seed)
    g = synth.TRUE_GLOBALS
    extra = [true[4 + 3 * k:7 + 3 * k] for k in range(P, len(d.peaks))]
    if extra:
        V = sum(synth._body(d.w, g['r'], *e) for e in extra)
        I = sum(synth._body_kk(d.w, g['r'], *e) for e in extra)
        du, dv = synth._rotate_inv(V, I, g['p0'], g['p1'])
        d.u, d.v = d.u - du, d.v - dv
        d.peaks = utils.Peaks(d.peaks[:P])
    return d, true[:4 + 3 * P]


def starts_for(N, P, seeds, nonuniform=False, swarm=True, scale=0.01):
    """Spectra of P peaks, each refined from the swarm's answer of fit_batch(swarmsize=64, maxiter=40) (with
    ``swarm``) and from the true vector perturbed by ``scale`` (clipped into the box)."""
    datas, trues = zip(*[multiplet(N, P, s) for s in seeds])
    if nonuniform:
        rng = np.random.default_rng(5)
        for d in datas:
            d.w = d.w + rng.uniform(-0.3, 0.3, N) * (d.w[1] - d.w[0])
    bounds = [d.generate_solution_bounds() for d in datas]
    LB = np.array([b[0] for b in bounds], dtype=np.float64)
    UB = np.array([b[1] for b in bounds], dtype=np.float64)
    wts = np.stack([utils.compute_weights(d.w, d.peaks) for d in datas])
    rng = np.random.default_rng(N + P)
    X = [np.clip(np.array(trues) * (1 + scale * rng.standard_normal((len(seeds), 4 + 3 * P))), LB, UB)]
    copies = 1
    if swarm:
        fits = core.fit_batch(datas, LB, UB, options=small_fit_options(rng='device', seed=1))
        X.insert(0, np.stack([f.params for f in fits]))
        wts = np.stack([f.weights for f in fits])
        copies = 2
    ws, us, vs = (np.stack([getattr(d, k) for d in datas] * copies) for k in ('w', 'u', 'v'))
    return (ws, us, vs, np.concatenate([wts] * copies), np.concatenate(X), np.concatenate([LB] * copies),
            np.concatenate([UB] * copies))


def check_invariants(ws, us, vs, wts, X0, LB, UB, got):
    x, f, passes, accepted, status = got
    assert np.all((x >= LB) & (x <= UB))
    N = ws.shape[1]
    with _cabi.Context(len(X0), N, (X0.shape[1] - 4) // 3) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        f0 = np.sqrt(ctx.normal_equations(X0)[3][:, 0] / N)
    assert np.all(f <= f0)
    none = accepted == 0
    assert np.array_equal(x[none], X0[none]) and np.array_equal(f[none], f0[none])


# (N, P, non-uniform axis, swarm starts, perturbation of the true vector, max_iter).  At 1,000 x 64 (D = 196, the
# largest system) a 64 x 40 swarm stops too far off for 50 passes, and even from 0.1 % the reference needs about 75.
SHAPES = [(4096, 6, False, True, 0.01, 50), (3000, 36, False, True, 0.01, 50), (1000, 64, False, False, 1e-3, 200),
          (4096, 6, True, True, 0.01, 50)]


@pytest.mark.parametrize('N,P,nonuniform,swarm,scale,max_iter', SHAPES,
                         ids=['4096x6', '3000x36', '1000x64', '4096x6_nonuniform'])
def test_parity_with_reference(N, P, nonuniform, swarm, scale, max_iter):
    ws, us, vs, wts, X0, LB, UB = starts_for(N, P, (41, 42) if P <= 6 else (41,), nonuniform, swarm, scale)
    got = device_refine(ws, us, vs, wts, X0, LB, UB, max_iter=max_iter)
    check_invariants(ws, us, vs, wts, X0, LB, UB, got)
    x, f, passes, accepted, status = got
    worst_f = worst_x = 0.0
    for b in range(len(X0)):
        rx, rf, rp, ra, rs = rr.refine(X0[b], LB[b], UB[b], ws[b], us[b], vs[b], wts[b], max_iter=max_iter)
        assert same_outcome(status[b], rs), (b, status[b], rs, passes[b], rp)
        se, _ = stderr_at(rx, ws[b], us[b], vs[b], wts[b], LB[b], UB[b])
        ef, ex = abs(f[b] / rf - 1), np.max(np.abs(x[b] - rx) / se)
        assert ef <= 1e-12 and ex <= 1e-3, (b, ef, ex)
        worst_f, worst_x = max(worst_f, ef / 1e-12), max(worst_x, ex / 1e-3)
        print('refine %d x %d start %d: passes %d (reference %d), accepted %d, status %d' % (N, P, b, passes[b], rp,
                                                                                              accepted[b], status[b]))
    print('refine %d x %d: worst objective error/tolerance %.3g, parameter error/tolerance %.3g' % (N, P, worst_f,
                                                                                                     worst_x))


def test_optimum_outside_the_box_against_scipy():
    """One area's upper bound below its true value: the GPU reaches at least scipy's bounded optimum, sits exactly on
    the bound there, and compute_uncertainties flags it."""
    from scipy.optimize import least_squares
    data, true = synth.multiplet(4096, 6, seed=43)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    bound = 6 + 3 * 2
    up[bound] = 0.9 * true[bound]
    x0 = np.clip(true * (1 + 0.01 * np.random.default_rng(1).standard_normal(true.size)), lo, up)
    wts = utils.compute_weights(data.w, data.peaks)
    x, f, passes, accepted, status = device_refine(data.w[None], data.u[None], data.v[None], wts[None], x0[None],
                                                   lo[None], up[None])
    assert status[0] in AT_MINIMUM
    assert x[0, bound] == up[bound]

    def fun(p):
        return wts * lin.residual_jacobian(p, data.w, data.u, data.v)[0]

    def jac(p):
        return wts[:, None] * lin.residual_jacobian(p, data.w, data.u, data.v)[1]

    sp = least_squares(fun, x0, jac=jac, bounds=(lo, up), method='trf', x_scale='jac', ftol=1e-15, xtol=1e-15,
                       gtol=1e-15)
    f_sp = np.sqrt(np.mean(fun(sp.x) ** 2))
    assert f[0] <= f_sp * (1 + 1e-12), (f[0], f_sp)
    fit = utils.FitUtility(data, lo, up, summary=False)
    fit.weights, fit.params, fit.error = wts, x[0], f[0]
    se = fit.compute_uncertainties()
    assert fit.uncertainty_info['at_bound'][bound]
    free = np.arange(true.size) != bound
    assert np.all(np.abs(x[0] - sp.x)[free] <= 1e-3 * se[free]), np.abs(x[0] - sp.x) / se


def test_no_accepted_step_and_frozen_peak():
    """max_iter = 1: the pass at the start only, x and f untouched.  A zero-area satellite held at its upper bound 0
    keeps its width and centre bit for bit."""
    data, true = synth.multiplet(2048, 6, seed=44)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    wts = utils.compute_weights(data.w, data.peaks)
    x0 = np.clip(true * (1 + 1e-3 * np.random.default_rng(0).standard_normal(true.size)), lo, up)
    zero = [4 + 3 * 5, 5 + 3 * 5, 6 + 3 * 5]
    lo[zero[2]], up[zero[2]], x0[zero[2]] = -1.0, 0.0, 0.0
    args = (data.w[None], data.u[None], data.v[None], wts[None], x0[None], lo[None], up[None])
    x, f, passes, accepted, status = device_refine(*args, max_iter=1)
    assert status[0] == _cabi.REFINE_MAX_ITER and passes[0] == 1 and accepted[0] == 0
    assert x.tobytes() == x0[None].tobytes()
    got = device_refine(*args)
    check_invariants(*args, got)
    x, f, passes, accepted, status = got
    assert status[0] in AT_MINIMUM and accepted[0] >= 1
    assert x[0, zero].tobytes() == x0[zero].tobytes()
    rx, rf, rp, ra, rs = rr.refine(x0, lo, up, data.w, data.u, data.v, wts)
    assert same_outcome(status[0], rs) and abs(f[0] / rf - 1) <= 1e-12


def test_nonfinite_start():
    data, true = synth.multiplet(1024, 6, seed=4)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    wts = utils.compute_weights(data.w, data.peaks)
    x0 = true.copy()
    lo[4], x0[4] = 0.0, 0.0
    x, f, passes, accepted, status = device_refine(data.w[None], data.u[None], data.v[None], wts[None], x0[None],
                                                   lo[None], up[None])
    assert status[0] == _cabi.REFINE_NONFINITE and passes[0] == 1 and accepted[0] == 0
    assert x.tobytes() == x0[None].tobytes()


def test_deterministic_alone_in_a_batch_and_in_fp32():
    ws, us, vs, wts, X0, LB, UB = starts_for(4096, 6, (45, 46))
    first = device_refine(ws, us, vs, wts, X0, LB, UB)
    assert len(set(first[2].tolist())) > 1             # members finish at different passes
    again = device_refine(ws, us, vs, wts, X0, LB, UB)
    f32 = device_refine(ws, us, vs, wts, X0, LB, UB, precision=_cabi.FP32)
    for a, b, c in zip(first, again, f32):
        assert a.tobytes() == b.tobytes() and a.tobytes() == c.tobytes()
    for b in range(len(X0)):
        s = slice(b, b + 1)
        alone = device_refine(ws[s], us[s], vs[s], wts[s], X0[s], LB[s], UB[s])
        for a, one in zip(first, alone):
            assert a[s].tobytes() == one.tobytes()


def test_refined_errors_are_calibrated():
    """256 noise realisations, each refined on the device from its true vector plus 50 standard errors: the spread
    of the estimates matches the mean sandwich error."""
    N, P, R, sigma = 4096, 6, 256, 1e-4
    base, true = synth.multiplet(N, P, seed=0, noise=0)
    wts = utils.compute_weights(base.w, base.peaks)
    lo, up = (np.array(a, dtype=np.float64) for a in base.generate_solution_bounds())
    rng = np.random.default_rng(1)
    us = base.u[None] + rng.normal(0, sigma, (R, N))
    vs = base.v[None] + rng.normal(0, sigma, (R, N))
    ws, W = np.repeat(base.w[None], R, axis=0), np.repeat(wts[None], R, axis=0)
    with _cabi.Context(R, N, P) as ctx:
        ctx.set_spectra(ws, us, vs, W)
        H, M, g, ssr = ctx.normal_equations(true[None].repeat(R, axis=0))
        se0 = np.sqrt(np.diag(utils.covariance_from_normal(H[0], M[0], g[0], ssr[0], N, true, lo, up)[0]))
        X0 = np.clip(true + 50 * se0 * rng.choice([-1.0, 1.0], (R, true.size)), lo, up)
        X, f, passes, accepted, status = ctx.refine(X0, lo, up)
        H, M, g, ssr = ctx.normal_equations(X)
    assert np.all(np.isin(status, AT_MINIMUM)), np.bincount(status)
    print('calibration: passes %d..%d' % (passes.min(), passes.max()))
    sand = np.array([np.sqrt(np.diag(utils.covariance_from_normal(H[b], M[b], g[b], ssr[b], N, X[b], lo, up)[0]))
                     for b in range(R)])
    ratio = X.std(axis=0, ddof=1) / sand.mean(axis=0)
    assert np.all((ratio > 0.8) & (ratio < 1.2)), ratio


def test_fit_with_refine_equals_fit_then_refine():
    data, _ = synth.multiplet(2048, 6, seed=2)
    lo, up = data.generate_solution_bounds()
    np.random.seed(3)
    a = core.fit(data, lo, up, summary=False, options=small_fit_options(refine=True))
    np.random.seed(3)
    b = core.fit(data, lo, up, summary=False, options=small_fit_options())
    swarm_params, swarm_error = b.params.copy(), b.error
    b.refine()
    assert a.params.tobytes() == b.params.tobytes() and a.error == b.error
    assert a.refine_info['start_params'].tobytes() == swarm_params.tobytes()
    assert a.refine_info['start_error'] == swarm_error and a.refine_info['accepted'] >= 1
    assert a.error < swarm_error
    # the area fraction: finite error, and within 0.1 of it of the numpy reference's from the same swarm point
    fe = a.area_fraction_stderr()
    assert np.isfinite(fe) and fe > 0
    ref = utils.FitUtility(data, lo, up, summary=False)
    ref.params = rr.refine(swarm_params, lo, up, data.w, data.u, data.v, a.weights)[0]
    assert abs(a.calculate_area_fraction() - ref.calculate_area_fraction()) <= 0.1 * fe


def test_fit_batch_with_refine_equals_refine_batch():
    for N, P in ((2048, 6), (3000, 36)):
        datas = [synth.multiplet(N, P, seed=s)[0] for s in (5, 6, 7)]
        bounds = [d.generate_solution_bounds() for d in datas]
        lows, ups = [b[0] for b in bounds], [b[1] for b in bounds]
        refined = core.fit_batch(datas, lows, ups, options=small_fit_options(rng='device', seed=3, refine=True))
        plain = core.fit_batch(datas, lows, ups, options=small_fit_options(rng='device', seed=3))
        utils.refine_batch(plain)
        for r, p in zip(refined, plain):
            assert r.params.tobytes() == p.params.tobytes() and r.error == p.error
            assert r.refine_info['passes'] == p.refine_info['passes']
            assert r.refine_info['status'] == p.refine_info['status']


def raw_refine(ctx, x, lb, ub, max_iter=50, xtol=1e-6):
    """The library call itself, past the checks Context.refine makes first."""
    x, lb, ub = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, lb, ub))
    return _cabi.lib().nmrfit_ctx_refine(ctx._h, _cabi.ptr(x), _cabi.ptr(lb), _cabi.ptr(ub), int(max_iter),
                                         ctypes.c_double(xtol), None, None, None, None, None)


def test_error_paths():
    data, true = synth.multiplet(512, 6, seed=1)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    f = utils.FitUtility(data, lo, up, summary=False, options=small_fit_options(maxiter=2))
    with pytest.raises(RuntimeError):
        f.refine()
    f = utils.FitUtility(data, lo, up, fit_im=True, summary=False, options=small_fit_options(maxiter=2))
    f.fit()
    with pytest.raises(NotImplementedError):
        f.refine()
    with pytest.raises(NotImplementedError):
        core.fit_batch([data], [lo], [up], fit_im=True, options=small_fit_options(maxiter=2, refine=True))
    with _cabi.Context(1, 1024, 65) as ctx:
        D = 4 + 3 * 65
        assert raw_refine(ctx, np.zeros((1, D)), -np.ones((1, D)), np.ones((1, D))) == -1
        assert 'at most 64 peaks' in _cabi.lib().nmrfit_last_error().decode()
    wts = utils.compute_weights(data.w, data.peaks)
    with _cabi.Context(1, 512, 6) as ctx:
        ctx.set_spectra(data.w[None], data.u[None], data.v[None], wts[None])
        x = np.clip(true, lo, up)[None]
        outside = x.copy()
        outside[0, 6] = up[6] * 1.5
        bad_box = up[None].copy()
        bad_box[0, 4] = lo[4]
        for args, msg in (((outside, lo[None], up[None]), 'inside its box'),
                          ((x, lo[None], bad_box), 'below its upper bound'),
                          ((x, lo[None], up[None], 0), 'max_iter'),
                          ((x, lo[None], up[None], 50, 0.0), 'xtol')):
            assert raw_refine(ctx, *args) == -1
            assert msg in _cabi.lib().nmrfit_last_error().decode()
        with pytest.raises(ValueError, match='inside its box'):
            ctx.refine(outside, lo, up)
        assert ctx.refine(x, lo, up)[4][0] in AT_MINIMUM                 # the context still works
