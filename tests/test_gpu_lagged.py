"""Correlated-noise passes on the GPU (csrc/lagged.cu, DESIGN K14) against the long-double reference (lagged_ref.py)
on every branch of their launch plan, their determinism, the calibration of the correlated standard errors over
processed-noise realisations, and FitUtility.compute_uncertainties(noise='correlated')."""
import numpy as np
import pytest

from nmrfit_b200 import _cabi, core, synth, utils
from nmrfit_b200.containers import Data
import lagged_ref as lag
import linearisation_ref as lin

pytestmark = pytest.mark.gpu

AT_MINIMUM = (_cabi.REFINE_CONVERGED, _cabi.REFINE_STALLED)
ERR_ARG, ERR_STATE = -1, -3                       # NMRFIT_ERR_ARG, NMRFIT_ERR_STATE


def worst_ratio(err, tol):
    """max(err / tol); where the tolerance is 0 only an exact 0 passes."""
    return float(np.max(np.divide(err, tol, out=np.where(err == 0, 0.0, np.inf), where=tol > 0)))


def sweep_batch(N, P, L, seed=51):
    """Three spectra of 6 ceil(P/6) peaks, the first P of them in the model: at the true vector; on a perturbed axis at
    a perturbed true vector; with zero weights over a third of the points (across chunk boundaries) at a perturbed
    true vector.  rho: a tapered geometric decay, an alternating-sign decay, and uniform(-1, 1) values."""
    rng = np.random.default_rng(N + P + L)
    D = 4 + 3 * P
    ws, us, vs, wts, X = [], [], [], [], []
    for i in range(3):
        d, true = synth.multiplet(N, 6 * -(-P // 6), seed=seed + i)
        w = d.w + (rng.uniform(-0.3, 0.3, N) * (d.w[1] - d.w[0]) if i == 1 and N > 1 else 0.0)
        wt = utils.compute_weights(d.w, d.peaks)
        if i == 2:
            wt[N // 5:N // 5 + N // 3] = 0.0
        x = true[:D] if i == 0 else true[:D] * (1 + 0.02 * rng.standard_normal(D))
        ws.append(w); us.append(d.u); vs.append(d.v); wts.append(wt); X.append(x)
    k = np.arange(L + 1)
    rho = np.stack([utils.bartlett_taper(0.8 ** k), (-0.7) ** k, np.r_[1.0, rng.uniform(-1, 1, L)]])
    return tuple(np.stack(a) for a in (ws, us, vs, wts, X)) + (rho,)


def device_passes(ws, us, vs, wts, X, rho, precision=_cabi.FP64):
    B, N = ws.shape
    with _cabi.Context(B, N, (X.shape[1] - 4) // 3, precision=precision) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        r = ctx.residual_acf(X, rho.shape[1] - 1)
        M = ctx.normal_m_lagged(X, rho)
        _, Mw, _, ssr = ctx.normal_equations(X)
    return r, M, Mw, ssr


@pytest.mark.parametrize('N,P,L', list(lag.SWEEP), ids=['%dx%d_L%d' % s for s in lag.SWEEP])
def test_parity_across_the_launch_plan(N, P, L):
    """r_k to 1e-12 r_0, r_0 to K12's ssr[1], M_rho to 1e-12 (sum |rho_k| over |k| <= L) sqrt(M_jj M_ll) of K12's M,
    on every branch of lagged_plan (lag.SWEEP).  The reference sums in long double."""
    plan = _cabi.lagged_plan(N, P, L)
    want = lag.SWEEP[(N, P, L)]
    assert {k: plan[k] for k in want} == want, plan
    ws, us, vs, wts, X, rho = sweep_batch(N, P, L)
    r, M, Mw, ssr = device_passes(ws, us, vs, wts, X, rho)
    worst_r = worst_m = 0.0
    for b in range(len(X)):
        r_ref = lag.residual_acf(X[b], ws[b], us[b], vs[b], L)
        ratio = worst_ratio(np.abs(r[b] - r_ref), 1e-12 * r_ref[0])
        assert ratio <= 1, ('r', b, ratio)
        assert abs(r[b, 0] - ssr[b, 1]) <= 1e-12 * ssr[b, 1]
        worst_r = max(worst_r, ratio)
        _, Mw_ref, _, _ = lin.normal_equations(X[b], ws[b], us[b], vs[b], wts[b], accumulate=np.longdouble)
        d = np.sqrt(np.diag(Mw_ref))
        tol = 1e-12 * (abs(rho[b, 0]) + 2 * np.abs(rho[b, 1:]).sum()) * np.outer(d, d)
        ratio = worst_ratio(np.abs(M[b] - lag.m_lagged(X[b], ws[b], us[b], vs[b], wts[b], rho[b])), tol)
        assert ratio <= 1, ('M', b, ratio)
        worst_m = max(worst_m, ratio)
        assert np.array_equal(M[b], M[b].T)
    print('lagged %d x %d, L = %d: worst error/tolerance r %.3g, M %.3g' % (N, P, L, worst_r, worst_m))


@pytest.mark.parametrize('N,P', [(37, 1), (20000, 6), (3000, 12), (4100, 24), (1000, 64)])
def test_lag_zero_is_the_m_of_the_normal_equations(N, P):
    ws, us, vs, wts, X, _ = sweep_batch(N, P, 0)
    r, M, Mw, ssr = device_passes(ws, us, vs, wts, X, np.ones((len(X), 1)))
    for b in range(len(X)):
        d = np.sqrt(np.diag(Mw[b]))
        assert worst_ratio(np.abs(M[b] - Mw[b]), 1e-12 * np.outer(d, d)) <= 1
        assert abs(r[b, 0] - ssr[b, 1]) <= 1e-12 * ssr[b, 1]


def test_deterministic_alone_in_a_batch_and_in_fp32():
    for N, P, L in ((20000, 6, 32), (4100, 24, 40), (1000, 64, 45)):
        ws, us, vs, wts, X, rho = sweep_batch(N, P, L)
        first = device_passes(ws, us, vs, wts, X, rho)
        again = device_passes(ws, us, vs, wts, X, rho)
        f32 = device_passes(ws, us, vs, wts, X, rho, precision=_cabi.FP32)
        for a, b, c in zip(first, again, f32):
            assert a.tobytes() == b.tobytes() and a.tobytes() == c.tobytes()
        for b in range(len(X)):
            s = slice(b, b + 1)
            alone = device_passes(ws[s], us[s], vs[s], wts[s], X[s], rho[s])
            for a, one in zip(first, alone):
                assert a[s].tobytes() == one.tobytes()
        M = first[1]
        assert np.array_equal(M, np.transpose(M, (0, 2, 1)))


def calibration_run(noise_u, noise_v, seed=0):
    """256 realisations of multiplet(4096, 6) plus the given noise, each refined from the true vector: the refined
    estimates and their fits with weights set."""
    N, P = 4096, 6
    base, true = synth.multiplet(N, P, seed=seed, noise=0)
    wts = utils.compute_weights(base.w, base.peaks)
    lo, up = (np.array(a, dtype=np.float64) for a in base.generate_solution_bounds())
    R = noise_u.shape[0]
    us, vs = base.u[None] + noise_u, base.v[None] + noise_v
    with _cabi.Context(R, N, P) as ctx:
        ctx.set_spectra(np.repeat(base.w[None], R, axis=0), us, vs, np.repeat(wts[None], R, axis=0))
        X, f, passes, accepted, status = ctx.refine(np.repeat(true[None], R, axis=0), lo, up)
    assert np.all(np.isin(status, AT_MINIMUM)), np.bincount(status)
    fits = []
    for b in range(R):
        fit = utils.FitUtility(Data(base.w, us[b], vs[b]), lo, up, summary=False)
        fit.params, fit.weights = X[b], wts
        fits.append(fit)
    return X, fits


def test_correlated_errors_are_calibrated():
    """Processed noise (white complex FID noise, exponential broadening of 3 points, 2x zero-fill, FFT): the spread of
    the refined estimates matches the mean correlated error (L = 32) for every parameter, while the white errors miss
    every area by more than 1.5x.  Control: on white noise the correlated errors are calibrated too."""
    R, sigma = 256, 1e-4
    nu, nv = synth.processed_noise(4096, sigma, broadening=3.0, zero_fill=2, n_realisations=R, seed=1)
    rng = np.random.default_rng(2)
    for name, (du, dv) in (('processed', (nu, nv)), ('white', (rng.normal(0, sigma, (R, 4096)),
                                                                rng.normal(0, sigma, (R, 4096))))):
        X, fits = calibration_run(du, dv)
        white = np.array(utils.compute_uncertainties_batch(fits))
        corr = np.array(utils.compute_uncertainties_batch(fits, noise='correlated'))
        spread = X.std(axis=0, ddof=1)
        ratio_c = spread / corr.mean(axis=0)
        ratio_w = spread / white.mean(axis=0)
        print('calibration %s: spread / correlated error %s; spread / white error (areas) %s'
              % (name, np.round(ratio_c, 3), np.round(ratio_w[6::3], 3)))
        assert np.all((ratio_c > 0.8) & (ratio_c < 1.2)), (name, ratio_c)
        if name == 'processed':
            assert np.all(ratio_w[6::3] > 1.5), ratio_w[6::3]
            assert fits[0].uncertainty_info['max_lag'] == 32 and fits[0].uncertainty_info['noise_acf'][1] > 0.8


def small_fit_options(**kw):
    opt = dict(swarmsize=64, maxiter=40)
    opt.update(kw)
    return opt


def processed_data(N, P, seed):
    d, _ = synth.multiplet(N, P, seed=seed, noise=0)
    nu, nv = synth.processed_noise(N, 1e-4, broadening=3.0, n_realisations=1, seed=seed)
    d.u, d.v = d.u + nu[0], d.v + nv[0]
    return d


def test_fit_refine_then_correlated_uncertainties():
    data = processed_data(4096, 6, 3)
    lo, up = data.generate_solution_bounds()
    f = utils.FitUtility(data, lo, up, summary=False, options=small_fit_options(refine=True))
    f.fit()
    se_white = f.compute_uncertainties().copy()
    cov_white = f.covariance.copy()
    assert f.compute_uncertainties(noise='white').tobytes() == se_white.tobytes()
    assert f.covariance.tobytes() == cov_white.tobytes()
    frac_white = f.area_fraction_stderr()
    se = f.compute_uncertainties(noise='correlated')
    info = f.uncertainty_info
    assert np.all(np.isfinite(se)) and not info['singular']
    assert np.all(info['inflation'] > 1), info['inflation']
    assert np.array_equal(info['inflation'], se / se_white)
    assert info['max_lag'] == 32 and info['noise_acf'].shape == (33,) and info['noise_acf'][0] == 1.0
    assert f.area_fraction_stderr() > frac_white                 # follows the covariance
    # a known correlation, as given
    rho = np.r_[1.0, 9.0 / (9.0 + np.arange(1, 17) ** 2)]
    se_k = f.compute_uncertainties(noise='correlated', noise_acf=rho)
    assert np.array_equal(f.uncertainty_info['noise_acf'], rho) and f.uncertainty_info['max_lag'] == 16
    assert np.all(np.isfinite(se_k)) and np.all(se_k > se_white)


def test_batch_equals_per_fit():
    for N, P in ((2048, 6), (3000, 36)):
        datas = [processed_data(N, P, s) for s in (5, 6, 7)]
        bounds = [d.generate_solution_bounds() for d in datas]
        fits = core.fit_batch(datas, [b[0] for b in bounds], [b[1] for b in bounds],
                              options=small_fit_options(rng='device', seed=3, refine=True))
        batch = [s.copy() for s in utils.compute_uncertainties_batch(fits, noise='correlated', max_lag=40)]
        covs = [f.covariance.copy() for f in fits]
        infos = [dict(f.uncertainty_info) for f in fits]
        for f, s, c, i in zip(fits, batch, covs, infos):
            assert f.compute_uncertainties(noise='correlated', max_lag=40).tobytes() == s.tobytes()
            assert f.covariance.tobytes() == c.tobytes()
            assert f.uncertainty_info['noise_acf'].tobytes() == i['noise_acf'].tobytes()
            assert f.uncertainty_info['inflation'].tobytes() == i['inflation'].tobytes()


def raw_acf(ctx, x, L, out=None):
    return _cabi.lib().nmrfit_ctx_residual_acf(ctx._h, _cabi.ptr(x), int(L),
                                               _cabi.ptr(np.empty((ctx.B, L + 1)) if out is None else out), None)


def raw_m(ctx, x, rho, L):
    return _cabi.lib().nmrfit_ctx_normal_m_lagged(ctx._h, _cabi.ptr(x), _cabi.ptr(rho), int(L),
                                                  _cabi.ptr(np.empty((ctx.B, ctx.D, ctx.D))), None)


def last_error():
    return _cabi.lib().nmrfit_last_error().decode()


def test_error_paths():
    data, true = synth.multiplet(512, 6, seed=1)
    lo, up = data.generate_solution_bounds()
    f = utils.FitUtility(data, lo, up, fit_im=True, summary=False, options=small_fit_options(maxiter=2))
    f.fit()
    with pytest.raises(NotImplementedError):
        f.compute_uncertainties(noise='correlated')
    with _cabi.Context(1, 512, 65) as ctx:
        x = np.zeros((1, ctx.D))
        with pytest.raises(ValueError, match='at most 64 peaks'):
            ctx.residual_acf(x, 4)
        assert raw_acf(ctx, x, 4) == ERR_ARG and 'at most 64 peaks' in last_error()
        assert raw_m(ctx, x, np.ones((1, 5)), 4) == ERR_ARG and 'at most 64 peaks' in last_error()
    wts = utils.compute_weights(data.w, data.peaks)
    with _cabi.Context(1, 512, 6) as ctx:
        x = true[None].copy()
        assert raw_acf(ctx, x, 4) == ERR_STATE and 'every spectrum must be set' in last_error()
        ctx.set_spectra(data.w[None], data.u[None], data.v[None], wts[None])
        for L, msg in ((504, 'cap of 503 at 6 peaks'), (512, 'below the number of points'), (-1, '>= 0')):
            with pytest.raises(ValueError, match=msg):
                ctx.residual_acf(x, L)
            assert raw_acf(ctx, x, L) == ERR_ARG and msg in last_error()
            if L >= 0:
                with pytest.raises(ValueError, match=msg):
                    ctx.normal_m_lagged(x, np.ones(L + 1))
                assert raw_m(ctx, x, np.ones((1, L + 1)), L) == ERR_ARG and msg in last_error()
        assert raw_m(ctx, x, np.array([[1.0, np.nan]]), 1) == ERR_ARG and 'finite' in last_error()
        assert _cabi.lib().nmrfit_ctx_residual_acf(ctx._h, None, 2, None, None) == ERR_ARG
        assert raw_m(ctx, None, np.ones((1, 2)), 1) == ERR_ARG and 'non-NULL' in last_error()
        f = utils.FitUtility(data, lo, up, summary=False)
        f.params, f.weights = true, wts
        for kw, msg in ((dict(noise_acf=np.r_[1.0, np.zeros(504)]), 'cap of 503'),
                        (dict(noise_acf=np.r_[1.0, np.zeros(512)]), 'below the number of points')):
            with pytest.raises(ValueError, match=msg):
                f.compute_uncertainties(noise='correlated', **kw)
        # max_lag above N - 1 is cut to N - 1 (here above the cap as well: refused, naming the cap)
        with pytest.raises(ValueError, match='cap of 503'):
            f.compute_uncertainties(noise='correlated', max_lag=10_000)
        r = ctx.residual_acf(x, 8)                                      # the context still works
        assert np.all(np.isfinite(r)) and r[0, 0] > 0
