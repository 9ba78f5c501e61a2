"""Normal equations of the objective on the GPU (csrc/normal_eq.cu) against the numpy reference
(linearisation_ref.py), their determinism, the calibration of the sandwich standard errors over noise realisations, and FitUtility.compute_uncertainties."""
import numpy as np
import pytest

from conftest import load_golden
from nmrfit_b200 import _cabi, core, synth, utils
import linearisation_ref as lin

pytestmark = pytest.mark.gpu

CASES = ['c1_4096x6', 'ragged_1000x6', 'tiny_257x6', 'p12_2048', 'p24_1536', 'c4_65536x24']


def device_normal(ws, us, vs, wts, X, precision=_cabi.FP64):
    B, N = ws.shape
    with _cabi.Context(B, N, (X.shape[1] - 4) // 3, precision=precision) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        return ctx.normal_equations(X)


def assert_parity(got, want):
    H, M, g, ssr = got
    Ho, Mo, go, so = want
    for X, Xo in ((H, Ho), (M, Mo)):
        d = np.sqrt(np.diag(Xo))
        assert np.all(np.abs(X - Xo) <= 1e-12 * np.outer(d, d)), np.max(np.abs(X - Xo) / np.outer(d, d))
    assert np.all(np.abs(g - go) <= 1e-10 * np.sqrt(np.diag(Ho) * so[0]))
    assert np.all(np.abs(ssr / so - 1) <= 1e-10)


@pytest.mark.parametrize('case', CASES)
def test_parity_with_reference(case):
    gd = load_golden('objective_' + case)
    xs = np.concatenate([gd['true'][None], gd['xs'][:3]])
    B = len(xs)
    rep = lambda a: np.repeat(a[None], B, axis=0)
    got = device_normal(rep(gd['w']), rep(gd['u']), rep(gd['v']), rep(gd['weights']), xs)
    for b, x in enumerate(xs):
        assert_parity([a[b] for a in got], lin.normal_equations(x, gd['w'], gd['u'], gd['v'], gd['weights']))


def test_parity_on_a_nonuniform_axis_and_a_mixed_batch():
    gd = load_golden('objective_c1_4096x6')
    rng = np.random.default_rng(0)
    w_pert = gd['w'] + rng.uniform(-0.3, 0.3, gd['w'].size) * (gd['w'][1] - gd['w'][0])
    spectra = [synth.multiplet(4096, 6, seed=s) for s in (11, 12)]
    ws = np.stack([w_pert] + [d.w for d, _ in spectra])
    us = np.stack([gd['u']] + [d.u for d, _ in spectra])
    vs = np.stack([gd['v']] + [d.v for d, _ in spectra])
    wts = np.stack([gd['weights']] + [utils.compute_weights(d.w, d.peaks) for d, _ in spectra])
    X = np.stack([gd['xs'][0], spectra[0][1], gd['xs'][5]])
    got = device_normal(ws, us, vs, wts, X)
    for b in range(3):
        assert_parity([a[b] for a in got], lin.normal_equations(X[b], ws[b], us[b], vs[b], wts[b]))


@pytest.mark.parametrize('case', ['c1_4096x6', 'p24_1536'])
def test_ssr_is_the_library_objective(case):
    gd = load_golden('objective_' + case)
    N, P = gd['w'].size, (gd['true'].size - 4) // 3
    xs = gd['xs'][:4]
    with _cabi.Context(4, N, P) as ctx:
        ctx.set_spectra(*(np.repeat(gd[k][None], 4, axis=0) for k in ('w', 'u', 'v', 'weights')))
        _, _, _, ssr = ctx.normal_equations(xs)
        for algo in (_cabi.ALGO_GENERAL, _cabi.ALGO_UNIFORM):
            ctx.set_algorithm(algo)
            f = ctx.objective_host(xs[:, None, :])[:, 0]
            assert np.all(np.abs(np.sqrt(ssr[:, 0] / N) / f - 1) <= 1e-10)


def test_deterministic_and_independent_of_the_batch():
    gd = load_golden('objective_p24_1536')
    spectra = [synth.multiplet(1536, 24, seed=s) for s in (3, 4, 5)]
    ws, us, vs = (np.stack([getattr(d, k) for d, _ in spectra]) for k in ('w', 'u', 'v'))
    wts = np.stack([utils.compute_weights(d.w, d.peaks) for d, _ in spectra])
    X = np.stack([gd['xs'][1], spectra[1][1], gd['xs'][2]])
    first = device_normal(ws, us, vs, wts, X)
    again = device_normal(ws, us, vs, wts, X)
    for a, b in zip(first, again):
        assert np.array_equal(a, b)
    for b in range(3):
        alone = device_normal(ws[b:b + 1], us[b:b + 1], vs[b:b + 1], wts[b:b + 1], X[b:b + 1])
        for a, s in zip(first, alone):
            assert np.array_equal(a[b], s[0])
    f32 = device_normal(ws, us, vs, wts, X, precision=_cabi.FP32)     # the pass is FP64 on FP32 contexts too
    for a, b in zip(first, f32):
        assert np.array_equal(a, b)
    H = first[0]
    assert np.array_equal(H, np.transpose(H, (0, 2, 1)))


def test_sandwich_errors_are_calibrated():
    """Gauss-Newton to the least-squares optimum of 256 noise realisations: the spread of the estimates matches the
    sandwich standard errors, and not the weighted-residual form s_w^2 H^-1 for every satellite area."""
    N, P, R, sigma = 4096, 6, 256, 1e-4
    base, true = synth.multiplet(N, P, seed=0, noise=0)
    wts = utils.compute_weights(base.w, base.peaks)
    rng = np.random.default_rng(1)
    us = base.u[None] + rng.normal(0, sigma, (R, N))
    vs = base.v[None] + rng.normal(0, sigma, (R, N))
    X = np.repeat(true[None], R, axis=0)
    lo, up = base.generate_solution_bounds()
    with _cabi.Context(R, N, P) as ctx:
        ctx.set_spectra(np.repeat(base.w[None], R, axis=0), us, vs, np.repeat(wts[None], R, axis=0))
        for _ in range(8):
            H, M, g, ssr = ctx.normal_equations(X)
            X = X - np.stack([np.linalg.solve(H[b], g[b]) for b in range(R)])
        H, M, g, ssr = ctx.normal_equations(X)
    sand = np.array([np.sqrt(np.diag(utils.covariance_from_normal(H[b], M[b], g[b], ssr[b], N, X[b], lo, up)[0]))
                     for b in range(R)])
    weighted = np.array([np.sqrt(ssr[b, 0] / (N - X.shape[1]) * np.diag(np.linalg.inv(H[b]))) for b in range(R)])
    emp = X.std(axis=0, ddof=1)
    ratio = emp / sand.mean(axis=0)
    assert np.all((ratio > 0.8) & (ratio < 1.2)), ratio
    areas = true[6::3]
    sats = 6 + 3 * np.nonzero(areas < areas.mean())[0]
    r_w = emp[sats] / weighted.mean(axis=0)[sats]
    assert np.any((r_w < 0.67) | (r_w > 1.5)), r_w


def small_fit_options(**kw):
    opt = dict(swarmsize=64, maxiter=40)
    opt.update(kw)
    return opt


def test_fit_then_uncertainties():
    data, true = synth.multiplet(2048, 6, seed=2)
    lo, up = data.generate_solution_bounds()
    f = utils.FitUtility(data, lo, up, summary=False, options=small_fit_options())
    with pytest.raises(RuntimeError):
        f.compute_uncertainties()
    f.fit()
    se = f.compute_uncertainties()
    assert se.shape == (len(true),) and np.all(np.isfinite(se)) and np.all(se > 0)
    assert f.covariance.shape == (len(true), len(true)) and not f.uncertainty_info['singular']
    fe = f.area_fraction_stderr()
    assert np.isfinite(fe) and fe > 0


def test_batch_equals_per_fit():
    datas = [synth.multiplet(2048, 6, seed=s)[0] for s in (5, 6, 7)]
    bounds = [d.generate_solution_bounds() for d in datas]
    fits = core.fit_batch(datas, [b[0] for b in bounds], [b[1] for b in bounds],
                          options=small_fit_options(rng='device', seed=3))
    batch = [s.copy() for s in utils.compute_uncertainties_batch(fits)]
    covs = [f.covariance.copy() for f in fits]
    for f, s, c in zip(fits, batch, covs):
        assert np.array_equal(f.compute_uncertainties(), s)
        assert np.array_equal(f.covariance, c)


def test_error_paths():
    data, _ = synth.multiplet(512, 6, seed=1)
    lo, up = data.generate_solution_bounds()
    f = utils.FitUtility(data, lo, up, fit_im=True, summary=False, options=small_fit_options(maxiter=2))
    f.fit()
    with pytest.raises(NotImplementedError):
        f.compute_uncertainties()
    with _cabi.Context(1, 512, 65) as ctx:
        with pytest.raises(_cabi.NmrfitError, match='at most 64 peaks') as e:
            ctx.normal_equations(np.zeros((1, 4 + 3 * 65)))
        assert e.value.code == -1
