"""Normal equations of the objective on the GPU (csrc/normal_eq.cu) against the numpy reference
(linearisation_ref.py) on every branch of the launch plan and at adversarial parameters, their determinism, the calibration of the sandwich standard errors over noise realisations, and FitUtility.compute_uncertainties."""
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


def worst_ratio(err, tol):
    """max(err / tol); where the tolerance is 0 only an exact 0 passes."""
    return float(np.max(np.divide(err, tol, out=np.where(err == 0, 0.0, np.inf), where=tol > 0)))


def assert_parity(got, want):
    """H and M to 1e-12 sqrt(X_jj X_kk), g to 1e-10 sqrt(H_jj ssr_w), the sums of squares to 1e-10 relative.
    Returns the largest error/tolerance ratio."""
    H, M, g, ssr = got
    Ho, Mo, go, so = want
    dh, dm = np.sqrt(np.diag(Ho)), np.sqrt(np.diag(Mo))
    checks = (('H', np.abs(H - Ho), 1e-12 * np.outer(dh, dh)), ('M', np.abs(M - Mo), 1e-12 * np.outer(dm, dm)),
              ('g', np.abs(g - go), 1e-10 * np.sqrt(np.diag(Ho) * so[0])), ('ssr', np.abs(ssr - so), 1e-10 * so))
    worst = 0.0
    for name, err, tol in checks:
        r = worst_ratio(err, tol)
        assert r <= 1, (name, r)
        worst = max(worst, r)
    return worst


def sweep_batch(N, P, seeds):
    """One synthetic spectrum per seed, of 6 ceil(P/6) peaks (synth.multiplet builds groups of 6), with its weights,
    and one parameter vector each, keeping the first P peaks (the normal equations are defined at any x): the true
    vector, a random particle of the spectrum's box, and a perturbed true vector, in turn."""
    rng = np.random.default_rng(N + P)
    D = 4 + 3 * P
    ws, us, vs, wts, X = [], [], [], [], []
    for i, s in enumerate(seeds):
        d, true = synth.multiplet(N, 6 * -(-P // 6), seed=s)
        lo, up = d.generate_solution_bounds()
        if i % 3 == 0:
            x = true[:D]
        elif i % 3 == 1:
            x = synth.particles(lo, up, 1, seed=s)[0, :D]
        else:
            x = true[:D] * (1 + 0.05 * rng.standard_normal(D)) + np.r_[0.3, -0.2, 0.0, 1e-3, np.zeros(3 * P)]
        ws.append(d.w); us.append(d.u); vs.append(d.v); wts.append(utils.compute_weights(d.w, d.peaks)); X.append(x)
    return tuple(np.stack(a) for a in (ws, us, vs, wts, X))


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


@pytest.mark.parametrize('N,P', list(lin.SWEEP), ids=['%dx%d' % s for s in lin.SWEEP])
def test_parity_across_the_launch_plan(N, P):
    """Every branch of normal_eq_plan (lin.SWEEP): point groups other than 6, one and several task slices, 16- to
    128-point tiles, rows without a padding column, ragged tiles and ragged last chunks, a chunk grown past 16,384
    points.  The reference sums in long double."""
    plan = _cabi.normal_equations_plan(N, P)
    want = lin.SWEEP[(N, P)]
    assert {k: plan[k] for k in want} == want, plan
    ws, us, vs, wts, X = sweep_batch(N, P, (21,) if N > 1_000_000 else (21, 22, 23))
    got = device_normal(ws, us, vs, wts, X)
    worst = max(assert_parity([a[b] for a in got], lin.normal_equations(X[b], ws[b], us[b], vs[b], wts[b],
                                                                        accumulate=np.longdouble))
                for b in range(len(X)))
    print('normal equations %d x %d: worst error/tolerance %.3g' % (N, P, worst))


ZERO_AREA_PEAK = 3


def adversarial_batch(N, P):
    """One spectrum and three parameter vectors at the edges of the lineshape and phase arithmetic.  Spectrum 2 has
    a stretch of zero weights and a peak of area 0."""
    ws, us, vs, wts, X = sweep_batch(N, P, (31,))
    w = ws[0]
    window = w[-1] - w[0]
    X = np.repeat(X, 3, axis=0)
    width, loc, area = (lambda k: 4 + 3 * k), (lambda k: 5 + 3 * k), (lambda k: 6 + 3 * k)
    # r = 0; widths of 1e-6 of the window and of twice the window; phases on both sides of 2^31, where sincos
    # leaves its fast argument reduction (the fast path is taken for |x| < 2^31 in the PTX it compiles to)
    X[0, 2] = 0.0
    X[0, width(0)], X[0, width(1)] = 1e-6 * window, 2 * window
    X[0, 0], X[0, 1] = 2.0 ** 31 - 1.0, 3.0
    # r = 1; centres exactly on a grid point (one of them 1e-6 of the window wide) and outside the window; every
    # phase on the slow path
    X[1, 2] = 1.0
    X[1, loc(0)], X[1, loc(1)], X[1, loc(2)] = w[N // 3], w[-1] + 0.1 * window, w[N // 2]
    X[1, width(2)] = 1e-6 * window
    X[1, 0], X[1, 1] = -5e9, 40.0
    # zero weights over a third of the spectrum, across chunk boundaries; a peak of area 0, whose width and
    # location drop out of the residual
    X[2, area(ZERO_AREA_PEAK)] = 0.0
    ws, us, vs, wts = (np.repeat(a, 3, axis=0) for a in (ws, us, vs, wts))
    wts[2, N // 5:N // 5 + N // 3] = 0.0
    return ws, us, vs, wts, X


@pytest.mark.parametrize('N,P', [(5000, 11), (2500, 28)], ids=['5000x11', '2500x28'])
def test_parity_at_adversarial_parameters(N, P):
    """Point groups (5000 x 11: ng = 2) and task slices (2500 x 28: 2 slices), both with ragged last chunks."""
    ws, us, vs, wts, X = adversarial_batch(N, P)
    got = device_normal(ws, us, vs, wts, X)
    worst = max(assert_parity([a[b] for a in got], lin.normal_equations(X[b], ws[b], us[b], vs[b], wts[b],
                                                                        accumulate=np.longdouble))
                for b in range(len(X)))
    print('normal equations %d x %d, adversarial: worst error/tolerance %.3g' % (N, P, worst))
    # the zero-area peak: exactly zero rows and columns for its width and location, and a singular covariance
    H, M, g, ssr = (a[2] for a in got)
    zero = [4 + 3 * ZERO_AREA_PEAK, 5 + 3 * ZERO_AREA_PEAK]
    for Z in (H, M):
        assert np.all(Z[zero, :] == 0) and np.all(Z[:, zero] == 0)
    assert np.all(g[zero] == 0)
    C, info = utils.covariance_from_normal(H, M, g, ssr, N, X[2], X[2] - 1, X[2] + 1)
    assert info['singular'] and np.all(np.isnan(C))


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
    # one task slice, then several (2 and 5 slices per chunk, ragged last chunks)
    batches = [(ws, us, vs, wts, X)] + [sweep_batch(N, P, (3, 4, 5)) for N, P in ((2500, 28), (1000, 64))]
    for ws, us, vs, wts, X in batches:
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
    # 36 peaks: two task slices per chunk and a ragged last chunk (3,000 = 11 x 256 + 184)
    for N, P in ((2048, 6), (3000, 36)):
        data, true = synth.multiplet(N, P, seed=2)
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
        if P == 36:
            # against the covariance of the reference normal equations at the fitted point, to 1e-11 of the
            # condition number of the Jacobi-scaled H that covariance_from_normal factorises
            H, M, g, ssr = lin.normal_equations(f.params, data.w, data.u, data.v, f.weights, accumulate=np.longdouble)
            C, info = utils.covariance_from_normal(H, M, g, ssr, N, f.params, lo, up)
            s = 1 / np.sqrt(np.diag(H))
            cond = np.linalg.cond(s[:, None] * H * s[None, :])
            se_ref = np.sqrt(np.diag(C))
            assert not info['singular']
            assert np.all(np.abs(se - se_ref) <= 1e-11 * cond * se_ref), (cond, np.max(np.abs(se / se_ref - 1)))


def test_batch_equals_per_fit():
    for N, P in ((2048, 6), (3000, 36)):
        datas = [synth.multiplet(N, P, seed=s)[0] for s in (5, 6, 7)]
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
