"""Robust refinement (DESIGN K16) without a GPU: the loss derivatives, scipy's loss rows, the reference refinement
against scipy, Huber's covariance (its linear identity and its ties), and every refusal the Python layer makes before
a CUDA call."""
import numpy as np
import pytest

from nmrfit_b200 import _cabi, core, synth, utils
import linearisation_ref as lin
import robust_ref as rr

ROBUST = ('huber', 'soft_l1', 'cauchy')


@pytest.mark.parametrize('loss', rr.LOSSES)
def test_derivatives_match_finite_differences(loss):
    z = np.array([0.01, 0.3, 0.7, 1.5, 4.0, 30.0, 900.0])
    h = 1e-6 * z
    rho, d1, d2 = rr.loss_terms(z, loss)
    rp, d1p, _ = rr.loss_terms(z + h, loss)
    rm, d1m, _ = rr.loss_terms(z - h, loss)
    assert np.allclose((rp - rm) / (2 * h), d1, rtol=1e-8, atol=0)
    assert np.allclose((d1p - d1m) / (2 * h), d2, rtol=1e-6, atol=1e-12)
    # psi(r) = rho'(r^2) r at c = 1, psi' against its finite difference
    r = np.sqrt(z)
    hr = 1e-6 * r
    psi = lambda t: rr.loss_terms(t * t, loss)[1] * t
    assert np.allclose((psi(r + hr) - psi(r - hr)) / (2 * hr), rr.psi_prime(z, loss), rtol=1e-6, atol=1e-12)
    assert np.all(d1 > 0)


def test_closed_forms_of_psi_prime():
    z = np.array([0.2, 0.9, 1.1, 5.0, 50.0])
    assert np.allclose(rr.psi_prime(z, 'huber'), np.where(z <= 1, 1.0, 0.0), rtol=0, atol=1e-15)
    assert np.allclose(rr.psi_prime(z, 'soft_l1'), (1 + z) ** -1.5, rtol=1e-14)
    assert np.allclose(rr.psi_prime(z, 'cauchy'), (1 - z) / (1 + z) ** 2, rtol=1e-13, atol=1e-16)


@pytest.mark.parametrize('loss', ROBUST)
def test_rows_are_scipys_losses(loss):
    """At unit weights the reference's rows, passed to least_squares as a callable loss, give the same fit as scipy's
    built-in loss of that name (public API only): a straight line with outliers, from the same start."""
    from scipy.optimize import least_squares
    rng = np.random.default_rng(7)
    t = np.linspace(0, 1, 200)
    y = 2.0 + 3.0 * t + rng.normal(0, 0.05, t.size)
    y[::17] += rng.uniform(0.5, 2.0, y[::17].size)
    fun = lambda p: p[0] + p[1] * t - y
    jac = lambda p: np.stack([np.ones_like(t), t], axis=1)
    rows = lambda z: np.array(rr.loss_terms(z, loss))
    opts = dict(method='trf', ftol=1e-14, xtol=1e-14, gtol=1e-14, f_scale=0.07)
    want = least_squares(fun, [0.0, 0.0], jac=jac, loss=loss, **opts)
    got = least_squares(fun, [0.0, 0.0], jac=jac, loss=rows, **opts)
    assert got.cost == pytest.approx(want.cost, rel=1e-13)
    assert np.allclose(got.x, want.x, rtol=1e-10, atol=0)
    assert got.nfev == want.nfev


def small_problem(N=600, impurity=True, seed=3):
    data, true = synth.multiplet(N, 6, seed=seed, noise=1e-4, jitter=False)
    if impurity:
        rr.impurity(data, true)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    wts = utils.compute_weights(data.w, data.peaks)
    return data, true, lo, up, wts


@pytest.mark.parametrize('loss', ROBUST)
def test_reference_refinement_reaches_scipy(loss):
    data, true, lo, up, wts = small_problem()
    c = 2e-4
    x0 = np.clip(true * (1 + 1e-3 * np.random.default_rng(2).standard_normal(true.size)), lo, up)
    x, f, passes, accepted, status = rr.refine(x0, lo, up, data.w, data.u, data.v, wts, loss, c, max_iter=100)
    assert status in (rr.CONVERGED, rr.STALLED) and accepted > 0
    sp = rr.scipy_fit(x0, lo, up, data.w, data.u, data.v, wts, loss, c)
    N = data.w.size
    assert f * f * N <= 2 * sp.cost * (1 + 1e-9)
    assert rr.robust_pass(x, data.w, data.u, data.v, wts, loss, c)[2] == pytest.approx(f * f * N, rel=1e-14)


def test_linear_pass_is_the_normal_equations():
    data, true, lo, up, wts = small_problem(impurity=False)
    H, _, g, ssr = lin.normal_equations(true, data.w, data.u, data.v, wts, accumulate=np.longdouble)
    Hr, gr, s = rr.robust_pass(true, data.w, data.u, data.v, wts, 'linear', None)
    assert np.array_equal(H, Hr) and np.array_equal(g, gr) and s == ssr[0]


def test_huber_inside_its_scale_is_least_squares():
    data, true, lo, up, wts = small_problem(impurity=False)
    H, _, g, ssr = lin.normal_equations(true, data.w, data.u, data.v, wts, accumulate=np.longdouble)
    Hr, gr, s = rr.robust_pass(true, data.w, data.u, data.v, wts, 'huber', 1.0)      # every |res| far below c
    assert np.array_equal(H, Hr) and np.array_equal(g, gr) and s == pytest.approx(ssr[0], rel=1e-15)


@pytest.mark.parametrize('tied', [False, True], ids=['untied', 'tied'])
def test_linear_moments_give_the_least_squares_covariance_bit_for_bit(tied):
    data, true, lo, up, wts = small_problem(impurity=False)
    ties = synth.satellite_ties(6) if tied else None
    x = true if ties is None else ties.expand(true[ties.free()])
    H, M, g, ssr = lin.normal_equations(x, data.w, data.u, data.v, wts, accumulate=np.longdouble)
    m = rr.moments(x, data.w, data.u, data.v, wts, 'linear', None)
    C0, i0 = utils.covariance_from_normal(H, M, g, ssr, data.w.size, x, lo, up, ties=ties)
    C1, i1 = utils.covariance_from_normal(H, M, g, ssr, data.w.size, x, lo, up, ties=ties, moments=m)
    assert C0.tobytes() == C1.tobytes()
    assert i1['robust_factor'] == 1.0 and 'robust_factor' not in i0
    C2, _ = rr.covariance(x, data.w, data.u, data.v, wts, 'linear', None, lo, up, ties=ties)
    assert C0.tobytes() == C2.tobytes()


@pytest.mark.parametrize('loss', ROBUST)
def test_tied_robust_covariance_is_t_c_theta_t(loss):
    data, true, lo, up, wts = small_problem()
    ties = synth.satellite_ties(6)
    x = ties.expand(true[ties.free()])
    H, M, g, ssr = lin.normal_equations(x, data.w, data.u, data.v, wts, accumulate=np.longdouble)
    m = rr.moments(x, data.w, data.u, data.v, wts, loss, 2e-4)
    C, info = utils.covariance_from_normal(H, M, g, ssr, data.w.size, x, lo, up, ties=ties, moments=m)
    T, _ = ties.matrix()
    Ht, Mt, gt = ties.project(H, M, g)
    free = ties.free()
    Ct, it = utils.covariance_from_normal(Ht, Mt, gt, ssr, data.w.size, x[free], lo[free], up[free], moments=m)
    assert np.allclose(C, T @ Ct @ T.T, rtol=1e-12, atol=0)
    d, N = free.size, data.w.size
    assert info['robust_factor'] == it['robust_factor']
    assert it['robust_factor'] * ssr[1] / (N - d) == pytest.approx(utils.robust_scale(m, N, d), rel=1e-14)


def test_robust_scale_and_its_failure():
    N, d = 1000, 10
    m = np.array([1.0, 2.0, 3.0, 800.0, 700.0])
    E = 0.8
    K = 1 + (d / N) * (0.7 - E * E) / (E * E)
    assert utils.robust_scale(m, N, d) == pytest.approx(K * K * (3.0 / (N - d)) / (E * E), rel=1e-15)
    assert np.isnan(utils.robust_scale(np.array([1.0, 2.0, 3.0, -5.0, 7.0]), N, d))
    data, true, lo, up, wts = small_problem(impurity=False)
    H, M, g, ssr = lin.normal_equations(true, data.w, data.u, data.v, wts)
    C, info = utils.covariance_from_normal(H, M, g, ssr, data.w.size, true, lo, up,
                                           moments=np.array([1.0, 1.0, 1.0, 0.0, 1.0]))
    assert info['singular'] and np.all(np.isnan(C))


# ---- refusals before any CUDA call ----------------------------------------------------------------------------------
@pytest.mark.parametrize('loss,f_scale,match', [
    ('tukey', 1.0, 'unknown loss'), (7, 1.0, 'unknown loss'), (True, 1.0, 'unknown loss'),
    ('huber', None, 'needs f_scale'), ('huber', 0.0, 'spectrum 0: f_scale'), ('cauchy', -1.0, 'spectrum 0'),
    ('soft_l1', [1.0, np.nan, 1.0], 'spectrum 1: f_scale'), ('huber', [1.0, np.inf, 1.0], 'spectrum 1'),
    ('huber', [1.0, 2.0], 'shape')])
def test_check_loss_refusals(loss, f_scale, match):
    with pytest.raises(ValueError, match=match):
        _cabi.check_loss(loss, f_scale, 3)


def test_check_loss_accepts():
    assert _cabi.check_loss('linear', None, 2) == (_cabi.LOSS_LINEAR, None)
    assert _cabi.check_loss(_cabi.LOSS_LINEAR, -1.0, 2) == (_cabi.LOSS_LINEAR, None)   # not read for linear
    code, fs = _cabi.check_loss('cauchy', 2.0, 3)
    assert code == _cabi.LOSS_CAUCHY and np.array_equal(fs, [2.0, 2.0, 2.0])


class _Fitted(utils.FitUtility):
    def __init__(self, fit_im=False):
        data, true, lo, up, wts = small_problem(N=256, impurity=False)
        super().__init__(data, lo, up, fit_im=fit_im, summary=False)
        self.params, self.error, self.weights = true.copy(), 1e-4, wts


def test_refine_refusals_before_cuda():
    f = _Fitted()
    with pytest.raises(ValueError, match='needs f_scale'):
        f.refine(loss='huber')
    with pytest.raises(ValueError, match='unknown loss'):
        utils.refine_batch([f, _Fitted()], loss='l1', f_scale=1.0)
    with pytest.raises(ValueError, match='spectrum 1'):
        utils.refine_batch([f, _Fitted()], loss='huber', f_scale=[1.0, 0.0])
    with pytest.raises(NotImplementedError, match='fit_im'):
        _Fitted(fit_im=True).refine(loss='huber', f_scale=1.0)


def test_correlated_noise_after_robust_refinement_is_refused():
    f = _Fitted()
    f.loss = dict(name='huber', f_scale=1.0)
    with pytest.raises(NotImplementedError, match='robust'):
        f.compute_uncertainties(noise='correlated')


@pytest.mark.parametrize('opts,match', [(dict(loss='huber', f_scale=1.0), 'need'), (dict(f_scale=1.0), 'need'),
                                        (dict(refine=True, loss='huber'), 'needs f_scale'),
                                        (dict(refine=True, loss='bisquare', f_scale=1.0), 'unknown loss')])
def test_fit_option_refusals(opts, match):
    data, true, lo, up, wts = small_problem(N=256, impurity=False)
    with pytest.raises(ValueError, match=match):
        utils.FitUtility(data, lo, up, summary=False, options=opts).fit()
    with pytest.raises(ValueError, match=match):
        core.fit_batch([data, data], [lo, lo], [up, up], options=opts)
