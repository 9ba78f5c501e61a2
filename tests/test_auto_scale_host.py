"""Automatic scale of the robust losses (DESIGN K17) without a GPU: the constants' Gaussian efficiency, the noise-level
formula against scipy, and every refusal of ``f_scale='auto'`` the Python layer makes before a CUDA call."""
import numpy as np
import pytest
from scipy.integrate import quad
from scipy.stats import median_abs_deviation, norm

from nmrfit_b200 import _cabi, core, synth, utils
import robust_ref as rr

ROBUST = ('huber', 'soft_l1', 'cauchy')


@pytest.mark.parametrize('loss', ROBUST)
def test_auto_scale_k_gives_95_percent_efficiency(loss):
    """(E psi')^2 / E psi^2 under N(0, 1) at c = AUTO_SCALE_K[loss], split at c where Huber's psi' jumps."""
    k = utils.AUTO_SCALE_K[loss]
    psi = lambda r: rr.loss_terms((r / k) ** 2, loss)[1] * r
    dpsi = lambda r: rr.psi_prime((r / k) ** 2, loss)

    def half(f):
        return sum(quad(lambda r: f(r) * norm.pdf(r), a, b, epsabs=1e-13, epsrel=1e-12)[0]
                   for a, b in ((0.0, k), (k, np.inf)))
    eff = (2 * half(dpsi)) ** 2 / (2 * half(lambda r: psi(r) ** 2))
    assert abs(eff - 0.95) < 1e-4, eff


def test_normal_mad_is_scipys_quantile():
    from scipy.special import ndtri
    assert utils.NORMAL_MAD == ndtri(0.75)


@pytest.mark.parametrize('n', [1, 2, 7, 1000, 4097])
def test_sigma_formula_is_scipys_bit_for_bit(n):
    rng = np.random.default_rng(n)
    for r in (rng.standard_normal(n) * 1e-4, rng.standard_t(2, n), np.where(rng.random(n) < 0.3, 5.0, 0.0) +
              rng.standard_normal(n)):
        med = np.median(r)
        mad = np.median(np.abs(r - med))
        assert (mad / utils.NORMAL_MAD).tobytes() == np.float64(median_abs_deviation(r, scale='normal')).tobytes()


# ---- refusals before any CUDA call ----------------------------------------------------------------------------------
@pytest.fixture
def no_cuda(monkeypatch):
    """Any call into the library fails the test."""
    def refuse():
        raise AssertionError('a CUDA call was made')
    monkeypatch.setattr(_cabi, 'lib', refuse)


@pytest.mark.parametrize('f_scale', [['auto', 1.0, 1.0], [1.0, 'auto', 2.0], np.array(['auto', 'auto', 'auto'])])
def test_auto_in_a_list_is_refused(f_scale, no_cuda):
    with pytest.raises(ValueError, match='give it once'):
        utils.check_loss_scale('huber', f_scale, 3)


@pytest.mark.parametrize('f_scale', ['Auto', 'mad', ''])
def test_other_strings_are_refused(f_scale, no_cuda):
    with pytest.raises(ValueError, match="or 'auto'"):
        utils.check_loss_scale('cauchy', f_scale, 2)


def test_check_loss_scale_accepts(no_cuda):
    for loss in ROBUST:
        assert utils.check_loss_scale(loss, 'auto', 4) == (_cabi.LOSSES[loss], 'auto')
    assert utils.check_loss_scale('linear', 'auto', 2) == (_cabi.LOSS_LINEAR, None)     # not read for linear
    assert utils.check_loss_scale('linear', 'anything', 2) == (_cabi.LOSS_LINEAR, None)
    code, fs = utils.check_loss_scale('huber', [1.0, 2.0], 2)
    assert code == _cabi.LOSS_HUBER and np.array_equal(fs, [1.0, 2.0])
    with pytest.raises(ValueError, match='needs f_scale'):
        utils.check_loss_scale('huber', None, 2)
    with pytest.raises(ValueError, match='unknown loss'):
        utils.check_loss_scale('tukey', 'auto', 2)


def small_problem(N=256):
    data, true = synth.multiplet(N, 6, seed=3, noise=1e-4, jitter=False)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    return data, true, lo, up, utils.compute_weights(data.w, data.peaks)


class _Fitted(utils.FitUtility):
    def __init__(self):
        data, true, lo, up, wts = small_problem()
        super().__init__(data, lo, up, summary=False)
        self.params, self.error, self.weights = true.copy(), 1e-4, wts


def test_refine_refusals_before_cuda(no_cuda):
    f = _Fitted()
    with pytest.raises(ValueError, match='give it once'):
        utils.refine_batch([f, _Fitted()], loss='huber', f_scale=['auto', 1.0])
    with pytest.raises(ValueError, match="or 'auto'"):
        f.refine(loss='soft_l1', f_scale='median')
    assert f.params is not None and getattr(f, 'refine_info', None) is None


@pytest.mark.parametrize('opts,match', [
    (dict(loss='huber', f_scale='auto'), 'need'), (dict(f_scale='auto'), 'need'),
    (dict(refine=True, loss='huber', f_scale=['auto', 'auto']), 'give it once'),
    (dict(refine=True, loss='cauchy', f_scale='noise'), "or 'auto'")])
def test_fit_option_refusals(opts, match, no_cuda):
    data, true, lo, up, wts = small_problem()
    with pytest.raises(ValueError, match=match):
        utils.FitUtility(data, lo, up, summary=False, options=opts).fit()
    with pytest.raises(ValueError, match=match):
        core.fit_batch([data, data], [lo, lo], [up, up], options=opts)


def test_noise_level_needs_a_fit(no_cuda):
    data, true, lo, up, wts = small_problem()
    f = utils.FitUtility(data, lo, up, summary=False)
    f.params = None
    with pytest.raises(RuntimeError, match='fit'):
        f.noise_level()
    assert utils.noise_level_batch([]).shape == (0,)
