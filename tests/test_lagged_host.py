"""Host side of the correlated-noise standard errors (DESIGN K14): the launch plan of csrc/lagged.cu, the long-double
reference of lagged_ref.py against dense products, the positive semidefiniteness the Bartlett taper guarantees, and
the argument checks made before any CUDA call (no GPU)."""
import numpy as np
import pytest
from scipy.linalg import toeplitz

from conftest import load_golden
from nmrfit_b200 import synth, utils
import lagged_ref as lag
import linearisation_ref as lin
from test_cabi_symbols import built  # noqa: F401  (builds the library; the plan query makes no CUDA call)

PLAN_POINTS = (1, 37, 255, 256, 257, 1000, 4096, 5000, 65536, 2_100_000)


def test_lagged_plan_invariants(built):
    """What csrc/lagged.cu relies on, for every peak count it accepts, at several lags up to the cap: the CTA fits
    __launch_bounds__(512), the point groups or task slices cover every 4x4 block of the upper triangle, the tile and
    its two halos fit the shared memory the launch opts into, and the chunks cover the spectrum."""
    from nmrfit_b200 import _cabi
    for P in range(1, 65):
        D = 4 + 3 * P
        nb = -(-D // 4)
        ep = 4 * nb
        cap = _cabi.lagged_plan(1000, P)['max_lag']
        assert cap >= 32 and (P > 12 or cap >= 128), (P, cap)
        # the cap is the largest lag whose 16-point tile fits in 200 KiB
        stage = lambda tp, L: (2 * tp + 2 * L) * ep + tp * P + 8 * P + L + 1
        assert stage(16, cap) <= 25600 < stage(16, cap + 1), (P, cap)
        for N in PLAN_POINTS:
            for L in sorted({0, 1, 32, cap // 2, cap}):
                p = _cabi.lagged_plan(N, P, L)
                where = (N, P, L, p)
                ng, tasks, tps, threads, tp, ch = (p[k] for k in ('point_groups', 'tasks', 'tasks_per_slice',
                                                                  'threads', 'tile_points', 'chunk_points'))
                assert p['max_lag'] == cap, where                        # a function of P alone
                assert tasks == nb * (nb + 1) // 2, where
                assert threads % 32 == 0 and 0 < threads <= 512, where
                if ng > 1:
                    assert p['slices'] == 1 and tps == tasks and ng * tasks <= threads, where
                else:
                    assert tps <= threads and p['slices'] * tps >= tasks and (p['slices'] - 1) * tps < tasks, where
                assert tp in (16, 32, 64, 128), where
                assert tp == 16 or stage(tp, L) <= 12288, where           # about 96 KB: two CTAs per SM
                assert ch >= 256 and ch & (ch - 1) == 0 and ch % tp == 0, where
                assert p['n_chunks'] == -(-N // ch) and p['n_chunks'] <= 128, where
                assert p['smem_bytes'] == 8 * max(stage(tp, L), 16 * threads) <= 200 * 1024, where
                assert p['scratch_doubles'] == p['n_chunks'] * tasks * 16, where
                assert p['acf_n_chunks'] == -(-N // p['acf_chunk_points']), where
                assert p['acf_scratch_doubles'] == p['acf_n_chunks'] * (L + 1), where


def test_lagged_plan_pins_and_refusals(built):
    """The branch every shape of the GPU parity sweep must take, the sizes DESIGN §4 K14 states, and the refusals."""
    from nmrfit_b200 import _cabi
    for (N, P, L), want in lag.SWEEP.items():
        got = _cabi.lagged_plan(N, P, L)
        assert {k: got[k] for k in want} == want, (N, P, L, got)
    c3 = _cabi.lagged_plan(16384, 6, 32)
    assert (c3['tile_points'], c3['chunk_points'], c3['n_chunks']) == (128, 8192, 2)
    assert [_cabi.lagged_plan(1000, P)['max_lag'] for P in (1, 6, 12, 24, 64)] == [1489, 503, 296, 147, 45]
    for N, P, L in ((0, 6, 0), (-5, 6, 0), (100, 0, 0), (100, 65, 0), (100, 6, -1), (100, 6, 504), (100, 64, 46)):
        with pytest.raises(_cabi.NmrfitError) as e:
            _cabi.lagged_plan(N, P, L)
        assert e.value.code == -1
    with pytest.raises(_cabi.NmrfitError, match='cap of 45 at 64 peaks'):
        _cabi.lagged_plan(1000, 64, 46)


def small_problem(N=300, seed=3):
    d, true = synth.multiplet(N, 6, seed=seed)
    wts = utils.compute_weights(d.w, d.peaks)
    x = true * (1 + 0.01 * np.random.default_rng(seed).standard_normal(true.size))
    return d, x, wts


def scaled_err(got, want):
    d = np.sqrt(np.abs(np.diag(want)))
    return np.max(np.abs(got - want) / np.outer(d, d))


def test_banded_reference_is_the_dense_product():
    d, x, wts = small_problem()
    rng = np.random.default_rng(0)
    for L in (0, 1, 7, 40, d.w.size - 1):
        rho = np.r_[1.0, rng.uniform(-1, 1, L)]
        got = lag.m_lagged(x, d.w, d.u, d.v, wts, rho)
        want = lag.m_dense(x, d.w, d.u, d.v, wts, rho)
        assert scaled_err(got, want) < 1e-12 * np.sum(np.abs(np.r_[rho, rho[1:]])), L


def test_acf_reference_is_the_direct_sum():
    d, x, wts = small_problem()
    res, _ = lin.residual_jacobian(x, d.w, d.u, d.v)
    r = lag.residual_acf(x, d.w, d.u, d.v, 20)
    n = res.size
    for k in (0, 1, 5, 20):
        assert r[k] == pytest.approx(sum(res[i] * res[i + k] for i in range(n - k)), rel=1e-12, abs=1e-15 * r[0])
    _, _, _, ssr = lin.normal_equations(x, d.w, d.u, d.v, wts, accumulate=np.longdouble)
    assert r[0] == pytest.approx(ssr[1], rel=1e-14)


def test_lag_zero_reproduces_m():
    g = load_golden('objective_c1_4096x6')
    for x in (g['true'], g['xs'][0]):
        _, M, _, _ = lin.normal_equations(x, g['w'], g['u'], g['v'], g['weights'], accumulate=np.longdouble)
        got = lag.m_lagged(x, g['w'], g['u'], g['v'], g['weights'], [1.0])
        assert scaled_err(got, M) < 1e-14


def test_tapered_estimate_is_positive_semidefinite():
    """From random residuals (white, strongly correlated, alternating): the tapered rho is a PSD Toeplitz sequence and
    M_rho is PSD, at every lag up to N - 1; the untapered estimate is not PSD for some of them."""
    d, x, wts = small_problem(N=200)
    n = d.w.size
    rng = np.random.default_rng(1)
    untapered_fails = 0
    for kind in ('white', 'smooth', 'alternating'):
        e = rng.standard_normal(n)
        if kind == 'smooth':
            e = np.convolve(e, np.exp(-np.arange(12) / 3.0), mode='same')
        elif kind == 'alternating':
            e = e + 3 * (-1.0) ** np.arange(n) * np.convolve(rng.standard_normal(n), np.ones(5), mode='same')
        r = np.array([np.sum(e[:n - k] * e[k:]) for k in range(n)])
        for L in (1, 8, 32, 120, n - 1):
            rho = utils.bartlett_taper(r[:L + 1] / r[0])
            T = toeplitz(np.r_[rho, np.zeros(n - L - 1)])
            assert np.linalg.eigvalsh(T).min() > -1e-12 * np.abs(rho).sum(), (kind, L)
            M = lag.m_lagged(x, d.w, d.u, d.v, wts, rho)
            ev = np.linalg.eigvalsh(0.5 * (M + M.T))
            assert ev.min() > -1e-12 * ev.max(), (kind, L, ev.min() / ev.max())
            raw = toeplitz(np.r_[r[:L + 1] / r[0], np.zeros(n - L - 1)])
            untapered_fails += np.linalg.eigvalsh(raw).min() < -1e-9
    assert untapered_fails > 0


def test_bartlett_weights():
    rho = np.array([1.0, 0.5, -0.25, 0.125])
    assert np.array_equal(utils.bartlett_taper(rho), rho * np.array([1.0, 0.75, 0.5, 0.25]))
    assert np.array_equal(utils.bartlett_taper(np.ones((2, 1))), np.ones((2, 1)))


def fitted():
    g = load_golden('objective_ragged_1000x6')
    f = utils.FitUtility(type('Data', (), dict(w=g['w'], u=g['u'], v=g['v']))(), g['lower'], g['upper'])
    f.params, f.weights = g['true'], g['weights']
    return f


@pytest.mark.parametrize('kwargs,match', [
    (dict(noise='pink'), 'noise must be'),
    (dict(noise='white', max_lag=-1), 'max_lag must be an integer'),
    (dict(noise='white', max_lag=2.5), 'max_lag must be an integer'),
    (dict(noise='white', noise_acf=[1.0, 0.5]), "noise='correlated' only"),
    (dict(noise='correlated', max_lag=-3), 'max_lag must be an integer'),
    (dict(noise='correlated', noise_acf=[0.9, 0.5]), 'rho_0 = 1'),
    (dict(noise='correlated', noise_acf=[1.0, 1.5]), r'\|rho_k\| <= 1'),
    (dict(noise='correlated', noise_acf=[1.0, np.nan]), 'finite'),
    (dict(noise='correlated', noise_acf=np.ones((2, 3))), 'shape'),
    (dict(noise='correlated', noise_acf=np.r_[1.0, np.zeros(1000)]), 'below the number of points'),
    (dict(noise='correlated', noise_acf=np.r_[1.0, np.zeros(504)]), 'cap of 503 at 6 peaks'),
])
def test_noise_arguments_are_refused_before_any_device_call(built, kwargs, match):
    """Every check raises ValueError on the host; a CUDA call here would fail differently (no GPU)."""
    f = fitted()
    with pytest.raises(ValueError, match=match):
        f.compute_uncertainties(**kwargs)
    with pytest.raises(ValueError, match=match):
        utils.compute_uncertainties_batch([f], **kwargs)


def test_lagged_context_checks(built):
    """Context.residual_acf / normal_m_lagged refuse bad lags and rho before any CUDA call (the checks are module
    functions, so no context is needed to run them)."""
    from nmrfit_b200 import _cabi
    assert _cabi.check_lag(32, 4096, 6) == 32
    for L, N, P, match in ((-1, 100, 6, '>= 0'), (100, 100, 6, 'below the number'), (46, 1000, 64, 'cap of 45'),
                           (0, 100, 65, 'at most 64 peaks'), (1.5, 100, 6, 'integer')):
        with pytest.raises(ValueError, match=match):
            _cabi.check_lag(L, N, P)
    rho = _cabi.check_rho([1.0, -0.5], 3, 100, 6)
    assert rho.shape == (3, 2) and rho.flags['C_CONTIGUOUS'] and np.array_equal(rho[2], [1.0, -0.5])
    for bad, match in (([1.0, np.inf], 'finite'), (np.ones((2, 2)), 'shape'), (np.ones((3, 2, 1)), 'shape')):
        with pytest.raises(ValueError, match=match):
            _cabi.check_rho(bad, 3, 100, 6)
