"""Host side of the parameter uncertainties: the reference residual Jacobian (linearisation_ref.py) against
complex-step derivatives, and the sandwich covariance and area-fraction error in numpy (no GPU)."""
import numpy as np
import pytest

from conftest import load_golden
from nmrfit_b200 import utils
import linearisation_ref as lin
from oracle import nmrfit_oracle as orc
from test_cabi_symbols import built  # noqa: F401  (builds the library; the plan query makes no CUDA call)

LN2 = np.log(2.0)


def residual_complex(x, w, u, v):
    """The residual written with operations that carry a complex step through every parameter."""
    n, P = w.size, (x.size - 4) // 3
    p0, p1, r, yoff = x[:4]
    phi = p0 + p1 * np.arange(n) / n
    fit = 0
    for k in range(P):
        width, loc, a = x[4 + 3 * k:7 + 3 * k]
        d = w - loc
        t = 2 * d / width
        s = 2 * np.sqrt(LN2) * d / width
        fit = fit + yoff + a * (r * (2 / (np.pi * width)) / (1 + t * t) + (1 - r) * (2 / width) * np.sqrt(LN2 / np.pi) * np.exp(-s * s))
    return u * np.cos(phi) - v * np.sin(phi) - fit


def perturbed_axis(w, seed=0):
    rng = np.random.default_rng(seed)
    h = w[1] - w[0]
    return w + rng.uniform(-0.3, 0.3, w.size) * h


CASES = [('objective_c1_4096x6', False), ('objective_p24_1536', False), ('objective_c1_4096x6', True)]


@pytest.mark.parametrize('case,nonuniform', CASES)
def test_reference_jacobian_matches_complex_step(case, nonuniform):
    g = load_golden(case)
    w = perturbed_axis(g['w']) if nonuniform else g['w']
    for x in (g['true'], g['xs'][0], g['xs'][1]):
        res, A = lin.residual_jacobian(x, w, g['u'], g['v'])
        data_scale = np.max(np.abs(g['u']) + np.abs(g['v']))       # the residual cancels data against model
        assert np.max(np.abs(res - residual_complex(x.astype(complex), w, g['u'], g['v']).real)) <= 1e-13 * data_scale
        for j in range(x.size):
            xc = x.astype(complex)
            xc[j] += 1e-30j
            cs = residual_complex(xc, w, g['u'], g['v']).imag / 1e-30
            scale = np.max(np.abs(A[:, j]))
            assert np.max(np.abs(cs - A[:, j])) <= 1e-13 * scale, (j, np.max(np.abs(cs - A[:, j])) / scale)


@pytest.mark.parametrize('case', ['objective_c1_4096x6', 'objective_p24_1536', 'objective_ragged_1000x6'])
def test_reference_residual_is_the_objective(case):
    g = load_golden(case)
    for x in g['xs'][:4]:
        res, _ = lin.residual_jacobian(x, g['w'], g['u'], g['v'])
        assert np.sqrt(np.square(np.multiply(g['weights'], res)).mean()) == orc.objective(x, g['w'], g['u'], g['v'],
                                                                                           g['weights'])


def test_reference_normal_equations_are_the_weighted_sums():
    g = load_golden('objective_ragged_1000x6')
    x, wts = g['xs'][0], g['weights']
    res, A = lin.residual_jacobian(x, g['w'], g['u'], g['v'])
    H, M, gr, ssr = lin.normal_equations(x, g['w'], g['u'], g['v'], wts)
    J = wts[:, None] * A
    for got, want in ((H, J.T @ J), (M, (wts[:, None] * J).T @ (wts[:, None] * J))):
        d = np.sqrt(np.diag(want))
        assert np.max(np.abs(got - want) / np.outer(d, d)) < 1e-13
    assert np.max(np.abs(gr - J.T @ (wts * res)) / np.sqrt(np.diag(H) * ssr[0])) < 1e-13
    assert np.isclose(ssr[0], np.sum((wts * res) ** 2), rtol=1e-14) and np.isclose(ssr[1], np.sum(res ** 2), rtol=1e-14)


def normal_at(g, x, weights):
    return lin.normal_equations(x, g['w'], g['u'], g['v'], weights)


def test_covariance_unit_weights_is_s2_hinv():
    g = load_golden('objective_c1_4096x6')
    x = g['true']
    H, M, gr, ssr = normal_at(g, x, np.ones_like(g['w']))
    C, info = utils.covariance_from_normal(H, M, gr, ssr, g['w'].size, x, g['lower'], g['upper'])
    s2 = ssr[1] / (g['w'].size - x.size)
    want = s2 * np.linalg.inv(H)
    assert not info['singular'] and info['dof'] == g['w'].size - x.size
    assert info['sigma'] == pytest.approx(np.sqrt(s2), rel=1e-15)
    assert np.array_equal(info['gradient'], gr)
    scale = np.sqrt(np.outer(np.diag(want), np.diag(want)))
    assert np.max(np.abs(C - want) / scale) < 1e-12
    assert np.array_equal(C, C.T)


def test_covariance_sandwich_with_weights():
    g = load_golden('objective_c1_4096x6')
    x = g['true']
    H, M, gr, ssr = normal_at(g, x, g['weights'])
    C, info = utils.covariance_from_normal(H, M, gr, ssr, g['w'].size, x, g['lower'], g['upper'])
    Hi = np.linalg.inv(H)
    want = ssr[1] / (g['w'].size - x.size) * Hi @ M @ Hi
    scale = np.sqrt(np.outer(np.diag(want), np.diag(want)))
    assert np.max(np.abs(C - want) / scale) < 1e-9
    assert np.all(np.diag(C) > 0)


def test_zero_area_is_singular():
    g = load_golden('objective_c1_4096x6')
    x = g['true'].copy()
    x[6] = 0.0                                    # the first peak's width and location no longer matter
    H, M, gr, ssr = normal_at(g, x, g['weights'])
    C, info = utils.covariance_from_normal(H, M, gr, ssr, g['w'].size, x, g['lower'], g['upper'])
    assert info['singular'] and np.all(np.isnan(C)) and C.shape == (x.size, x.size)
    # a rank-deficient H with a non-zero diagonal fails in the factorisation instead
    H2 = H.copy()
    H2[:, 7] = H2[7, :] = H[:, 8]
    H2[7, 7] = H[8, 8]
    H2[7, 8] = H2[8, 7] = H[8, 8]
    C2, info2 = utils.covariance_from_normal(H2, M, gr, ssr, g['w'].size, g['true'], g['lower'], g['upper'])
    assert info2['singular'] and np.all(np.isnan(C2))


def test_at_bound_flags():
    g = load_golden('objective_c1_4096x6')
    x = g['true'].copy()
    lo, up = g['lower'], g['upper']
    x[4] = lo[4]
    x[8] = up[8] - 1e-12 * (up[8] - lo[8])
    x[10] = lo[10] + 1e-6 * (up[10] - lo[10])     # close, but not within 1e-9 of the box width
    H, M, gr, ssr = normal_at(g, g['true'], g['weights'])
    _, info = utils.covariance_from_normal(H, M, gr, ssr, g['w'].size, x, lo, up)
    want = np.zeros(x.size, dtype=bool)
    want[[4, 8]] = True
    assert np.array_equal(info['at_bound'], want)


def test_area_fraction_stderr_is_the_delta_method():
    g = load_golden('objective_p24_1536')
    x = g['true']
    f = utils.FitUtility(None, g['lower'], g['upper'])
    f.params = x.copy()
    rng = np.random.default_rng(5)
    B = rng.normal(size=(x.size, x.size))
    f.covariance = (B @ B.T) * 1e-6 * np.outer(np.abs(x) + 1e-3, np.abs(x) + 1e-3)
    grad = np.zeros(x.size)
    for j in range(6, x.size, 3):
        h = 1e-6 * abs(x[j])
        xp, xm = x.copy(), x.copy()
        xp[j] += h
        xm[j] -= h
        grad[j] = (orc.area_fraction(orc.get_areas(xp)) - orc.area_fraction(orc.get_areas(xm))) / (2 * h)
    want = np.sqrt(grad @ f.covariance @ grad)
    assert f.area_fraction_stderr() == pytest.approx(want, rel=1e-8)


PLAN_POINTS = (1, 37, 255, 256, 257, 1000, 4096, 5000, 65536, 2_100_000)


def test_normal_equations_plan_invariants(built):
    """What csrc/normal_eq.cu relies on, for every peak count it accepts: the CTA fits __launch_bounds__(512), the
    point groups or task slices cover every 4x4 block, the tile keeps the staged rows near 48 KB, the chunks cover
    the spectrum in at most 128 partials, and the shared memory holds both the staged tile and the end-of-chunk
    reduction within the 200 KiB the launch opts into."""
    from nmrfit_b200 import _cabi
    for P in range(1, 65):
        E = 5 + 3 * P
        nb = -(-E // 4)
        ep = 4 * nb
        for N in PLAN_POINTS:
            p = _cabi.normal_equations_plan(N, P)
            where = (N, P, p)
            ng, tasks, tps, threads, tp, ch = (p[k] for k in ('point_groups', 'tasks', 'tasks_per_slice', 'threads',
                                                              'tile_points', 'chunk_points'))
            assert tasks == nb * (nb + 1), where                      # upper triangles of both matrices
            assert threads % 32 == 0 and 0 < threads <= 512, where
            if ng > 1:
                assert p['slices'] == 1 and tps == tasks and ng * tasks <= threads, where
            else:
                assert ng == 1 and tps <= threads, where
                assert p['slices'] * tps >= tasks and (p['slices'] - 1) * tps < tasks, where
            assert tp in (16, 32, 64, 128), where
            assert tp == 16 or 2 * tp * ep <= 6144, where
            assert ch >= 256 and ch & (ch - 1) == 0 and ch % tp == 0, where
            assert p['n_chunks'] == -(-N // ch) and p['n_chunks'] <= 128, where
            stage = 2 * tp * ep + 2 * tp * P + 8 * P                  # rows, model values, d/dr terms, peak constants
            assert p['smem_bytes'] == 8 * max(stage, 16 * threads) <= 200 * 1024, where
            assert p['scratch_doubles'] == p['n_chunks'] * tasks * 16, where


def test_normal_equations_plan_pins(built):
    """The sizes DESIGN §4 K12 states, and the branch every shape of the GPU parity sweep must take."""
    from nmrfit_b200 import _cabi
    c3 = _cabi.normal_equations_plan(16384, 6)
    assert (c3['n_chunks'], c3['chunk_points']) == (4, 4096)
    assert round(c3['scratch_doubles'] * 8 * 1024 / 1e6) == 22            # MB for 1,024 spectra
    c4 = _cabi.normal_equations_plan(65536, 24)
    assert (c4['n_chunks'], c4['chunk_points']) == (128, 512)
    assert round(c4['scratch_doubles'] * 8 / 1e6, 1) == 6.9
    for (N, P), want in lin.SWEEP.items():
        got = _cabi.normal_equations_plan(N, P)
        assert {k: got[k] for k in want} == want, (N, P, got)
    for N, P in ((0, 6), (-5, 6), (100, 0), (100, 65)):
        with pytest.raises(_cabi.NmrfitError) as e:
            _cabi.normal_equations_plan(N, P)
        assert e.value.code == -1


def test_compute_uncertainties_errors_before_any_device_call():
    g = load_golden('objective_tiny_257x6')
    f = utils.FitUtility(None, g['lower'], g['upper'])
    with pytest.raises(RuntimeError, match='fit'):
        f.compute_uncertainties()
    f.params = g['true']
    f.fit_im = True
    with pytest.raises(NotImplementedError):
        f.compute_uncertainties()
