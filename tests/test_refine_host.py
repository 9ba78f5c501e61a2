"""Host side of the refinement (DESIGN K13): the numpy restatement of bounded Levenberg-Marquardt
(refine_ref.refine) from a swarm's answer, its frozen-set and non-finite rules, and the argument checks
``Context.refine`` makes before any CUDA call (no GPU)."""
import numpy as np
import pytest

from nmrfit_b200 import _cabi, synth, utils
import linearisation_ref as lin
import refine_ref as rr
from oracle import nmrfit_oracle as orc, pso_oracle


def stderr_at(x, d, wts, lo, up):
    H, M, g, ssr = lin.normal_equations(x, d.w, d.u, d.v, wts, accumulate=np.longdouble)
    C, info = utils.covariance_from_normal(H, M, g, ssr, d.w.size, x, lo, up)
    return np.sqrt(np.diag(C)), info


def test_reference_refines_the_configs0_swarm_to_the_optimum():
    """configs[0]: 4,096 points, 6 peaks, pyswarm's 100 x 100 swarm seeded with 0 (the oracle's restatement).  The
    swarm stops at 16.6x the optimum's RMS, 5 to 733 standard errors off in every parameter; refinement converges in
    at most 10 passes."""
    d, _ = synth.multiplet(4096, 6, seed=0)
    lo, up = d.generate_solution_bounds()
    wts = utils.compute_weights(d.w, d.peaks)
    np.random.seed(0)
    xs, fs = pso_oracle.pso(orc.objective, lo, up, args=(d.w, d.u, d.v, wts, False), swarmsize=100, maxiter=100,
                            omega=-0.2134, phip=-0.3344, phig=2.3259)[:2]
    x, f, passes, accepted, status = rr.refine(xs, lo, up, d.w, d.u, d.v, wts)
    assert status == rr.CONVERGED and passes <= 10 and accepted >= 1, (status, passes)
    # the optimum, with a tolerance no step can meet
    x_opt, f_opt, _, _, _ = rr.refine(x, lo, up, d.w, d.u, d.v, wts, max_iter=100, xtol=1e-12)
    assert f * f < 1.0001 * f_opt * f_opt
    assert round(fs / f_opt, 1) == 16.6
    se, _ = stderr_at(x_opt, d, wts, lo, up)
    off = np.abs(xs - x_opt) / se
    assert round(off.min()) == 5 and round(off.max()) == 733, off
    assert np.all(np.abs(x - x_opt) <= 1e-3 * se)


def test_reference_frozen_set():
    """An area whose optimum lies above its upper bound, started on that bound, stays there.  A satellite of area 0
    held at its upper bound 0 keeps its width and centre bit for bit (H_jj = 0 for both)."""
    d, true = synth.multiplet(2048, 6, seed=3)
    lo, up = (np.array(a) for a in d.generate_solution_bounds())
    wts = utils.compute_weights(d.w, d.peaks)
    x0 = np.clip(true * (1 + 1e-3 * np.random.default_rng(0).standard_normal(true.size)), lo, up)
    bound = 6 + 3 * 1
    lo_b, up_b, x_b = lo.copy(), up.copy(), x0.copy()
    up_b[bound] = 0.95 * true[bound]
    x_b[bound] = up_b[bound]
    g = lin.normal_equations(x_b, d.w, d.u, d.v, wts)[2]
    assert g[bound] < 0
    x, f, passes, accepted, status = rr.refine(x_b, lo_b, up_b, d.w, d.u, d.v, wts)
    assert status == rr.CONVERGED and accepted >= 1
    assert x[bound] == up_b[bound] and np.all((x >= lo_b) & (x <= up_b))

    zero = [4 + 3 * 5, 5 + 3 * 5, 6 + 3 * 5]
    lo_z, up_z, x_z = lo.copy(), up.copy(), x0.copy()
    lo_z[zero[2]], up_z[zero[2]], x_z[zero[2]] = -1.0, 0.0, 0.0
    H = lin.normal_equations(x_z, d.w, d.u, d.v, wts)[0]
    assert H[zero[0], zero[0]] == 0 and H[zero[1], zero[1]] == 0
    x, f, passes, accepted, status = rr.refine(x_z, lo_z, up_z, d.w, d.u, d.v, wts)
    assert status == rr.CONVERGED and accepted >= 1
    assert x[zero].tobytes() == x_z[zero].tobytes() and np.all((x >= lo_z) & (x <= up_z))


def test_reference_nonfinite_start():
    d, true = synth.multiplet(1024, 6, seed=4)
    lo, up = (np.array(a) for a in d.generate_solution_bounds())
    wts = utils.compute_weights(d.w, d.peaks)
    x0 = true.copy()
    lo[4] = 0.0
    x0[4] = 0.0                                          # width 0: 1/width is infinite
    x, f, passes, accepted, status = rr.refine(x0, lo, up, d.w, d.u, d.v, wts)
    assert status == rr.NONFINITE and passes == 1 and accepted == 0
    assert x.tobytes() == x0.tobytes()


def test_context_refine_checks_arguments_before_any_cuda_call(monkeypatch):
    def no_library():
        raise AssertionError('the library was called')
    monkeypatch.setattr(_cabi, 'lib', no_library)
    ctx = object.__new__(_cabi.Context)
    ctx._h = None
    ctx.B, ctx.N, ctx.P, ctx.D = 2, 100, 2, 10
    x = np.zeros((2, 10))
    lo, up = -np.ones(10), np.ones(10)
    bad = [
        (dict(x=np.zeros((2, 9))), 'x must have shape'),
        (dict(x=np.zeros(10)), 'x must have shape'),
        (dict(lb=-np.ones(9)), 'lb and ub'),
        (dict(x=np.full((2, 10), 2.0)), 'inside its box'),
        (dict(x=np.full((2, 10), np.nan)), 'inside its box'),
        (dict(lb=np.ones(10)), 'below its upper bound'),
        (dict(ub=np.r_[np.ones(9), -1.0]), 'below its upper bound'),
        (dict(max_iter=0), 'max_iter'),
        (dict(xtol=0.0), 'xtol'),
        (dict(xtol=np.nan), 'xtol'),
    ]
    for kw, msg in bad:
        args = dict(x=x, lb=lo, ub=up, max_iter=50, xtol=1e-6)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            ctx.refine(**args)
    ctx.P, ctx.D = 65, 4 + 3 * 65
    with pytest.raises(ValueError, match='at most 64 peaks'):
        ctx.refine(np.zeros((2, ctx.D)), -np.ones(ctx.D), np.ones(ctx.D))
    ctx.P, ctx.D, ctx.N = 2, 10, 10
    with pytest.raises(ValueError, match='degrees of freedom'):
        ctx.refine(x, lo, up)


def test_refine_needs_a_least_squares_fit():
    d, _ = synth.multiplet(512, 6, seed=1)
    lo, up = d.generate_solution_bounds()
    f = utils.FitUtility(d, lo, up, summary=False)
    with pytest.raises(RuntimeError, match='call fit'):
        f.refine()
    f = utils.FitUtility(d, lo, up, fit_im=True, summary=False, options={'refine': True})
    with pytest.raises(NotImplementedError):
        f.fit()                                          # refused before the swarm runs
    f.params, f.error = np.zeros(len(lo)), 1.0
    with pytest.raises(NotImplementedError):
        f.refine()
