"""Robust losses on the GPU across their whole scale (DESIGN K16).  What decides the arithmetic is z = (res / c)^2,
so every test here runs where test_gpu_robust.py does not: c from 1e-3 sigma (z >> 1 at almost every point) to
1e6 sigma (z ~ 1e-12), and c so small that z overflows.  The robust pass and the moments against robust_ref, the
limits the losses must reach as c grows (Huber is K12, every robust refinement is least squares), the standard errors
when almost no point lies inside c, and the refinement's refusal to move when z is not finite."""
import numpy as np
import pytest

from nmrfit_b200 import _cabi, synth, utils
import linearisation_ref as lin
import robust_ref as rr
from test_gpu_refine import AT_MINIMUM, multiplet, starts_for
from test_gpu_robust import ROBUST, SIGMA, record, worst

pytestmark = pytest.mark.gpu

SCALES = np.array([1e-3, 0.1, 1.345, 1e2, 1e4, 1e6])     # c / sigma
# (N, P, non-uniform axis): K12's plan branches of linearisation_ref.SWEEP (one tile, one slice, two task slices)
SHAPES = [(37, 1, False), (4096, 6, False), (3000, 36, False), (4096, 6, True)]
SHAPE_IDS = ['37x1', '4096x6', '3000x36', 'nonuniform']


def problem(N, P, nonuniform):
    """A multiplet with sigma = 1e-4 noise, its box and weights, and two points: the truth (the residual is the noise
    alone, so c sets z at every point alike) and the truth perturbed by 1e-3 (a misfit of up to ~1e3 sigma)."""
    d, true = multiplet(N, P, 41)
    if nonuniform:
        d.w = d.w + np.random.default_rng(5).uniform(-0.3, 0.3, N) * (d.w[1] - d.w[0])
    lo, up = (np.array(a, dtype=np.float64) for a in d.generate_solution_bounds())
    wts = utils.compute_weights(d.w, d.peaks)
    x = np.clip(true * (1 + 1e-3 * np.random.default_rng(N + P).standard_normal(true.size)), lo, up)
    return d, lo, up, wts, [np.clip(true, lo, up), x]


def rounding_spread(x, d, wts, loss, c):
    """How far the residual's own rounding can move each output: (H [D, D], g [D], cost, moments [5]).  The kernel and
    the reference each form res_i as a difference of terms of size |u_i| + |v_i|, so they may differ by
    delta_i = 16 eps (|u_i| + |v_i|) whatever the loss.  At c near or below that, z = (res/c)^2 is ill-conditioned
    (a point with |res| close to c dominates H_rho for small c, and its rho' moves by delta / |res| of itself), and
    each per-point term is moved by up to its change over res_i +- delta_i; those changes add in magnitude."""
    res, A = lin.residual_jacobian(x, d.w, d.u, d.v)
    delta = 16 * np.finfo(np.float64).eps * (np.abs(d.u) + np.abs(d.v))
    w2 = np.asarray(wts, dtype=np.float64) ** 2

    def terms(r):
        z = (r / c) ** 2
        rho, d1, _ = rr.loss_terms(z, loss)
        dpsi = rr.psi_prime(z, loss)
        return np.stack([w2 * d1, w2 * d1 * r, w2 * c * c * rho, w2 * r * r, (d1 * r) ** 2, dpsi, dpsi * dpsi])

    t = terms(res)
    dt = np.maximum(np.abs(terms(res + delta) - t), np.abs(terms(res - delta) - t))
    absA = np.abs(A)
    return absA.T @ (dt[0][:, None] * absA), absA.T @ dt[1], dt[2].sum(), dt[2:].sum(axis=1)


def context(d, wts, B):
    ctx = _cabi.Context(B, d.w.size, len(d.peaks))
    ctx.set_spectra(*(np.repeat(a[None], B, axis=0) for a in (d.w, d.u, d.v, wts)))
    return ctx


@pytest.mark.parametrize('loss', ROBUST)
@pytest.mark.parametrize('N,P,nonuniform', SHAPES, ids=SHAPE_IDS)
def test_pass_and_moments_across_the_scale(N, P, nonuniform, loss):
    """normal_equations_loss and loss_moments against the long-double reference at every c / sigma of SCALES, with
    test_gpu_robust's tolerances: H_rho 1e-12 sqrt(H_jj H_kk), g_rho and the cost 1e-10, the moments 1e-12 of the sum
    of their terms' magnitudes (the sum itself for all but sum psi', whose terms change sign for Cauchy).  To each is
    added what the rounding of the residual itself can do (rounding_spread): nothing at c >= 1.345 sigma, and at
    c = 1e-3 sigma more than the fixed tolerances for H_rho and for soft-L1's and Cauchy's moments."""
    d, lo, up, wts, xs = problem(N, P, nonuniform)
    X = np.repeat(np.array(xs), SCALES.size, axis=0)              # [x0 at every c, x1 at every c]
    cs = np.tile(SCALES * SIGMA, len(xs))
    with context(d, wts, len(X)) as ctx:
        H, g, cost = ctx.normal_equations_loss(X, loss, cs)
        m = ctx.loss_moments(X, loss, cs)
    ratios = {}
    for b, (x, c) in enumerate(zip(X, cs)):
        Ho, go, so = rr.robust_pass(x, d.w, d.u, d.v, wts, loss, c)
        mo = rr.moments(x, d.w, d.u, d.v, wts, loss, c)
        res = lin.residual_jacobian(x, d.w, d.u, d.v)[0].astype(np.longdouble)
        mag = mo.copy()
        mag[3] = float(np.sum(np.abs(rr.psi_prime((res / np.longdouble(c)) ** 2, loss))))
        eH, eg, es, em = rounding_spread(x, d, wts, loss, c)
        dh = np.sqrt(np.diag(Ho))
        r = dict(H=worst(np.abs(H[b] - Ho), 1e-12 * np.outer(dh, dh) + eH),
                 g=worst(np.abs(g[b] - go), 1e-10 * np.sqrt(np.diag(Ho) * so) + eg),
                 s=worst(np.abs(cost[b] - so), 1e-10 * so + es),
                 m=worst(np.abs(m[b] - mo), 1e-12 * mag + em + 1e-300))
        ratios['x%d c=%gsigma' % (b // SCALES.size, c / SIGMA)] = r
    print('%s %d x %d%s: worst error/tolerance %s' % (loss, N, P, ' nonuniform' if nonuniform else '', ratios))
    record('scales_%s_%dx%d%s' % (loss, N, P, '_nonuniform' if nonuniform else ''), ratios)
    bad = {k: r for k, r in ratios.items() if max(r.values()) > 1.0}
    assert not bad, bad


@pytest.mark.parametrize('N,P,nonuniform', SHAPES, ids=SHAPE_IDS)
def test_huber_inside_its_scale_is_k12(N, P, nonuniform):
    """With c above every |res_i|, Huber's rho' is 1 at every point, sqrt(rho') scales no row, and H_rho and g_rho are
    K12's H and g byte for byte.  The cost, formed as (w c sqrt(z))^2, agrees with sum w^2 res^2 to 1e-15."""
    d, lo, up, wts, xs = problem(N, P, nonuniform)
    amax = [np.abs(lin.residual_jacobian(x, d.w, d.u, d.v)[0]).max() for x in xs]
    X = np.repeat(np.array(xs), 2, axis=0)
    cs = np.array([c for a in amax for c in (1.001 * a, 1e6 * SIGMA)])
    assert np.all(cs > np.repeat(amax, 2))
    with context(d, wts, len(X)) as ctx:
        H0, M0, g0, ssr0 = ctx.normal_equations(X)
        H, g, cost = ctx.normal_equations_loss(X, 'huber', cs)
    assert H.tobytes() == H0.tobytes() and g.tobytes() == g0.tobytes()
    rel = np.abs(cost / ssr0[:, 0] - 1)
    print('huber inside its scale %d x %d: cost against K12 %s' % (N, P, rel))
    assert np.all(rel <= 1e-15), rel


def test_refinement_at_a_large_scale_is_least_squares():
    """At c = 1e6 sigma every point lies deep inside c (z ~ 1e-12), each loss is least squares to ~1e-12 and each
    robust refinement must end where refine() ends: within 1e-4 standard errors (a few xtol), with M-estimator errors
    within 1e-6 of the sandwich's, and with no more STALLED ends than refine() has.  At the optimum, whether the last
    tiny step is accepted (CONVERGED) or every damped retry rejected (STALLED) is decided by the last bits of the cost
    (test_gpu_refine.AT_MINIMUM), so a cost exact to rounding may stall on a different spectrum than least squares
    does.  A cost with more than rounding error makes the step test s_t < s_c noise well before the optimum: the
    refinement then stalls on every spectrum, about 1e-3 standard errors short of it."""
    ws, us, vs, wts, X0, LB, UB = starts_for(4096, 6, (41, 42))
    B, N = ws.shape
    c = 1e6 * SIGMA
    with _cabi.Context(B, N, 6) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        x_ls, _, _, _, st_ls = ctx.refine(X0, LB, UB)
        H, M, g, ssr = ctx.normal_equations(x_ls)
        se_ls = np.array([np.sqrt(np.diag(utils.covariance_from_normal(H[b], M[b], g[b], ssr[b], N, x_ls[b], LB[b],
                                                                       UB[b])[0])) for b in range(B)])
        stalled = int(np.sum(st_ls == _cabi.REFINE_STALLED))
        assert np.all(np.isin(st_ls, AT_MINIMUM)) and stalled <= B // 2, st_ls
        out = {}
        for loss in ROBUST:
            x, f, passes, accepted, status = ctx.refine(X0, LB, UB, loss=loss, f_scale=c,
                                                        max_iter=utils.default_max_iter(None, loss))
            Hr, Mr, gr, ssrr = ctx.normal_equations(x)
            mom = ctx.loss_moments(x, loss, c)
            se = np.array([np.sqrt(np.diag(utils.covariance_from_normal(Hr[b], Mr[b], gr[b], ssrr[b], N, x[b], LB[b],
                                                                        UB[b], moments=mom[b])[0]))
                           for b in range(B)])
            out[loss] = dict(status=status.tolist(), passes=passes.tolist(),
                             dx=float(np.max(np.abs(x - x_ls) / se_ls)), dse=float(np.max(np.abs(se / se_ls - 1))))
    print('refinement at c = 1e6 sigma against least squares (statuses %s): %s' % (st_ls.tolist(), out))
    record('large_scale_refinement', dict(least_squares=st_ls.tolist(), **out))
    for loss, o in out.items():
        status = np.array(o['status'])
        assert np.all(np.isin(status, AT_MINIMUM)) and np.sum(status == _cabi.REFINE_STALLED) <= stalled, (loss, o)
        assert o['dx'] <= 1e-4 and o['dse'] <= 1e-6, (loss, o)


@pytest.mark.parametrize('loss', ROBUST)
def test_uncertainties_when_almost_no_point_is_inside_the_scale(loss):
    """At c = 1e-3 sigma only the few points with |res| <= c count in Huber's sum psi' (none or 4 here), and Cauchy's
    sum psi' can be negative (psi' ~ -1/z beyond c).  compute_uncertainties() after such a refinement must not raise;
    it returns the reference's errors, or NaN with singular set exactly where the reference's sum psi' <= 0
    (utils.robust_scale).
    Each problem is taken at its truth (the loss set on the fit as refine() sets it) and after refine() from there."""
    c = 1e-3 * SIGMA
    cases = []
    for seed, N, P in ((3, 4096, 6), (4, 3000, 36)):
        data, true = multiplet(N, P, seed)
        lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
        for refined in (False, True):
            fit = utils.FitUtility(data, lo, up, summary=False)
            fit.params, fit.error = np.clip(true, lo, up), SIGMA
            fit.weights = utils.compute_weights(data.w, data.peaks)
            if refined:
                fit.refine(loss=loss, f_scale=c)
            else:
                fit.loss = dict(name=loss, f_scale=c)
            se = fit.compute_uncertainties()
            x, wts = fit.params, fit.weights
            mo = rr.moments(x, data.w, data.u, data.v, wts, loss, c)
            C, info = rr.covariance(x, data.w, data.u, data.v, wts, loss, c, lo, up)
            case = dict(shape='%dx%d' % (N, P), refined=refined, sum_psi_prime=float(mo[3]),
                        singular=bool(fit.uncertainty_info['singular']))
            cases.append(case)
            assert fit.uncertainty_info['singular'] == info['singular'], case
            if mo[3] <= 0:
                assert info['singular'] and np.all(np.isnan(se)), case
            else:
                assert np.all(np.isfinite(se)), case
                case['stderr_rel'] = float(np.max(np.abs(se / np.sqrt(np.diag(C)) - 1)))
                assert case['stderr_rel'] <= 1e-6, case
    print('uncertainties at c = 1e-3 sigma, %s: %s' % (loss, cases))
    record('tiny_scale_uncertainties_' + loss, cases)
    if loss != 'soft_l1':                 # both outcomes occur: one truth with sum psi' <= 0, one with sum psi' > 0
        truths = [case['sum_psi_prime'] for case in cases if not case['refined']]
        assert min(truths) <= 0 < max(truths), truths


@pytest.mark.parametrize('loss', ROBUST)
def test_refinement_when_z_overflows(loss):
    """f_scale = 1e-300 makes z = (res/c)^2 overflow at every point: the cost at the start is not finite, and the
    refinement ends NONFINITE with x as it was, through Context.refine and through FitUtility.refine alike."""
    ws, us, vs, wts, X0, LB, UB = starts_for(4096, 6, (41, 42), swarm=False)
    with _cabi.Context(len(X0), 4096, 6) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        cost = ctx.normal_equations_loss(X0, loss, 1e-300)[2]
        x, f, passes, accepted, status = ctx.refine(X0, LB, UB, loss=loss, f_scale=1e-300)
    assert not np.any(np.isfinite(cost)), cost
    assert np.all(status == _cabi.REFINE_NONFINITE), status
    assert x.tobytes() == X0.tobytes() and np.all(accepted == 0) and np.all(passes == 1)
    data, true = synth.multiplet(4096, 6, seed=41)
    lo, up = data.generate_solution_bounds()
    fit = utils.FitUtility(data, lo, up, summary=False)
    start = np.clip(true, lo, up)
    fit.params, fit.error, fit.weights = start.copy(), SIGMA, utils.compute_weights(data.w, data.peaks)
    fit.refine(loss=loss, f_scale=1e-300)
    assert fit.refine_info['status'] == _cabi.REFINE_NONFINITE and fit.params.tobytes() == start.tobytes()
    assert fit.error == SIGMA
