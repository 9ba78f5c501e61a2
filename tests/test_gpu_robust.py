"""Robust refinement on the GPU (DESIGN K16): the robust pass and the moments against the long-double restatement
(robust_ref) across K12's launch plan, the LINEAR identities, the refinement against robust_ref and scipy, determinism,
the calibration of Huber's covariance, the bias an unmodelled line leaves, the fit / fit_batch paths and the library's
refusals."""
import ctypes
import json
import os

import numpy as np
import pytest

from nmrfit_b200 import _cabi, core, synth, utils
import robust_ref as rr
from test_gpu_refine import AT_MINIMUM, multiplet, same_outcome, small_fit_options, starts_for
from test_gpu_ties import tied_starts

pytestmark = pytest.mark.gpu

ROBUST = ('huber', 'soft_l1', 'cauchy')
SIGMA = 1e-4                       # synth.multiplet's noise level
C_OF = dict(huber=1.345 * SIGMA, soft_l1=1.345 * SIGMA, cauchy=2.385 * SIGMA, linear=None)


def record(name, value):
    """Keep a measured number of this run in the JSON file NMRFIT_TEST_RECORD names, if it is set."""
    path = os.environ.get('NMRFIT_TEST_RECORD')
    if not path:
        return
    data = json.load(open(path)) if os.path.exists(path) else {}
    data[name] = value
    json.dump(data, open(path, 'w'), indent=1)


def worst(err, tol):
    return float(np.max(err / tol))


# (N, P, non-uniform axis): shapes pinned to K12's plan branches (linearisation_ref.SWEEP)
PASS_SHAPES = [(37, 1, False), (4096, 6, False), (3000, 36, False), (1000, 64, False), (4096, 6, True)]


@pytest.mark.parametrize('N,P,nonuniform', PASS_SHAPES, ids=['37x1', '4096x6', '3000x36', '1000x64', 'nonuniform'])
def test_pass_and_moments_parity(N, P, nonuniform):
    d, true = multiplet(N, P, 41)
    if nonuniform:
        d.w = d.w + np.random.default_rng(5).uniform(-0.3, 0.3, N) * (d.w[1] - d.w[0])
    if (N, P) == (3000, 36):
        assert _cabi.normal_equations_plan(N, P)['slices'] > 1
    lo, up = (np.array(a, dtype=np.float64) for a in d.generate_solution_bounds())
    wts = utils.compute_weights(d.w, d.peaks)
    x = np.clip(true * (1 + 1e-3 * np.random.default_rng(N + P).standard_normal(true.size)), lo, up)
    ratios = {}
    with _cabi.Context(1, N, P) as ctx:
        ctx.set_spectra(d.w[None], d.u[None], d.v[None], wts[None])
        H0, M0, g0, ssr0 = ctx.normal_equations(x[None])
        for loss in rr.LOSSES:
            c = C_OF[loss]
            H, g, cost = ctx.normal_equations_loss(x[None], loss, c)
            m = ctx.loss_moments(x[None], loss, c)
            if loss == 'linear':                         # K12's bytes
                assert H.tobytes() == H0.tobytes() and g.tobytes() == g0.tobytes()
                assert cost.tobytes() == ssr0[:, 0].copy().tobytes()
            Ho, go, so = rr.robust_pass(x, d.w, d.u, d.v, wts, loss, c)
            mo = rr.moments(x, d.w, d.u, d.v, wts, loss, c)
            dh = np.sqrt(np.diag(Ho))
            r = dict(H=worst(np.abs(H[0] - Ho), 1e-12 * np.outer(dh, dh)),
                     g=worst(np.abs(g[0] - go), 1e-10 * np.sqrt(np.diag(Ho) * so)),
                     s=worst(np.abs(cost[0] - so), 1e-10 * so),
                     m=worst(np.abs(m[0] - mo), 1e-12 * np.abs(mo) + 1e-300))
            ratios[loss] = r
            assert max(r.values()) <= 1.0, (loss, r)
            if loss != 'linear':
                assert mo[3] < N                          # some points are beyond the scale
    print('pass parity %d x %d: worst error/tolerance %s' % (N, P, ratios))
    record('pass_parity_%dx%d%s' % (N, P, '_nonuniform' if nonuniform else ''), ratios)


def raw_refine_loss(ctx, x, lb, ub, loss, f_scale, ties=(None, None, None), max_iter=50, xtol=1e-6):
    """nmrfit_ctx_refine_loss itself, past the checks Context.refine makes first: (status code, x, f, passes,
    accepted, status)."""
    B = x.shape[0]
    x, lb, ub = (np.array(a, dtype=np.float64, order='C') for a in (x, lb, ub))
    f = np.empty(B)
    passes, accepted, status = (np.empty(B, dtype=np.int32) for _ in range(3))
    fs = None if f_scale is None else np.ascontiguousarray(f_scale, dtype=np.float64)
    rc = _cabi.lib().nmrfit_ctx_refine_loss(ctx._h, _cabi.ptr(x), _cabi.ptr(lb), _cabi.ptr(ub),
                                            *[_cabi.ptr(t) for t in ties], int(loss), _cabi.ptr(fs), int(max_iter),
                                            ctypes.c_double(xtol), _cabi.ptr(f), _cabi.ptr(passes),
                                            _cabi.ptr(accepted), _cabi.ptr(status), None)
    return rc, x, f, passes, accepted, status


def raw_refine_ls(ctx, x, lb, ub, ties=None, max_iter=50, xtol=1e-6):
    """nmrfit_ctx_refine, or nmrfit_ctx_refine_tied with ``ties``: (status code, x, f, passes, accepted, status)."""
    B = x.shape[0]
    x, lb, ub = (np.array(a, dtype=np.float64, order='C') for a in (x, lb, ub))
    f = np.empty(B)
    passes, accepted, status = (np.empty(B, dtype=np.int32) for _ in range(3))
    outs = (int(max_iter), ctypes.c_double(xtol), _cabi.ptr(f), _cabi.ptr(passes), _cabi.ptr(accepted),
            _cabi.ptr(status), None)
    if ties is None:
        rc = _cabi.lib().nmrfit_ctx_refine(ctx._h, _cabi.ptr(x), _cabi.ptr(lb), _cabi.ptr(ub), *outs)
    else:
        m, s, o = (np.ascontiguousarray(t, dtype=d) for t, d in zip(ties, (np.int32, np.float64, np.float64)))
        rc = _cabi.lib().nmrfit_ctx_refine_tied(ctx._h, _cabi.ptr(x), _cabi.ptr(lb), _cabi.ptr(ub), _cabi.ptr(m),
                                                _cabi.ptr(s), _cabi.ptr(o), *outs)
    return rc, x, f, passes, accepted, status


def test_linear_refinement_is_nmrfit_ctx_refine_bit_for_bit():
    ws, us, vs, wts, X0, LB, UB = starts_for(4096, 6, (41, 42))
    with _cabi.Context(len(X0), 4096, 6) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        rc, *want = raw_refine_ls(ctx, X0, LB, UB)
        assert rc == 0
        rc, *got = raw_refine_loss(ctx, X0, LB, UB, _cabi.LOSS_LINEAR, None)
        assert rc == 0
        for a, b in zip(want, got):
            assert a.tobytes() == b.tobytes()
    ws, us, vs, wts, X0, LB, UB = tied_starts(4096, 6, (41, 42))
    ties = utils.batch_ties(synth.satellite_ties(6), len(X0), 6)[1]
    with _cabi.Context(len(X0), 4096, 6) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        rc, *want = raw_refine_ls(ctx, X0, LB, UB, ties=ties)
        assert rc == 0
        rc, *got = raw_refine_loss(ctx, X0, LB, UB, _cabi.LOSS_LINEAR, None, ties=ties)
        assert rc == 0
        for a, b in zip(want, got):
            assert a.tobytes() == b.tobytes()


def robust_stderr(x, w, u, v, wts, loss, c, lo, up, ties=None):
    return np.sqrt(np.diag(rr.covariance(x, w, u, v, wts, loss, c, lo, up, ties=ties)[0]))


def check_parity(ws, us, vs, wts, X0, LB, UB, loss, c, got, ties=None, max_iter=50):
    x, f, passes, accepted, status = got
    worst_f = worst_x = 0.0
    for b in range(len(X0)):
        rx, rf, rp, ra, rs = rr.refine(X0[b], LB[b], UB[b], ws[b], us[b], vs[b], wts[b], loss, c, max_iter=max_iter,
                                       ties=ties)
        assert same_outcome(status[b], rs), (b, status[b], rs, passes[b], rp)
        se = robust_stderr(rx, ws[b], us[b], vs[b], wts[b], loss, c, LB[b], UB[b], ties=ties)
        if ties is not None:
            se = se[ties.free()]
            ex = np.max(np.abs(x[b] - rx)[ties.free()] / se)
        else:
            ex = np.max(np.abs(x[b] - rx) / se)
        ef = abs(f[b] / rf - 1)
        assert ef <= 1e-12 and ex <= 1e-3, (b, ef, ex)
        worst_f, worst_x = max(worst_f, ef / 1e-12), max(worst_x, ex / 1e-3)
    return worst_f, worst_x


@pytest.mark.parametrize('loss', ROBUST)
def test_refinement_parity(loss):
    ws, us, vs, wts, X0, LB, UB = starts_for(4096, 6, (41, 42))
    c = C_OF[loss]
    with _cabi.Context(len(X0), 4096, 6) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        got = ctx.refine(X0, LB, UB, loss=loss, f_scale=c)
    assert np.all((got[0] >= LB) & (got[0] <= UB))
    w = check_parity(ws, us, vs, wts, X0, LB, UB, loss, c, got)
    print('refinement parity %s: worst f %.3g, x %.3g of tolerance; passes %s' % (loss, *w, got[2]))
    record('refine_parity_' + loss, dict(f=w[0], x=w[1], passes=got[2].tolist()))


def test_refinement_parity_with_ties():
    ws, us, vs, wts, X0, LB, UB = tied_starts(4096, 6, (41, 42))
    ties = synth.satellite_ties(6)
    c = C_OF['huber']
    arrays = utils.batch_ties(ties, len(X0), 6)[1]
    with _cabi.Context(len(X0), 4096, 6) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        got = ctx.refine(X0, LB, UB, ties=arrays, loss='huber', f_scale=c)
    w = check_parity(ws, us, vs, wts, X0, LB, UB, 'huber', c, got, ties=ties)
    print('tied refinement parity huber: worst f %.3g, x %.3g of tolerance' % w)
    record('refine_parity_huber_tied', dict(f=w[0], x=w[1]))


def impurity_problem(seed, area=None):
    data, true = synth.multiplet(4096, 6, seed=seed, noise=SIGMA, jitter=False)
    sats = rr.impurity(data, true, area=area)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    wts = utils.compute_weights(data.w, data.peaks)
    return data, true, lo, up, wts, sats


@pytest.mark.parametrize('bound', [False, True], ids=['free', 'binding_bound'])
def test_scipy_oracle_with_an_impurity(bound):
    data, true, lo, up, wts, sats = impurity_problem(7)
    c = C_OF['huber']
    if bound:                                          # the impurity pulls satellite 0's area up: cap it below
        up[6 + 3 * sats[0]] = true[6 + 3 * sats[0]] * 0.99
    x0 = np.clip(true, lo, up)
    with _cabi.Context(1, 4096, 6) as ctx:
        ctx.set_spectra(data.w[None], data.u[None], data.v[None], wts[None])
        x, f, passes, accepted, status = ctx.refine(x0[None], lo, up, loss='huber', f_scale=c, max_iter=100)
    assert status[0] in AT_MINIMUM
    sp = rr.scipy_fit(x0, lo, up, data.w, data.u, data.v, wts, 'huber', c)
    N = data.w.size
    cost_dev, cost_sp = f[0] ** 2 * N / 2, sp.cost
    se = robust_stderr(x[0], data.w, data.u, data.v, wts, 'huber', c, lo, up)
    dx = np.max(np.abs(x[0] - sp.x) / se)
    print('scipy oracle (%s): cost device %.15g scipy %.15g, max |dx|/se %.3g, passes %d'
          % ('bound' if bound else 'free', cost_dev, cost_sp, dx, passes[0]))
    record('scipy_oracle_' + ('bound' if bound else 'free'), dict(cost_device=cost_dev, cost_scipy=cost_sp, dx=dx))
    assert cost_dev <= cost_sp * (1 + 1e-10)
    assert dx <= 1e-2
    if bound:
        k = 6 + 3 * sats[0]
        assert x[0, k] == up[k] and sp.active_mask[k] == 1


def test_deterministic_alone_in_a_batch_and_in_fp32():
    ws, us, vs, wts, X0, LB, UB = starts_for(4096, 6, (45, 46))
    c = np.array([1.3e-4, 2.7e-4, 0.9e-4, 5e-4])

    def run(sl, cs, precision=_cabi.FP64):
        with _cabi.Context(len(X0[sl]), 4096, 6, precision=precision) as ctx:
            ctx.set_spectra(ws[sl], us[sl], vs[sl], wts[sl])
            out = ctx.refine(X0[sl], LB[sl], UB[sl], loss='huber', f_scale=cs)
            return out + (ctx.loss_moments(out[0], 'huber', cs), ctx.normal_equations_loss(out[0], 'huber', cs)[0])

    first = run(slice(None), c)
    f32 = run(slice(None), c, _cabi.FP32)
    for a, b in zip(first, f32):
        assert a.tobytes() == b.tobytes()
    for b in range(len(X0)):
        alone = run(slice(b, b + 1), c[b:b + 1])
        for a, one in zip(first, alone):
            assert a[b:b + 1].tobytes() == one.tobytes()


@pytest.fixture(scope='module')
def realisations():
    """256 white-noise realisations of the K16 setup, with and without the unmodelled line (area of one satellite),
    refined from the truth with least squares and with Huber at c = 1.345 sigma, each at the library's default max_iter
    (50 and utils.ROBUST_MAX_ITER).  Returns per case (X, stderr, passes)."""
    N, P, R = 4096, 6, 256
    base, true = synth.multiplet(N, P, seed=0, noise=0, jitter=False)
    wts = utils.compute_weights(base.w, base.peaks)
    lo, up = (np.array(a, dtype=np.float64) for a in base.generate_solution_bounds())
    rng = np.random.default_rng(11)
    noise_u, noise_v = rng.normal(0, SIGMA, (2, R, N))
    imp = synth.multiplet(N, P, seed=0, noise=0, jitter=False)[0]
    sats = rr.impurity(imp, true)
    ws, W = np.repeat(base.w[None], R, axis=0), np.repeat(wts[None], R, axis=0)
    X0 = np.repeat(true[None], R, axis=0)
    out = dict(true=true, sats=sats)
    c = C_OF['huber']
    with _cabi.Context(R, N, P) as ctx:
        for case, d in (('clean', base), ('impurity', imp)):
            ctx.set_spectra(ws, d.u[None] + noise_u, d.v[None] + noise_v, W)
            for loss in ('linear', 'huber'):
                X, f, passes, accepted, status = ctx.refine(X0, lo, up, loss=loss, f_scale=c,
                                                            max_iter=utils.default_max_iter(None, loss))
                assert np.all(np.isin(status, AT_MINIMUM)), np.bincount(status)
                H, M, g, ssr = ctx.normal_equations(X)
                mom = ctx.loss_moments(X, loss, c) if loss != 'linear' else [None] * R
                se = np.array([np.sqrt(np.diag(utils.covariance_from_normal(H[b], M[b], g[b], ssr[b], N, X[b], lo, up,
                                                                            moments=mom[b])[0])) for b in range(R)])
                out[case, loss] = (X, se, passes)
    return out


def test_huber_errors_are_calibrated(realisations):
    X, se, passes = realisations['clean', 'huber']
    ratio = X.std(axis=0, ddof=1) / se.mean(axis=0)
    Xi, sei, passes_i = realisations['impurity', 'huber']
    ratio_i = Xi.std(axis=0, ddof=1) / sei.mean(axis=0)
    print('huber calibration: spread / mean error %.3f..%.3f (clean), %.3f..%.3f (impurity); passes median %d, max '
          '%d, %d of %d past 50' % (ratio.min(), ratio.max(), ratio_i.min(), ratio_i.max(), np.median(passes),
                                   passes.max(), np.sum(passes > 50), passes.size))
    record('calibration', dict(clean=[float(ratio.min()), float(ratio.max())],
                               impurity=[float(ratio_i.min()), float(ratio_i.max())], ratio_clean=ratio.tolist(),
                               ratio_impurity=ratio_i.tolist(), passes_median=float(np.median(passes)),
                               passes_max=int(passes.max()), past_50=int(np.sum(passes > 50)),
                               passes_linear_max=int(realisations['clean', 'linear'][2].max()),
                               impurity_passes_median=float(np.median(passes_i)),
                               impurity_passes_max=int(passes_i.max()), impurity_past_50=int(np.sum(passes_i > 50))))
    assert np.all((ratio > 0.8) & (ratio < 1.2)), ratio


def test_huber_halves_the_satellite_bias(realisations):
    true, sats = realisations['true'], realisations['sats']
    idx = 6 + 3 * sats
    bias = {}
    for loss in ('linear', 'huber'):
        X = realisations['impurity', loss][0][:64]
        bias[loss] = X[:, idx].mean(axis=0) / true[idx] - 1
    ls, hu = np.max(np.abs(bias['linear'])), np.max(np.abs(bias['huber']))
    print('satellite-area bias (64 realisations): least squares %s, huber %s, worst ratio %.3f'
          % (np.round(100 * bias['linear'], 3), np.round(100 * bias['huber'], 3), hu / ls))
    record('bias', dict(linear=bias['linear'].tolist(), huber=bias['huber'].tolist(), ratio=hu / ls))
    assert hu <= 0.5 * ls


def test_fit_with_robust_refine_equals_fit_then_refine():
    data, true = synth.multiplet(2048, 6, seed=2)
    rr.impurity(data, true)
    lo, up = data.generate_solution_bounds()
    c = C_OF['huber']
    np.random.seed(3)
    a = core.fit(data, lo, up, summary=False, options=small_fit_options(refine=True, loss='huber', f_scale=c))
    np.random.seed(3)
    b = core.fit(data, lo, up, summary=False, options=small_fit_options())
    b.refine(loss='huber', f_scale=c)
    assert a.params.tobytes() == b.params.tobytes() and a.error == b.error
    assert a.loss == dict(name='huber', f_scale=c) and a.refine_info['loss'] == 'huber'
    assert a.refine_info['f_scale'] == c and a.refine_info['accepted'] >= 1
    assert a.refine_info['status'] in AT_MINIMUM              # the default max_iter of a robust loss reaches it
    with _cabi.Context(1, 2048, 6) as ctx:
        ctx.set_spectra(data.w[None], data.u[None], data.v[None], a.weights[None])
        ssr = ctx.normal_equations(a.params[None])[3]
        m = ctx.loss_moments(a.params[None], 'huber', c)
    assert a.error == pytest.approx(np.sqrt(ssr[0, 0] / 2048), rel=1e-12)
    assert a.refine_info['cost'] == m[0, 0]
    se = a.compute_uncertainties()
    info = a.uncertainty_info
    assert np.all(np.isfinite(se)) and info['loss'] == 'huber' and info['f_scale'] == c
    assert info['robust_factor'] > 0 and np.isfinite(a.area_fraction_stderr())
    with pytest.raises(NotImplementedError):
        a.compute_uncertainties(noise='correlated')
    # fit_batch: per-spectrum scales, against fit_batch then refine_batch
    datas = [synth.multiplet(2048, 6, seed=s)[0] for s in (5, 6, 7)]
    bounds = [d.generate_solution_bounds() for d in datas]
    lows, ups = [q[0] for q in bounds], [q[1] for q in bounds]
    cs = [1.2e-4, 2e-4, 3e-4]
    refined = core.fit_batch(datas, lows, ups, options=small_fit_options(rng='device', seed=3, refine=True,
                                                                         loss='cauchy', f_scale=cs))
    plain = core.fit_batch(datas, lows, ups, options=small_fit_options(rng='device', seed=3))
    utils.refine_batch(plain, loss='cauchy', f_scale=cs)
    for r, p, c in zip(refined, plain, cs):
        assert r.params.tobytes() == p.params.tobytes() and r.error == p.error
        assert r.refine_info['passes'] == p.refine_info['passes'] and r.loss == dict(name='cauchy', f_scale=c)
        assert r.refine_info['status'] in AT_MINIMUM
    utils.compute_uncertainties_batch(refined)
    for r in refined:
        assert r.uncertainty_info['loss'] == 'cauchy' and np.all(np.isfinite(r.stderr))


def test_library_refusals():
    data, true = synth.multiplet(512, 6, seed=1)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    wts = utils.compute_weights(data.w, data.peaks)
    x = np.clip(true, lo, up)[None].repeat(2, axis=0)
    lib = _cabi.lib()

    def last():
        return lib.nmrfit_last_error().decode()

    with _cabi.Context(2, 512, 6) as ctx:
        ctx.set_spectra(data.w[None].repeat(2, 0), data.u[None].repeat(2, 0), data.v[None].repeat(2, 0),
                        wts[None].repeat(2, 0))
        cases = ((dict(loss=9, f_scale=[1e-4, 1e-4]), 'unknown loss'),
                 (dict(loss=_cabi.LOSS_HUBER, f_scale=None), 'f_scale must be non-NULL'),
                 (dict(loss=_cabi.LOSS_HUBER, f_scale=[1e-4, 0.0]), 'spectrum 1: f_scale'),
                 (dict(loss=_cabi.LOSS_CAUCHY, f_scale=[np.nan, 1e-4]), 'spectrum 0: f_scale'),
                 (dict(loss=_cabi.LOSS_HUBER, f_scale=[1e-4, 1e-4], max_iter=0), 'max_iter'),
                 (dict(loss=_cabi.LOSS_HUBER, f_scale=[1e-4, 1e-4], ties=(np.zeros((2, 22), np.int32), None, None)),
                  'all NULL'))
        for kw, msg in cases:
            rc = raw_refine_loss(ctx, x, lo[None].repeat(2, 0), up[None].repeat(2, 0), **kw)[0]
            assert rc == -1 and msg in last(), (kw, last())
        xc = np.ascontiguousarray(x)
        out = np.empty((2, 5))
        assert lib.nmrfit_ctx_loss_moments(ctx._h, _cabi.ptr(xc), 5, None, _cabi.ptr(out), None) == -1
        assert 'unknown loss' in last()
        fs = np.array([1e-4, -1.0])
        assert lib.nmrfit_ctx_normal_equations_loss(ctx._h, _cabi.ptr(xc), _cabi.LOSS_SOFT_L1, _cabi.ptr(fs), None,
                                                    None, None, None) == -1
        assert 'spectrum 1: f_scale' in last()
        # LINEAR does not read f_scale
        assert lib.nmrfit_ctx_loss_moments(ctx._h, _cabi.ptr(xc), 0, None, _cabi.ptr(out), None) == 0
        with pytest.raises(ValueError, match='spectrum 1'):
            ctx.refine(x, lo, up, loss='huber', f_scale=[1e-4, 0.0])
        assert ctx.refine(x, lo, up, loss='huber', f_scale=1e-4, max_iter=200)[4][0] in AT_MINIMUM   # still works
    with _cabi.Context(1, 1024, 65) as ctx:
        D = 4 + 3 * 65
        assert raw_refine_loss(ctx, np.zeros((1, D)), -np.ones((1, D)), np.ones((1, D)), _cabi.LOSS_HUBER,
                               [1.0])[0] == -1
        assert 'at most 64 peaks' in last()
        out = np.empty((1, 5))
        assert lib.nmrfit_ctx_loss_moments(ctx._h, _cabi.ptr(np.zeros((1, D))), 1, _cabi.ptr(np.ones(1)),
                                           _cabi.ptr(out), None) == -1
        assert 'at most 64 peaks' in last()
