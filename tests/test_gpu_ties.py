"""Tied refinement on the GPU (nmrfit_ctx_refine_tied, DESIGN K15) against the numpy restatement (ties_ref) and scipy
on the reduced problem: the identity map against the untied refinement, exactness of fixed and linked entries,
determinism, the calibration of the tied errors, the library's refusals and the fit / fit_batch paths."""
import ctypes

import numpy as np
import pytest

from nmrfit_b200 import _cabi, core, synth, utils
import linearisation_ref as lin
import ties_ref as tr
from test_gpu_refine import (AT_MINIMUM, device_refine, multiplet, same_outcome, small_fit_options,
                             starts_for)

pytestmark = pytest.mark.gpu


def tied_refine(ws, us, vs, wts, X, LB, UB, ties, precision=_cabi.FP64, **kw):
    B, N = ws.shape
    arrays = ties if isinstance(ties, tuple) else utils.batch_ties(ties, B, (X.shape[1] - 4) // 3)[1]
    with _cabi.Context(B, N, (X.shape[1] - 4) // 3, precision=precision) as ctx:
        ctx.set_spectra(ws, us, vs, wts)
        return ctx.refine(X, LB, UB, ties=arrays, **kw)


@pytest.mark.parametrize('N,P,nonuniform', [(4096, 6, False), (3000, 36, False), (1000, 64, False),
                                            (4096, 6, True)], ids=['4096x6', '3000x36', '1000x64', 'nonuniform'])
def test_identity_map_is_the_untied_refinement(N, P, nonuniform):
    swarm = P <= 36
    ws, us, vs, wts, X0, LB, UB = starts_for(N, P, (41, 42) if P <= 6 else (41,), nonuniform, swarm,
                                             0.01 if swarm else 1e-3)
    kw = dict(max_iter=200 if P == 64 else 50)
    a = device_refine(ws, us, vs, wts, X0, LB, UB, **kw)
    b = tied_refine(ws, us, vs, wts, X0, LB, UB, utils.Ties(P), **kw)
    for u, t in zip(a, b):
        assert u.tobytes() == t.tobytes()


def tied_starts(N, P, seeds, nonuniform=False, swarm=True, scale=0.01):
    """Spectra whose true vectors satisfy ``ties`` (multiplet without jitter), refined from swarm answers and from
    the true vector perturbed by ``scale``."""
    datas, trues = zip(*[synth.multiplet(N, P, seed=s, jitter=False) for s in seeds])
    if nonuniform:
        rng = np.random.default_rng(5)
        for d in datas:
            d.w = d.w + rng.uniform(-0.3, 0.3, N) * (d.w[1] - d.w[0])
    bounds = [d.generate_solution_bounds() for d in datas]
    LB = np.array([b[0] for b in bounds], dtype=np.float64)
    UB = np.array([b[1] for b in bounds], dtype=np.float64)
    wts = np.stack([utils.compute_weights(d.w, d.peaks) for d in datas])
    rng = np.random.default_rng(N + P)
    X = [np.clip(np.array(trues) * (1 + scale * rng.standard_normal((len(seeds), 4 + 3 * P))), LB, UB)]
    copies = 1
    if swarm:
        fits = core.fit_batch(datas, LB, UB, options=small_fit_options(rng='device', seed=1))
        X.insert(0, np.stack([f.params for f in fits]))
        wts = np.stack([f.weights for f in fits])
        copies = 2
    ws, us, vs = (np.stack([getattr(d, k) for d in datas] * copies) for k in ('w', 'u', 'v'))
    return (ws, us, vs, np.concatenate([wts] * copies), np.concatenate(X), np.concatenate([LB] * copies),
            np.concatenate([UB] * copies))


def tied_stderr(t, x, w, u, v, wts, lo, up):
    H, M, g, ssr = lin.normal_equations(x, w, u, v, wts, accumulate=np.longdouble)
    return np.sqrt(np.diag(utils.covariance_from_normal(H, M, g, ssr, w.size, x, lo, up, ties=t)[0]))


def fixed_phases_equal_widths(P):
    g = synth.TRUE_GLOBALS
    t = utils.Ties(P).fix('p0', g['p0']).fix('p1', g['p1'])
    for k in range(1, P):
        t.link(('width', k), ('width', 0))
    return t


CASES = [('satellites_4096x6', 4096, 6, False, True, 0.01, 50), ('satellites_3000x36', 3000, 36, False, True, 0.01, 50),
         ('phases_widths_1000x64', 1000, 64, False, False, 1e-3, 200),
         ('satellites_nonuniform', 4096, 6, True, True, 0.01, 50)]


@pytest.mark.parametrize('name,N,P,nonuniform,swarm,scale,max_iter', CASES, ids=[c[0] for c in CASES])
def test_parity_with_reference(name, N, P, nonuniform, swarm, scale, max_iter):
    seeds = (41, 42) if P <= 6 else (41,)
    if 'phases' in name:                                 # any multiplet satisfies these ties: P need not be 6k
        ws, us, vs, wts, X0, LB, UB = starts_for(N, P, seeds, nonuniform, swarm, scale)
        t = fixed_phases_equal_widths(P)
    else:
        ws, us, vs, wts, X0, LB, UB = tied_starts(N, P, seeds, nonuniform, swarm, scale)
        t = synth.satellite_ties(P)
    x, f, passes, accepted, status = tied_refine(ws, us, vs, wts, X0, LB, UB, t, max_iter=max_iter)
    master, scale_, offset = t.arrays()
    free = t.free()
    group, _ = t.groups()
    linked = (master >= 0) & (master != np.arange(master.size))
    worst_f = worst_x = 0.0
    for b in range(len(X0)):
        # exactness: fixed entries are their values, dependents numpy's a * theta + c
        assert x[b, master == -1].tobytes() == offset[master == -1].tobytes()
        assert x[b, linked].tobytes() == (scale_[linked] * x[b, free][group[linked]] + offset[linked]).tobytes()
        rx, rf, rp, ra, rs = tr.refine(t, X0[b], LB[b], UB[b], ws[b], us[b], vs[b], wts[b], max_iter=max_iter)
        assert same_outcome(status[b], rs), (b, status[b], rs, passes[b], rp)
        se = tied_stderr(t, rx, ws[b], us[b], vs[b], wts[b], LB[b], UB[b])
        ef, ex = abs(f[b] / rf - 1), np.max(np.abs(x[b] - rx)[free] / se[free])
        assert ef <= 1e-12 and ex <= 1e-3, (b, ef, ex)
        worst_f, worst_x = max(worst_f, ef / 1e-12), max(worst_x, ex / 1e-3)
        print('%s start %d: passes %d (reference %d), status %d' % (name, b, passes[b], rp, status[b]))
    print('%s: worst objective error/tolerance %.3g, parameter error/tolerance %.3g' % (name, worst_f, worst_x))


@pytest.mark.parametrize('binding', [False, True], ids=['interior', 'dependent_box_binds'])
def test_against_scipy_on_the_reduced_problem(binding):
    """scipy's trf on theta within the reduced box.  With ``binding`` the upper satellite's area is linked to the
    lower one's with its own upper bound below the optimum, so the reduced box is set by the dependent's box."""
    from scipy.optimize import least_squares
    data, true = synth.multiplet(4096, 6, seed=43, jitter=False)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    t = synth.satellite_ties(6)
    dep = t.index('area', 4)                             # linked to area(0)
    if binding:
        up[dep] = 0.8 * true[dep]
    x0 = np.clip(true * (1 + 0.01 * np.random.default_rng(1).standard_normal(true.size)), lo, up)
    wts = utils.compute_weights(data.w, data.peaks)
    x, f, passes, accepted, status = tied_refine(data.w[None], data.u[None], data.v[None], wts[None], x0[None],
                                                 lo[None], up[None], t)
    assert status[0] in AT_MINIMUM
    master, scale, offset = t.arrays()
    free, rlo, rhi = _cabi.reduced_box(master, scale, offset, lo, up)
    T, c = t.matrix()

    def fun(th):
        return wts * lin.residual_jacobian(t.expand(th), data.w, data.u, data.v)[0]

    def jac(th):
        return (wts[:, None] * lin.residual_jacobian(t.expand(th), data.w, data.u, data.v)[1]) @ T

    th0 = np.clip(x0[free], rlo, rhi)
    sp = least_squares(fun, th0, jac=jac, bounds=(rlo, rhi), method='trf', x_scale='jac', ftol=1e-15, xtol=1e-15,
                       gtol=1e-15)
    f_sp = np.sqrt(np.mean(fun(sp.x) ** 2))
    assert f[0] <= f_sp * (1 + 1e-9), (f[0], f_sp)
    se = tied_stderr(t, x[0], data.w, data.u, data.v, wts, lo, up)[free]
    k = list(free).index(t.index('area', 0))
    if binding:
        assert x[0, free][k] == rhi[k] and rhi[k] == (up[dep] - offset[dep]) / scale[dep]
    inner = np.arange(free.size) != (k if binding else -1)
    assert np.all(np.abs(x[0, free] - sp.x)[inner] <= 1e-3 * se[inner]), np.abs(x[0, free] - sp.x) / se


def test_deterministic_mixed_maps_and_fp32():
    ws, us, vs, wts, X0, LB, UB = tied_starts(4096, 6, (45, 46))
    maps = [synth.satellite_ties(6), fixed_phases_equal_widths(6), None, synth.satellite_ties(6).fix('r', 0.55)]
    first = tied_refine(ws, us, vs, wts, X0, LB, UB, maps)
    again = tied_refine(ws, us, vs, wts, X0, LB, UB, maps)
    f32 = tied_refine(ws, us, vs, wts, X0, LB, UB, maps, precision=_cabi.FP32)
    for a, b, c in zip(first, again, f32):
        assert a.tobytes() == b.tobytes() and a.tobytes() == c.tobytes()
    for b in range(len(X0)):
        s = slice(b, b + 1)
        alone = tied_refine(ws[s], us[s], vs[s], wts[s], X0[s], LB[s], UB[s], [maps[b]])
        for a, one in zip(first, alone):
            assert a[s].tobytes() == one.tobytes()


def calibration(noise):
    N, P, R, sigma = 4096, 6, 256, 1e-4
    base, true = synth.multiplet(N, P, seed=0, noise=0)
    lo, up = (np.array(a, dtype=np.float64) for a in base.generate_solution_bounds())
    rng = np.random.default_rng(1)
    if noise == 'white':
        nu, nv = rng.normal(0, sigma, (R, N)), rng.normal(0, sigma, (R, N))
    else:
        nu, nv = synth.processed_noise(N, sigma, n_realisations=R, seed=1)
    t = synth.satellite_ties(P)
    tied, untied = [], []
    for ties in (t, None):
        fits = []
        for r in range(R):
            d, _ = synth.multiplet(N, P, seed=0, noise=0)
            d.u, d.v = base.u + nu[r], base.v + nv[r]
            f = utils.FitUtility(d, lo, up, summary=False)
            f.weights = utils.compute_weights(d.w, d.peaks)
            f.params, f.error = true.copy(), 1.0
            fits.append(f)
        utils.refine_batch(fits, ties=ties)
        utils.compute_uncertainties_batch(fits, noise=noise)
        (tied if ties is not None else untied).extend(fits)
    return t, tied, untied


@pytest.mark.parametrize('noise', ['white', 'correlated'])
def test_tied_errors_are_calibrated(noise):
    t, tied, untied = calibration(noise)
    assert all(f.refine_info['status'] in AT_MINIMUM for f in tied)
    free = t.free()
    X = np.stack([f.params for f in tied])[:, free]
    se = np.stack([f.stderr for f in tied])[:, free]
    ratio = X.std(axis=0, ddof=1) / se.mean(axis=0)
    print('calibration (%s): spread / tied error %s' % (noise, np.round(ratio, 3)))
    assert np.all((ratio > 0.8) & (ratio < 1.2)), ratio
    assert all(f.uncertainty_info['dof'] == 4096 - free.size for f in tied)
    ft = np.mean([f.area_fraction_stderr() for f in tied])
    fu = np.mean([f.area_fraction_stderr() for f in untied])
    print('calibration (%s): area fraction error tied / untied = %.4f' % (noise, ft / fu))
    assert ft < fu


def raw_refine_tied(ctx, x, lb, ub, m, s, o, max_iter=50, xtol=1e-6):
    """The library call itself, past the checks Context.refine makes first."""
    x, lb, ub, s, o = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, lb, ub, s, o))
    m = np.ascontiguousarray(m, dtype=np.int32)
    return _cabi.lib().nmrfit_ctx_refine_tied(ctx._h, _cabi.ptr(x), _cabi.ptr(lb), _cabi.ptr(ub), _cabi.ptr(m),
                                              _cabi.ptr(s), _cabi.ptr(o), int(max_iter), ctypes.c_double(xtol),
                                              None, None, None, None, None)


def test_library_refusals():
    data, true = synth.multiplet(512, 6, seed=1, jitter=False)
    lo, up = (np.array(a, dtype=np.float64) for a in data.generate_solution_bounds())
    wts = utils.compute_weights(data.w, data.peaks)
    D = true.size
    with _cabi.Context(1, 512, 6) as ctx:
        ctx.set_spectra(data.w[None], data.u[None], data.v[None], wts[None])

        def ident():
            return np.arange(D, dtype=np.int32), np.ones(D), np.zeros(D)
        cases = []
        m, s, o = ident(); m[5] = 22; cases.append(((m, s, o), 'out of range'))
        m, s, o = ident(); m[5], m[4] = 4, 7; cases.append(((m, s, o), 'no chains'))
        m, s, o = ident(); m[5], m[4] = 4, -1; cases.append(((m, s, o), 'is fixed'))
        m, s, o = ident(); m[5], s[5] = 4, 0.0; cases.append(((m, s, o), 'non-zero'))
        m, s, o = ident(); m[5], s[5] = 4, np.inf; cases.append(((m, s, o), 'non-zero'))
        m, s, o = ident(); m[5], o[5] = -1, np.nan; cases.append(((m, s, o), 'offset is not finite'))
        m, s, o = ident(); m[6], s[6] = 9, -1.0; cases.append(((m, s, o), 'parameter 6 and its master 9'))
        for (m, s, o), msg in cases:
            assert raw_refine_tied(ctx, true[None], lo[None], up[None], m, s, o) == -1
            assert msg in _cabi.lib().nmrfit_last_error().decode(), (msg, _cabi.lib().nmrfit_last_error())
        assert raw_refine_tied(ctx, true[None], lo[None], up[None], *ident(), max_iter=0) == -1
        t = synth.satellite_ties(6)
        x, f, passes, accepted, status = ctx.refine(true[None] * 1.001, lo, up, ties=t.arrays())
        assert status[0] in AT_MINIMUM                   # the context still works
    with _cabi.Context(1, 10, 6) as ctx:                 # d = 10 free parameters, N = 10 < D = 22
        ctx.set_spectra(data.w[None, :10], data.u[None, :10], data.v[None, :10], wts[None, :10])
        m, s, o = synth.satellite_ties(6).arrays()
        m[:2] = -1
        o[:2] = true[:2]
        assert raw_refine_tied(ctx, true[None], lo[None], up[None], m, s, o) == -1
        assert 'more points than free parameters' in _cabi.lib().nmrfit_last_error().decode()


def test_fit_with_ties_equals_fit_then_refine():
    data, true = synth.multiplet(2048, 6, seed=2, jitter=False)
    lo, up = data.generate_solution_bounds()
    t = synth.satellite_ties(6)
    np.random.seed(3)
    a = core.fit(data, lo, up, summary=False, options=small_fit_options(refine=True, ties=t))
    np.random.seed(3)
    b = core.fit(data, lo, up, summary=False, options=small_fit_options())
    b.refine(ties=t)
    assert a.params.tobytes() == b.params.tobytes() and a.error == b.error and a.ties is t
    a.compute_uncertainties()
    assert a.uncertainty_info['dof'] == 2048 - t.free().size
    assert np.isfinite(a.area_fraction_stderr())
    datas = [synth.multiplet(2048, 6, seed=s, jitter=False)[0] for s in (5, 6, 7)]
    bounds = [d.generate_solution_bounds() for d in datas]
    lows, ups = [b[0] for b in bounds], [b[1] for b in bounds]
    per = [t, None, synth.satellite_ties(6).fix('yoff', 0.0)]
    refined = core.fit_batch(datas, lows, ups, options=small_fit_options(rng='device', seed=3, refine=True,
                                                                          ties=per))
    plain = core.fit_batch(datas, lows, ups, options=small_fit_options(rng='device', seed=3))
    utils.refine_batch(plain, ties=per)
    for r, p in zip(refined, plain):
        assert r.params.tobytes() == p.params.tobytes() and r.error == p.error
        assert r.refine_info['passes'] == p.refine_info['passes'] and r.ties is p.ties
    with pytest.raises(ValueError, match='refine'):
        core.fit(data, lo, up, summary=False, options=small_fit_options(ties=t))
    with pytest.raises(NotImplementedError):
        core.fit(data, lo, up, fit_im=True, summary=False, options=small_fit_options(refine=True, ties=t))
