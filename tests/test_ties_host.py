"""Host side of fixed and linked parameters (DESIGN K15): the checks of ``utils.Ties`` and ``_cabi.check_ties``, the
projection of the normal equations, the expansion, the covariance of the tied model and the numpy tied refinement
(ties_ref) against the untied one (no GPU)."""
import numpy as np
import pytest

from nmrfit_b200 import _cabi, synth, utils
import linearisation_ref as lin
import refine_ref as rr
import ties_ref as tr


def spectrum(N=2048, seed=3):
    d, true = synth.multiplet(N, 6, seed=seed, jitter=False)   # the satellite ties hold for its true vector
    lo, up = (np.array(a, dtype=np.float64) for a in d.generate_solution_bounds())
    return d, true, lo, up, utils.compute_weights(d.w, d.peaks)


def test_ties_refuses_malformed_maps():
    t = utils.Ties(6)
    for call, msg in ((lambda: t.link(5, 5), 'itself'),
                      (lambda: t.link(5, 22), 'index must be'),
                      (lambda: t.link(5, -1), 'index must be'),
                      (lambda: t.link(5, 4, scale=0.0), 'non-zero'),
                      (lambda: t.link(5, 4, scale=np.inf), 'finite'),
                      (lambda: t.link(5, 4, offset=np.nan), 'offset'),
                      (lambda: t.fix(0, np.nan), 'offset'),
                      (lambda: t.index('area', 6), 'peak must be'),
                      (lambda: t.index('p0', 1), 'global'),
                      (lambda: t.index('height', 0), 'unknown')):
        with pytest.raises(ValueError, match=msg):
            call()
    t.link(5, 4)
    with pytest.raises(ValueError, match='no chains'):
        t.link(7, 5)                                     # 5 is linked
    with pytest.raises(ValueError, match='no chains'):
        t.link(4, 8)                                     # 4 is a master
    with pytest.raises(ValueError, match='cannot be fixed'):
        t.fix(4, 1.0)
    t.fix(0, 0.25)
    with pytest.raises(ValueError, match='is fixed'):
        t.link(1, 0)
    assert t.index(('area', 2)) == 12 and t.index('yoff') == 3


def raw_map(D):
    return np.arange(D, dtype=np.int32), np.ones(D), np.zeros(D)


def test_check_ties_refuses_what_the_library_refuses():
    d, true, lo, up, wts = spectrum()
    D, N, P = true.size, d.w.size, 6
    cases = []
    m, s, o = raw_map(D); m[5] = 22; cases.append(((m, s, o), 'out of range'))
    m, s, o = raw_map(D); m[5] = -2; cases.append(((m, s, o), 'out of range'))
    m, s, o = raw_map(D); m[5], m[4] = 4, 7; cases.append(((m, s, o), 'no chains'))
    m, s, o = raw_map(D); m[5], m[4] = 4, -1; cases.append(((m, s, o), 'is fixed'))
    m, s, o = raw_map(D); m[5], s[5] = 4, 0.0; cases.append(((m, s, o), 'non-zero'))
    m, s, o = raw_map(D); m[5], s[5] = 4, np.nan; cases.append(((m, s, o), 'non-zero'))
    m, s, o = raw_map(D); m[5], o[5] = -1, np.inf; cases.append(((m, s, o), 'offset is not finite'))
    m, s, o = raw_map(D); m[5], o[5] = 4, np.nan; cases.append(((m, s, o), 'offset is not finite'))
    # a dependent whose box, mapped through a negative scale, misses its master's box
    m, s, o = raw_map(D); m[6], s[6] = 9, -1.0; cases.append(((m, s, o), 'parameter 6 and its master 9'))
    # intervals that overlap in one point only
    m, s, o = raw_map(D); m[12] = 9
    point = lo.copy(); point[12] = up[9]
    cases.append(((m, s, o), 'parameter 12 and its master 9: the reduced box is empty', point))
    for case in cases:
        (mm, ss, oo), msg = case[:2]
        with pytest.raises(ValueError, match=msg):
            _cabi.check_ties(mm, ss, oo, case[2] if len(case) > 2 else lo, up, 1, N, P)
    # a negative scale whose mapped box does overlap: the interval is swapped
    m, s, o = raw_map(D); m[18], s[18], o[18] = 6, -1.0, up[18] + lo[6] + 0.5 * (up[6] - lo[6])
    free, rlo, rhi = _cabi.reduced_box(m, s, o, lo, up)
    k = list(free).index(6)
    assert rlo[k] == max(lo[6], (up[18] - o[18]) / -1.0) and rhi[k] == min(up[6], (lo[18] - o[18]) / -1.0)
    assert rhi[k] > rlo[k]
    with pytest.raises(ValueError, match='degrees of freedom'):
        _cabi.check_ties(*raw_map(D), lo, up, 1, D, P)
    m, s, o = raw_map(D); m[4:] = -1; o[4:] = true[4:]
    _cabi.check_ties(m, s, o, lo, up, 1, 5, P)          # d = 4 < N = 5
    with pytest.raises(ValueError, match='shape'):
        _cabi.check_ties(*raw_map(D - 1), lo, up, 1, N, P)


def test_projection_equals_the_reduced_model():
    d, true, lo, up, wts = spectrum()
    t = synth.satellite_ties(6).fix('p1', true[1])
    x = t.expand(true[t.free()])
    H, M, g, ssr = lin.normal_equations(x, d.w, d.u, d.v, wts, accumulate=np.longdouble)
    Ht, Mt, gt = t.project(H, M, g)
    T, c = t.matrix()
    res, A = lin.residual_jacobian(x, d.w, d.u, d.v)
    At = (A @ T).astype(np.longdouble)
    w2 = np.asarray(wts, dtype=np.longdouble) ** 2
    X = np.asarray(At.T @ (w2[:, None] * At), dtype=np.float64)
    tol = 1e-12 * np.sqrt(np.outer(np.diag(X), np.diag(X)))
    assert np.all(np.abs(Ht - X) <= tol), np.max(np.abs(Ht - X) / tol)
    gX = np.asarray(At.T @ (w2 * np.asarray(res, dtype=np.longdouble)), dtype=np.float64)
    assert np.all(np.abs(gt - gX) <= 1e-12 * np.sqrt(np.diag(X) * ssr[0]))
    I = utils.Ties(6)
    for a, b in zip(I.project(H, M, g), (H, M, g)):
        assert a.tobytes() == b.tobytes()


def test_expansion_is_numpys_and_stays_in_the_box():
    d, true, lo, up, wts = spectrum()
    t = synth.satellite_ties(6)
    t.link(('area', 3), ('area', 2), scale=-0.5, offset=0.01)
    master, scale, offset = t.arrays()
    free, rlo, rhi = _cabi.reduced_box(master, scale, offset, lo, up)
    linked = (master >= 0) & (master != np.arange(true.size))
    group, _ = t.groups()
    for theta in (rlo, rhi, 0.5 * (rlo + rhi)):
        x = t.expand(theta)
        assert x[free].tobytes() == theta.tobytes()
        want = scale[linked] * theta[group[linked]] + offset[linked]
        assert x[linked].tobytes() == want.tobytes()
        # dependents leave their own box at a reduced bound only by the rounding of a * t + c
        slack = 4 * np.spacing(np.abs(x) + np.abs(offset))
        assert np.all(x[linked] >= lo[linked] - slack[linked]) and np.all(x[linked] <= up[linked] + slack[linked])


def test_covariance_of_the_tied_model():
    d, true, lo, up, wts = spectrum()
    H, M, g, ssr = lin.normal_equations(true, d.w, d.u, d.v, wts, accumulate=np.longdouble)
    C0, i0 = utils.covariance_from_normal(H, M, g, ssr, d.w.size, true, lo, up)
    C1, i1 = utils.covariance_from_normal(H, M, g, ssr, d.w.size, true, lo, up, ties=utils.Ties(6))
    assert C0.tobytes() == C1.tobytes() and i0['dof'] == i1['dof']
    assert i0['at_bound'].tobytes() == i1['at_bound'].tobytes() and i0['sigma'] == i1['sigma']
    t = synth.satellite_ties(6).fix('p0', true[0])
    x = t.expand(true[t.free()])
    H, M, g, ssr = lin.normal_equations(x, d.w, d.u, d.v, wts, accumulate=np.longdouble)
    C, info = utils.covariance_from_normal(H, M, g, ssr, d.w.size, x, lo, up, ties=t)
    assert info['dof'] == d.w.size - t.free().size
    assert np.all(C[0] == 0) and np.all(C[:, 0] == 0)
    se = np.sqrt(np.diag(C))
    master, scale, _ = t.arrays()
    for j in range(1, true.size):
        assert se[j] == abs(scale[j]) * se[master[j]] or master[j] == j
    assert np.all(se[t.free()[1:]] > 0)


def test_reference_with_the_identity_map_is_the_untied_reference():
    d, true, lo, up, wts = spectrum(seed=5)
    x0 = np.clip(true * (1 + 0.01 * np.random.default_rng(2).standard_normal(true.size)), lo, up)
    a = rr.refine(x0, lo, up, d.w, d.u, d.v, wts)
    b = tr.refine(utils.Ties(6), x0, lo, up, d.w, d.u, d.v, wts)
    assert a[0].tobytes() == b[0].tobytes() and a[1:] == b[1:]


def test_reference_tied_refinement_converges_to_a_tied_point():
    d, true, lo, up, wts = spectrum(N=4096, seed=0)
    t = synth.satellite_ties(6)
    x0 = np.clip(true * (1 + 0.01 * np.random.default_rng(3).standard_normal(true.size)), lo, up)
    x, f, passes, accepted, status = tr.refine(t, x0, lo, up, d.w, d.u, d.v, wts)
    assert status in (tr.CONVERGED, tr.STALLED) and accepted >= 1
    assert x.tobytes() == t.expand(x[t.free()]).tobytes()
    fu = rr.refine(x0, lo, up, d.w, d.u, d.v, wts)[1]
    assert fu <= f                                       # the constrained optimum is no better than the free one


def test_ties_need_refine_and_fit_im_stays_refused():
    d, true, lo, up, wts = spectrum(N=512, seed=1)
    f = utils.FitUtility(d, lo, up, summary=False, options={'ties': synth.satellite_ties(6)})
    with pytest.raises(ValueError, match='refine'):
        f.fit()
    f = utils.FitUtility(d, lo, up, fit_im=True, summary=False,
                         options={'refine': True, 'ties': synth.satellite_ties(6)})
    with pytest.raises(NotImplementedError):
        f.fit()
    from nmrfit_b200 import core
    with pytest.raises(ValueError, match='refine'):
        core.fit_batch([d], [lo], [up], options={'ties': synth.satellite_ties(6)})


def test_context_refine_checks_ties_before_any_cuda_call(monkeypatch):
    def no_library():
        raise AssertionError('the library was called')
    monkeypatch.setattr(_cabi, 'lib', no_library)
    ctx = object.__new__(_cabi.Context)
    ctx._h = None
    ctx.B, ctx.N, ctx.P, ctx.D = 2, 100, 2, 10
    m, s, o = raw_map(10)
    m[5] = 12
    with pytest.raises(ValueError, match='spectrum 0, parameter 5: master 12 is out of range'):
        ctx.refine(np.zeros((2, 10)), -np.ones(10), np.ones(10), ties=(m, s, o))
    m = np.stack([np.arange(10), np.r_[np.arange(9), 7]])
    m[1, 7] = -1
    with pytest.raises(ValueError, match='spectrum 1, parameter 9: its master 7 is fixed'):
        ctx.refine(np.zeros((2, 10)), -np.ones(10), np.ones(10), ties=(m, s, o))
