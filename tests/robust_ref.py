"""Reference robust refinement for the tests of the K16 passes (DESIGN K16): the robust normal equations, the loss
moments, K13's Levenberg-Marquardt rules on them (with or without ties) and Huber's covariance, in numpy with the sums
in long double on the residual and Jacobian of linearisation_ref.py.  Test infrastructure only."""
import numpy as np

import linearisation_ref as lin
from nmrfit_b200 import _cabi, utils

CONVERGED, STALLED, MAX_ITER, NONFINITE = 1, 2, 3, 4
LOSSES = ('linear', 'huber', 'soft_l1', 'cauchy')


def loss_terms(z, loss):
    """``(rho, rho', rho'')`` of ``loss`` at z >= 0 (scipy.optimize.least_squares' convention), in z's dtype."""
    z = np.asarray(z)
    one = np.ones_like(z)
    if loss == 'linear':
        return z.copy(), one, np.zeros_like(z)
    if loss == 'huber':
        inner = z <= 1
        s = np.sqrt(np.where(inner, one, z))
        return np.where(inner, z, 2 * s - 1), np.where(inner, one, 1 / s), np.where(inner, 0 * z, -0.5 / (s * s * s))
    if loss == 'soft_l1':
        t = 1 + z
        return 2 * (np.sqrt(t) - 1), 1 / np.sqrt(t), -0.5 / (t * np.sqrt(t))
    if loss == 'cauchy':
        t = 1 + z
        return np.log1p(z), 1 / t, -1 / (t * t)
    raise ValueError(loss)


def psi_prime(z, loss):
    """psi'(r) = rho'(z) + 2 z rho''(z) at z = (r/c)^2."""
    _, d1, d2 = loss_terms(z, loss)
    return d1 + 2 * z * d2


def _terms(x, w, u, v, weights, loss, c):
    res, A = lin.residual_jacobian(x, w, u, v)
    ld = np.longdouble
    r, A, wt, c = res.astype(ld), A.astype(ld), np.asarray(weights, dtype=ld), ld(c)
    z = (r / c) ** 2
    rho, d1, d2 = loss_terms(z, loss)
    return r, A, wt * wt, c, z, rho, d1, d2


def robust_pass(x, w, u, v, weights, loss, c):
    """``(H_rho, g_rho, s_rho)`` = (sum w^2 rho' A^T A, sum w^2 rho' res A, sum w^2 c^2 rho), summed in long double;
    for ``linear`` c is not used."""
    r, A, w2, c, z, rho, d1, _ = _terms(x, w, u, v, weights, loss, 1.0 if loss == 'linear' else c)
    k = w2 * d1
    H = A.T @ (k[:, None] * A)
    g = A.T @ (k * r)
    s = np.sum(w2 * r * r) if loss == 'linear' else np.sum(w2 * c * c * rho)
    return np.asarray(H, dtype=np.float64), np.asarray(g, dtype=np.float64), float(s)


def moments(x, w, u, v, weights, loss, c):
    """(cost, sum w^2 res^2, sum psi^2, sum psi', sum psi'^2) in long double, psi = rho' res."""
    r, _, w2, c, z, rho, d1, d2 = _terms(x, w, u, v, weights, loss, 1.0 if loss == 'linear' else c)
    psi, dpsi = d1 * r, d1 + 2 * z * d2
    cost = np.sum(w2 * r * r) if loss == 'linear' else np.sum(w2 * c * c * rho)
    return np.array([cost, np.sum(w2 * r * r), np.sum(psi * psi), np.sum(dpsi), np.sum(dpsi * dpsi)],
                    dtype=np.float64)


def refine(x, lb, ub, w, u, v, weights, loss, c, max_iter=50, xtol=1e-6, ties=None):
    """K13's bounded Levenberg-Marquardt, rule for rule as csrc/refine.cu runs it, on ``robust_pass`` (projected by
    ``ties.project`` over the free parameters when ``ties`` is given, as ties_ref does).  Returns
    ``(x, f, passes, accepted, status)`` with f = sqrt(s_rho / N)."""
    if ties is None:
        th = np.array(x, dtype=np.float64)
        lo, hi = np.asarray(lb, dtype=np.float64), np.asarray(ub, dtype=np.float64)
        expand = np.copy
    else:
        master, scale, offset = ties.arrays()
        free, lo, hi = _cabi.reduced_box(master, scale, offset, np.asarray(lb, dtype=np.float64),
                                         np.asarray(ub, dtype=np.float64))
        th = np.fmin(np.fmax(np.asarray(x, dtype=np.float64)[free], lo), hi)
        expand = ties.expand
    N, d = w.size, th.size

    def npass(t):
        H, g, s = robust_pass(expand(t), w, u, v, weights, loss, c)
        if ties is not None:
            H, _, g = ties.project(H, H, g)
        return H, g, s

    H, g, s = npass(th)
    passes, accepted = 1, 0
    if not (np.all(np.isfinite(H)) and np.all(np.isfinite(g)) and np.isfinite(s)):
        return expand(th), np.sqrt(s / N), passes, accepted, NONFINITE
    lam, status = 1e-3, 0
    while True:
        if passes >= max_iter:
            status = MAX_ITER
            break
        diag = np.diag(H)
        fr = ~((diag == 0) | ((th == lo) & (g > 0)) | ((th == hi) & (g < 0)))
        idx = np.nonzero(fr)[0]
        sc = 1.0 / np.sqrt(diag[idx])
        while True:
            A = sc[:, None] * H[np.ix_(idx, idx)] * sc[None, :] + lam * np.eye(idx.size)
            try:
                L = np.linalg.cholesky(A)
                break
            except np.linalg.LinAlgError:
                lam *= 10.0
                if lam > 1e16:
                    status = STALLED
                    break
        if status:
            break
        y = np.linalg.solve(L.T, np.linalg.solve(L, -(sc * g[idx])))
        tt = th.copy()
        tt[idx] = np.minimum(np.maximum(th[idx] + sc * y, lo[idx]), hi[idx])
        Ht, gt, st = npass(tt)
        passes += 1
        if np.isfinite(st) and st < s:
            small = np.all(np.abs(tt - th) * np.sqrt(diag * (N - d) / s) <= xtol)
            th, H, g, s = tt, Ht, gt, st
            lam = max(lam / 10.0, 1e-12)
            accepted += 1
            if small:
                status = CONVERGED
                break
        else:
            lam *= 10.0
            if lam > 1e16:
                status = STALLED
                break
    return expand(th), np.sqrt(s / N), passes, accepted, status


def covariance(x, w, u, v, weights, loss, c, lower, upper, ties=None):
    """Huber's covariance at ``x`` from the long-double normal equations and moments: ``covariance_from_normal`` with
    the moments of ``loss`` (None for linear, the least-squares computation)."""
    H, M, g, ssr = lin.normal_equations(x, w, u, v, weights, accumulate=np.longdouble)
    m = None if loss == 'linear' else moments(x, w, u, v, weights, loss, c)
    return utils.covariance_from_normal(H, M, g, ssr, w.size, x, lower, upper, ties=ties, moments=m)


def scipy_fit(x0, lb, ub, w, u, v, weights, loss, c, **kw):
    """The independent oracle: scipy ``least_squares(method='trf')`` on the unweighted residual with ``f_scale=c`` and
    a callable loss returning w^2 [rho, rho', rho''], whose cost is s_rho / 2 exactly.  Returns scipy's result."""
    from scipy.optimize import least_squares
    w2 = np.asarray(weights, dtype=np.float64) ** 2

    def rho(z):
        return w2 * np.array([np.asarray(t, dtype=np.float64) for t in loss_terms(z, loss)])

    opts = dict(method='trf', ftol=1e-15, xtol=1e-15, gtol=1e-15, max_nfev=2000, x_scale='jac')
    opts.update(kw)
    return least_squares(lambda x: lin.residual_jacobian(x, w, u, v)[0], x0,
                         jac=lambda x: lin.residual_jacobian(x, w, u, v)[1], bounds=(lb, ub), loss=rho, f_scale=c,
                         **opts)


def impurity(data, true, sat=0, area=None, offset=0.012, width=0.0015, r=0.9):
    """The unmodelled line of DESIGN K16's experiment added to ``data`` (in place): a pseudo-Voigt of ``width`` and
    mixing ``r`` at ``offset`` to the right of satellite ``sat`` of ``synth.multiplet``, with the area of that satellite
    unless ``area`` is given.  The line is added to the phased real part only (u, v rotated back by the true phase).
    Returns the satellites' indices in the peak list."""
    from oracle.nmrfit_oracle import voigt
    areas = true[6::3]
    sats = np.flatnonzero(areas < areas.mean())
    k = sats[sat]
    line = voigt(data.w, r, 0.0, width, true[5 + 3 * k] + offset, areas[k] if area is None else area)
    phi = true[0] + true[1] * np.arange(data.w.size) / data.w.size
    data.u = data.u + line * np.cos(phi)
    data.v = data.v - line * np.sin(phi)
    return sats
