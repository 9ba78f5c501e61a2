"""Reference tied refinement for the tests of csrc/refine.cu with a tie map (DESIGN K15): bounded Levenberg-Marquardt
over the free parameters theta of x = T theta + c, in numpy on the long-double normal equations of
linearisation_ref.py, rule for rule as the kernel runs it and step for step as refine_ref.refine.  Test
infrastructure only."""
import numpy as np

import linearisation_ref as lin
from nmrfit_b200 import _cabi

CONVERGED, STALLED, MAX_ITER, NONFINITE = 1, 2, 3, 4


def start(ties, x, lb, ub):
    """The library's start: the free entries of ``x`` clipped into the reduced box (NaN to its lower end), then
    expanded.  Returns ``(theta, lo, hi)``."""
    master, scale, offset = ties.arrays()
    free, lo, hi = _cabi.reduced_box(master, scale, offset, np.asarray(lb, dtype=np.float64),
                                     np.asarray(ub, dtype=np.float64))
    return np.fmin(np.fmax(np.asarray(x, dtype=np.float64)[free], lo), hi), lo, hi


def refine(ties, x, lb, ub, w, u, v, weights, max_iter=50, xtol=1e-6):
    """Tied bounded Levenberg-Marquardt on ``linearisation_ref.normal_equations(..., np.longdouble)``, projected by
    ``ties.project`` (the kernel's summation order).  Returns ``(x, f, passes, accepted, status)`` with x expanded and
    f = sqrt(s/N)."""
    th, lo, hi = start(ties, x, lb, ub)
    N, d = w.size, th.size

    def npass(t):
        H, M, g, ssr = lin.normal_equations(ties.expand(t), w, u, v, weights, accumulate=np.longdouble)
        Ht, _, gt = ties.project(H, M, g)
        return Ht, gt, ssr[0]

    H, g, s = npass(th)
    passes, accepted = 1, 0
    if not (np.all(np.isfinite(H)) and np.all(np.isfinite(g)) and np.isfinite(s)):
        return ties.expand(th), np.sqrt(s / N), passes, accepted, NONFINITE
    lam, status = 1e-3, 0
    while True:
        if passes >= max_iter:
            status = MAX_ITER
            break
        diag = np.diag(H)
        free = ~((diag == 0) | ((th == lo) & (g > 0)) | ((th == hi) & (g < 0)))
        idx = np.nonzero(free)[0]
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
    return ties.expand(th), np.sqrt(s / N), passes, accepted, status
