"""Reference refinement for the tests of csrc/refine.cu (DESIGN K13): bounded Levenberg-Marquardt in numpy on the
long-double normal equations of linearisation_ref.py, rule for rule as the kernel runs it.  Test infrastructure only."""
import numpy as np

import linearisation_ref as lin


CONVERGED, STALLED, MAX_ITER, NONFINITE = 1, 2, 3, 4


def refine(x, lb, ub, w, u, v, weights, max_iter=50, xtol=1e-6):
    """Bounded Levenberg-Marquardt (DESIGN K13) on ``linearisation_ref.normal_equations(..., np.longdouble)``, rule
    for rule as csrc/refine.cu runs it.  Returns ``(x, f, passes, accepted, status)`` with f = sqrt(s/N)."""
    x, lb, ub = (np.array(a, dtype=np.float64) for a in (x, lb, ub))
    N, D = w.size, x.size

    def npass(at):
        H, _, g, ssr = lin.normal_equations(at, w, u, v, weights, accumulate=np.longdouble)
        return H, g, ssr[0]

    H, g, s = npass(x)
    passes, accepted = 1, 0
    if not (np.all(np.isfinite(H)) and np.all(np.isfinite(g)) and np.isfinite(s)):
        return x, np.sqrt(s / N), passes, accepted, NONFINITE
    lam, status = 1e-3, 0
    while True:
        if passes >= max_iter:
            status = MAX_ITER
            break
        diag = np.diag(H)
        free = ~((diag == 0) | ((x == lb) & (g > 0)) | ((x == ub) & (g < 0)))
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
        xt = x.copy()
        xt[idx] = np.minimum(np.maximum(x[idx] + sc * y, lb[idx]), ub[idx])
        Ht, gt, st = npass(xt)
        passes += 1
        if np.isfinite(st) and st < s:
            small = np.all(np.abs(xt - x) * np.sqrt(diag * (N - D) / s) <= xtol)
            x, H, g, s = xt, Ht, gt, st
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
    return x, np.sqrt(s / N), passes, accepted, status
