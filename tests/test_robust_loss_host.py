"""The robust losses of DESIGN K16 (nmrfit_b200/csrc/robust_loss.cuh compiled for the host, and the test reference
tests/robust_ref.py) against mpmath at 40 digits, at every z = (res / c)^2 a finite f_scale can give: z = 0, the
smallest subnormal, a log grid over [1e-300, 1e300], and 1 - ulp, 1, 1 + ulp (Huber's branch point and the zero of
Cauchy's psi').  Tolerance: 4 ulp of the exact value for rho and rho'; 4 ulp of max(|psi'|, rho') for psi' =
rho' + 2 z rho'', whose exact value falls far below rho' where the loss is flat (Huber beyond c, soft-L1 and Cauchy at
large z) and crosses zero at Cauchy's z = 1."""
import ctypes

import mpmath
import numpy as np
import pytest

import robust_ref as rr
from test_host_math import P, dp, hm  # noqa: F401  (hm: the host build of the device headers)

ROBUST = ('huber', 'soft_l1', 'cauchy')
CODE = dict(linear=0, huber=1, soft_l1=2, cauchy=3)          # NMRFIT_LOSS_*
ULPS = 4


def z_grid():
    one = np.float64(1.0)
    edges = [0.0, 5e-324, np.nextafter(one, 0), one, np.nextafter(one, 2)]
    grid = np.logspace(-300, 300, 1201)
    wiggle = 10.0 ** np.random.default_rng(16).uniform(-300, 300, 800)
    near_one = 1 + np.linspace(-1e-3, 1e-3, 41)
    return np.unique(np.concatenate([edges, grid, wiggle, near_one]))


def exact(z, loss):
    """(rho, rho', psi') of ``loss`` at the double z, in mpmath at 40 digits, each in a form without cancellation."""
    with mpmath.workdps(40):
        z = mp(z)
        t = 1 + z
        if loss == 'linear':
            return z, mpmath.mpf(1), mpmath.mpf(1)
        if loss == 'huber':
            if z <= 1:
                return z, mpmath.mpf(1), mpmath.mpf(1)
            s = mpmath.sqrt(z)
            return 2 * s - 1, 1 / s, mpmath.mpf(0)
        if loss == 'soft_l1':
            s = mpmath.sqrt(t)
            return 2 * z / (s + 1), 1 / s, 1 / (t * s)
        if loss == 'cauchy':
            return mpmath.log1p(z), 1 / t, (1 - z) / (t * t)
    raise ValueError(loss)


def mp(x):
    """The finite float64 or long double x as an mpf, exactly."""
    m, e = np.frexp(x)
    return mpmath.ldexp(mpmath.mpf(int(np.ldexp(m, 64))), int(e) - 64)


def ulp(v, dtype):
    """The spacing of ``dtype``'s numbers at the mpf v >= 0 (subnormal spacing below the normal range)."""
    fi = np.finfo(dtype)
    e = mpmath.frexp(v)[1] if v != 0 else fi.minexp
    return mpmath.ldexp(1, max(e, fi.minexp + 1) - fi.nmant - 1)


def ulp_errors(got, z, loss, dtype):
    """[3, z.size]: the errors of ``got`` = (rho, rho', psi') in ulps (``dtype``'s) of the tolerance's scale."""
    out = np.empty((3, z.size))
    with mpmath.workdps(40):
        for i, q in enumerate(z):
            rho, d1, dpsi = exact(q, loss)
            for k, (want, scale) in enumerate(((rho, abs(rho)), (d1, d1), (dpsi, max(abs(dpsi), d1)))):
                g = dtype(got[k][i])
                out[k, i] = float(abs(mp(g) - want) / ulp(scale, dtype)) if np.isfinite(g) else np.inf
    return out


def device_terms(hm, z, loss):
    hm.h_loss.argtypes = [ctypes.c_int, dp, ctypes.c_int, dp, dp, dp]
    z = np.ascontiguousarray(z, dtype=np.float64)
    rho, d1, dpsi = np.empty_like(z), np.empty_like(z), np.empty_like(z)
    hm.h_loss(CODE[loss], P(z), z.size, P(rho), P(d1), P(dpsi))
    return rho, d1, dpsi


@pytest.mark.parametrize('loss', rr.LOSSES)
def test_device_loss_terms_against_mpmath(hm, loss):
    z = z_grid()
    err = ulp_errors(device_terms(hm, z, loss), z, loss, np.float64)
    worst = err.max(axis=1)
    print('%s: worst error in ulps rho %.2f, rho\' %.2f, psi\' %.2f' % (loss, *worst))
    for k, name in enumerate(('rho', "rho'", "psi'")):
        i = int(np.argmax(err[k]))
        assert err[k, i] <= ULPS, (loss, name, z[i], err[k, i])


@pytest.mark.parametrize('dtype', [np.float64, np.longdouble], ids=['float64', 'longdouble'])
@pytest.mark.parametrize('loss', rr.LOSSES)
def test_reference_loss_terms_against_mpmath(loss, dtype):
    """robust_ref.loss_terms and psi_prime in long double, where the GPU tests use them, and in float64, where
    scipy_fit hands the terms to scipy.  rho'' is checked through rho' + 2 z rho'' in long double only: at large z it
    (~z^-1.5 or -z^-2) leaves float64's range before rho' does."""
    z = z_grid().astype(dtype)
    with np.errstate(over='ignore'):
        rho, d1, d2 = rr.loss_terms(z, loss)
        dpsi = rr.psi_prime(z, loss)
    assert rho.dtype == d1.dtype == d2.dtype == dpsi.dtype == dtype
    err = ulp_errors((rho, d1, dpsi), z, loss, dtype)
    if dtype == np.longdouble:
        err = np.concatenate([err, ulp_errors((rho, d1, d1 + 2 * z * d2), z, loss, dtype)[2:]])
    for k, name in enumerate(('rho', "rho'", "psi'", "rho' + 2 z rho''")[:len(err)]):
        i = int(np.argmax(err[k]))
        assert err[k, i] <= ULPS, (loss, name, float(z[i]), err[k, i])
