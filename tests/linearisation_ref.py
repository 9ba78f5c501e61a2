"""Reference linearisation of the real-part objective, for the tests of the parameter-uncertainty pass
(csrc/normal_eq.cu).  numpy float64 (the sums optionally in long double), test infrastructure only.  The residual is built from the oracle's own ``ps2``
and ``voigt`` in the oracle objective's operation order, so that its weighted RMS is ``oracle.objective`` bit for bit;
the Jacobian is in closed form (checked against complex-step derivatives in test_uncertainty_host.py)."""
import numpy as np

from oracle.nmrfit_oracle import LN2, ps2, voigt


def residual_jacobian(x, w, u, v):
    """Residual ``res = v_data - v_fit`` built exactly as ``objective`` builds it (so that
    ``np.sqrt(np.square(np.multiply(weights, res)).mean())`` IS the objective) and its Jacobian ``A = d res / dx``
    [N, D] in closed form, with d = w - loc, t = 2d/width, s = 2 sqrt(ln2) d/width: d/dp0 = -i_data,
    d/dp1 = -i_data * i/N, d/dr = -sum a (L - G), d/dyoff = -P (yoff enters once per peak), and per peak
    d/da = -(r L + (1-r) G), d/dloc = -a (r L 2t/(1+t^2) 2/width + (1-r) G 2s 2 sqrt(ln2)/width),
    d/dwidth = -a (r (L/width)(t^2-1)/(1+t^2) + (1-r)(G/width)(2s^2-1))."""
    x = np.asarray(x, dtype=np.float64)
    p0, p1, r, yoff = x[:4]
    n = w.shape[-1]
    n_peaks = (x.size - 4) // 3
    v_data, i_data = ps2(u, v, p0=p0, p1=p1)
    v_fit = np.zeros_like(v_data)
    A = np.zeros((n, x.size))
    A[:, 0] = -i_data
    A[:, 1] = -i_data * (np.arange(n) / n)
    A[:, 3] = -n_peaks
    for k in range(4, len(x), 3):
        width, loc, a = x[k], x[k + 1], x[k + 2]
        v_fit = v_fit + voigt(w, r, yoff, width, loc, a)
        d = w - loc
        t = 2 * d / width
        s = 2 * np.sqrt(LN2) * d / width
        lor = (2 / (np.pi * width)) / (1 + t * t)
        gau = (2 / width) * np.sqrt(LN2 / np.pi) * np.exp(-s * s)
        A[:, 2] -= a * (lor - gau)
        A[:, k] = -a * (r * (lor / width) * (t * t - 1) / (1 + t * t) + (1 - r) * (gau / width) * (2 * s * s - 1))
        A[:, k + 1] = -a * (r * lor * 2 * t / (1 + t * t) * (2 / width) + (1 - r) * gau * 2 * s * (2 * np.sqrt(LN2) / width))
        A[:, k + 2] = -(r * lor + (1 - r) * gau)
    return v_data - v_fit, A


def normal_equations(x, w, u, v, weights, accumulate=np.float64):
    """(H, M, g, ssr) of ``residual_jacobian``: H = A^T W^2 A, M = A^T W^4 A, g = A^T W^2 res,
    ssr = (sum (weights res)^2, sum res^2).  The residual and Jacobian are float64; the products and sums are formed
    in ``accumulate`` and the results returned as float64.  With ``np.longdouble`` the sums no longer depend on the
    host's BLAS kernels (numpy's own loops run them) and carry at least 11 more bits than the kernel's FP64 sums, so a
    comparison measures the kernel's error alone."""
    res, A = residual_jacobian(x, w, u, v)
    res, A, wt = (np.asarray(a, dtype=accumulate) for a in (res, A, weights))
    w2 = wt * wt
    H = A.T @ (w2[:, None] * A)
    M = A.T @ ((w2 * w2)[:, None] * A)
    g = A.T @ (w2 * res)
    ssr = np.array([np.sum(w2 * res * res), np.sum(res * res)])
    return tuple(np.asarray(a, dtype=np.float64) for a in (H, M, g, ssr))


# Launch plans of the GPU parity sweep (test_gpu_uncertainty.py): (n_points, n_peaks) -> the plan each shape must
# take (_cabi.normal_equations_plan) and the branch of csrc/normal_eq.cu it covers.  test_uncertainty_host.py pins
# the same table without a GPU, so a plan change that moves a shape off its branch fails there first.
SWEEP = {
    (37, 1): dict(point_groups=42, slices=1, tile_points=128, n_chunks=1),         # N below one tile, E = 8
    (3000, 2): dict(point_groups=21, slices=1, tile_points=128, n_chunks=1),       # ragged tile
    (777, 9): dict(point_groups=3, slices=1, tile_points=64, n_chunks=1),          # E = 32
    (20000, 6): dict(point_groups=6, slices=1, tile_points=128, n_chunks=5),       # last chunk 3,616
    (5000, 11): dict(point_groups=2, slices=1, tile_points=64, n_chunks=3),        # last chunk 904
    (5000, 24): dict(point_groups=1, slices=1, tile_points=32, n_chunks=10),       # last chunk 392
    (6000, 27): dict(point_groups=1, slices=1, tile_points=32, n_chunks=12, tasks_per_slice=506, threads=512),
    (2500, 28): dict(point_groups=1, slices=2, tile_points=32, n_chunks=5),        # first multi-slice shape
    (1000, 31): dict(point_groups=1, slices=2, tile_points=16, n_chunks=4),        # first 16-point tiles
    (6000, 36): dict(point_groups=1, slices=2, tile_points=16, n_chunks=24),
    (9000, 48): dict(point_groups=1, slices=3, tile_points=16, n_chunks=36, threads=512),    # last chunk 40
    (4100, 57): dict(point_groups=1, slices=4, tile_points=16, n_chunks=17),       # E = 176, last chunk 4
    (1000, 64): dict(point_groups=1, slices=5, tile_points=16, n_chunks=4),        # the 64-peak limit
    (2100000, 1): dict(point_groups=42, slices=1, tile_points=128, chunk_points=32768, n_chunks=65),
}
