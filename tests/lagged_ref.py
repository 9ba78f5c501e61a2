"""Reference residual autocorrelation and lag-weighted M, for the tests of the correlated-noise passes
(csrc/lagged.cu, DESIGN K14).  Built on ``linearisation_ref.residual_jacobian`` (float64); the products and sums are
formed in long double, so that a comparison measures the kernel's error alone.  Test infrastructure only."""
import numpy as np
from scipy.linalg import toeplitz

import linearisation_ref as lin


def residual_acf(x, w, u, v, max_lag):
    """r_k = sum_{i=0}^{N-1-k} res_i res_{i+k}, k = 0..max_lag, by direct sums."""
    res, _ = lin.residual_jacobian(x, w, u, v)
    r = res.astype(np.longdouble)
    n = r.size
    return np.array([np.sum(r[:n - k] * r[k:]) for k in range(max_lag + 1)], dtype=np.float64)


def m_lagged(x, w, u, v, weights, rho):
    """M_rho = sum_i a_i^T z_i with a_i = w_i^2 A_i and z_i = rho_0 a_i + sum_{k >= 1} rho_k (a_{i+k} + a_{i-k}), rows
    outside [0, N) zero: the shifted sums, then a^T z."""
    _, A = lin.residual_jacobian(x, w, u, v)
    wt = np.asarray(weights, dtype=np.longdouble)
    a = (wt * wt)[:, None] * A.astype(np.longdouble)
    rho = np.asarray(rho, dtype=np.longdouble)
    z = rho[0] * a
    for k in range(1, rho.size):
        z[:-k] += rho[k] * a[k:]
        z[k:] += rho[k] * a[:-k]
    return np.asarray(a.T @ z, dtype=np.float64)


def m_dense(x, w, u, v, weights, rho):
    """The same as a dense product, A^T W^2 T W^2 A with T the banded Toeplitz matrix of rho (small N only)."""
    _, A = lin.residual_jacobian(x, w, u, v)
    n = A.shape[0]
    col = np.zeros(n)
    col[:len(rho)] = rho[:n]
    w2 = np.asarray(weights, dtype=np.float64) ** 2
    a = w2[:, None] * A
    return a.T @ toeplitz(col) @ a


# Launch plans of the GPU parity sweep (test_gpu_lagged.py): (n_points, n_peaks, max_lag) -> the plan each shape must
# take (_cabi.lagged_plan) and the branch of csrc/lagged.cu it covers.  test_lagged_host.py pins the same table
# without a GPU, so a plan change that moves a shape off its branch fails there first.
SWEEP = {
    (37, 1, 0): dict(point_groups=85, slices=1, tile_points=128, n_chunks=1, acf_n_chunks=1),    # L = 0, ragged tile
    (37, 1, 36): dict(point_groups=85, slices=1, tile_points=128, n_chunks=1, acf_n_chunks=1),   # N = L + 1
    # L at the cap of one peak: halo of 1,489 rows around 16-point tiles, and across three residual chunks
    (5000, 1, 1489): dict(point_groups=85, slices=1, tile_points=16, n_chunks=1, acf_n_chunks=10, max_lag=1489),
    (20000, 6, 32): dict(point_groups=12, slices=1, tile_points=128, n_chunks=3, acf_n_chunks=40),   # halos cross chunks
    (5000, 6, 200): dict(point_groups=12, slices=1, tile_points=32, n_chunks=1, acf_n_chunks=10),    # L > tile
    (3000, 12, 128): dict(point_groups=4, slices=1, tile_points=16, n_chunks=2, acf_n_chunks=6),     # L > tile, 2 chunks
    (4100, 24, 40): dict(point_groups=1, slices=1, tile_points=32, n_chunks=9, acf_n_chunks=9),      # last chunk 4 < L
    (1000, 64, 1): dict(point_groups=1, slices=3, tile_points=16, n_chunks=4, acf_n_chunks=2),       # L = 1, 64 peaks
    (1000, 64, 45): dict(point_groups=1, slices=3, tile_points=16, n_chunks=4, acf_n_chunks=2, max_lag=45),  # the cap
}
