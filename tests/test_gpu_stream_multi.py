"""The streamed kernel's several-particles-per-warp evaluation (objective_stream.cu, eval_region_multi): the lanes of a
warp hold different particles, so their near peaks, exact-path peaks and phases differ inside one warp.  It must give
the one-group kernel's bits whatever the particles of a warp have in common."""
import numpy as np
import pytest

from conftest import relerr
from nmrfit_b200 import _cabi, synth, utils
from oracle import nmrfit_oracle as orc

pytestmark = pytest.mark.gpu


def _mixed_particles(data, true, n):
    """Random particles with, every few particles, one that takes a different path through the kernel: a peak too
    narrow for the recurrences (exact path), a peak moved far off the window, a large phase."""
    lo, up = data.generate_solution_bounds()
    xs = synth.particles(lo, up, n, seed=11)
    xs[0] = true
    for i in range(1, n, 3):
        xs[i, 4 + 3 * (i % 6)] = 1e-6
    for i in range(2, n, 7):
        xs[i, 5 + 3 * (i % 6)] = data.w[0] - 0.5
    for i in range(3, n, 5):
        xs[i, 0], xs[i, 1] = 50.0, -80.0
    return xs


@pytest.mark.parametrize('n_points', [4096, 1000, 16384])     # four, two and two far-field cells per region
def test_warps_of_mixed_particles_agree_with_one_group_kernel(n_points):
    data, true = synth.multiplet(n_points, 6, seed=5 + n_points)
    wts = utils.compute_weights(data.w, data.peaks)
    xs = _mixed_particles(data, true, 61)
    with _cabi.Context(1, n_points, 6) as ctx:
        ctx.set_spectrum(0, data.w, data.u, data.v, wts)
        ctx.set_variant(0)
        want = ctx.objective_host(xs)
        assert np.all(np.isfinite(want))
        assert relerr(want, orc.objective_swarm(xs, data.w, data.u, data.v, wts)) < 1e-10
        for stages, sp in ((0, 0), (2, 4), (3, 5), (2, 8), (2, 6)):
            ctx.set_variant(1, stages, 2)
            ctx.set_tuning(0, 0, 0, sp)
            assert ctx.get_variant(len(xs))[0] == 1
            assert np.array_equal(ctx.objective_host(xs), want), (stages, sp)
