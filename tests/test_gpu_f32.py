"""Opt-in FP32 objective (precision='fp32'): <= 1e-5 relative against the reference objective on identical
particle positions (north-star tolerance), on uniform and non-uniform axes, and a whole fit in FP32."""
import numpy as np
import pytest

from conftest import load_golden, relerr
import nmrfit_b200
from nmrfit_b200 import _cabi, equations, synth, utils
from oracle import nmrfit_oracle as orc

pytestmark = pytest.mark.gpu
TOL32 = 1e-5
OBJ_CASES = ['c1_4096x6', 'ragged_1000x6', 'p12_2048', 'tiny_257x6', 'p24_1536']


@pytest.mark.parametrize('case', OBJ_CASES)
def test_fp32_matches_reference_golden(case):
    g = load_golden('objective_' + case)
    n_peaks = (g['xs'].shape[1] - 4) // 3
    with _cabi.Context(1, g['w'].size, n_peaks, precision=_cabi.FP32) as ctx:
        ctx.set_spectrum(0, g['w'], g['u'], g['v'], g['weights'])
        assert ctx.get_algorithm() == _cabi.ALGO_UNIFORM
        f = ctx.objective_host(g['xs'])
        assert relerr(f, g['f']) < TOL32
        ctx.set_algorithm(_cabi.ALGO_GENERAL)            # the any-axis FP32 kernel on the same data
        assert relerr(ctx.objective_host(g['xs']), g['f']) < TOL32
    f = equations.objective_batch(g['xs'], g['w'], g['u'], g['v'], g['weights'], precision=_cabi.FP32)
    assert relerr(f, g['f']) < TOL32


@pytest.mark.parametrize('threads,r', [(128, 4), (128, 8), (128, 16), (256, 4), (256, 8), (256, 16)])
def test_fp32_uniform_variants(threads, r):
    g = load_golden('objective_ragged_1000x6')
    runs = min(r, 8)                                     # the FP32 kernel is built for 4 and 8 points per thread
    with _cabi.Context(1, g['w'].size, 6, precision=_cabi.FP32) as ctx:
        ctx.set_spectrum(0, g['w'], g['u'], g['v'], g['weights'])
        for sp in (1, 5, 16):
            ctx.set_tuning(threads, r, 0, sp)
            t = ctx.get_tuning(len(g['xs']))
            assert (t['threads'], t['points_per_thread']) == (threads, runs)
            assert t['n_point_tiles'] == -(-g['w'].size // (threads * runs))
            assert relerr(ctx.objective_host(g['xs']), g['f']) < TOL32


def test_fp32_non_uniform_axis_and_extreme_widths():
    data, true = synth.multiplet(1500, 6, seed=12)
    w = data.w + 1e-6 * np.sin(np.arange(1500))          # not uniform
    wts = utils.compute_weights(data.w, data.peaks)
    lo, up = data.generate_solution_bounds()
    xs = synth.particles(lo, up, 12, seed=2)
    want = orc.objective_swarm(xs, w, data.u, data.v, wts)
    with _cabi.Context(1, 1500, 6, precision=_cabi.FP32) as ctx:
        ctx.set_spectrum(0, w, data.u, data.v, wts)
        assert ctx.get_algorithm() == _cabi.ALGO_GENERAL
        t = ctx.get_tuning(len(xs))                      # the any-axis FP32 kernel's fixed geometry
        assert (t['threads'], t['points_per_thread'], t['n_point_tiles']) == (256, 4, 2)
        assert relerr(ctx.objective_host(xs), want) < TOL32
    # uniform axis, widths that leave the recurrence (exact FP64 path inside the FP32 kernel) and far-away peaks
    xs = []
    for width in (1e-6, 2e-4, 0.05, 10.0):
        y = true.copy(); y[4::3] = width; xs.append(y)
    y = true.copy(); y[5::3] = 100.0; xs.append(y)
    xs = np.array(xs)
    want = orc.objective_swarm(xs, data.w, data.u, data.v, wts)
    got = equations.objective_batch(xs, data.w, data.u, data.v, wts, precision=_cabi.FP32)
    assert np.all(np.isfinite(got)) and relerr(got, want) < TOL32


def test_fp32_full_size_c2_and_fit_im_refused():
    N, P, S = 32768, 12, 1024
    data, true = synth.multiplet(N, P, seed=2000)
    wts = utils.compute_weights(data.w, data.peaks)
    lo, up = data.generate_solution_bounds()
    xs = synth.particles(lo, up, S, seed=7)
    xs[0] = true
    with _cabi.Context(1, N, P) as c64, _cabi.Context(1, N, P, precision=_cabi.FP32) as c32:
        for c in (c64, c32):
            c.set_spectrum(0, data.w, data.u, data.v, wts)
        f64, f32 = c64.objective_host(xs), c32.objective_host(xs)
        assert relerr(f32, f64) < TOL32
        assert f32[0] == f32.min()                       # the generating parameters still win
        with pytest.raises(_cabi.NmrfitError, match='FP32'):
            c32.objective_host(xs[:4], _cabi.IM_REFERENCE)


def test_fit_in_fp32_lands_on_the_fp64_fit():
    g = load_golden('fit_lite_1024x6')
    from conftest import peaks_from_golden
    data = nmrfit_b200.containers.Data(g['w'], g['u'], g['v'])
    data.peaks = peaks_from_golden(g)
    opts = dict(swarmsize=int(g['swarmsize']), maxiter=int(g['maxiter']))
    fits = {}
    for prec in ('fp64', 'fp32'):
        np.random.seed(int(g['seed']))
        fits[prec] = nmrfit_b200.fit(data, g['lower'], g['upper'], summary=False, options=dict(opts, precision=prec))
    # same random stream, objective values differ by ~1e-7: the swarm follows the same path until two particles
    # are closer than that, so the two results agree to much better than the fit's own uncertainty
    assert abs(fits['fp32'].error / fits['fp64'].error - 1) < 1e-3
    assert np.allclose(fits['fp32'].get_areas(), fits['fp64'].get_areas(), rtol=5e-2)
