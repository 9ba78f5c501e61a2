"""The oracle's restatement of the auto peak selector (oracle/nmrfit_oracle.auto_peaks, with oracle/peakutils_oracle.py
for the absent peakutils) against the golden fixtures produced by the reference's own AutoPeakSelector
(tests/golden/make_golden.py: the unmodified class, scipy.integrate.simps bound to simpson, peakutils.baseline bound
to the restated algorithm - PARITY UNPINNED for that one piece)."""
import numpy as np
import pytest

from conftest import load_golden, relerr
from oracle import nmrfit_oracle as orc, peakutils_oracle

CASES = ['peaks_1024x6', 'peaks_2500x12', 'peaks_4096x6', 'peaks_desc_1500x6',
         'peaks_c3_16384x6']      # the last: a BASELINE configs[2] spectrum (1,638,400 upsampled samples, window 88,554)


def _close(got, want, scale):
    got, want = np.asarray(got, dtype=float), np.asarray(want, dtype=float)
    return got.shape == want.shape and np.max(np.abs(got - want), initial=0.0) <= 1e-13 * scale


@pytest.mark.parametrize('case', CASES)
def test_auto_peaks_matches_the_reference_class(case):
    g = load_golden(case)
    peaks, aux = orc.auto_peaks(g['w'], g['V'], float(g['thresh']), float(g['window']))
    pr = g['probe']
    assert np.array_equal(aux['wu'][pr], g['wu_probe']) and np.array_equal(aux['uu'][pr], g['uu_probe'])
    # The Savitzky-Golay coefficients (a least-squares solve) and peakutils' baseline (pinv, dot) go through BLAS /
    # LAPACK, whose summation order depends on the host CPU: the smoothed signal, the baselines and the heights and
    # areas built on them agree to rounding (at most 3e-14 of their scale between OpenBLAS's x86 kernel sets); every
    # index, location, width and bound is exact.
    scale = np.abs(g['V']).max()
    assert _close(aux['us'][pr], g['us_probe'], scale) and _close(aux['baseline'], g['baseline'], scale)
    assert [p.i for p in aux['pre']] == list(g['pre_i'])
    assert [p.i for p in peaks] == list(g['i'])
    for key in ('loc', 'width'):
        assert np.array_equal([getattr(p, key) for p in peaks], g[key]), key
    assert _close([p.height for p in peaks], g['height'], scale)
    assert _close([p.area for p in peaks], g['area'], np.abs(g['area']).max())
    assert _close([p.baseline for p in peaks], g['local_baseline'], scale)
    assert np.array_equal([p.bounds for p in peaks], g['bounds'])
    assert [p.idx_lo for p in peaks] == list(g['idx_lo']) and [p.idx_hi for p in peaks] == list(g['idx_hi'])


def test_argrelmax_restatement_equals_scipy():
    import scipy.signal
    rng = np.random.default_rng(0)
    for n, order in ((50, 1), (500, 7), (3000, 40), (3000, 5000), (64, 200)):
        x = rng.normal(size=n)
        x[rng.integers(0, n, 5)] = x.max()                  # ties: never a strict maximum
        assert np.array_equal(orc.argrelmax_clip(x, order), scipy.signal.argrelmax(x, order=order)[0])


def test_degree_zero_baseline_closed_form():
    """The loop the device runs: clip to the running mean until it moves by < 0.1 % - equals the general algorithm."""
    rng = np.random.default_rng(1)
    for n in (40, 1000, 20000):
        y = rng.normal(0, 1e-3, n) + np.exp(-0.5 * ((np.arange(n) - n / 2) / (n / 30)) ** 2)
        b, it = peakutils_oracle.baseline0(y)
        assert abs(b / peakutils_oracle.baseline(y, 0)[0] - 1) < 1e-12
    y = np.full(10, 1.0004)                                 # first mean within 0.1 % of the initial coefficient 1.0
    assert peakutils_oracle.baseline(y, 0)[0] == y[0] == peakutils_oracle.baseline0(y)[0]
