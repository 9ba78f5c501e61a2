"""Deterministic synthetic multiplet spectra (inputs only; SURVEY.md section 8d).

Nothing here is on the timed path: it builds the (w, u, v) arrays, the ``Peak``
records and the true parameter vector that tests and ``bench.py`` feed to the
CUDA path.  The lineshape is evaluated once on the host with numpy/scipy purely
to synthesise data (the reference has no sample data: ``examples/`` is
git-ignored, .gitignore:2).

"propcar-like" group = two 1H main lines flanked by four 13C satellites at 1 %
of a main line's area (README.md:50 speaks of 6 peaks; the isotope-ratio use
case is utils.py:35-55 / plot.py:129-227).
"""
import numpy as np
from scipy.special import dawsn

from .utils import Peak, Peaks
from .containers import Data

W_LO, W_HI = 3.23, 3.60            # README.md:37 bounds the propcar window here
_OFFS = np.array([-0.115, -0.085, -0.015, 0.015, 0.085, 0.115])   # -> 3.30 ... 3.53 for one group
_IS_MAIN = np.array([False, False, True, True, False, False])
TRUE_GLOBALS = dict(p0=0.25, p1=0.05, r=0.55, yoff=0.0)
_SQLN2 = np.sqrt(np.log(2.0))


def _body(w, r, width, loc, a):
    t = (w - loc) / (0.5 * width)
    s = (w - loc) * (2 * _SQLN2) / width
    lor = (2 / (np.pi * width)) / (1 + t * t)
    gau = (2 / width) * np.sqrt(np.log(2.0) / np.pi) * np.exp(-s * s)
    return a * (r * lor + (1 - r) * gau)


def _body_kk(w, r, width, loc, a):
    t = (w - loc) / (0.5 * width)
    s = (w - loc) * (2 * _SQLN2) / width
    lor = (2 / (np.pi * width)) * t / (1 + t * t)
    gau = (2 / width) * np.sqrt(np.log(2.0) / np.pi) * (2 / np.sqrt(np.pi)) * dawsn(s)
    return a * (r * lor + (1 - r) * gau)


def _rotate_inv(V, I, p0, p1):
    n = V.shape[-1]
    phi = p0 + (p1 * np.arange(n) / n)
    c, s = np.cos(phi), np.sin(phi)
    return V * c + I * s, -V * s + I * c


def multiplet(n_points, n_peaks=6, seed=0, noise=1e-4, jitter=None):
    """Return ``(data, true_params)`` for one synthetic spectrum.

    ``n_peaks`` must be a multiple of 6 (one propcar-like group per 6 peaks,
    groups tiled evenly across the window).  ``jitter`` (default: on when more
    than one group or seed != 0) draws centres U(-0.002, 0.002) and widths
    U(0.003, 0.005) from ``default_rng(seed)``; noise is N(0, noise^2) on u and v
    from the same generator.  ``data.peaks`` carry loc/width/area/height/bounds
    as AutoPeakSelector would fill them (utils.py:760-770 conventions:
    bounds = loc -/+ 2 widths).
    """
    if n_peaks % 6:
        raise ValueError('n_peaks must be a multiple of 6')
    groups = n_peaks // 6
    rng = np.random.default_rng(seed)
    if jitter is None:
        jitter = groups > 1 or seed != 0
    w = np.linspace(W_LO, W_HI, n_points)
    span = W_HI - W_LO
    locs, widths, areas = [], [], []
    for g in range(groups):
        centre = W_LO + span * (g + 0.5) / groups
        for k in range(6):
            loc = centre + _OFFS[k] / groups
            width = 0.004 + 0.0002 * (k % 2)
            if jitter:
                loc += rng.uniform(-0.002, 0.002) / groups
                width = rng.uniform(0.003, 0.005)
            locs.append(loc)
            widths.append(width)
            areas.append(1.0 if _IS_MAIN[k] else 0.01)
    locs, widths, areas = map(np.array, (locs, widths, areas))
    g0 = TRUE_GLOBALS
    V = sum(_body(w, g0['r'], widths[k], locs[k], areas[k]) for k in range(n_peaks))
    scale = 1.0 / V.max()                     # core.py:53 normalises by the maximum
    areas = areas * scale
    V = V * scale
    I = sum(_body_kk(w, g0['r'], widths[k], locs[k], areas[k]) for k in range(n_peaks))
    u, v = _rotate_inv(V, I, g0['p0'], g0['p1'])
    if noise:
        u = u + rng.normal(0.0, noise, n_points)
        v = v + rng.normal(0.0, noise, n_points)

    data = Data(w, u, v)
    data.p0, data.p1 = g0['p0'], g0['p1']
    peaks = Peaks()
    for k in range(n_peaks):
        pk = Peak()
        pk.loc, pk.width, pk.area = float(locs[k]), float(widths[k]), float(areas[k])
        pk.height = float(V[np.argmin(np.abs(w - pk.loc))])
        pk.bounds = [pk.loc - 2 * pk.width, pk.loc + 2 * pk.width]
        peaks.append(pk)
    data.peaks = peaks
    data.roibounds = [pk.bounds for pk in peaks]

    true = [g0['p0'], g0['p1'], g0['r'], g0['yoff']]
    for k in range(n_peaks):
        true.extend([widths[k], locs[k], areas[k]])
    return data, np.array(true)


# each main line's 13C satellites, (main, lower satellite, upper satellite) by position within a group: the pairs
# sit at -/+ J/2 = -/+ 0.1 (per group) around their main line
_SATELLITES = ((2, 0, 4), (3, 1, 5))


def satellite_ties(n_peaks):
    """The natural ties of ``multiplet``'s propcar-like groups (``utils.Ties``): for each main line m with satellites
    s- and s+, width(s-) = width(s+) = width(m), area(s+) = area(s-) and loc(s-/+) = loc(m) -/+ J/2, with J/2 the
    offset ``_OFFS`` puts between them (scaled by the number of groups, as ``multiplet`` scales it).  The true vector
    of ``multiplet(..., jitter=False)`` satisfies them; jittered centres leave the satellites' boxes off the tie."""
    from .utils import Ties
    if n_peaks % 6:
        raise ValueError('n_peaks must be a multiple of 6')
    groups = n_peaks // 6
    t = Ties(n_peaks)
    for g in range(groups):
        for m, lo, hi in _SATELLITES:
            assert _IS_MAIN[m] and not _IS_MAIN[lo] and not _IS_MAIN[hi]
            km, kl, kh = 6 * g + m, 6 * g + lo, 6 * g + hi
            for s in (kl, kh):
                t.link(('width', s), ('width', km))
                t.link(('loc', s), ('loc', km), offset=(_OFFS[s % 6] - _OFFS[m]) / groups)
            t.link(('area', kh), ('area', kl))
    return t


def processed_noise(n_points, sigma, broadening=3.0, zero_fill=2, n_realisations=1, seed=0):
    """Noise of a processed spectrum, for ``u`` and ``v``: white complex noise on an FID of n_points / zero_fill
    samples, exponential line broadening of ``broadening`` spectral points (the FWHM it gives a Lorentzian line;
    0 for none), zero-filled to n_points, FFT.  Scaled so that the real part has standard deviation ``sigma``.
    Its real part then has the autocorrelation rho_k ~ b^2 / (b^2 + k^2) at b = broadening.  Returns
    ``(noise_u, noise_v)``, each [n_realisations, n_points], from ``default_rng(seed)``."""
    rng = np.random.default_rng(seed)
    n_fid = n_points // zero_fill
    window = np.exp(-np.pi * broadening * np.arange(n_fid) / n_points)
    fid = (rng.standard_normal((n_realisations, n_fid)) + 1j * rng.standard_normal((n_realisations, n_fid))) * window
    spec = np.fft.fft(fid, n=n_points, axis=1) * (sigma / np.sqrt(np.sum(window * window)))
    return spec.real, spec.imag


def particles(lower, upper, n_particles, seed=7):
    """Objective-parity particle positions: lb + U(0,1)*(ub-lb), default_rng(seed)."""
    lb = np.asarray(lower, dtype=float)
    ub = np.asarray(upper, dtype=float)
    return lb + np.random.default_rng(seed).random((n_particles, lb.size)) * (ub - lb)
