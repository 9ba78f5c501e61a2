"""Fit driver, mirroring ``nmrfit.utils`` for the hot path.

``FitUtility`` keeps the reference's constructor, methods and result attributes
(utils.py:96-339); what changes is underneath: the swarm lives on the GPU and a
generation is one batched launch instead of ``swarmsize`` Python callbacks.

``Peak`` / ``Peaks`` are the plain records the driver reads (utils.py:14-93).
``AutoPeakSelector`` (utils.py:670-783) and its batched form ``select_peaks_batch`` run on the GPU
(csrc/peaks.cu).  The interactive, matplotlib-driven selectors of the reference (BoundsSelector,
PeakSelector: utils.py:342-667) are outside the accelerated path and are not provided.
"""
import numpy as np

from . import _cabi
from . import equations
from . import swarm as _swarm


class Peaks(list):
    """List of ``Peak`` records (utils.py:14-55)."""

    def average_height(self):
        return sum(abs(p.height) for p in self) / len(self)

    def split(self):
        """(main peaks, satellites) by height relative to the average."""
        h = self.average_height()
        mains, sats = Peaks(), Peaks()
        for p in self:
            (mains if abs(p.height) >= h else sats).append(p)
        return mains, sats


class Peak:
    """Metadata of one peak: ``loc``, ``height``, ``bounds`` [lo, hi], ``width`` (FWHM), ``area``."""

    def __repr__(self):
        return 'Peak(loc=%s, height=%s, bounds=[%s, %s], width=%s, area=%s)' % (
            getattr(self, 'loc', None), getattr(self, 'height', None),
            *(getattr(self, 'bounds', [None, None])), getattr(self, 'width', None), getattr(self, 'area', None))


def compute_weights(w, peaks, expon=0.5):
    """Frequency-dependent residual weights (utils.py:191-224): 1 everywhere,
    (tallest/|height|)**expon inside each peak's index window (later peaks
    overwrite earlier ones), then 10 Jacobi smoothing sweeps.  Host-side: it runs
    once per fit and costs microseconds."""
    n_pk = len(peaks)
    lo = np.zeros(n_pk, dtype=int)
    hi = np.zeros(n_pk, dtype=int)
    mag = np.zeros(n_pk)
    for i, pk in enumerate(peaks):
        a = int(np.argmin(np.abs(w - pk.bounds[0])))
        b = int(np.argmin(np.abs(w - pk.bounds[1])))
        lo[i], hi[i] = min(a, b), max(a, b)
        mag[i] = np.abs(pk.height)
    tallest = np.amax(mag)
    weights = np.ones(len(w))
    for i in range(n_pk):
        weights[lo[i]:hi[i] + 1] = np.power(tallest / mag[i], expon)
    return equations.laplace1d(weights)


def peak_windows(peaks_list, expon=0.5):
    """Inputs of the device weights kernel for a batch: ``bounds`` [B, K, 2] (``Peak.bounds``) and ``values``
    [B, K] = (tallest/|height|)**expon per spectrum (utils.py:206-221) - the only host arithmetic left."""
    B, K = len(peaks_list), len(peaks_list[0])
    bounds = np.empty((B, K, 2))
    mag = np.empty((B, K))
    for b, peaks in enumerate(peaks_list):
        if len(peaks) != K:
            raise ValueError('every spectrum of a batch must have the same number of peaks')
        for k, pk in enumerate(peaks):
            bounds[b, k, 0], bounds[b, k, 1] = pk.bounds[0], pk.bounds[1]
            mag[b, k] = np.abs(pk.height)
    values = np.power(np.amax(mag, axis=1, keepdims=True) / mag, expon)
    return bounds, values


class FitUtility:
    """Interface used to perform a fit of the data (drop-in for utils.py:96-339).

    Attributes after ``fit()``: ``params`` (ndarray D), ``error`` (float),
    ``weights``; after ``generate_result()``: ``w, u, v, V, I`` and the per-peak
    lists ``real_contribs`` / ``imag_contribs``.

    ``options`` understands the reference's keys (``swarmsize`` 204, ``maxiter``
    2000, ``omega`` -0.2134, ``phip`` -0.3344, ``phig`` 2.3259; utils.py:177-181)
    plus optional extras that do not exist upstream:
      ``rng``       'host' (default): numpy's legacy global stream in pyswarm's order, so
                    ``np.random.seed(k)`` gives the reference's trajectory - the stream is continued ON THE
                    DEVICE from np.random's own state (bit-identical numbers, state handed back);
                    'host_arrays': the same numbers drawn on the host and copied; 'device': Philox on the GPU.
      ``seed``      Philox seed for rng='device'.
      ``minstep``, ``minfunc``   pyswarm's stop tolerances (1e-8).
      ``precision`` 'fp64' (default) or 'fp32'.
      ``chunk``     generations queued between host checks of the stop flag.
      ``fused``     'auto' (default) | 'off' | 'require': run the generations of a small swarm in one
                    cooperative launch (bit-identical to the per-step kernels).
      ``device``    CUDA device index.
      ``refine``    True: ``refine()`` after the swarm (default False).
      ``ties``      a ``Ties`` the refinement holds (``refine(ties=...)``; needs ``refine``: the swarm does not
                    honour ties).  ``fit_batch`` takes one ``Ties`` for every spectrum or a list of them.
      ``loss``, ``f_scale``   a robust loss the refinement minimises (``refine(loss=..., f_scale=...)``; needs
                    ``refine``: the swarm keeps the reference's objective).  ``fit_batch`` takes one f_scale for every
                    spectrum or one per spectrum; f_scale 'auto' estimates each spectrum's scale from its
                    least-squares residuals (``refine(f_scale='auto')``).
    ``processes`` is accepted and ignored (the GPU evaluates every particle at once).
    """

    def __init__(self, data, lower, upper, expon=0.5, dynamic_weighting=True, fit_im=False, processes=1,
                 summary=True, options={}):
        self.data = data
        self.lower = lower
        self.upper = upper
        self.expon = expon
        self.dynamic_weighting = dynamic_weighting
        self.fit_im = fit_im
        self.summary = summary
        self.processes = processes
        self.options = options

    def fit(self):
        """Minimise the objective over the box [lower, upper] with the swarm (then ``refine()`` with
        ``options['refine']``)."""
        if self.options.get('refine', False):
            _check_refinable(self)
            check_loss_scale(self.options.get('loss', 'linear'), self.options.get('f_scale'), 1)
        else:
            check_unrefined_options(self.options)
        self.weights = self._compute_weights()
        if self.dynamic_weighting is False:
            self.weights = np.ones_like(self.weights)

        opt = self.options
        xopt, fopt, info = _swarm.pso_single(
            self.data.w, self.data.u, self.data.v, self.weights, self.lower, self.upper,
            fit_im=self.fit_im,
            swarmsize=opt.get('swarmsize', 204), maxiter=opt.get('maxiter', 2000),
            omega=opt.get('omega', -0.2134), phip=opt.get('phip', -0.3344), phig=opt.get('phig', 2.3259),
            minstep=opt.get('minstep', 1e-8), minfunc=opt.get('minfunc', 1e-8),
            rng=opt.get('rng', 'host'), seed=opt.get('seed', 0), precision=opt.get('precision', 'fp64'),
            chunk=opt.get('chunk', 16), device=opt.get('device', None), fused=opt.get('fused', 'auto'))

        self.params = xopt
        self.error = fopt
        self.fit_info = info
        if opt.get('refine', False):
            self.refine(ties=opt.get('ties'), loss=opt.get('loss', 'linear'), f_scale=opt.get('f_scale'))

        if self.summary is True:
            self._print_summary()

    def _compute_weights(self):
        return compute_weights(self.data.w, self.data.peaks, self.expon)

    def generate_result(self, scale=1):
        """Evaluate the fitted curves, optionally upsampled by ``scale`` (utils.py:226-295)."""
        if scale == 1.0:
            w = self.data.w
        else:
            w = np.linspace(self.data.w.min(), self.data.w.max(), int(scale * self.data.w.shape[0]))

        p0, p1 = self.params[0], self.params[1]
        # the reference re-phases the data object here (utils.py:252)
        self.data.shift_phase(method='manual', p0=p0, p1=p1)

        params = _cabi.as_f64(self.params)
        n_peaks = (params.size - 4) // 3
        w = _cabi.as_f64(w)
        n = w.size
        # one result block (pinned and pooled when large: _cabi.result_empty), carved into the six outputs
        block = _cabi.result_empty((2 * n_peaks + 4) * n)
        real = block[:n_peaks * n].reshape(n_peaks, n)
        imag = block[n_peaks * n:2 * n_peaks * n].reshape(n_peaks, n)
        V, I, u, v = (block[(2 * n_peaks + k) * n:(2 * n_peaks + k + 1) * n] for k in range(4))
        dev = self.options.get('device', None)
        _cabi.check(_cabi.lib().nmrfit_generate_result_host(
            _cabi.default_device() if dev is None else int(dev), _cabi.ptr(params), n_peaks, _cabi.ptr(w), n,
            _cabi.ptr(real), _cabi.ptr(imag), _cabi.ptr(V), _cabi.ptr(I), _cabi.ptr(u), _cabi.ptr(v)))

        self.u = u
        self.v = v
        self.V = V
        self.I = I
        self.w = w
        self.real_contribs = [real[k] for k in range(n_peaks)]
        self.imag_contribs = [imag[k] for k in range(n_peaks)]

    def calculate_area_fraction(self):
        """Satellite area / total area, satellites = areas below the mean (utils.py:297-310)."""
        areas = self.get_areas()
        m = np.mean(areas)
        mains = areas[areas >= m].sum()
        sats = areas[areas < m].sum()
        return sats / (mains + sats)

    def get_areas(self):
        """Fitted areas: every third parameter from index 6 (utils.py:322)."""
        return np.array([self.params[i] for i in range(6, len(self.params), 3)])

    def refine(self, max_iter=None, xtol=1e-6, ties=None, loss='linear', f_scale=None):
        """Refine the swarm's ``params`` to the least-squares optimum of the weighted residual within the box, by
        bounded Levenberg-Marquardt on the GPU (see ``refine_batch``).  Replaces ``params`` and ``error`` (which
        becomes sqrt(s/N) from the normal equations at the new point; both stay bit for bit as they were if no step
        was accepted) and sets ``refine_info`` = dict(start_params, start_error, passes, accepted, status), status one
        of ``_cabi.REFINE_CONVERGED``, ``_STALLED``, ``_MAX_ITER``, ``_NONFINITE``.

        ``ties`` (a ``Ties``) refines the constrained model: fixed parameters keep their values, linked ones follow
        their masters, and the free ones are refined within the reduced box (DESIGN K15).  The ties used are kept
        as ``self.ties``, so that ``compute_uncertainties()`` and ``area_fraction_stderr()`` give the errors of that
        model.

        ``loss`` ('linear', 'huber', 'soft_l1' or 'cauchy', scipy's convention) with ``f_scale`` c > 0, in units of the
        data, minimises the robust cost sum w^2 c^2 rho((res/c)^2) instead (DESIGN K16): a point whose unweighted
        residual is far beyond c, such as an unmodelled impurity line, then has bounded influence.  c = 1.345 sigma for
        'huber' and 2.385 sigma for 'cauchy' keep 95 % efficiency on Gaussian noise of level sigma.  The loss is kept as
        ``self.loss`` = dict(name, f_scale) (None for linear), so that ``compute_uncertainties()`` gives the robust
        covariance; ``error`` stays the weighted RMSE sqrt(sum w^2 res^2 / N) at the new point, and ``refine_info``
        gains ``loss``, ``f_scale`` and ``cost`` (the robust cost at the returned point; N error^2 for linear).
        Iteratively reweighted steps converge linearly while points lie beyond c, so a robust refinement takes more
        passes than least squares (DESIGN K16): ``max_iter`` None is 50 for linear and ``ROBUST_MAX_ITER`` = 200 for a
        robust loss.  The loop stops as soon as every spectrum has finished, so the larger cap costs nothing then.

        ``f_scale='auto'`` sets c from the data (DESIGN K17): a least-squares refinement first (``max_iter`` None is 50
        there), then sigma = MAD / 0.6744897501960817 of its unweighted residuals over all points (``noise_level()``,
        as ``scipy.stats.median_abs_deviation(scale='normal')``; the median ignores the few points an impurity line
        spoils, where the least-squares sigma does not), c = ``AUTO_SCALE_K[loss]`` * sigma, and the robust
        refinement from the least-squares point with that c.  The result is that of ``refine()`` followed by
        ``refine(loss=loss, f_scale=c)`` bit for bit, except that ``refine_info`` keeps the start of the first stage
        and gains ``scale`` = dict(sigma, median, k, lsq_passes, lsq_accepted, lsq_status).  ValueError naming the
        spectrum, with no fit changed, if a sigma is 0 or not finite (more than half of the residuals equal, or the
        least-squares stage ended ``REFINE_NONFINITE``).

        Raises RuntimeError before ``fit()`` and NotImplementedError with ``fit_im``."""
        refine_batch([self], max_iter, xtol, ties=None if ties is None else [ties], loss=loss, f_scale=f_scale)
        return self.params

    def noise_level(self):
        """The noise level sigma = MAD / 0.6744897501960817 of the unweighted residuals at ``params`` over all points
        (``noise_level_batch``): one device pass, no refinement."""
        return float(noise_level_batch([self])[0])

    def compute_uncertainties(self, noise='white', max_lag=32, noise_acf=None):
        """Standard errors of ``params`` from the linearised least-squares problem at the fitted point (one pass
        over the spectrum on the GPU, see ``compute_uncertainties_batch``).  Sets ``covariance`` [D, D], ``stderr``
        [D] and ``uncertainty_info``, and returns ``stderr``.

        The errors assume that ``params`` is the least-squares optimum; the swarm stops short of it, and ``refine()``
        takes ``params`` there first.  ``noise='correlated'`` accounts for noise that is correlated from point to point,
        as line broadening makes it (see ``compute_uncertainties_batch`` for it and for ``max_lag`` and ``noise_acf``).

        After ``refine(ties=...)`` the errors are those of the tied model (``self.ties``, see
        ``covariance_from_normal``): 0 for a fixed parameter, |scale| times its master's for a linked one.  After a
        robust ``refine(loss=...)`` they are Huber's M-estimator covariance (``covariance_from_normal(moments=...)``);
        ``noise='correlated'`` is then refused with NotImplementedError.

        Raises RuntimeError before ``fit()``, NotImplementedError with ``fit_im`` (that objective is a sum of two
        RMSEs, not a least-squares problem) and ValueError when the spectrum has no more points than parameters or
        an argument is out of range."""
        compute_uncertainties_batch([self], noise=noise, max_lag=max_lag, noise_acf=noise_acf)
        return self.stderr

    def area_fraction_stderr(self):
        """Standard error of ``calculate_area_fraction()`` by the delta method, with the split into main peaks and
        satellites held fixed: for f = S/T, df/da_k = (1 - f)/T for a satellite and -f/T for a main peak.  Computes
        the covariance first if it is missing."""
        if getattr(self, 'covariance', None) is None:
            self.compute_uncertainties()
        areas = self.get_areas()
        m = np.mean(areas)
        total = areas.sum()
        frac = areas[areas < m].sum() / total
        grad = np.zeros(len(self.params))
        grad[6::3] = np.where(areas < m, (1 - frac) / total, -frac / total)
        return float(np.sqrt(grad @ self.covariance @ grad))

    def _print_summary(self):
        import pandas as pd
        res = np.array(self.params)
        res_globals = pd.DataFrame(res[:4].reshape((1, -1)), columns=['p0', 'p1', 'r', 'y-off'])
        res_peaks = pd.DataFrame(res[4:].reshape((-1, 3)), columns=['width', 'location', 'area'])
        print('\nFit Summary:')
        print('------------')
        print('Global parameters')
        print(res_globals.to_string(index=False))
        print('\nPeak parameters')
        print(res_peaks.to_string(index=False))
        print("Error:\t", self.error)


# ---- parameter uncertainties (not in the reference) ---------------------------------------------------------------
def covariance_from_normal(H, M, g, ssr, n_points, params, lower, upper, ties=None, moments=None):
    """Sandwich covariance of the weighted least-squares estimate from the normal equations of one spectrum
    (``Context.normal_equations``): ``C = s^2 H^-1 M H^-1`` with ``s^2 = sum res^2 / (N - D)``.

    The dynamic weights emphasise small peaks; they are not inverse noise levels, while the spectral noise is the
    same at every point of the unweighted data.  So the noise level comes from the unweighted residuals and the
    weights enter through H (= A^T W^2 A) and M (= A^T W^4 A); with unit weights M = H and C = s^2 H^-1.  The estimate
    assumes independent noise from point to point: zero-filled or apodised spectra have correlated noise, and the
    errors are then optimistic.

    H^-1 comes from a Cholesky factorisation of the Jacobi-scaled ``S H S``, S = diag(H_jj^-1/2) (H itself spans
    many decades).  If that fails, or some H_jj = 0 (a parameter the residual does not depend on, such as the width
    of a peak of area 0), ``C`` is all NaN and ``info['singular']`` is True.

    Returns ``(C [D, D], info)``, info = dict(sigma, dof, gradient=g, at_bound, singular); ``at_bound[j]`` flags a
    parameter within 1e-9 of its box width of a bound, where the linearisation says little.

    ``ties`` (a ``Ties``): the covariance of the tied model x = T theta + c (DESIGN K15).  H, M and g are projected
    onto the d free parameters (H_theta = T^T H T, summed member by member as the refinement does, so the identity
    map gives this function's untied result bit for bit), s^2 = sum res^2 / (N - d), and ``C = T C_theta T^T``: a
    fixed parameter has error 0 and a linked one |scale| times its master's.  ``dof`` is N - d; ``at_bound`` is judged
    on the reduced box and a linked parameter carries its master's flag.

    ``moments`` (``Context.loss_moments`` at ``params``: cost, sum w^2 res^2, sum psi^2, sum psi', sum psi'^2): the
    covariance of a robust fit (DESIGN K16, Huber 1981 section 7.6), s^2 replaced by
    K^2 [sum psi^2 / (N - D)] / [sum psi' / N]^2 with K = 1 + (D/N) Var(psi') / E[psi']^2; H and M stay those of K12.
    ``info`` then gains ``robust_factor``, that scalar over s^2 (``sigma`` stays s).  sum psi' <= 0 (a Cauchy fit with
    gross misfit) makes ``C`` all NaN and ``singular`` True.  None is the least-squares computation, bit for bit."""
    if ties is not None:
        return _tied_covariance(H, M, g, ssr, n_points, params, lower, upper, ties, moments)
    H, M, g = np.asarray(H, dtype=np.float64), np.asarray(M, dtype=np.float64), np.asarray(g, dtype=np.float64)
    x, lb, ub = (np.asarray(a, dtype=np.float64) for a in (params, lower, upper))
    D = H.shape[0]
    dof = int(n_points) - D
    sigma2 = float(ssr[1]) / dof
    tol = 1e-9 * (ub - lb)
    info = dict(sigma=float(np.sqrt(sigma2)), dof=dof, gradient=g.copy(),
                at_bound=(np.abs(x - lb) <= tol) | (np.abs(ub - x) <= tol), singular=False)
    if moments is not None:
        scalar = robust_scale(moments, n_points, D)
        info['robust_factor'] = scalar / sigma2
        if not np.isfinite(scalar):
            info['singular'] = True
            return np.full((D, D), np.nan), info
        sigma2 = scalar
    diag = np.diag(H)
    if not np.all(np.isfinite(H)) or np.any(diag <= 0):
        info['singular'] = True
        return np.full((D, D), np.nan), info
    s = 1.0 / np.sqrt(diag)
    try:
        L = np.linalg.cholesky(s[:, None] * H * s[None, :])
    except np.linalg.LinAlgError:
        info['singular'] = True
        return np.full((D, D), np.nan), info
    Linv = np.linalg.solve(L, np.eye(D))
    Hinv = s[:, None] * (Linv.T @ Linv) * s[None, :]
    C = sigma2 * (Hinv @ M @ Hinv)
    return 0.5 * (C + C.T), info


def robust_scale(moments, n_points, d):
    """Huber's scale of the sandwich for an M-estimator with d free parameters from ``moments`` (cost, sum w^2 res^2,
    sum psi^2, sum psi', sum psi'^2): K^2 [sum psi^2 / (N - d)] / [sum psi' / N]^2, K = 1 + (d/N) Var(psi') / E[psi']^2.
    NaN when sum psi' <= 0.  For the linear loss (psi = res, psi' = 1) it is sum res^2 / (N - d)."""
    m = np.asarray(moments, dtype=np.float64)
    N = float(n_points)
    if not m[3] > 0:
        return float('nan')
    mean = m[3] / N
    K = 1.0 + (d / N) * (m[4] / N - mean * mean) / (mean * mean)
    return float(K * K * (m[2] / (N - d)) / (mean * mean))


def _tied_covariance(H, M, g, ssr, n_points, params, lower, upper, ties, moments=None):
    """``covariance_from_normal`` with ``ties``: the untied computation on the free parameters, then expanded."""
    x, lb, ub = (np.asarray(a, dtype=np.float64) for a in (params, lower, upper))
    master, scale, offset = ties.arrays()
    free, lo, hi = _cabi.reduced_box(master, scale, offset, lb, ub)
    Ht, Mt, gt = ties.project(H, M, g)
    Ct, info = covariance_from_normal(Ht, Mt, gt, ssr, n_points, x[free], lo, hi, moments=moments)
    group, a = ties.groups()
    D = len(master)
    tied = group >= 0
    C = np.zeros((D, D))
    C[np.ix_(tied, tied)] = (a[tied, None] * a[None, tied]) * Ct[np.ix_(group[tied], group[tied])]
    at_bound = np.zeros(D, dtype=bool)
    at_bound[tied] = info['at_bound'][group[tied]]
    info.update(gradient=np.asarray(g, dtype=np.float64).copy(), at_bound=at_bound)
    return C, info


class Ties:
    """Fixed and linked parameters of a model of ``n_peaks`` peaks (D = 4 + 3 n_peaks), for the refinement and the
    standard errors (DESIGN K15).  Every parameter starts free; ``fix(j, value)`` holds x_j = value, and
    ``link(j, master, scale, offset)`` makes x_j = scale * x_master + offset, where the master must stay free (one
    master per dependent, no chains).  Indices come from ``index``.  The free parameters theta, in index order, are
    what the refinement moves: x = T theta + c (``matrix``, ``expand``).  Malformed ties raise ValueError at once."""

    GLOBALS = ('p0', 'p1', 'r', 'yoff')
    PEAK = ('width', 'loc', 'area')

    def __init__(self, n_peaks):
        self.n_peaks = int(n_peaks)
        self.D = 4 + 3 * self.n_peaks
        self.master = np.arange(self.D, dtype=np.int32)
        self.scale = np.ones(self.D)
        self.offset = np.zeros(self.D)

    def index(self, name, peak=None):
        """Index of ``'p0'``, ``'p1'``, ``'r'``, ``'yoff'``, or of ``'width'``, ``'loc'``, ``'area'`` of ``peak``
        (also given as ``(name, peak)``)."""
        if isinstance(name, tuple):
            name, peak = name
        if name in self.GLOBALS:
            if peak is not None:
                raise ValueError('%r is a global parameter: it takes no peak' % name)
            return self.GLOBALS.index(name)
        if name not in self.PEAK:
            raise ValueError('unknown parameter %r: one of %s' % (name, ', '.join(self.GLOBALS + self.PEAK)))
        if isinstance(peak, bool) or not isinstance(peak, (int, np.integer)) or not 0 <= peak < self.n_peaks:
            raise ValueError('peak must be an integer in [0, %d), got %r' % (self.n_peaks, peak))
        return 4 + 3 * int(peak) + self.PEAK.index(name)

    def _param(self, j):
        if isinstance(j, (str, tuple)):
            return self.index(j)
        if isinstance(j, bool) or not isinstance(j, (int, np.integer)) or not 0 <= j < self.D:
            raise ValueError('parameter index must be an integer in [0, %d), got %r' % (self.D, j))
        return int(j)

    def _dependents(self, j):
        return [i for i in range(self.D) if i != j and self.master[i] == j]

    def fix(self, j, value):
        """Hold parameter ``j`` at ``value`` (finite)."""
        j = self._param(j)
        if not np.isfinite(value):
            raise ValueError('parameter %d: offset is not finite' % j)
        if self._dependents(j):
            raise ValueError('parameter %d: it is the master of %s and cannot be fixed' % (j, self._dependents(j)))
        self.master[j], self.scale[j], self.offset[j] = -1, 1.0, float(value)
        return self

    def link(self, j, master, scale=1.0, offset=0.0):
        """x_j = ``scale`` * x_master + ``offset``; ``scale`` finite and non-zero (for zero, use ``fix``), ``offset``
        finite, ``master`` a free parameter other than j."""
        j, m = self._param(j), self._param(master)
        if m == j:
            raise ValueError('parameter %d cannot be linked to itself' % j)
        if not np.isfinite(scale) or scale == 0:
            raise ValueError('parameter %d: scale must be finite and non-zero (fix the parameter instead of a zero '
                             'scale)' % j)
        if not np.isfinite(offset):
            raise ValueError('parameter %d: offset is not finite' % j)
        if self.master[m] == -1:
            raise ValueError('parameter %d: its master %d is fixed' % (j, m))
        if self.master[m] != m:
            raise ValueError('parameter %d: its master %d is itself linked (no chains)' % (j, m))
        if self._dependents(j):
            raise ValueError('parameter %d: it is the master of %s and cannot be linked (no chains)'
                             % (j, self._dependents(j)))
        self.master[j], self.scale[j], self.offset[j] = m, float(scale), float(offset)
        return self

    def arrays(self):
        """``(master [D] int32, scale [D], offset [D])`` as ``Context.refine(ties=...)`` and the C ABI take them."""
        return self.master.copy(), self.scale.copy(), self.offset.copy()

    def free(self):
        """Indices of the free parameters theta, ascending."""
        return np.flatnonzero(self.master == np.arange(self.D))

    def groups(self):
        """``(group [D], a [D])``: the index into theta of each parameter's master (-1 for a fixed parameter) and its
        scale (1 for a free one, 0 for a fixed one)."""
        free = self.free()
        pos = np.full(self.D, -1)
        pos[free] = np.arange(free.size)
        group = np.where(self.master >= 0, pos[np.maximum(self.master, 0)], -1)
        a = np.where(self.master == np.arange(self.D), 1.0, np.where(self.master < 0, 0.0, self.scale))
        return group, a

    def matrix(self):
        """``(T [D, d], c [D])`` with x = T theta + c."""
        group, a = self.groups()
        T = np.zeros((self.D, self.free().size))
        tied = group >= 0
        T[np.flatnonzero(tied), group[tied]] = a[tied]
        c = np.where(self.master == np.arange(self.D), 0.0, self.offset)
        return T, c

    def expand(self, theta):
        """x [D] from the free parameters ``theta`` [d]: x_j = scale_j * theta + offset_j for a linked parameter (as
        numpy's ``a * t + c``, which the refinement's expansion reproduces bit for bit), the value for a fixed one."""
        theta = np.asarray(theta, dtype=np.float64)
        free = self.free()
        if theta.shape != (free.size,):
            raise ValueError('theta must have shape (%d,), got %s' % (free.size, theta.shape))
        group, a = self.groups()
        x = self.offset.copy()
        x[free] = theta
        linked = (self.master >= 0) & (self.master != np.arange(self.D))
        x[linked] = self.scale[linked] * theta[group[linked]] + self.offset[linked]
        return x

    def project(self, H, M, g):
        """``(T^T H T, T^T M T, T^T g)`` summed as the refinement sums them: over each group's members in ascending
        index (the master with scale 1), starting from the first term, so that the identity map returns H, M and g
        exactly."""
        H, M, g = (np.asarray(v, dtype=np.float64) for v in (H, M, g))
        free = self.free()
        members = [np.flatnonzero((self.master == j)) for j in free]   # the master is its own member
        a = [np.where(mem == j, 1.0, self.scale[mem]) for mem, j in zip(members, free)]
        d, width = free.size, max(len(m) for m in members)
        mem = np.array([np.r_[m, np.full(width - len(m), -1)] for m in members])
        sc = np.array([np.r_[s, np.zeros(width - len(s))] for s in a])
        out = []
        for X in (H, M):
            Xt = None
            for p in range(width):
                for q in range(width):
                    ok = (mem[:, p] >= 0)[:, None] & (mem[:, q] >= 0)[None, :]
                    t = (sc[:, p][:, None] * sc[:, q][None, :]) * X[np.ix_(np.maximum(mem[:, p], 0),
                                                                           np.maximum(mem[:, q], 0))]
                    Xt = t if Xt is None else np.where(ok, Xt + t, Xt)
            out.append(Xt)
        gt = sc[:, 0] * g[mem[:, 0]]
        for p in range(1, width):
            gt = np.where(mem[:, p] >= 0, gt + sc[:, p] * g[np.maximum(mem[:, p], 0)], gt)
        return out[0], out[1], gt


def bartlett_taper(rho):
    """``rho_k (1 - k/(L+1))`` along the last axis of ``rho`` [..., L+1]: the Bartlett (triangle) window.  The biased
    autocorrelation of a sequence and the triangle are both positive-semidefinite sequences, and so is their
    product (Schur), so the lag-weighted M formed from a tapered estimate is positive semidefinite by construction."""
    rho = np.asarray(rho, dtype=np.float64)
    L = rho.shape[-1] - 1
    return rho * (1.0 - np.arange(L + 1) / (L + 1))


def _check_noise_args(noise, max_lag, noise_acf, B, N, P):
    """The checks ``compute_uncertainties_batch`` makes before any CUDA call: returns (L, rho) with rho None unless
    ``noise_acf`` is given (then [B, L+1]); ValueError otherwise."""
    if noise not in ('white', 'correlated'):
        raise ValueError("noise must be 'white' or 'correlated', got %r" % (noise,))
    if isinstance(max_lag, bool) or not isinstance(max_lag, (int, np.integer)) or max_lag < 0:
        raise ValueError('max_lag must be an integer >= 0, got %r' % (max_lag,))
    if noise == 'white':
        if noise_acf is not None:
            raise ValueError("noise_acf is used with noise='correlated' only")
        return 0, None
    if noise_acf is None:
        return _cabi.check_lag(min(int(max_lag), N - 1), N, P), None
    rho = _cabi.check_rho(noise_acf, B, N, P)
    if not np.all(rho[:, 0] == 1.0):
        raise ValueError('noise_acf must have rho_0 = 1')
    if not np.all(np.abs(rho) <= 1.0):
        raise ValueError('noise_acf must have |rho_k| <= 1')
    return rho.shape[1] - 1, rho


def stack_fits(fits, fields):
    """The device inputs of a batch of fits of equal length and peak count: ``W, U, V, weights`` [B, N] from each
    fit's data and weights, then one [B, D] array per attribute named in ``fields``, all float64."""
    N, D = len(fits[0].data.w), len(fits[0].params)
    for f in fits:
        if len(f.data.w) != N or len(f.params) != D:
            raise ValueError('every fit of a batch must have the same number of points and peaks')
    rows = [(f.data.w, f.data.u, f.data.v, f.weights) + tuple(getattr(f, k) for k in fields) for f in fits]
    return tuple(np.stack([_cabi.as_f64(a) for a in arrs]) for arrs in zip(*rows))


def compute_uncertainties_batch(fits, noise='white', max_lag=32, noise_acf=None):
    """``compute_uncertainties()`` for many fits of equal length and peak count (what ``fit_batch`` returns) in one
    device pass: the normal equations of every spectrum at its fitted ``params`` with its fit's ``weights``, then
    ``covariance_from_normal`` per fit.  Sets ``covariance``, ``stderr`` and ``uncertainty_info`` on every fit and
    returns the list of ``stderr``.

    ``noise='white'`` (the default) assumes noise independent from point to point.  ``noise='correlated'`` uses
    ``C = s^2 H^-1 M_rho H^-1`` with ``M_rho = sum_i sum_{|k| <= L} rho_|k| a_i^T a_{i+k}``, a_i = w_i^2 A_i
    (``Context.normal_m_lagged``, DESIGN K14), and L = min(max_lag, N - 1):
      * by default rho is estimated from the residuals at ``params`` (``Context.residual_acf``), rho_k = r_k / r_0,
        and tapered by ``bartlett_taper``, which keeps M_rho positive semidefinite;
      * ``noise_acf`` [L+1] or [B, L+1] (rho_0 = 1, |rho_k| <= 1) is a known correlation used as given, with no
        taper, for example the autocorrelation of a signal-free region of the full spectrum.
    s^2 stays sum res^2 / (N - D).  These errors assume stationary noise and a residual that is noise: call
    ``refine()`` first, because after an unrefined swarm the lineshape misfit shows up as correlation.  s^2 and the
    estimated rho carry biases of order D * sum(rho) / N (a few per cent in s^2 at 4,096 points and 6 peaks with
    sum(rho) near 10).  At a correlation length of 3 points, the taper at the default L = 32 loses 4-7 % of the
    standard error, 2-4 % at L = 64.

    ``uncertainty_info`` also holds ``noise``, ``noise_acf`` (the rho used, [L+1]; [1.] for white noise),
    ``max_lag`` (L) and ``inflation`` (the correlated over the white standard error of each parameter; ones for
    white noise)."""
    fits = list(fits)
    if not fits:
        return []
    for f in fits:
        if getattr(f, 'params', None) is None:
            raise RuntimeError('compute_uncertainties needs a fitted model: call fit() first')
        if f.fit_im:
            raise NotImplementedError('uncertainties are not available with fit_im: that objective is a sum of two '
                                      'RMSEs, not a least-squares problem')
    W, U, V, weights, X = stack_fits(fits, ('params',))
    N, D = W.shape[1], X.shape[1]
    ties = [getattr(f, 'ties', None) for f in fits]
    losses = [getattr(f, 'loss', None) for f in fits]
    if noise == 'correlated' and any(lo is not None for lo in losses):
        raise NotImplementedError("noise='correlated' is not available after a robust refinement: the lag-weighted "
                                  "meat of psi is a separate derivation")
    d = max(D if t is None else t.free().size for t in ties)
    if N <= d:
        raise ValueError('the spectrum has %d points for %d parameters: no residual degrees of freedom' % (N, d))
    B, P = len(fits), (D - 4) // 3
    L, rho = _check_noise_args(noise, max_lag, noise_acf, B, N, P)
    with _cabi.pooled_context(B, N, P, device=fits[0].options.get('device')) as ctx:
        ctx.set_spectra(W, U, V, weights)
        H, M, g, ssr = ctx.normal_equations(X)
        moments = [None] * B
        for name in sorted({lo['name'] for lo in losses if lo is not None}):
            use = [lo is not None and lo['name'] == name for lo in losses]
            m = ctx.loss_moments(X, name, [lo['f_scale'] if u else 1.0 for lo, u in zip(losses, use)])
            for b in np.flatnonzero(use):
                moments[b] = m[b]
        if noise == 'correlated':
            if rho is None:
                r = ctx.residual_acf(X, L)
                r0 = r[:, :1]
                rho = bartlett_taper(np.where(r0 > 0, r / np.where(r0 > 0, r0, 1.0), np.eye(1, L + 1)))
            M_rho = ctx.normal_m_lagged(X, rho)
    for b, f in enumerate(fits):
        f.covariance, f.uncertainty_info = covariance_from_normal(H[b], M[b], g[b], ssr[b], N, f.params, f.lower,
                                                                  f.upper, ties=ties[b], moments=moments[b])
        f.stderr = np.sqrt(np.diag(f.covariance))
        lo = losses[b]
        f.uncertainty_info.update(loss='linear' if lo is None else lo['name'], f_scale=None if lo is None else
                                  lo['f_scale'], robust_factor=f.uncertainty_info.get('robust_factor', 1.0))
        inflation = np.ones(D)
        if noise == 'correlated':
            white = f.stderr
            f.covariance, f.uncertainty_info = covariance_from_normal(H[b], M_rho[b], g[b], ssr[b], N, f.params,
                                                                      f.lower, f.upper, ties=ties[b])
            f.stderr = np.sqrt(np.diag(f.covariance))
            with np.errstate(divide='ignore', invalid='ignore'):
                inflation = f.stderr / white
            if ties[b] is not None:
                inflation[ties[b].master == -1] = 1.0             # a fixed parameter: 0 / 0
        f.uncertainty_info.update(noise=noise, noise_acf=np.ones(1) if rho is None else rho[b].copy(), max_lag=L,
                                  inflation=inflation)
    return [f.stderr for f in fits]


def _check_refinable(f, fitted=False):
    if fitted and getattr(f, 'params', None) is None:
        raise RuntimeError('refine needs a fitted model: call fit() first')
    if f.fit_im:
        raise NotImplementedError('refinement is not available with fit_im: that objective is a sum of two RMSEs, '
                                  'not a least-squares problem')


def apply_refinement(fits, x, fval, passes, accepted, status, ties=None, loss='linear', f_scale=None, moments=None):
    """Store the result of ``Context.refine`` on the fits it refined (see ``FitUtility.refine``), with the ``ties``
    of each (a list, or None for none).  For a robust ``loss`` (a name), ``f_scale`` [B] and ``moments``
    (``Context.loss_moments`` at the returned x) are required: ``error`` then comes from moments[:, 1] and the cost from
    moments[:, 0]."""
    robust = loss != 'linear'
    N = len(fits[0].data.w) if fits else 0
    for b, f in enumerate(fits):
        f.ties = None if ties is None else ties[b]
        f.loss = dict(name=loss, f_scale=float(f_scale[b])) if robust else None
        f.refine_info = dict(start_params=np.array(f.params, dtype=np.float64), start_error=f.error,
                             passes=int(passes[b]), accepted=int(accepted[b]), status=int(status[b]), loss=loss,
                             f_scale=float(f_scale[b]) if robust else None,
                             cost=float(moments[b, 0]) if robust else N * float(fval[b]) ** 2)
        if accepted[b] > 0:
            f.params = x[b].copy()
            f.error = float(np.sqrt(moments[b, 1] / N)) if robust else float(fval[b])


ROBUST_MAX_ITER = 200
NORMAL_MAD = 0.6744897501960817          # scipy.special.ndtri(0.75): E MAD = NORMAL_MAD sigma for Gaussian noise
# c / sigma of each robust loss at 95 % asymptotic efficiency on Gaussian noise, (E psi')^2 / E psi^2 = 0.95
AUTO_SCALE_K = {'huber': 1.345, 'soft_l1': 1.287, 'cauchy': 2.385}
AUTO_SCALE_LIST = ("f_scale 'auto' estimates the scale of every spectrum of the call: give it once, not in a list "
                   "of scales")


def check_loss_scale(loss, f_scale, B):
    """``_cabi.check_loss`` that also takes ``f_scale='auto'`` for a robust loss: returns ``(code, 'auto')`` then, else
    what ``check_loss`` returns.  ValueError for any other string and for 'auto' inside a list of scales.  With the
    linear loss ``f_scale`` is not read."""
    code, _ = _cabi.check_loss(loss, 1.0, B)
    if code == _cabi.LOSS_LINEAR:
        return code, None
    if isinstance(f_scale, str):
        if f_scale != 'auto':
            raise ValueError("f_scale must be a number, one number per spectrum, or 'auto', got %r" % f_scale)
        return code, 'auto'
    if isinstance(f_scale, (list, tuple, np.ndarray)) and \
            any(isinstance(v, str) for v in np.ravel(np.asarray(f_scale, dtype=object))):
        raise ValueError(AUTO_SCALE_LIST)
    return _cabi.check_loss(code, f_scale, B)


def noise_level_batch(fits):
    """``noise_level()`` for many fits of equal length and peak count in one device pass: sigma = MAD / NORMAL_MAD of
    each spectrum's unweighted residuals at its ``params`` (``Context.residual_scale``, DESIGN K17), as
    ``scipy.stats.median_abs_deviation(res, scale='normal')``.  Returns sigma [B]."""
    fits = list(fits)
    if not fits:
        return np.empty(0)
    for f in fits:
        if getattr(f, 'params', None) is None:
            raise RuntimeError('noise_level needs a fitted model: call fit() first')
        if f.fit_im:
            raise NotImplementedError('noise_level is not available with fit_im: that objective is a sum of two '
                                      'RMSEs, not one residual')
    W, U, V, weights, X = stack_fits(fits, ('params',))
    with _cabi.pooled_context(len(fits), W.shape[1], (X.shape[1] - 4) // 3,
                              device=fits[0].options.get('device')) as ctx:
        ctx.set_spectra(W, U, V, weights)
        return ctx.residual_scale(X)[1] / NORMAL_MAD


def default_max_iter(max_iter, loss):
    """``max_iter`` of the refinement: as given, else 50 for the linear loss and ``ROBUST_MAX_ITER`` for a robust one
    (``loss`` a name or ``_cabi.LOSS_*`` code)."""
    if max_iter is not None:
        return max_iter
    return 50 if loss in ('linear', _cabi.LOSS_LINEAR) else ROBUST_MAX_ITER


def refine_with_loss(ctx, fits, x, lb, ub, ties=None, ties_per=None, loss='linear', f_scale=None, max_iter=None,
                     xtol=1e-6):
    """``ctx.refine`` (its spectra and weights set) and ``apply_refinement``, with the moments pass at the result for a
    robust loss.  ``loss`` and ``f_scale`` must have passed ``check_loss_scale``; ``max_iter`` None is
    ``default_max_iter``.  ``f_scale='auto'`` runs the two stages of ``FitUtility.refine``: the least-squares
    refinement, the scale from the MAD of its residuals, then the robust refinement from its result."""
    code, fs = check_loss_scale(loss, f_scale, len(fits))
    name = [k for k, v in _cabi.LOSSES.items() if v == code][0]
    if isinstance(fs, str):
        starts = [(np.array(f.params, dtype=np.float64), f.error) for f in fits]
        lsq = ctx.refine(x, lb, ub, ties=ties, max_iter=default_max_iter(max_iter, 'linear'), xtol=xtol)
        med, mad = ctx.residual_scale(lsq[0])
        sigma = mad / NORMAL_MAD
        for b in range(len(fits)):                       # every scale is checked before any fit changes
            if lsq[4][b] == _cabi.REFINE_NONFINITE or not (np.isfinite(sigma[b]) and sigma[b] > 0):
                raise ValueError("spectrum %d: f_scale='auto' needs a noise level > 0 from the least-squares residuals,"
                                 " got sigma = MAD / %r = %r (least-squares status %d)"
                                 % (b, NORMAL_MAD, sigma[b], lsq[4][b]))
        apply_refinement(fits, *lsq, ties=ties_per)
        fs = AUTO_SCALE_K[name] * sigma
        refine_with_loss(ctx, fits, lsq[0], lb, ub, ties=ties, ties_per=ties_per, loss=code, f_scale=fs,
                         max_iter=max_iter, xtol=xtol)
        for b, f in enumerate(fits):
            f.refine_info.update(start_params=starts[b][0], start_error=starts[b][1],
                                 scale=dict(sigma=float(sigma[b]), median=float(med[b]), k=AUTO_SCALE_K[name],
                                            lsq_passes=int(lsq[2][b]), lsq_accepted=int(lsq[3][b]),
                                            lsq_status=int(lsq[4][b])))
        return
    out = ctx.refine(x, lb, ub, ties=ties, loss=code, f_scale=fs, max_iter=default_max_iter(max_iter, code),
                     xtol=xtol)
    moments = None if code == _cabi.LOSS_LINEAR else ctx.loss_moments(out[0], code, fs)
    apply_refinement(fits, *out, ties=ties_per, loss=name, f_scale=fs, moments=moments)


TIES_NEED_REFINE = "options['ties'] needs options['refine'] = True: the swarm does not honour ties"
LOSS_NEEDS_REFINE = ("options['loss'] and options['f_scale'] need options['refine'] = True: the swarm keeps the "
                     "reference's objective")


def check_unrefined_options(opt):
    """ValueError for options that only the refinement honours, given without options['refine']."""
    if opt.get('ties') is not None:
        raise ValueError(TIES_NEED_REFINE)
    if opt.get('loss') is not None or opt.get('f_scale') is not None:
        raise ValueError(LOSS_NEEDS_REFINE)


def batch_ties(ties, B, P):
    """``ties`` as ``refine_batch`` takes it (None, one ``Ties`` for every spectrum, or a list of ``Ties`` or None)
    -> ``(list of B Ties or None, (master, scale, offset) [B, D] or None)``.  None entries of a list are untied
    (the identity map)."""
    if ties is None:
        return [None] * B, None
    per = list(ties) if isinstance(ties, (list, tuple)) else [ties] * B
    if len(per) != B:
        raise ValueError('ties must be one Ties or a list of %d, got %d' % (B, len(per)))
    full = [Ties(P) if t is None else t for t in per]
    for t in full:
        if not isinstance(t, Ties) or t.n_peaks != P:
            raise ValueError('every tie set must be a Ties of %d peaks' % P)
    return per, tuple(np.stack(a) for a in zip(*[t.arrays() for t in full]))


def refine_batch(fits, max_iter=None, xtol=1e-6, ties=None, loss='linear', f_scale=None):
    """``refine()`` for many fits of equal length and peak count (what ``fit_batch`` returns) in one device call:
    the spectra and each fit's ``weights`` go to a pooled context, and every spectrum runs bounded Levenberg-Marquardt
    (``Context.refine``, DESIGN K13) from its ``params`` within its box.  ``ties``: one ``Ties`` for every fit, or a
    list with one ``Ties`` (or None) per fit (DESIGN K15); each fit keeps its own as ``ties``.  ``loss`` and
    ``f_scale`` (a scalar, one per fit, or 'auto' for each fit's own, DESIGN K17) and ``max_iter`` (None:
    ``default_max_iter``) as ``FitUtility.refine`` (DESIGN K16).  Returns the list of refined ``params``."""
    fits = list(fits)
    if not fits:
        return []
    for f in fits:
        _check_refinable(f, fitted=True)
    W, U, V, weights, X, LB, UB = stack_fits(fits, ('params', 'lower', 'upper'))
    N, D = W.shape[1], X.shape[1]
    per, arrays = batch_ties(ties, len(fits), (D - 4) // 3)
    check_loss_scale(loss, f_scale, len(fits))
    cap = default_max_iter(max_iter, loss)
    if arrays is None:
        _cabi.check_refine_args(X, LB, UB, cap, xtol, len(fits), N, (D - 4) // 3)
    else:
        _cabi.check_refine_args(X, LB, UB, cap, xtol, len(fits), N, (D - 4) // 3, box=False)
        _cabi.check_ties(*arrays, LB, UB, len(fits), N, (D - 4) // 3)
    with _cabi.pooled_context(len(fits), N, (D - 4) // 3, device=fits[0].options.get('device')) as ctx:
        ctx.set_spectra(W, U, V, weights)
        refine_with_loss(ctx, fits, X, LB, UB, ties=arrays, ties_per=per, loss=loss, f_scale=f_scale,
                         max_iter=max_iter, xtol=xtol)
    return [f.params for f in fits]


# ---- automatic peak selection (utils.py:670-783) on the GPU ----------------------------------------------------
_SG_TABLES = None


def _sg_tables():
    """Savitzky-Golay(11, 4) coefficients and edge maps handed to the device: scipy's own when scipy is importable
    (what the reference would compute: utils.py:716), else the library's built-in copy (None)."""
    global _SG_TABLES
    if _SG_TABLES is None:
        try:
            import scipy.signal
            c = scipy.signal.savgol_coeffs(11, 4)
            pinv = np.linalg.pinv(np.vander(np.arange(11.0), 5))
            left = np.vander(np.arange(0, 5.0), 5) @ pinv
            right = np.vander(np.arange(6, 11.0), 5) @ pinv
            _SG_TABLES = (np.concatenate([c, left.ravel(), right.ravel()]),)
        except ImportError:
            _SG_TABLES = (None,)
    return _SG_TABLES[0]


def _ascending(w, u):
    """interp1d sorts its abscissae (stable argsort) before interpolating (utils.py:711): mirror it on the host."""
    w, u = _cabi.as_f64(w), _cabi.as_f64(u)
    if w.size > 1 and np.all(w[1:] > w[:-1]):
        return w, u
    ind = np.argsort(w, kind='mergesort')
    return np.ascontiguousarray(w[ind]), np.ascontiguousarray(u[ind])


def select_peaks_batch(ws, us, thresh=0.0, window=0.02, upsample=100, max_peaks=64, device=None, details=False):
    """``AutoPeakSelector(w, u, thresh, window).find_peaks()`` for every spectrum of a batch in one pass on the GPU.

    ``ws``, ``us``: [B, N] (or [N]) axis and phased real part of each spectrum.  Returns a list of ``Peaks`` (one per
    spectrum; ``Peak`` records with ``loc, i, height, width, bounds, baseline, area, idx``), or with ``details`` also the
    global baselines and the maxima before the width screen.  Raises ValueError where the reference does (a maximum
    without a half-height crossing of either kind: utils.py:752-753 take the argmin of an empty sequence)."""
    ws, us = np.atleast_2d(np.asarray(ws, dtype=np.float64)), np.atleast_2d(np.asarray(us, dtype=np.float64))
    if ws.shape != us.shape:
        raise ValueError('ws and us must have the same shape')
    B, N = ws.shape
    rows = [_ascending(ws[b], us[b]) for b in range(B)]
    W = np.ascontiguousarray(np.stack([r[0] for r in rows]))
    U = np.ascontiguousarray(np.stack([r[1] for r in rows]))
    with _cabi.PeakPicker(B, N, upsample=upsample, max_peaks=max_peaks, device=device) as pk:
        n_max, idx, val, base = pk.maxima(W, U, window, sg_coeffs=_sg_tables())
        n_keep = np.zeros(B, dtype=np.int32)
        keep_i = np.zeros((B, max_peaks), dtype=np.int64)
        keep_h = np.zeros((B, max_peaks))
        pre = []
        for b in range(B):
            order = np.argsort(idx[b, :n_max[b]])            # argrelmax returns ascending indices (utils.py:731)
            i_b, h_b = idx[b, :n_max[b]][order], val[b, :n_max[b]][order] - base[b]      # :737
            sel = h_b > thresh                              # :738
            n_keep[b] = int(sel.sum())
            keep_i[b, :n_keep[b]], keep_h[b, :n_keep[b]] = i_b[sel], h_b[sel]
            pre.append((i_b[sel], h_b[sel]))
        out = pk.measure(n_keep, keep_i, keep_h)
    result = []
    for b in range(B):
        peaks = Peaks()
        for k in range(n_keep[b]):
            if out['ok'][b, k] < 0:
                raise ValueError('attempt to get argmin of an empty sequence')       # as the reference does here
            if out['ok'][b, k] == 0:
                continue                                    # utils.py:755: x_left >= x_right, the peak is dropped
            p = Peak()
            p.loc, p.i = float(out['loc'][b, k]), int(keep_i[b, k])
            p.width = float(out['width'][b, k])
            p.bounds = [float(out['bounds'][b, k, 0]), float(out['bounds'][b, k, 1])]
            lo, hi = (int(t) for t in out['idx_range'][b, k])
            p.idx = (np.arange(lo, hi + 1),)                # what np.where returns (utils.py:763)
            p.baseline = float(out['baseline'][b, k])
            p.height = float(out['height'][b, k])
            p.area = float(out['area'][b, k])
            peaks.append(p)
        result.append(peaks)
    if details:
        return result, dict(baseline=base, pre=pre)
    return result


class AutoPeakSelector:
    """Drop-in for the reference's AutoPeakSelector (utils.py:670-783) with the arithmetic on the GPU: same constructor,
    ``find_maxima`` / ``find_width`` / ``find_peaks``, ``peaks`` and ``baseline`` attributes.  The upsampled arrays
    (``w``, ``u``, ``u_smoothed``: 100x the input, utils.py:713-716) stay on the device; ``plot`` is not provided."""

    def __init__(self, w, u, thresh, window):
        self.thresh = thresh
        self.window = window
        self._w, self._u = np.asarray(w, dtype=np.float64), np.asarray(u, dtype=np.float64)
        self.peaks = Peaks()
        self.baseline = None
        self._found = None

    def _run(self):
        if self._found is None:
            peaks, aux = select_peaks_batch(self._w[None], self._u[None], self.thresh, self.window, details=True)
            self._found = peaks[0]
            self.baseline = float(aux['baseline'][0])
            self._pre = aux['pre'][0]

    def find_maxima(self):
        self._run()
        w_lo, w_hi, M = self._w.min(), self._w.max(), self._w.size * 100
        step = (w_hi - w_lo) / (M - 1)
        self.peaks = Peaks()
        for i, h in zip(*self._pre):
            p = Peak()
            p.i, p.height = int(i), float(h)
            p.loc = float(w_hi if i == M - 1 else i * step + w_lo)     # np.linspace's own expression (utils.py:713)
            self.peaks.append(p)

    def find_width(self):
        self._run()
        self.peaks = self._found

    def find_peaks(self):
        self.find_maxima()
        self.find_width()
