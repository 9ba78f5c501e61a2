"""ctypes binding of libnmrfit_b200.so (include/nmrfit_b200.h).

There is no CPU fallback: if the shared library has not been built
(``python -c 'import __graft_entry__ as g; g.build()'``) or no CUDA device is
usable, the first call raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('NMRFIT_B200_LIB') or os.path.join(_HERE, 'csrc', 'libnmrfit_b200.so')

OK = 0
FP64, FP32 = 0, 1
REAL_ONLY, IM_REFERENCE, IM_SUM = 0, 1, 2
ALGO_AUTO, ALGO_GENERAL, ALGO_UNIFORM = 0, 1, 2
FUSED_AUTO, FUSED_OFF, FUSED_REQUIRE = 0, 1, 2
RUNNING, STOP_MINFUNC, STOP_MINSTEP, STOP_MAXITER, STOP_PEER_LOST = 0, 1, 2, 3, 4
REFINE_CONVERGED, REFINE_STALLED, REFINE_MAX_ITER, REFINE_NONFINITE = 1, 2, 3, 4
LOSS_LINEAR, LOSS_HUBER, LOSS_SOFT_L1, LOSS_CAUCHY = 0, 1, 2, 3
LOSSES = {'linear': LOSS_LINEAR, 'huber': LOSS_HUBER, 'soft_l1': LOSS_SOFT_L1, 'cauchy': LOSS_CAUCHY}

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)


class NmrfitError(RuntimeError):
    """A libnmrfit_b200 call returned a non-zero status."""

    def __init__(self, code, message):
        super().__init__('libnmrfit_b200 error %d: %s' % (code, message))
        self.code = code


class PsoOpts(ctypes.Structure):
    _fields_ = [('swarmsize', ctypes.c_int), ('maxiter', ctypes.c_int),
                ('omega', ctypes.c_double), ('phip', ctypes.c_double), ('phig', ctypes.c_double),
                ('minstep', ctypes.c_double), ('minfunc', ctypes.c_double),
                ('fit_im', ctypes.c_int), ('bounds_per_spectrum', ctypes.c_int),
                ('seed', ctypes.c_ulonglong), ('particle_offset', ctypes.c_longlong),
                ('spectrum_offset', ctypes.c_longlong)]


# name -> (restype, argtypes); every symbol include/nmrfit_b200.h declares
_vp, _i, _d = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
SIGNATURES = {
    'nmrfit_abi_version': (_i, []),
    'nmrfit_last_error': (ctypes.c_char_p, []),
    'nmrfit_device_count': (_i, [c_int_p]),
    'nmrfit_ctx_create': (_i, [ctypes.POINTER(_vp), _i, _i, _i, _i, _i]),
    'nmrfit_ctx_destroy': (None, [_vp]),
    'nmrfit_ctx_set_spectrum': (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    'nmrfit_ctx_set_spectra': (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp]),
    'nmrfit_ctx_compute_weights': (_i, [_vp, _vp, _vp, _i, _i, _d, _vp, _vp]),
    'nmrfit_ctx_normal_equations': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'nmrfit_normal_eq_plan': (_i, [_i, _i, c_int_p]),
    'nmrfit_ctx_refine': (_i, [_vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp, _vp, _vp]),
    'nmrfit_ctx_refine_tied': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp, _vp, _vp]),
    'nmrfit_ctx_normal_equations_loss': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    'nmrfit_ctx_loss_moments': (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    'nmrfit_ctx_refine_loss': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _d, _vp, _vp, _vp, _vp, _vp]),
    'nmrfit_ctx_residual_acf': (_i, [_vp, _vp, _i, _vp, _vp]),
    'nmrfit_ctx_residuals': (_i, [_vp, _vp, _vp, _vp]),
    'nmrfit_ctx_residual_scale': (_i, [_vp, _vp, _vp, _vp]),
    'nmrfit_ctx_normal_m_lagged': (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    'nmrfit_lagged_plan': (_i, [_i, _i, _i, c_int_p]),
    'nmrfit_ctx_set_algorithm': (_i, [_vp, _i]),
    'nmrfit_ctx_get_algorithm': (_i, [_vp, _i, c_int_p]),
    'nmrfit_ctx_set_tuning': (_i, [_vp, _i, _i, _i, _i]),
    'nmrfit_ctx_get_tuning': (_i, [_vp, _i, c_int_p, c_int_p, c_int_p, c_int_p, c_int_p]),
    'nmrfit_ctx_set_variant': (_i, [_vp, _i, _i, _i]),
    'nmrfit_ctx_get_variant': (_i, [_vp, _i, c_int_p, c_int_p]),
    'nmrfit_ctx_set_far_cells': (_i, [_vp, _i]),
    'nmrfit_ctx_set_fused': (_i, [_vp, _i]),
    'nmrfit_ctx_fused_launches': (_i, [_vp, ctypes.POINTER(ctypes.c_longlong)]),
    'nmrfit_ctx_fused_timing': (_i, [_vp, _i, _vp]),
    'nmrfit_ctx_profile': (_i, [_vp, _i]),
    'nmrfit_ctx_profile_read': (_i, [_vp, c_double_p, ctypes.POINTER(ctypes.c_longlong)]),
    'nmrfit_ctx_profile_read_split': (_i, [_vp, c_double_p, c_double_p, ctypes.POINTER(ctypes.c_longlong)]),
    'nmrfit_objective_batch': (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    'nmrfit_objective_batch_host': (_i, [_vp, _vp, _i, _i, _vp]),
    'nmrfit_ctx_mt19937_shape': (_i, [_vp, ctypes.c_longlong]),
    'nmrfit_ctx_mt19937': (_i, [_vp, _vp, c_int_p, ctypes.c_longlong, ctypes.POINTER(_vp), ctypes.POINTER(_vp), _vp]),
    'nmrfit_pso_begin': (_i, [_vp, _vp, _vp, ctypes.POINTER(PsoOpts), _vp, _vp, _vp]),
    'nmrfit_pso_advance': (_i, [_vp, _vp, _vp, _vp]),
    'nmrfit_pso_step': (_i, [_vp, _vp, _vp, _vp]),
    'nmrfit_pso_peer_export': (_i, [_vp, _i, _i, _vp, ctypes.POINTER(_vp)]),
    'nmrfit_pso_peer_open': (_i, [_vp, _vp, _vp]),
    'nmrfit_pso_commit_peers': (_i, [_vp, _vp]),
    'nmrfit_pso_step_peers': (_i, [_vp, _vp, _vp, _vp]),
    'nmrfit_pso_peer_error': (_i, [_vp, c_int_p]),
    'nmrfit_pso_run_peers': (_i, [_vp, _i, _vp, _vp, c_int_p, c_int_p, _vp]),
    'nmrfit_pso_peer_timeout': (_i, [_vp, _d]),
    'nmrfit_objective_spectrum_host': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    'nmrfit_ctx_mt19937_begin': (_i, [_vp, _vp, _i, ctypes.c_longlong, ctypes.POINTER(_vp), ctypes.POINTER(_vp)]),
    'nmrfit_ctx_mt19937_end': (_i, [_vp, _vp, ctypes.POINTER(_i)]),
    'nmrfit_comm_init_all': (_i, [_vp, _i]),
    'nmrfit_comm_commit': (_i, [_vp, _i]),
    'nmrfit_comm_run': (_i, [_vp, _i, _i, _vp, _vp, ctypes.POINTER(_i), ctypes.POINTER(_i)]),
    'nmrfit_pso_record': (_i, [_vp, ctypes.POINTER(_vp), c_int_p]),
    'nmrfit_pso_commit': (_i, [_vp, _vp, _i, _vp]),
    'nmrfit_pso_run': (_i, [_vp, _i, _vp, _vp, c_int_p, _vp]),
    'nmrfit_pso_get_best': (_i, [_vp, _vp, _vp, _vp, _vp]),
    'nmrfit_pso_get_state': (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    'nmrfit_ps2': (_i, [_vp, _vp, _i, _d, _d, _i, _vp, _vp, _vp]),
    'nmrfit_ps2_host': (_i, [_i, _vp, _vp, _i, _d, _d, _i, _vp, _vp]),
    'nmrfit_voigt': (_i, [_vp, _i, _d, _d, _d, _d, _d, _vp, _vp]),
    'nmrfit_voigt_host': (_i, [_i, _vp, _i, _d, _d, _d, _d, _d, _vp]),
    'nmrfit_kk': (_i, [_vp, _i, _d, _d, _d, _d, _d, _vp, _vp]),
    'nmrfit_kk_host': (_i, [_i, _vp, _i, _d, _d, _d, _d, _d, _vp]),
    'nmrfit_generate_result': (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'nmrfit_generate_result_host': (_i, [_i, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    'nmrfit_phase_create': (_i, [ctypes.POINTER(_vp), _i, _i, _i, _vp, _vp]),
    'nmrfit_phase_destroy': (None, [_vp]),
    'nmrfit_phase_brute': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    'nmrfit_phase_acme': (_i, [_vp, _vp, _i, _vp]),
    'nmrfit_peaks_create': (_i, [ctypes.POINTER(_vp), _i, _i, _i, _i, _i]),
    'nmrfit_peaks_destroy': (None, [_vp]),
    'nmrfit_peaks_maxima': (_i, [_vp, _vp, _vp, _d, _vp, _i, _d, _vp, _vp, _vp, _vp]),
    'nmrfit_peaks_measure': (_i, [_vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'nmrfit_peaks_probe': (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp]),
    'nmrfit_host_alloc': (_i, [ctypes.c_size_t, ctypes.POINTER(_vp)]),
    'nmrfit_host_free': (_i, [_vp]),
    'nmrfit_fp64_peak': (_i, [_i, _i, _i, c_double_p, c_double_p]),
    'nmrfit_launch_count': (ctypes.c_longlong, []),
}

_lib = None


def lib():
    """The loaded library (loads on first use; raises if it is not built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                'libnmrfit_b200.so is not built (%s). Build it with '
                '`python -c "import __graft_entry__ as g; g.build()"` from the repo root. '
                'nmrfit_b200 has no CPU fallback.' % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)       # AttributeError here = header and library disagree
            fn.restype = res
            fn.argtypes = args
        if handle.nmrfit_abi_version() != 2:
            raise ImportError('libnmrfit_b200.so ABI version mismatch')
        _lib = handle
    return _lib


def check(status):
    if status != OK:
        raise NmrfitError(status, lib().nmrfit_last_error().decode('utf-8', 'replace'))


def as_f64(a):
    """C-contiguous float64 view/copy of ``a``."""
    return np.ascontiguousarray(a, dtype=np.float64)


def ptr(a):
    """void* of a numpy array, a torch tensor (``data_ptr``), an int address, or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return ctypes.c_void_p(a.ctypes.data)
    if hasattr(a, 'data_ptr'):
        return ctypes.c_void_p(a.data_ptr())
    return ctypes.c_void_p(int(a))


def device_count():
    n = ctypes.c_int(0)
    check(lib().nmrfit_device_count(ctypes.byref(n)))
    return n.value


NORMAL_EQ_PLAN_KEYS = ('point_groups', 'slices', 'tasks', 'tasks_per_slice', 'threads', 'tile_points', 'chunk_points',
                       'n_chunks', 'smem_bytes', 'scratch_doubles')


def normal_equations_plan(n_points, n_peaks):
    """Launch plan of ``Context.normal_equations`` for ``n_points`` points and ``n_peaks`` peaks (host only, no CUDA
    call): a dict of ``NORMAL_EQ_PLAN_KEYS``.  ``scratch_doubles`` is per spectrum."""
    out = (ctypes.c_int * len(NORMAL_EQ_PLAN_KEYS))()
    check(lib().nmrfit_normal_eq_plan(int(n_points), int(n_peaks), out))
    return dict(zip(NORMAL_EQ_PLAN_KEYS, out))


LAGGED_PLAN_KEYS = ('point_groups', 'slices', 'tasks', 'tasks_per_slice', 'threads', 'tile_points', 'chunk_points',
                    'n_chunks', 'smem_bytes', 'scratch_doubles', 'max_lag', 'acf_chunk_points', 'acf_n_chunks',
                    'acf_scratch_doubles')


def lagged_plan(n_points, n_peaks, max_lag=0):
    """Launch plan of ``Context.residual_acf`` and ``Context.normal_m_lagged`` (host only, no CUDA call): a dict of
    ``LAGGED_PLAN_KEYS``; ``max_lag`` is the largest lag the passes take at ``n_peaks``.  Scratch sizes are per
    spectrum."""
    out = (ctypes.c_int * len(LAGGED_PLAN_KEYS))()
    check(lib().nmrfit_lagged_plan(int(n_points), int(n_peaks), int(max_lag), out))
    return dict(zip(LAGGED_PLAN_KEYS, out))


def check_lag(max_lag, N, P):
    """The lag checks of the lagged passes (the library makes them again): returns int(max_lag), else ValueError."""
    if P > 64:
        raise ValueError('the lagged passes support at most 64 peaks (D <= 196), got %d' % P)
    if isinstance(max_lag, bool) or int(max_lag) != max_lag:
        raise ValueError('max_lag must be an integer, got %r' % (max_lag,))
    L = int(max_lag)
    if L < 0:
        raise ValueError('max_lag must be >= 0')
    if L >= N:
        raise ValueError('max_lag must be below the number of points, %d' % N)
    cap = lagged_plan(N, P)['max_lag']
    if L > cap:
        raise ValueError('max_lag %d is above the cap of %d at %d peaks' % (L, cap, P))
    return L


def check_rho(rho, B, N, P):
    """``rho`` [L+1] (every spectrum) or [B, L+1] as a fresh C-contiguous [B, L+1] float64 array, with its lag
    checked and every value finite.  ValueError otherwise."""
    rho = np.asarray(rho, dtype=np.float64)
    if rho.ndim not in (1, 2) or rho.shape[-1] < 1 or (rho.ndim == 2 and rho.shape[0] != B):
        raise ValueError('rho must have shape (L+1,) or (%d, L+1), got %s' % (B, rho.shape))
    check_lag(rho.shape[-1] - 1, N, P)
    if not np.all(np.isfinite(rho)):
        raise ValueError('every rho must be finite')
    return np.array(np.broadcast_to(rho, (B, rho.shape[-1])), dtype=np.float64, order='C')


def check_refine_args(x, lb, ub, max_iter, xtol, B, N, P, box=True):
    """The checks ``Context.refine`` makes before any CUDA call (the library makes them again): returns fresh
    C-contiguous float64 copies of ``x`` [B, D] and of ``lb``, ``ub`` broadcast to [B, D].  ValueError otherwise.
    ``box=False`` leaves the box, the start and the degrees of freedom to ``check_ties``."""
    D = 4 + 3 * P
    if P > 64:
        raise ValueError('refinement supports at most 64 peaks (D <= 196), got %d' % P)
    if box and N <= D:
        raise ValueError('the spectrum has %d points for %d parameters: no residual degrees of freedom' % (N, D))
    x = np.array(x, dtype=np.float64, order='C')
    if x.shape != (B, D):
        raise ValueError('x must have shape (%d, %d), got %s' % (B, D, x.shape))
    try:
        lb, ub = (np.ascontiguousarray(np.broadcast_to(np.asarray(a, dtype=np.float64), (B, D))) for a in (lb, ub))
    except ValueError:
        raise ValueError('lb and ub must have shape (%d, %d) or (%d,)' % (B, D, D)) from None
    if int(max_iter) < 1:
        raise ValueError('max_iter must be >= 1')
    if not float(xtol) > 0:
        raise ValueError('xtol must be > 0')
    if not box:
        return x, lb, ub
    if not np.all(ub > lb):
        raise ValueError('every lower bound must be below its upper bound')
    if not np.all((x >= lb) & (x <= ub)):
        raise ValueError('the start must lie inside its box')
    return x, lb, ub


def reduced_box(master, scale, offset, lb, ub):
    """The box of the free parameters of one tie map [D] (DESIGN K15): ``(free, lo, hi)``, ``free`` their indices in
    ascending order and [lo, hi] each one's own box intersected with the box of every dependent mapped through its tie,
    computed as the library computes it.  ``lb``, ``ub`` are [D], or [n, D] for n spectra sharing the map (then lo, hi
    are [n, d]).  ValueError, naming the parameter and its master, where a box is empty or a single point.  The map
    itself must have passed ``check_tie_map``."""
    lb, ub = np.asarray(lb, dtype=np.float64), np.asarray(ub, dtype=np.float64)
    D = len(master)
    free = np.flatnonzero(master == np.arange(D))
    lo, hi = lb[..., free].copy(), ub[..., free].copy()
    for m, j in enumerate(free):
        if not np.all(hi[..., m] > lo[..., m]):
            raise ValueError('parameter %d (a master or free): its box is empty or a single point' % j)
        for i in np.flatnonzero(master == j):
            if i == j:
                continue
            li, ui = (lb[..., i] - offset[i]) / scale[i], (ub[..., i] - offset[i]) / scale[i]
            if scale[i] < 0:
                li, ui = ui, li
            lo[..., m], hi[..., m] = np.maximum(lo[..., m], li), np.minimum(hi[..., m], ui)
            if not np.all((hi[..., m] > lo[..., m]) & ~np.isnan(li) & ~np.isnan(ui)):
                raise ValueError('parameter %d and its master %d: the reduced box is empty or a single point' % (i, j))
    return free, lo, hi


def check_tie_map(master, scale, offset):
    """One tie map [D] (``master`` int, ``scale``, ``offset`` float64; DESIGN K15): ValueError, naming the parameter,
    for a master out of [-1, D), a chain, a fixed master, a zero or non-finite scale of a linked parameter and a
    non-finite offset of a fixed or linked one."""
    D = len(master)
    for j in range(D):
        m = int(master[j])
        if m < -1 or m >= D:
            raise ValueError('parameter %d: master %d is out of range (-1 fixed, j free, else a free parameter below '
                             '%d)' % (j, m, D))
        if m == j:
            continue
        if not np.isfinite(offset[j]):
            raise ValueError('parameter %d: offset is not finite' % j)
        if m == -1:
            continue
        if not np.isfinite(scale[j]) or scale[j] == 0:
            raise ValueError('parameter %d: scale must be finite and non-zero (fix the parameter instead of a zero '
                             'scale)' % j)
        if master[m] == -1:
            raise ValueError('parameter %d: its master %d is fixed' % (j, m))
        if master[m] != m:
            raise ValueError('parameter %d: its master %d is itself linked (no chains)' % (j, m))


def check_ties(master, scale, offset, lb, ub, B, N, P):
    """The checks ``Context.refine(ties=...)`` makes before any CUDA call, as ``nmrfit_ctx_refine_tied`` makes them:
    ``master``, ``scale``, ``offset`` of shape [D] (every spectrum) or [B, D], ``lb``, ``ub`` [B, D] or [D].  Returns
    C-contiguous [B, D] int32 / float64 / float64 copies of the map, else ValueError naming the spectrum and the
    parameter (a malformed map, an empty or single-point reduced box, or no more points than free parameters)."""
    D = 4 + 3 * P
    try:
        master = np.broadcast_to(np.asarray(master), (B, D))
        scale, offset, lb, ub = (np.broadcast_to(np.asarray(a, dtype=np.float64), (B, D))
                                 for a in (scale, offset, lb, ub))
    except ValueError:
        raise ValueError('the tie arrays, lb and ub must have shape (%d, %d) or (%d,)' % (B, D, D)) from None
    if master.dtype.kind not in 'iu' and not np.all(master == np.round(master)):
        raise ValueError('tie masters must be integers')
    master = np.ascontiguousarray(master, dtype=np.int32)
    # each distinct map is checked once, its reduced box over all the spectra that carry it at once; a refusal is
    # then located spectrum by spectrum for its message
    maps = np.concatenate([master.view(np.uint32).astype(np.uint64), scale.view(np.uint64), offset.view(np.uint64)],
                          axis=1)
    _, first, which = np.unique(maps, axis=0, return_index=True, return_inverse=True)
    for k, b0 in enumerate(first):
        group = np.flatnonzero(which.ravel() == k)
        m, s, o = master[b0], scale[b0], offset[b0]
        try:
            check_tie_map(m, s, o)
            free = reduced_box(m, s, o, lb[group], ub[group])[0]
        except ValueError:
            for b in group:
                try:
                    check_tie_map(m, s, o)
                    reduced_box(m, s, o, lb[b], ub[b])
                except ValueError as e:
                    raise ValueError('spectrum %d, %s' % (b, e)) from None
        if N <= free.size:
            raise ValueError('spectrum %d: %d points for %d free parameters: no residual degrees of freedom'
                             % (group[0], N, free.size))
    return master, np.ascontiguousarray(scale), np.ascontiguousarray(offset)


def check_loss(loss, f_scale, B):
    """The loss checks of the robust entry points (the library makes them again): ``loss`` a ``LOSS_*`` code or one of
    ``LOSSES``' names, ``f_scale`` a scalar or [B], finite and > 0, for a robust loss (not read for linear).  Returns
    ``(code, f_scale as a fresh [B] float64 array, or None for linear)``, else ValueError naming the spectrum."""
    if isinstance(loss, str):
        if loss not in LOSSES:
            raise ValueError('unknown loss %r: one of %s' % (loss, ', '.join(LOSSES)))
        loss = LOSSES[loss]
    if isinstance(loss, bool) or not isinstance(loss, (int, np.integer)) or loss not in LOSSES.values():
        raise ValueError('unknown loss %r: one of %s or their LOSS_* codes' % (loss, ', '.join(LOSSES)))
    if loss == LOSS_LINEAR:
        return LOSS_LINEAR, None
    if f_scale is None:
        raise ValueError('a robust loss needs f_scale, the scale c of the residual in units of the data')
    try:
        fs = np.array(np.broadcast_to(np.asarray(f_scale, dtype=np.float64), (B,)), dtype=np.float64)
    except (TypeError, ValueError):
        raise ValueError('f_scale must be a scalar or have shape (%d,)' % B) from None
    bad = np.flatnonzero(~(np.isfinite(fs) & (fs > 0)))
    if bad.size:
        raise ValueError('spectrum %d: f_scale must be finite and > 0, got %r' % (bad[0], fs[bad[0]]))
    return int(loss), fs


def default_device():
    """LOCAL_RANK under torchrun, else NMRFIT_DEVICE, else 0."""
    for key in ('NMRFIT_DEVICE', 'LOCAL_RANK'):
        if os.environ.get(key):
            return int(os.environ[key])
    return 0


class _Handle:
    """Owner of one library handle ``_h``, freed by the C function named ``_destroy`` on ``close()``, at the end of a
    ``with`` block or when the owner is collected."""

    _destroy = None

    def close(self):
        if getattr(self, '_h', None) is not None and self._h:
            getattr(lib(), self._destroy)(self._h)
            self._h = ctypes.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class Context(_Handle):
    """Owner of one ``nmrfit_ctx``: a batch of spectra resident on one GPU."""

    _destroy = 'nmrfit_ctx_destroy'

    def __init__(self, n_spectra, n_points, n_peaks, device=None, precision=FP64):
        self._h = ctypes.c_void_p()
        self.device = default_device() if device is None else int(device)
        self.B, self.N, self.P = int(n_spectra), int(n_points), int(n_peaks)
        self.D = 4 + 3 * self.P
        self.precision = precision
        check(lib().nmrfit_ctx_create(ctypes.byref(self._h), self.device, self.B, self.N, self.P, precision))
        self._keep = []

    # -- spectra
    def set_spectrum(self, b, w, u, v, weights):
        arrs = [as_f64(a) for a in (w, u, v, weights)]
        for a in arrs:
            if a.shape != (self.N,):
                raise ValueError('spectrum arrays must have shape (%d,), got %s' % (self.N, a.shape))
        check(lib().nmrfit_ctx_set_spectrum(self._h, int(b), *[ptr(a) for a in arrs]))

    def set_spectra(self, w, u, v, weights=None, b0=0):
        """Bulk upload: ``w, u, v`` (and optionally ``weights``) are [count, N] arrays for spectra b0..b0+count-1."""
        arrs = [as_f64(a) for a in (w, u, v)]
        count = arrs[0].shape[0]
        wts = None if weights is None else as_f64(weights)
        for a in arrs + ([wts] if wts is not None else []):
            if a.shape != (count, self.N):
                raise ValueError('spectra arrays must have shape (%d, %d), got %s' % (count, self.N, a.shape))
        check(lib().nmrfit_ctx_set_spectra(self._h, int(b0), count, *[ptr(a) for a in arrs], ptr(wts)))

    def compute_weights(self, peak_bounds, peak_values, sweeps=10, omega=0.33333333, want_host=True, stream=None):
        """Residual weights of every spectrum on the device (utils.py:191-224).  ``peak_bounds`` [B, K, 2],
        ``peak_values`` [B, K].  Returns the [B, N] weights when ``want_host``."""
        pb, pv = as_f64(peak_bounds), as_f64(peak_values)
        if pb.ndim != 3 or pb.shape[0] != self.B or pb.shape[2] != 2 or pv.shape != pb.shape[:2]:
            raise ValueError('peak_bounds must be [%d, K, 2] and peak_values [%d, K]' % (self.B, self.B))
        out = result_empty(self.B * self.N).reshape(self.B, self.N) if want_host else None
        check(lib().nmrfit_ctx_compute_weights(self._h, ptr(pb), ptr(pv), pb.shape[1], int(sweeps), float(omega),
                                               ptr(out), ptr(stream)))
        return out

    def _params(self, x):
        """One parameter vector per spectrum, ``x`` [B, D], as float64 for the post-fit passes."""
        x = as_f64(x)
        if x.shape != (self.B, self.D):
            raise ValueError('x must have shape (%d, %d), got %s' % (self.B, self.D, x.shape))
        return x

    def normal_equations(self, x, stream=None):
        """Normal equations of the objective at ``x`` [B, D] (one parameter vector per spectrum) over the spectra and
        weights the context holds: returns host arrays ``H`` [B, D, D] = sum w^2 A^T A, ``M`` [B, D, D] = sum w^4 A^T A,
        ``g`` [B, D] = sum w^2 res A and ``ssr`` [B, 2] = (sum w^2 res^2, sum res^2), with res = Vdata - Vfit and
        A = d res / dx (include/nmrfit_b200.h)."""
        x = self._params(x)
        H = np.empty((self.B, self.D, self.D))
        M = np.empty((self.B, self.D, self.D))
        g = np.empty((self.B, self.D))
        ssr = np.empty((self.B, 2))
        check(lib().nmrfit_ctx_normal_equations(self._h, ptr(x), ptr(H), ptr(M), ptr(g), ptr(ssr), ptr(stream)))
        return H, M, g, ssr

    def normal_equations_loss(self, x, loss, f_scale=None, stream=None):
        """Robust normal equations at ``x`` [B, D] (DESIGN K16): returns host arrays ``H`` [B, D, D] =
        sum w^2 rho' A^T A, ``g`` [B, D] = sum w^2 rho' res A and ``cost`` [B] = sum w^2 c^2 rho, with z = (res/c)^2,
        c = ``f_scale`` (scalar or [B]) and ``loss`` a ``LOSS_*`` code or name.  For linear they are
        ``normal_equations``' H, g and ssr[:, 0] bit for bit."""
        loss, fs = check_loss(loss, f_scale, self.B)
        x = self._params(x)
        H = np.empty((self.B, self.D, self.D))
        g = np.empty((self.B, self.D))
        cost = np.empty(self.B)
        check(lib().nmrfit_ctx_normal_equations_loss(self._h, ptr(x), loss, ptr(fs), ptr(H), ptr(g), ptr(cost),
                                                     ptr(stream)))
        return H, g, cost

    def loss_moments(self, x, loss, f_scale=None, stream=None):
        """Moments of the loss at ``x`` [B, D] (DESIGN K16): [B, 5] = (cost, sum w^2 res^2, sum psi^2, sum psi',
        sum psi'^2), psi = rho'(z) res and psi' = rho' + 2 z rho'' unweighted.  Arguments as ``normal_equations_loss``."""
        loss, fs = check_loss(loss, f_scale, self.B)
        x = self._params(x)
        out = np.empty((self.B, 5))
        check(lib().nmrfit_ctx_loss_moments(self._h, ptr(x), loss, ptr(fs), ptr(out), ptr(stream)))
        return out

    def refine(self, x, lb, ub, max_iter=50, xtol=1e-6, stream=None, ties=None, loss=LOSS_LINEAR, f_scale=None):
        """Bounded Levenberg-Marquardt refinement of ``x`` [B, D] (one start per spectrum) to the least-squares optimum
        of the weighted residual within [``lb``, ``ub``] ([B, D], or [D] for every spectrum), looping on the device
        (include/nmrfit_b200.h, DESIGN K13).  Returns ``(x, f, passes, accepted, status)``: the refined [B, D] (the
        start, bit for bit, where no step was accepted), sqrt(s/N) there [B], the passes of the normal equations,
        the accepted steps and the ``REFINE_*`` status [B].

        ``ties`` = ``(master, scale, offset)``, each [D] or [B, D] (``utils.Ties.arrays()``), refines the free
        parameters of the tied model instead (DESIGN K15): fixed and linked parameters
        follow from them, the start's free entries are clipped into the reduced box and the returned x is expanded.

        ``loss`` (a ``LOSS_*`` code or name) with ``f_scale`` (scalar or [B]) minimises the robust cost
        sum w^2 c^2 rho((res/c)^2) instead (``nmrfit_ctx_refine_loss``, DESIGN K16); f is then sqrt(cost/N).  Linear is
        the least-squares refinement bit for bit."""
        loss, fs = check_loss(loss, f_scale, self.B)
        if ties is None:
            x, lb, ub = check_refine_args(x, lb, ub, max_iter, xtol, self.B, self.N, self.P)
        else:
            x, lb, ub = check_refine_args(x, lb, ub, max_iter, xtol, self.B, self.N, self.P, box=False)
            master, scale, offset = check_ties(*ties, lb, ub, self.B, self.N, self.P)
        f = np.empty(self.B)
        passes, accepted, status = (np.empty(self.B, dtype=np.int32) for _ in range(3))
        tie_ptrs = (None, None, None) if ties is None else (ptr(master), ptr(scale), ptr(offset))
        check(lib().nmrfit_ctx_refine_loss(self._h, ptr(x), ptr(lb), ptr(ub), *tie_ptrs, loss, ptr(fs), int(max_iter),
                                           float(xtol), ptr(f), ptr(passes), ptr(accepted), ptr(status), ptr(stream)))
        return x, f, passes, accepted, status

    def residual_acf(self, x, max_lag, stream=None):
        """Residual autocorrelation at ``x`` [B, D] over the spectra the context holds: returns ``r`` [B, L+1] on the
        host, r_k = sum_{i < N-k} res_i res_{i+k} (the biased form; r_0 is ``normal_equations``' ssr[:, 1]).
        ``max_lag`` = L, 0 <= L < N and at most ``lagged_plan(N, P)['max_lag']``."""
        L = check_lag(max_lag, self.N, self.P)
        x = self._params(x)
        r = np.empty((self.B, L + 1))
        check(lib().nmrfit_ctx_residual_acf(self._h, ptr(x), L, ptr(r), ptr(stream)))
        return r

    def residuals(self, x, stream=None):
        """The unweighted residuals res = Vdata - Vfit at ``x`` [B, D] over the spectra the context holds, the residual
        of ``normal_equations``: returns [B, N] on the host (DESIGN K17)."""
        x = self._params(x)
        res = np.empty((self.B, self.N))
        check(lib().nmrfit_ctx_residuals(self._h, ptr(x), ptr(res), ptr(stream)))
        return res

    def residual_scale(self, x, stream=None):
        """The median of the residuals at ``x`` [B, D] and their median absolute deviation, each as ``np.median`` gives
        it (exact selection on the device, DESIGN K17): returns ``(median [B], MAD [B])``.  MAD / 0.6744897501960817
        (``utils.NORMAL_MAD``) is the normal-consistent noise level, ``scipy.stats.median_abs_deviation(res,
        scale='normal')``."""
        x = self._params(x)
        out = np.empty((self.B, 2))
        check(lib().nmrfit_ctx_residual_scale(self._h, ptr(x), ptr(out), ptr(stream)))
        return out[:, 0].copy(), out[:, 1].copy()

    def normal_m_lagged(self, x, rho, stream=None):
        """Lag-weighted M at ``x`` [B, D]: returns [B, D, D] = sum_i sum_{|k| <= L} rho_|k| a_i^T a_{i+k}, a_i = w_i^2 A_i
        (rows outside the spectrum are zero), from ``rho`` [L+1] or [B, L+1].  With rho = [1] it is ``normal_equations``'
        M.  The result is exactly symmetric."""
        rho = check_rho(rho, self.B, self.N, self.P)
        x = self._params(x)
        M = np.empty((self.B, self.D, self.D))
        check(lib().nmrfit_ctx_normal_m_lagged(self._h, ptr(x), ptr(rho), rho.shape[1] - 1, ptr(M), ptr(stream)))
        return M

    def set_algorithm(self, algorithm=ALGO_AUTO):
        """ALGO_AUTO (default), ALGO_GENERAL (any axis) or ALGO_UNIFORM (require the uniform-axis kernel)."""
        check(lib().nmrfit_ctx_set_algorithm(self._h, int(algorithm)))

    def get_algorithm(self, fit_im=REAL_ONLY):
        """Which objective kernel a launch with this ``fit_im`` would run."""
        a = ctypes.c_int(0)
        check(lib().nmrfit_ctx_get_algorithm(self._h, int(fit_im), ctypes.byref(a)))
        return a.value

    def set_tuning(self, threads=0, points_per_thread=0, exp_table_bits=0, particles_per_cta=0):
        check(lib().nmrfit_ctx_set_tuning(self._h, threads, points_per_thread, exp_table_bits, particles_per_cta))

    def get_tuning(self, n_particles):
        vals = [ctypes.c_int(0) for _ in range(5)]
        check(lib().nmrfit_ctx_get_tuning(self._h, int(n_particles), *[ctypes.byref(v) for v in vals]))
        keys = ('threads', 'points_per_thread', 'exp_table_bits', 'particles_per_cta', 'n_point_tiles')
        return dict(zip(keys, (v.value for v in vals)))

    def set_variant(self, variant=-1, stages=0, occupancy=0):
        """FP64 uniform-axis evaluation kernel: -1 library's choice, 0 one particle group per CTA, 1 streamed
        (``stages`` ring slots, ``occupancy`` 2 or 3 CTAs of 256 threads per SM; 0 = auto)."""
        check(lib().nmrfit_ctx_set_variant(self._h, int(variant), int(stages), int(occupancy)))

    def set_far_cells(self, cells=0):
        """Far-field cells per region (0 = by axis length, or 1, 2, 4); applies to every FP64 uniform-axis kernel."""
        check(lib().nmrfit_ctx_set_far_cells(self._h, int(cells)))

    def get_variant(self, n_particles):
        v, st = ctypes.c_int(0), ctypes.c_int(0)
        check(lib().nmrfit_ctx_get_variant(self._h, int(n_particles), ctypes.byref(v), ctypes.byref(st)))
        return v.value, st.value

    def set_fused(self, mode=FUSED_AUTO):
        """FUSED_AUTO: ``pso_run`` uses the one-launch fused swarm kernel whenever the shape allows;
        FUSED_OFF: always the per-step kernels; FUSED_REQUIRE: fail if the fused kernel cannot run."""
        check(lib().nmrfit_ctx_set_fused(self._h, int(mode)))

    def fused_timing(self, enable=True, read=False):
        """Per-phase cycle counters of the fused swarm kernel (CTA 0): move, constants, objective, tile sums,
        publish, barrier, argmin, commit.  ``read`` returns what accumulated since they were enabled."""
        out = np.zeros(8, dtype=np.int64) if read else None
        check(lib().nmrfit_ctx_fused_timing(self._h, int(bool(enable)), ptr(out)))
        return out

    def fused_launches(self):
        n = ctypes.c_longlong(0)
        check(lib().nmrfit_ctx_fused_launches(self._h, ctypes.byref(n)))
        return n.value

    def profile(self, enable=True):
        check(lib().nmrfit_ctx_profile(self._h, int(bool(enable))))

    def profile_read(self):
        """(summed objective-kernel milliseconds, launches) since the last read."""
        ms, n = ctypes.c_double(0), ctypes.c_longlong(0)
        check(lib().nmrfit_ctx_profile_read(self._h, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, n.value

    def profile_read_split(self):
        """(prepare-pass ms, evaluation-kernel ms, launches) since the last read."""
        a, b, n = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_longlong(0)
        check(lib().nmrfit_ctx_profile_read_split(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(n)))
        return a.value, b.value, n.value

    # -- objective
    def objective_host(self, x, fit_im=REAL_ONLY):
        """x: [B, S, D] (or [S, D] when B == 1) host array -> f [B, S] (or [S])."""
        x = as_f64(x)
        squeeze = x.ndim == 2
        if squeeze:
            if self.B != 1:
                raise ValueError('x must be [n_spectra, n_particles, D]')
            x = x[None]
        if x.ndim != 3 or x.shape[0] != self.B or x.shape[2] != self.D:
            raise ValueError('x must have shape [%d, S, %d], got %s' % (self.B, self.D, x.shape))
        f = np.empty((self.B, x.shape[1]), dtype=np.float64)
        check(lib().nmrfit_objective_batch_host(self._h, ptr(x), x.shape[1], int(fit_im), ptr(f)))
        return f[0] if squeeze else f

    def objective_with_spectrum(self, x, w, u, v, weights, fit_im=REAL_ONLY):
        """``set_spectrum(0, ...)`` + ``objective_host(x)`` in one call (contexts of one spectrum): x [S, D] -> f [S].
        With page-locked ``x`` the comparison of the spectrum with the context's copy overlaps the evaluation."""
        x = as_f64(x)
        if x.ndim != 2 or x.shape[1] != self.D:
            raise ValueError('x must have shape [S, %d], got %s' % (self.D, x.shape))
        arrs = [as_f64(a) for a in (w, u, v, weights)]
        for a in arrs:
            if a.shape != (self.N,):
                raise ValueError('spectrum arrays must have shape (%d,), got %s' % (self.N, a.shape))
        f = np.empty(x.shape[0], dtype=np.float64)
        check(lib().nmrfit_objective_spectrum_host(self._h, *[ptr(a) for a in arrs], ptr(x), x.shape[0], int(fit_im), ptr(f)))
        return f

    def objective_device(self, x_dev, n_particles, f_dev, fit_im=REAL_ONLY, stream=None):
        """Asynchronous: x_dev/f_dev are device pointers (ints) or torch CUDA tensors."""
        check(lib().nmrfit_objective_batch(self._h, ptr(x_dev), int(n_particles), int(fit_im), ptr(f_dev),
                                           ptr(stream)))

    # -- swarm
    def pso_begin(self, lb, ub, opts, r_pos=None, r_vel=None, stream=None):
        lb, ub = as_f64(lb), as_f64(ub)
        per = 1 if lb.ndim == 2 else 0
        want = (self.B, self.D) if per else (self.D,)
        if lb.shape != want or ub.shape != want:
            raise ValueError('lb/ub must have shape %s' % (want,))
        opts.bounds_per_spectrum = per
        r_pos = self._rand(r_pos, opts.swarmsize)
        r_vel = self._rand(r_vel, opts.swarmsize)
        check(lib().nmrfit_pso_begin(self._h, ptr(lb), ptr(ub), ctypes.byref(opts), ptr(r_pos), ptr(r_vel),
                                     ptr(stream)))
        self._swarmsize = opts.swarmsize

    def _rand(self, r, S, gens=None):
        if r is None or not isinstance(r, np.ndarray):
            return r
        r = as_f64(r)
        n = self.B * S * self.D * (1 if gens is None else gens)
        if r.size != n:
            raise ValueError('random array has %d elements, expected %d' % (r.size, n))
        return r

    def pso_advance(self, rp=None, rg=None, stream=None):
        rp, rg = self._rand(rp, self._swarmsize), self._rand(rg, self._swarmsize)
        check(lib().nmrfit_pso_advance(self._h, ptr(rp), ptr(rg), ptr(stream)))

    def pso_step(self, rp=None, rg=None, stream=None):
        """One whole single-context generation (advance + commit), asynchronous."""
        rp, rg = self._rand(rp, self._swarmsize), self._rand(rg, self._swarmsize)
        check(lib().nmrfit_pso_step(self._h, ptr(rp), ptr(rg), ptr(stream)))

    def legacy_uniform_pairs(self, n_pairs, elements, stream=None):
        """The next ``2 * n_pairs`` arrays of ``elements`` doubles of numpy's GLOBAL legacy stream (np.random.rand /
        np.random.uniform), generated on the device: returns two device addresses - arrays 0, 2, 4, ... and arrays
        1, 3, 5, ... back to back - and advances ``np.random``'s state exactly as drawing them on the host would."""
        kind, key, pos, has_gauss, cached = np.random.get_state()
        if kind != 'MT19937':
            raise RuntimeError('numpy legacy generator is not MT19937')
        key = np.ascontiguousarray(key, dtype=np.uint32).copy()
        p = ctypes.c_int(int(pos))
        a, b = ctypes.c_void_p(), ctypes.c_void_p()
        check(lib().nmrfit_ctx_mt19937_shape(self._h, int(elements)))
        check(lib().nmrfit_ctx_mt19937(self._h, ptr(key), ctypes.byref(p), 2 * int(n_pairs), ctypes.byref(a),
                                       ctypes.byref(b), ptr(stream)))
        np.random.set_state((kind, key, p.value, has_gauss, cached))
        return a.value, b.value

    def legacy_uniform_pairs_begin(self, n_pairs, elements):
        """``legacy_uniform_pairs`` in two halves: queue the generation of the next ``2 * n_pairs`` arrays from
        np.random's CURRENT state and return at once (the state is not advanced yet); ``legacy_uniform_pairs_end``
        waits, advances np.random and returns the two device addresses."""
        kind, key, pos, has_gauss, cached = np.random.get_state()
        if kind != 'MT19937':
            raise RuntimeError('numpy legacy generator is not MT19937')
        key = np.ascontiguousarray(key, dtype=np.uint32)
        a, b = ctypes.c_void_p(), ctypes.c_void_p()
        check(lib().nmrfit_ctx_mt19937_shape(self._h, int(elements)))
        check(lib().nmrfit_ctx_mt19937_begin(self._h, ptr(key), int(pos), 2 * int(n_pairs), ctypes.byref(a), ctypes.byref(b)))
        return (a.value, b.value, kind, has_gauss, cached)

    def legacy_uniform_pairs_end(self, pending, advance=True):
        """Wait for a ``legacy_uniform_pairs_begin``; ``advance=False`` drops the draw (np.random keeps its state)."""
        a, b, kind, has_gauss, cached = pending
        if not advance:
            check(lib().nmrfit_ctx_mt19937_end(self._h, None, None))
            return None
        key = np.empty(624, dtype=np.uint32)
        p = ctypes.c_int(0)
        check(lib().nmrfit_ctx_mt19937_end(self._h, ptr(key), ctypes.byref(p)))
        np.random.set_state((kind, key, p.value, has_gauss, cached))
        return a, b

    # -- record exchange over peer memory
    def peer_export(self, n_ranks, rank):
        """Allocate this context's exchange window; returns (ipc_handle bytes[64], base address)."""
        handle = ctypes.create_string_buffer(64)
        base = ctypes.c_void_p()
        check(lib().nmrfit_pso_peer_export(self._h, int(n_ranks), int(rank), handle, ctypes.byref(base)))
        self._peer_ranks = int(n_ranks)
        return handle.raw, base.value

    def peer_open(self, ipc_handles=None, local_bases=None):
        """ipc_handles: list of 64-byte handles (one per rank) from other processes; local_bases: list of base
        addresses of other contexts of THIS process (None entries fall back to the handle)."""
        R = self._peer_ranks
        hbuf = None
        if ipc_handles is not None:
            hbuf = ctypes.create_string_buffer(b''.join(bytes(h) for h in ipc_handles), 64 * R)
        lb = None
        if local_bases is not None:
            lb = (ctypes.c_void_p * R)(*[ctypes.c_void_p(b) if b else None for b in local_bases])
        check(lib().nmrfit_pso_peer_open(self._h, hbuf, lb))

    def pso_commit_peers(self, stream=None):
        check(lib().nmrfit_pso_commit_peers(self._h, ptr(stream)))

    def pso_step_peers(self, rp=None, rg=None, stream=None):
        rp, rg = self._rand(rp, self._swarmsize), self._rand(rg, self._swarmsize)
        check(lib().nmrfit_pso_step_peers(self._h, ptr(rp), ptr(rg), ptr(stream)))

    def pso_run_peers(self, n_generations, rp_all=None, rg_all=None, stream=None):
        """A chunk of sharded generations in one call (records exchanged over peer memory inside the finish kernel);
        synchronises.  Returns (spectra still running, 1 if a wait for a peer expired)."""
        rp_all = self._rand(rp_all, self._swarmsize, n_generations)
        rg_all = self._rand(rg_all, self._swarmsize, n_generations)
        running, lost = ctypes.c_int(0), ctypes.c_int(0)
        check(lib().nmrfit_pso_run_peers(self._h, int(n_generations), ptr(rp_all), ptr(rg_all), ctypes.byref(running),
                                         ctypes.byref(lost), ptr(stream)))
        return running.value, lost.value

    def peer_timeout(self, milliseconds):
        check(lib().nmrfit_pso_peer_timeout(self._h, float(milliseconds)))

    def peer_error(self):
        e = ctypes.c_int(0)
        check(lib().nmrfit_pso_peer_error(self._h, ctypes.byref(e)))
        return e.value

    def pso_record(self):
        p, n = ctypes.c_void_p(), ctypes.c_int(0)
        check(lib().nmrfit_pso_record(self._h, ctypes.byref(p), ctypes.byref(n)))
        return p.value, n.value

    def pso_commit(self, recs_dev=None, n_ranks=1, stream=None):
        check(lib().nmrfit_pso_commit(self._h, ptr(recs_dev), int(n_ranks), ptr(stream)))

    def pso_run(self, n_generations, rp_all=None, rg_all=None, stream=None):
        rp_all = self._rand(rp_all, self._swarmsize, n_generations)
        rg_all = self._rand(rg_all, self._swarmsize, n_generations)
        running = ctypes.c_int(0)
        check(lib().nmrfit_pso_run(self._h, int(n_generations), ptr(rp_all), ptr(rg_all), ctypes.byref(running),
                                   ptr(stream)))
        return running.value

    def pso_best(self):
        x = np.empty((self.B, self.D))
        f = np.empty(self.B)
        it = np.empty(self.B, dtype=np.int32)
        stop = np.empty(self.B, dtype=np.int32)
        check(lib().nmrfit_pso_get_best(self._h, ptr(x), ptr(f), ptr(it), ptr(stop)))
        return x, f, it, stop

    def pso_state(self):
        S = self._swarmsize
        out = dict(x=np.empty((self.B, S, self.D)), v=np.empty((self.B, S, self.D)), p=np.empty((self.B, S, self.D)),
                   fx=np.empty((self.B, S)), fp=np.empty((self.B, S)))
        check(lib().nmrfit_pso_get_state(self._h, *[ptr(out[k]) for k in ('x', 'v', 'p', 'fx', 'fp')]))
        return out


class PhaseScorer(_Handle):
    """Device copies of a batch of spectra (u, v: [B, N] or [N]) for phase estimation (csrc/phase.cu)."""

    _destroy = 'nmrfit_phase_destroy'

    def __init__(self, u, v, device=None):
        u, v = as_f64(np.atleast_2d(u)), as_f64(np.atleast_2d(v))
        if u.shape != v.shape or u.ndim != 2:
            raise ValueError('u and v must have the same [B, N] shape')
        self.B, self.N = u.shape
        self._h = ctypes.c_void_p()
        dev = default_device() if device is None else int(device)
        check(lib().nmrfit_phase_create(ctypes.byref(self._h), dev, self.B, self.N, ptr(u), ptr(v)))

    def brute(self, candidates, details=False):
        """First smallest baseline error among the upward candidates, per spectrum (containers.py:98-110)."""
        c = as_f64(candidates)
        best, berr = np.empty(self.B), np.empty(self.B)
        err = np.empty((self.B, c.size)) if details else None
        ok = np.empty((self.B, c.size), dtype=np.int32) if details else None
        check(lib().nmrfit_phase_brute(self._h, ptr(c), c.size, ptr(best), ptr(berr), ptr(err), ptr(ok)))
        return (best, berr, err, ok.astype(bool)) if details else best

    def acme(self, ph_radians):
        """ACME score [B, K] for candidates [(p0, p1), ...] in radians (proc_autophase.py:142-187)."""
        ph = as_f64(np.atleast_2d(ph_radians))
        if ph.shape[1] != 2:
            raise ValueError('ph must be [K, 2]')
        score = np.empty((self.B, ph.shape[0]))
        check(lib().nmrfit_phase_acme(self._h, ptr(ph), ph.shape[0], ptr(score)))
        return score


class Communicator:
    """The contexts of ONE process as the ranks of a particle-sharded swarm (nmrfit_comm_*: no collective library; the
    best records cross between the contexts' windows inside the finish kernel).  ``ctxs[r]`` begins its own shard with
    ``particle_offset`` = the shard's first global particle index; then ``commit()`` and ``run(n)``."""

    def __init__(self, ctxs):
        self.ctxs = list(ctxs)
        self._arr = (ctypes.c_void_p * len(self.ctxs))(*[c._h for c in self.ctxs])
        check(lib().nmrfit_comm_init_all(self._arr, len(self.ctxs)))

    def commit(self):
        check(lib().nmrfit_comm_commit(self._arr, len(self.ctxs)))

    def run(self, n_generations, rp_all=None, rg_all=None):
        """rp_all / rg_all: per-context arrays [n_generations][shard particles][D] (or None: device random numbers).
        Returns (spectra still running, 1 if a rank was lost)."""
        n = len(self.ctxs)
        keep, rp, rg = [], None, None
        if rp_all is not None:
            keep = [[c._rand(a, c._swarmsize, n_generations) for c, a in zip(self.ctxs, arrs)] for arrs in (rp_all, rg_all)]
            rp = (ctypes.c_void_p * n)(*[ptr(a) for a in keep[0]])
            rg = (ctypes.c_void_p * n)(*[ptr(a) for a in keep[1]])
        running, lost = ctypes.c_int(0), ctypes.c_int(0)
        check(lib().nmrfit_comm_run(self._arr, n, int(n_generations), rp, rg, ctypes.byref(running), ctypes.byref(lost)))
        return running.value, lost.value


class PeakPicker(_Handle):
    """Device side of the automatic peak selection for a batch of spectra (csrc/peaks.cu): ``maxima`` then ``measure``."""

    _destroy = 'nmrfit_peaks_destroy'

    def __init__(self, n_spectra, n_points, upsample=100, max_peaks=64, device=None):
        self._h = ctypes.c_void_p()
        self.B, self.N, self.upsample, self.max_peaks = int(n_spectra), int(n_points), int(upsample), int(max_peaks)
        self.M = self.N * self.upsample
        dev = default_device() if device is None else int(device)
        check(lib().nmrfit_peaks_create(ctypes.byref(self._h), dev, self.B, self.N, self.upsample, self.max_peaks))

    def maxima(self, w, u, window, sg_coeffs=None, max_it=100, tol=1e-3):
        """-> (n_maxima [B], maxima [B, max_peaks] (unsorted upsampled indices), signal there, global baseline [B])"""
        w, u = as_f64(np.atleast_2d(w)), as_f64(np.atleast_2d(u))
        if w.shape != (self.B, self.N) or u.shape != (self.B, self.N):
            raise ValueError('w and u must have shape (%d, %d)' % (self.B, self.N))
        sg = None if sg_coeffs is None else as_f64(sg_coeffs)
        if sg is not None and sg.size != 121:
            raise ValueError('sg_coeffs must hold 11 + 2*5*11 values')
        n = np.zeros(self.B, dtype=np.int32)
        idx = np.zeros((self.B, self.max_peaks), dtype=np.int64)
        val = np.zeros((self.B, self.max_peaks))
        base = np.zeros(self.B)
        check(lib().nmrfit_peaks_maxima(self._h, ptr(w), ptr(u), float(window), ptr(sg), int(max_it), float(tol), ptr(n),
                                        ptr(idx), ptr(val), ptr(base)))
        return n, idx, val, base

    def measure(self, n_peaks, peak_i, peak_height, max_it=100, tol=1e-3):
        n_peaks = np.ascontiguousarray(n_peaks, dtype=np.int32)
        peak_i = np.ascontiguousarray(peak_i, dtype=np.int64)
        peak_height = as_f64(peak_height)
        shape = (self.B, self.max_peaks)
        if peak_i.shape != shape or peak_height.shape != shape or n_peaks.shape != (self.B,):
            raise ValueError('peak arrays must have shape %s' % (shape,))
        out = dict(ok=np.zeros(shape, dtype=np.int32), loc=np.zeros(shape), width=np.zeros(shape), bounds=np.zeros(shape + (2,)),
                   baseline=np.zeros(shape), height=np.zeros(shape), area=np.zeros(shape),
                   idx_range=np.zeros(shape + (2,), dtype=np.int64))
        check(lib().nmrfit_peaks_measure(self._h, ptr(n_peaks), ptr(peak_i), ptr(peak_height), int(max_it), float(tol),
                                         *[ptr(out[k]) for k in ('ok', 'loc', 'width', 'bounds', 'baseline', 'height', 'area',
                                                                 'idx_range')]))
        return out

    def probe(self, b, idx):
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        wu, uu, us = np.zeros(idx.size), np.zeros(idx.size), np.zeros(idx.size)
        check(lib().nmrfit_peaks_probe(self._h, int(b), ptr(idx), idx.size, ptr(wu), ptr(uu), ptr(us)))
        return wu, uu, us


# ---- pinned result buffers --------------------------------------------------------------------------
# Large results (generate_result at scale 16: 109 MB) are written into page-locked host memory taken from a small
# pool: the device-to-host copy runs at PCIe speed and there are no first-touch page faults.  A block goes back to the
# pool when the last numpy view of it is garbage collected.
import weakref

_PINNED_MIN = 4 << 20          # smaller results use ordinary numpy memory
_PINNED_KEEP = 512 << 20       # bytes kept in the pool; blocks beyond that are freed
_pinned_idle = {}              # block size -> [address, ...]
_pinned_bytes = 0


class _PinnedBlock:
    """Owner of one pinned allocation; numpy arrays made from it keep it alive through ``.base``."""

    def __init__(self, address, nbytes, count):
        self.address, self.nbytes = address, nbytes
        self.__array_interface__ = {'shape': (count,), 'typestr': '<f8', 'data': (address, False), 'version': 3}


def _pinned_release(address, nbytes):
    global _pinned_bytes
    if _pinned_bytes + nbytes <= _PINNED_KEEP:
        _pinned_idle.setdefault(nbytes, []).append(address)
        _pinned_bytes += nbytes
    else:
        try:
            lib().nmrfit_host_free(ctypes.c_void_p(address))
        except Exception:      # interpreter shutdown
            pass


def result_empty(count):
    """1-D float64 array of ``count`` elements for results: pinned and pooled when large, else ``np.empty``."""
    global _pinned_bytes
    nbytes = int(count) * 8
    if nbytes < _PINNED_MIN:
        return np.empty(int(count))
    size = (nbytes + (1 << 21) - 1) & ~((1 << 21) - 1)     # 2 MB buckets so that blocks are reusable
    idle = _pinned_idle.get(size)
    if idle:
        address = idle.pop()
        _pinned_bytes -= size
    else:
        p = ctypes.c_void_p()
        check(lib().nmrfit_host_alloc(size, ctypes.byref(p)))
        address = p.value
    block = _PinnedBlock(address, size, int(count))
    weakref.finalize(block, _pinned_release, address, size)
    return np.asarray(block)


# ---- context pool ---------------------------------------------------------------------------------
# Creating and destroying a context costs tens of milliseconds (pinned-host and device allocations, and
# every cudaFree synchronises) - far more than a small fit itself - so the fit drivers borrow contexts from
# this pool and hand them back with default settings.  A pooled context keeps its device buffers.
_pool = {}
_POOL_PER_KEY = 2
_POOL_KEYS = 8


class pooled_context:
    """``with pooled_context(B, N, P, device, precision) as ctx:`` - a cached context of that shape, or a new one."""

    def __init__(self, n_spectra, n_points, n_peaks, device=None, precision=FP64):
        dev = default_device() if device is None else int(device)
        self.key = (dev, int(n_spectra), int(n_points), int(n_peaks), int(precision))
        self.ctx = None

    def __enter__(self):
        idle = _pool.get(self.key)
        if idle:
            self.ctx = idle.pop()
        else:
            dev, B, N, P, prec = self.key
            self.ctx = Context(B, N, P, device=dev, precision=prec)
        return self.ctx

    def __exit__(self, exc_type, exc, tb):
        ctx, self.ctx = self.ctx, None
        if exc_type is not None:
            ctx.close()                    # do not reuse a context an error may have left half way
            return
        ctx.set_tuning()
        ctx.set_variant()
        ctx.set_far_cells()
        ctx.set_fused(FUSED_AUTO)
        ctx.set_algorithm(ALGO_AUTO)
        ctx.profile(False)
        if self.key not in _pool and len(_pool) >= _POOL_KEYS:
            _, old = _pool.popitem()
            for c in old:
                c.close()
        idle = _pool.setdefault(self.key, [])
        small = self.key[1] * self.key[2] * 32 <= (256 << 20)      # big batches give their memory back
        if small and len(idle) < _POOL_PER_KEY:
            idle.append(ctx)
        else:
            ctx.close()


def clear_pool():
    """Destroy every idle pooled context (frees their device memory)."""
    while _pool:
        _, idle = _pool.popitem()
        for c in idle:
            c.close()


def fp64_peak(device=None, iters=4096, repeats=10):
    """(burst, sustained) DFMA TFLOP/s of the device."""
    burst, sus = ctypes.c_double(0), ctypes.c_double(0)
    dev = default_device() if device is None else int(device)
    check(lib().nmrfit_fp64_peak(dev, iters, repeats, ctypes.byref(burst), ctypes.byref(sus)))
    return burst.value, sus.value


def launch_count():
    return int(lib().nmrfit_launch_count())
