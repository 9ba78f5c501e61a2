"""Public entry points, mirroring ``nmrfit.core`` (core.py)."""
import numpy as np

from . import containers
from . import utils
from . import swarm as _swarm
from . import _cabi

__all__ = ['load', 'fit', 'fit_batch', 'fit_batch_sharded']


def load(path, vendor='varian'):
    """Reading spectrometer files (core.py:9-61: nmrglue + FFT) is outside the
    accelerated path; build ``containers.Data(w, u, v)`` from arrays instead."""
    raise NotImplementedError(
        'nmrfit_b200 accelerates the fit path only; load the FID with the reference package '
        '(nmrglue) and wrap the arrays in nmrfit_b200.containers.Data(w, u, v)')


def fit(data, lower, upper, expon=0.5, dynamic_weighting=True, fit_im=False, processes=1, summary=True, options={}):
    """Perform a fit of NMR spectroscopy data (same signature as core.py:64).

    Returns the ``FitUtility`` holding ``params`` and ``error``.
    """
    f = utils.FitUtility(data, lower, upper, expon, dynamic_weighting, fit_im, processes, summary, options)
    f.fit()
    return f


def fit_batch(datas, lowers, uppers, expon=0.5, dynamic_weighting=True, fit_im=False, summary=False, options={}):
    """Fit many independent spectra (equal length and peak count) at once on one GPU.

    Equivalent to ``[fit(d, lo, up, ...) for d, lo, up in zip(...)]`` but all swarms
    advance together, one launch per generation.  With options['rng'] == 'host' and
    options['seeds'] = [k_0, k_1, ...], spectrum b reproduces the reference fit run
    after ``np.random.seed(k_b)``.  With options['refine'] every fit is then refined (``utils.refine_batch``) in the
    same context, where the spectra and weights already are, with options['ties'] (one ``utils.Ties`` for every
    spectrum or a list of them) and options['loss'] / options['f_scale'] (one scale for every spectrum, one per
    spectrum, or 'auto' for each spectrum's own from its least-squares residuals) if given.  Returns a list of ``FitUtility``.
    """
    fits = [utils.FitUtility(d, lo, up, expon, dynamic_weighting, fit_im, 1, summary, options)
            for d, lo, up in zip(datas, lowers, uppers)]
    opt = options
    refine = opt.get('refine', False)
    B = len(fits)
    if refine and fits:
        utils._check_refinable(fits[0])
        utils.check_loss_scale(opt.get('loss', 'linear'), opt.get('f_scale'), B)
    if not refine:
        utils.check_unrefined_options(opt)
    lb = np.array(lowers, dtype=np.float64)
    n_peaks = (lb.shape[1] - 4) // 3
    W, U, V = (np.stack([_cabi.as_f64(getattr(f.data, k)) for f in fits]) for k in ('w', 'u', 'v'))
    with _cabi.pooled_context(B, W.shape[1], n_peaks, device=opt.get('device'),
                              precision=_swarm._precision(opt.get('precision', 'fp64'))) as ctx:
        # weights (utils.py:191-224) are computed on the device, next to the spectra; as in the reference they
        # are computed first and only then replaced by ones when dynamic weighting is off (utils.py:171-173)
        ctx.set_spectra(W, U, V)
        bounds, values = utils.peak_windows([f.data.peaks for f in fits], expon)
        weights = ctx.compute_weights(bounds, values)
        if dynamic_weighting is False:
            weights = np.ones_like(weights)
            ctx.set_spectra(W, U, V, weights)
        x, fbest, it, stop = _swarm.pso_batch(
            None, lowers, uppers, fit_im=fit_im,
            swarmsize=opt.get('swarmsize', 204), maxiter=opt.get('maxiter', 2000),
            omega=opt.get('omega', -0.2134), phip=opt.get('phip', -0.3344), phig=opt.get('phig', 2.3259),
            minstep=opt.get('minstep', 1e-8), minfunc=opt.get('minfunc', 1e-8),
            rng=opt.get('rng', 'device'), seeds=opt.get('seeds'), seed=opt.get('seed', 0),
            chunk=opt.get('chunk', 16), fused=opt.get('fused', 'auto'), ctx=ctx,
            spectrum_offset=opt.get('spectrum_offset', 0))
        for b, f in enumerate(fits):
            f.weights = weights[b]
            f.params = x[b].copy()
            f.error = float(fbest[b])
            f.fit_info = dict(generations=int(it[b]), stop=int(stop[b]))
        if refine:
            per, arrays = utils.batch_ties(opt.get('ties'), B, n_peaks)
            utils.refine_with_loss(ctx, fits, x, lowers, uppers, ties=arrays, ties_per=per,
                                   loss=opt.get('loss', 'linear'), f_scale=opt.get('f_scale'))
    for f in fits:
        if summary is True:
            f._print_summary()
    return fits


def gather_fit_results(local, counts, group=None):
    """All-gather of per-rank result blocks ``local`` [count_r, K] (float64) into [sum(counts), K], rank order.
    Ranks hold different numbers of spectra, so blocks are padded to the largest count for the collective."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    K = local.shape[1]
    pad = np.zeros((max(counts), K))
    pad[:local.shape[0]] = local
    backend = dist.get_backend(group)
    dev = torch.device('cuda', torch.cuda.current_device()) if backend == 'nccl' else torch.device('cpu')
    mine = torch.from_numpy(pad).to(dev)
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine, group=group)
    return np.concatenate([parts[r].cpu().numpy()[:counts[r]] for r in range(world)])


def fit_batch_sharded(datas, lowers, uppers, expon=0.5, dynamic_weighting=True, fit_im=False, options={}, group=None,
                      fit_fn=None):
    """``fit_batch`` over the ranks of a ``torch.distributed`` group (one process per GPU): the spectra are split into
    contiguous blocks, every rank fits its block on its own GPU with no communication, and one final all-gather
    hands every rank all the fitted parameters (BASELINE config 3's flow).  Device random numbers are keyed by the
    GLOBAL spectrum index (``spectrum_offset``), so the result does not depend on the number of ranks.

    Returns ``(params [B, D], errors [B], generations [B], stop [B])`` - identical on every rank.
    ``fit_fn`` (default ``fit_batch``) exists so that the exchange logic can be tested without a GPU.
    """
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    B = len(datas)
    ranges = [_swarm.shard_range(B, r, world) for r in range(world)]
    off, cnt = ranges[rank]
    D = len(lowers[0])
    local = np.zeros((cnt, D + 3))
    if cnt:
        opt = dict(options)
        opt['spectrum_offset'] = int(opt.get('spectrum_offset', 0)) + off
        if opt.get('seeds') is not None:
            opt['seeds'] = list(opt['seeds'])[off:off + cnt]
        fits = (fit_fn or fit_batch)(datas[off:off + cnt], lowers[off:off + cnt], uppers[off:off + cnt], expon,
                                     dynamic_weighting, fit_im, False, opt)
        for i, f in enumerate(fits):
            local[i, :D] = f.params
            local[i, D] = f.error
            local[i, D + 1] = f.fit_info['generations']
            local[i, D + 2] = f.fit_info['stop']
    full = gather_fit_results(local, [c for _, c in ranges], group)
    return full[:, :D], full[:, D], full[:, D + 1].astype(int), full[:, D + 2].astype(int)
