"""Monte-Carlo prior scans -> ternary flavor histograms (``scripts/mc_unitary.py``, ``mc_x.py``,
``mc_texture.py`` + the histogram definition of ``plot.flavor_contour``, ``plot.py:364-370``).

The reference obtains prior samples by running emcee on a flat likelihood (``mc_unitary.py:121-131``),
maps ``angles_to_u`` / ``u_to_fr`` / ``flux_averaged_BSMu`` over the chain in Python
(``mc_unitary.py:189-192``, ``mc_x.py:186-192``, ``mc_texture.py:216-221``) and histograms at plot time.
Here a scan is ONE fused kernel per GPU: Philox4x32-10 draws (counter = global sample index) ->
flavor physics -> block-private shared-memory histogram.  Across GPUs the global index range is
split into contiguous shards -- the result is bit-identical for any number of ranks -- and the
per-rank histograms are summed by a single NCCL all-reduce.
"""

import ctypes as C
from argparse import Namespace

import numpy as np

from . import _lib
from . import model as _model
from .enums import ParamTag, PriorsCateg, Texture, enum_name
from .param import Param, ParamSet

__all__ = ['sm_paramset', 'scan_paramset', 'scan_model', 'scan_histogram', 'scan_samples', 'ternary_histogram',
           'shard_range', 'allreduce_counts', 'coverage_mask', 'scan_evidence', 'scan_evidence_grid', 'scan_evidence_sources', 'scan_profile_grid',
           'scan_profile_sources']

DEFAULT_BINNING = np.logspace(np.log10(6e4), np.log10(1e7), 21)  # fr.py:283-285


def sm_paramset(with_mass=True, gaussian=True):
    """The SM nuisance parameters of ``scripts/mc_texture.py:34-56`` / ``scripts/fr.py:38-49``:
    three mixing angles with LIMITEDGAUSS priors, a flat CP phase and (optionally) the two mass
    splittings with GAUSSIAN priors."""
    lg = PriorsCateg.LIMITEDGAUSS if gaussian else None
    g = PriorsCateg.GAUSSIAN if gaussian else None
    e = 1e-9
    tag = ParamTag.SM_ANGLES
    ps = [
        Param(name='s_12_2', value=0.307, seed=[0.26, 0.35], ranges=[0., 1.], std=0.013, prior=lg, tag=tag),
        Param(name='c_13_4', value=(1 - 0.02206) ** 2, seed=[0.950, 0.961], ranges=[0., 1.], std=0.00147, prior=lg, tag=tag),
        Param(name='s_23_2', value=0.538, seed=[0.31, 0.75], ranges=[0., 1.], std=0.069, prior=lg, tag=tag),
        Param(name='dcp', value=4.08404, seed=[0 + e, 2 * np.pi - e], ranges=[0., 2 * np.pi], std=2.0, tag=tag),
    ]
    if with_mass:
        ps += [
            Param(name='m21_2', value=7.40E-23, seed=[7.2E-23, 7.6E-23], ranges=[6.80E-23, 8.02E-23], std=2.1E-24, prior=g, tag=tag),
            Param(name='m3x_2', value=2.494E-21, seed=[2.46E-21, 2.53E-21], ranges=[2.399E-21, 2.593E-21], std=3.3E-23, prior=g, tag=tag),
        ]
    return ps


def scan_paramset(mode, dimension=6):
    """ParamSet of a scan mode.

    unitary  : 4 Haar-flat coordinates, uniform                      (mc_unitary.py:34-46)
    x        : 3 angles with LIMITEDGAUSS priors + dcp + x ~ U(0,1)  (mc_x.py:34-49)
    texture  : 6 SM params with priors + logLam ~ U(SCALE_BOUNDARIES) (mc_texture.py:34-67)
    anarchic : texture + 4 Haar-flat new-physics mixing coordinates   (Texture.NONE)
    """
    mode = mode.lower()
    if mode == 'unitary':
        return ParamSet(sm_paramset(with_mass=False, gaussian=False))
    if mode == 'x':
        return ParamSet(sm_paramset(with_mass=False) + [Param(name='astroX', value=0.5, seed=[0., 1.], ranges=[0., 1.], std=0.1, tag=ParamTag.SRCANGLES)])
    if mode in ('texture', 'anarchic'):
        ps = sm_paramset(with_mass=True)
        if mode == 'anarchic':
            tag = ParamTag.MMANGLES
            ps += [Param(name='np_s_12_2', value=0.5, ranges=[0., 1.], std=0.2, tag=tag),
                   Param(name='np_c_13_4', value=0.5, ranges=[0., 1.], std=0.2, tag=tag),
                   Param(name='np_s_23_2', value=0.5, ranges=[0., 1.], std=0.2, tag=tag),
                   Param(name='np_dcp', value=np.pi, ranges=[0., 2 * np.pi], std=0.2, tag=tag)]
        b = _model.SCALE_BOUNDARIES[int(dimension)]
        ps.append(Param(name='logLam', value=float(np.mean(b)), ranges=list(b), std=3, tag=ParamTag.SCALE))
        return ParamSet(ps)
    raise ValueError("scan mode must be 'unitary', 'x', 'texture' or 'anarchic', got {0!r}".format(mode))


def scan_model(mode, source_ratio=(1, 2, 0), dimension=6, texture=Texture.OET, binning=DEFAULT_BINNING, paramset=None):
    """Flat model of a scan (flat likelihood, as ``mc_*.py`` ``triangle_llh``: "return 1. # Flat LLH")."""
    mode = mode.lower()
    pset = paramset if paramset is not None else scan_paramset(mode, dimension)
    if mode == 'anarchic':
        texture = Texture.NONE
    args = Namespace(source_ratio=_np_norm(source_ratio), dimension=int(dimension), texture=texture,
                     binning=np.asarray(binning, dtype=np.float64), no_bsm=mode in ('unitary', 'x'))
    return _model.flatten(args, None, pset, likelihood='FLAT')


def _np_norm(x):
    x = np.asarray(x, dtype=np.float64)
    return x / x.sum()


def shard_range(count, rank, world_size, first_index=0):
    """Contiguous shard [first, first + n) of the global sample index range for ``rank``."""
    base, rem = divmod(int(count), int(world_size))
    n = base + (1 if rank < rem else 0)
    start = first_index + rank * base + min(rank, rem)
    return start, n


def _dist():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist
    except ImportError:
        pass
    return None


def allreduce_counts(*tensors):
    """Sum integer count tensors over the ranks of the initialised process group in place
    (NCCL on GPUs; any backend works -- the gloo CPU tests exercise exactly this call).  No-op
    without a process group.  This is the ONLY collective of the scan path."""
    dist = _dist()
    if dist is not None and dist.get_world_size() > 1:
        for t in tensors:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return tensors


def scan_histogram(fm, count, nb=25, seed=26, first_index=0, distributed=True, out=None, return_tensor=False):
    """Histogram of ``count`` prior samples: ``np.histogramdd(frs, bins=(nb+1,)*3, range=((0,1),)*3)``.

    With an initialised ``torch.distributed`` process group (and ``distributed=True``) the index range
    is sharded over the ranks and the counts are summed with one all-reduce; every rank returns the
    full histogram.  ``seed`` defaults to the reference scripts' ``--seed 26`` (``mc_unitary.py:97``)."""
    torch = _lib.torch_cuda()
    dist = _dist() if distributed else None
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    start, n = shard_range(count, rank, world, first_index)
    cells = (nb + 1) ** 3
    hist = out if out is not None else torch.zeros((cells,), dtype=torch.int64, device='cuda')
    kept = torch.zeros((1,), dtype=torch.int64, device='cuda')
    _lib.torch_ops().scan_hist(fm.blob, int(seed), int(start), int(n), int(nb), hist, kept)
    if dist and world > 1:
        allreduce_counts(hist, kept)
    h = hist.reshape(nb + 1, nb + 1, nb + 1)
    if return_tensor:
        return h, kept
    return h.cpu().numpy(), int(kept.item())


def scan_samples(fm, count, seed=26, first_index=0, return_tensor=False):
    """The drawn parameters ``theta[count, ndim]``, compositions ``fr[count, 3]`` and status bytes
    of a scan (what the reference saves with ``np.save``, ``mc_unitary.py:193``)."""
    torch = _lib.torch_cuda()
    theta = torch.empty((count, fm.ndim), dtype=torch.float64, device='cuda')
    fr = torch.empty((count, 3), dtype=torch.float64, device='cuda')
    st = torch.empty((count,), dtype=torch.uint8, device='cuda')
    cfg = _lib.ScanConfig(seed=int(seed), first_index=int(first_index), count=int(count), nb=0)
    _lib.check(_lib.load().gf_scan_samples(fm.ref, C.byref(cfg), _lib.ptr(theta), _lib.ptr(fr), _lib.ptr(st),
                                           _lib.stream_ptr(torch)))
    if return_tensor:
        return theta, fr, st
    return theta.cpu().numpy(), fr.cpu().numpy(), st.cpu().numpy()


def ternary_histogram(frs, nb=25, return_tensor=False):
    """``np.histogramdd(frs, bins=(nb+1,)*3, range=((0,1),)*3)`` (``plot.py:364-370``), bit-exact."""
    torch = _lib.torch_cuda()
    f = _lib.to_device(frs, torch, 3).reshape(-1, 3)
    hist = torch.zeros(((nb + 1) ** 3,), dtype=torch.int64, device='cuda')
    _lib.check(_lib.load().gf_ternary_hist(_lib.ptr(f), f.shape[0], int(nb), _lib.ptr(hist), _lib.stream_ptr(torch)))
    h = hist.reshape(nb + 1, nb + 1, nb + 1)
    return h if return_tensor else h.cpu().numpy()


def gaussian_weights(sigma, truncate=4.0):
    """SciPy's normalised 1-D Gaussian kernel for ``gaussian_filter(sigma)`` (``scipy.ndimage._filters._gaussian_kernel1d``
    with order 0): ``(radius, weights[-radius .. radius])`` with ``radius = int(truncate * sigma + 0.5)``."""
    radius = int(truncate * float(sigma) + 0.5)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (float(sigma) * float(sigma)) * x ** 2)
    return radius, phi / phi.sum()


def smooth_histogram(hist, hist_smooth, return_tensor=False):
    """``H = H / np.sum(H); H_s = gaussian_filter(H, sigma=hist_smooth)`` of ``plot.flavor_contour`` (``plot.py:372-375``)
    on the device, bit-identical to SciPy (separable, mode 'reflect', SciPy's accumulation order).  ``hist``: cubic
    histogram of counts; returns float64 of the same shape."""
    torch = _lib.torch_cuda()
    h = hist.to(device='cuda', dtype=torch.int64).contiguous() if isinstance(hist, torch.Tensor) else \
        torch.as_tensor(np.ascontiguousarray(hist, dtype=np.int64)).cuda()
    n1 = int(h.shape[0])
    if h.ndim != 3 or tuple(h.shape) != (n1, n1, n1):
        raise ValueError('smooth_histogram: a cubic 3-D histogram is expected, got shape %s' % (tuple(h.shape),))
    radius, w = gaussian_weights(hist_smooth)
    total = int(h.sum().item())
    out = torch.empty(h.shape, dtype=torch.float64, device='cuda')
    work = torch.empty(h.shape, dtype=torch.float64, device='cuda')
    wh = np.ascontiguousarray(w[:radius + 1], dtype=np.float64)        # outermost tap ... centre
    _lib.check(_lib.load().gf_hist_smooth(_lib.ptr(h), n1, total, wh.ctypes.data_as(C.c_void_p), radius, _lib.ptr(out), _lib.ptr(work),
                                          _lib.stream_ptr(torch)))
    return out if return_tensor else out.cpu().numpy()


def coverage_mask(hist, coverage, return_tensor=False, hist_smooth=0.05):
    """Highest-density region of a ternary histogram holding ``coverage`` per cent of the samples
    (``plot.flavor_contour``, ``plot.py:372-384``).  Returns ``(mask, info)``: ``mask`` has the shape of
    ``hist`` (1 inside the region); ``info = (content of the first excluded cell, number of masked
    cells, number of masked cells tied with the first excluded one)``.

    ``hist_smooth`` is the reference's 3-D smoothing width in bins (``gaussian_filter(H, sigma=hist_smooth)``,
    ``plot.py:375``).  Its default 0.05 -- like every value below 0.125 -- truncates to a one-tap kernel, the identity:
    the region is then found on the integer counts.  Larger values filter the normalised histogram on the device
    (``smooth_histogram``) and find the region on the smoothed field; ``info[0]`` is then a float."""
    torch = _lib.torch_cuda()
    if gaussian_weights(hist_smooth)[0] > 0:
        field = smooth_histogram(hist, hist_smooth, return_tensor=True)
        mask = torch.empty(field.numel(), dtype=torch.uint8, device='cuda')
        cstar, counts = C.c_double(), (C.c_uint64 * 2)()
        _lib.check(_lib.load().gf_coverage_mask_f64(_lib.ptr(field), field.numel(), float(coverage), _lib.ptr(mask), C.byref(cstar), counts,
                                                    _lib.stream_ptr(torch)))
        mask = mask.reshape(field.shape)
        return (mask if return_tensor else mask.cpu().numpy()), (float(cstar.value), int(counts[0]), int(counts[1]))
    if isinstance(hist, torch.Tensor):
        h = hist.to(device='cuda', dtype=torch.int64).contiguous()
    else:
        h = torch.as_tensor(np.ascontiguousarray(hist, dtype=np.int64)).cuda()
    mask = torch.empty(h.numel(), dtype=torch.uint8, device='cuda')
    info = (C.c_uint64 * 3)()
    _lib.check(_lib.load().gf_coverage_mask(_lib.ptr(h), h.numel(), float(coverage), _lib.ptr(mask), info, _lib.stream_ptr(torch)))
    mask = mask.reshape(h.shape)
    return (mask if return_tensor else mask.cpu().numpy()), tuple(int(x) for x in info)


def scan_evidence(fm, count, seed=26, first_index=0, distributed=True):
    """ln of the prior-mean likelihood, ln( (1/N) sum_i L(theta_i) ) with theta_i ~ priors: the
    Monte-Carlo evidence of a model up to its theta-independent prior-volume constant (what
    ``scripts/sens.py:232-294`` obtains from MultiNest per grid point).  Sharded over ranks like
    ``scan_histogram``; the (max, sum-exp) partials of the ranks are merged with two all-reduces."""
    torch = _lib.torch_cuda()
    dist = _dist() if distributed else None
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    start, n = shard_range(count, rank, world, first_index)
    lse = torch.tensor([-np.inf, 0.0], dtype=torch.float64, device='cuda')
    cfg = _lib.ScanConfig(seed=int(seed), first_index=int(start), count=int(n), nb=0)
    _lib.check(_lib.load().gf_scan_evidence(fm.ref, C.byref(cfg), _lib.ptr(lse), _lib.stream_ptr(torch)))
    if dist and world > 1:
        lse = _lse_allreduce(dist, lse)
    return float(_lnz(lse.cpu().numpy(), count))


def scan_evidence_grid(fm, scales, count, seed=26, first_index=0, distributed=True):
    """``scan_evidence`` at every frozen scale of ``scales`` (log10 Lambda) in ONE launch: each prior sample is drawn once
    and evaluated at all scales (``gf_scan_evidence_grid``; ``scripts/sens.py:199-201, 232-294`` runs one MultiNest job per
    scale).  The model must not sample the scale (``args.fixed_scale``).  Returns ``lnZ[len(scales)]``."""
    torch = _lib.torch_cuda()
    dist = _dist() if distributed else None
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    start, n = shard_range(count, rank, world, first_index)
    sc = torch.as_tensor(np.ascontiguousarray(scales, dtype=np.float64)).cuda()
    ns = int(sc.numel())
    lse = torch.empty((ns, 2), dtype=torch.float64, device='cuda')
    lse[:, 0] = -np.inf
    lse[:, 1] = 0.0
    lib = _lib.load()
    nbytes = int(lib.gf_scan_evidence_grid_workspace(ns))
    work = torch.empty(max(nbytes, 1), dtype=torch.uint8, device='cuda')
    cfg = _lib.ScanConfig(seed=int(seed), first_index=int(start), count=int(n), nb=0)
    _lib.check(lib.gf_scan_evidence_grid(fm.ref, C.byref(cfg), _lib.ptr(sc), ns, _lib.ptr(lse), _lib.ptr(work), nbytes, _lib.stream_ptr(torch)))
    if dist and world > 1:
        lse = _lse_allreduce(dist, lse)
    return _lnz(lse.cpu().numpy(), count)


def source_rows(sources, injected):
    """Validated ``(sources[nsrc, 3], injected[nsrc, 3])`` float64 arrays for ``scan_evidence_sources``: ``sources`` is one
    composition ``[3]`` or a list ``[nsrc, 3]``, ``injected`` one composition shared by all sources or one per source.  Every
    row must be finite and non-negative with a positive sum (it is normalised to unit sum on the device, as ``model.flatten``
    normalises ``args.source_ratio``).  Raises ValueError otherwise."""
    src = np.array(sources, dtype=np.float64, ndmin=2)
    if src.ndim != 2 or src.shape[1] != 3 or src.shape[0] < 1:
        raise ValueError('sources must be one composition [3] or a list [nsrc, 3], got shape %s' % (np.shape(sources),))
    inj = np.array(injected, dtype=np.float64, ndmin=2)
    if inj.ndim != 2 or inj.shape[1] != 3 or inj.shape[0] not in (1, src.shape[0]):
        raise ValueError('injected must be one composition [3] or one per source [%d, 3], got shape %s' % (src.shape[0], np.shape(injected)))
    inj = np.ascontiguousarray(np.broadcast_to(inj, src.shape))
    for name, a in (('source', src), ('injected composition', inj)):
        bad = ~(np.all(np.isfinite(a) & (a >= 0), axis=1) & (a.sum(axis=1) > 0))
        if bad.any():
            j = int(np.nonzero(bad)[0][0])
            raise ValueError('%s %d = %s: entries must be finite and non-negative with a positive sum' % (name, j, a[j].tolist()))
    return np.ascontiguousarray(src), inj


def _sources_launch(lib, fm, cfg, sc, ns, src, inj, lse, stream):
    """Enqueue ``gf_scan_evidence_sources`` for ``src`` / ``inj`` (any length: split into calls of at most ``GF_SRC_MAX``)
    into ``lse`` [nsrc, ns, 2] (a contiguous CUDA tensor)."""
    torch = _lib.torch_cuda()
    for j0 in range(0, src.shape[0], _lib.GF_SRC_MAX):
        s, i = src[j0:j0 + _lib.GF_SRC_MAX], inj[j0:j0 + _lib.GF_SRC_MAX]
        n = s.shape[0]
        nbytes = int(lib.gf_scan_evidence_sources_workspace(ns, n))
        work = _workspace(torch, nbytes)
        _lib.check(lib.gf_scan_evidence_sources(fm.ref, C.byref(cfg), _lib.ptr(sc), ns, s.ctypes.data_as(C.c_void_p),
                                                i.ctypes.data_as(C.c_void_p), n, C.c_void_p(lse.data_ptr() + 16 * ns * j0),
                                                _lib.ptr(work), nbytes, stream))


_WORK = {}


def _workspace(torch, nbytes):
    """Scratch of the evidence-grid kernels, one buffer per (device, stream), grown on demand and reused by later calls (the
    kernels leave it reusable by the next launch on the same stream)."""
    key = (torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream)
    buf = _WORK.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = _WORK[key] = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device='cuda')
    return buf


def _lse_allreduce(dist, lse):
    """Merge per-rank (max, sum-exp) pairs [..., 2] with two all-reduces: the max, then the sums rescaled to it."""
    torch = _lib.torch_cuda()
    gmax = lse[..., 0].clone()
    dist.all_reduce(gmax, op=dist.ReduceOp.MAX)
    part = torch.where(torch.isfinite(gmax), lse[..., 1] * torch.exp(lse[..., 0] - gmax), torch.zeros_like(gmax))
    dist.all_reduce(part, op=dist.ReduceOp.SUM)
    return torch.stack([gmax, part], dim=-1)


def _lnz(h, count):
    """ln( (1/count) sum ) of (max, sum-exp) pairs [..., 2]; -inf where no sample carried weight."""
    with np.errstate(divide='ignore'):
        return np.where(h[..., 1] > 0, h[..., 0] + np.log(h[..., 1]) - np.log(count), -np.inf)


def scan_evidence_sources(fm, scales, sources, injected, count, seed=26, first_index=0, distributed=True):
    """``scan_evidence_grid`` for many source compositions at once: ``lnZ[nsrc, len(scales)]``, row j the evidence grid of a
    model whose source is ``sources[j]`` and whose injected composition is ``injected[j]`` (or the one shared ``injected``
    [3]).  ONE launch per ``GF_SRC_MAX`` sources (``gf_scan_evidence_sources``): every prior sample is drawn and run through
    the eigen stage once per scale, then scored for every source.  The model's own source and injected composition are
    ignored; it must not sample the scale or the source and must have the Gaussian likelihood.  Sharded over ranks and merged
    like ``scan_evidence_grid``."""
    src, inj = source_rows(sources, injected)
    torch = _lib.torch_cuda()
    dist = _dist() if distributed else None
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    start, n = shard_range(count, rank, world, first_index)
    sc = torch.as_tensor(np.ascontiguousarray(scales, dtype=np.float64).ravel()).cuda()
    ns = int(sc.numel())
    lse = torch.empty((src.shape[0], ns, 2), dtype=torch.float64, device='cuda')
    lse[..., 0] = -np.inf
    lse[..., 1] = 0.0
    cfg = _lib.ScanConfig(seed=int(seed), first_index=int(start), count=int(n), nb=0)
    _sources_launch(_lib.load(), fm, cfg, sc, ns, src, inj, lse, _lib.stream_ptr(torch))
    if dist and world > 1:
        lse = _lse_allreduce(dist, lse)
    return _lnz(lse.cpu().numpy(), count)


# defaults of the profile optimiser, from the host-harness study recorded in DESIGN.md (K3c)
PROFILE_NSTARTS = 64
PROFILE_MAX_EVALS = 6000
PROFILE_FTOL = 1e-10
PROFILE_XTOL = 1e-7


def scan_profile_grid(fm, scales, nstarts=PROFILE_NSTARTS, seed=27, task0=0, max_evals=PROFILE_MAX_EVALS, ftol=PROFILE_FTOL,
                      xtol=PROFILE_XTOL):
    """Profile likelihood at every frozen scale of ``scales`` (log10 Lambda) in ONE launch (``gf_profile_grid``): the maximum of
    ``ln_prob`` over the model's columns inside their prior box, by bounded Nelder-Mead from ``nstarts`` starts per scale (the
    prior means, then prior draws).  The model must not sample the scale (``args.fixed_scale``).  ``task0`` is the global index
    of ``scales[0]``: a scale's result depends on ``(seed, task0 + s, nstarts)`` only, however the scales are split over calls.
    Returns a dict of NumPy arrays: ``best`` [ns], ``argmax`` [ns, ndim], ``fr`` [ns, 3] (composition at the argmax),
    ``status`` [ns] (its GF_ST_* bits), ``nevals`` [ns] (objective evaluations over all starts), ``nconverged`` [ns]
    (starts that converged before ``max_evals``)."""
    torch = _lib.torch_cuda()
    best, argmax, fr, st, counts = _profile_launch(torch, fm, scales, nstarts, seed, task0, max_evals, ftol, xtol)
    c = counts.cpu().numpy()
    return dict(best=best.cpu().numpy(), argmax=argmax.cpu().numpy(), fr=fr.cpu().numpy(), status=st.cpu().numpy(), nevals=c[:, 0],
                nconverged=c[:, 1])


def _profile_setup(torch, fm, scales, lead, nstarts, seed, task0, max_evals, ftol, xtol):
    """(scales on the device, their number, ProfileConfig, outputs) of a profile launch; the outputs (best, argmax, fr, status,
    counts) are CUDA tensors with the leading axes ``lead`` before the scale axis."""
    sc = torch.as_tensor(np.ascontiguousarray(scales, dtype=np.float64).ravel()).cuda()
    ns = int(sc.numel())
    shape = tuple(lead) + (ns,)
    out = (torch.empty(shape, dtype=torch.float64, device='cuda'), torch.empty(shape + (fm.ndim,), dtype=torch.float64, device='cuda'),
           torch.empty(shape + (3,), dtype=torch.float64, device='cuda'), torch.empty(shape, dtype=torch.uint8, device='cuda'),
           torch.empty(shape + (2,), dtype=torch.int64, device='cuda'))
    cfg = _lib.ProfileConfig(seed=int(seed), task0=int(task0), nstarts=int(nstarts), max_evals=int(max_evals), ftol=float(ftol),
                             xtol=float(xtol))
    return sc, ns, cfg, out


def _profile_launch(torch, fm, scales, nstarts, seed, task0, max_evals=PROFILE_MAX_EVALS, ftol=PROFILE_FTOL, xtol=PROFILE_XTOL):
    """Enqueue ``gf_profile_grid`` on torch's current stream: (best, argmax, fr, status, counts) as CUDA tensors."""
    sc, ns, cfg, out = _profile_setup(torch, fm, scales, (), nstarts, seed, task0, max_evals, ftol, xtol)
    _lib.check(_lib.load().gf_profile_grid(fm.ref, C.byref(cfg), _lib.ptr(sc), ns, *(_lib.ptr(t) for t in out), _lib.stream_ptr(torch)))
    return out


def scan_profile_sources(fm, scales, sources, injected, nstarts=PROFILE_NSTARTS, seed=27, task0=0, max_evals=PROFILE_MAX_EVALS, ftol=PROFILE_FTOL,
                         xtol=PROFILE_XTOL):
    """``scan_profile_grid`` for many source compositions at once: row j is the profile of a model whose source is
    ``sources[j]`` and whose injected composition is ``injected[j]`` (or the one shared ``injected`` [3]), from the same starts
    at every scale.  ONE launch per ``GF_SRC_MAX`` sources (``gf_profile_sources``: one block per (scale, source)).  The model's
    own source and injected composition are ignored; it must not sample the scale or the source and must have the Gaussian
    likelihood.  Returns the dict of ``scan_profile_grid`` with a leading ``[nsrc]`` axis."""
    src, inj = source_rows(sources, injected)
    torch = _lib.torch_cuda()
    out = _profile_sources_launch(torch, fm, scales, src, inj, nstarts, seed, task0, max_evals, ftol, xtol)
    best, argmax, fr, st, counts = (t.cpu().numpy() for t in out)
    return dict(best=best, argmax=argmax, fr=fr, status=st, nevals=counts[..., 0], nconverged=counts[..., 1])


def _profile_sources_launch(torch, fm, scales, src, inj, nstarts, seed, task0, max_evals=PROFILE_MAX_EVALS, ftol=PROFILE_FTOL, xtol=PROFILE_XTOL):
    """Enqueue ``gf_profile_sources`` on torch's current stream for the validated rows ``src`` / ``inj`` (any number: split into
    calls of at most ``GF_SRC_MAX``): (best, argmax, fr, status, counts) as CUDA tensors with a leading [nsrc] axis."""
    sc, ns, cfg, out = _profile_setup(torch, fm, scales, (src.shape[0],), nstarts, seed, task0, max_evals, ftol, xtol)
    lib, stream = _lib.load(), _lib.stream_ptr(torch)
    for j0 in range(0, src.shape[0], _lib.GF_SRC_MAX):
        s, i = src[j0:j0 + _lib.GF_SRC_MAX], inj[j0:j0 + _lib.GF_SRC_MAX]
        _lib.check(lib.gf_profile_sources(fm.ref, C.byref(cfg), _lib.ptr(sc), ns, s.ctypes.data_as(C.c_void_p), i.ctypes.data_as(C.c_void_p),
                                          s.shape[0], *(_lib.ptr(t[j0]) for t in out), stream))
    return out
