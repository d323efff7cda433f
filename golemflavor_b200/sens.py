"""Sensitivity sweep over (operator dimension, new-physics scale) grid points
(``scripts/sens.py:184-314``: one HTCondor job per (dimension, Lambda-segment), ``submitter/sens_dag.py:76-95``).

The reference fixes the scale parameter at each grid value (``sens.py:261-266``: ``scale_prm.value = scale``
and the sampler runs over all *non-SCALE* params) and runs MultiNest with the proprietary GolemFit
likelihood.  Here every grid point is an independent emcee-style chain of the Gaussian flavor-ratio
posterior with log10(Lambda) FROZEN at the grid value: all chains of one dimension run in ONE launch of
the device-resident ensemble sampler (``gf_ensemble_run``), grid points are sharded over the ranks of
the process group with no communication during sampling, and only the per-point summaries are
gathered at the end (``all_gather`` of a few numbers per chain).
"""

from argparse import Namespace

import numpy as np

from . import _lib, llh
from . import model as _model
from .enums import ParamTag, Texture
from .mcmc import DeviceEnsembleSampler
from .param import Param, ParamSet
from .scan import (DEFAULT_BINNING, PROFILE_NSTARTS, _check_groups, _dist, _group_lnz, _lnz, _lse_allreduce, _profile_launch, _profile_sources_launch,
                   _sources_launch, _workspace, shard_range, sm_paramset, source_rows)

__all__ = ['scale_grid', 'sweep_paramset', 'sweep', 'evidence_grid', 'evidence_source_grid', 'evidence_error', 'profile_grid', 'profile_source_grid',
           'get_limit', 'limits', 'limit_table', 'BAYES_K', 'FREQ_CL']


def scale_grid(dimension, segments):
    """``eval_scales``: the null point -100 followed by ``segments - 1`` equidistant values inside
    ``SCALE_BOUNDARIES[dimension]`` (``sens.py:199-201``)."""
    lo, hi = _model.SCALE_BOUNDARIES[int(dimension)]
    return np.concatenate([[-100.0], np.linspace(lo, hi, int(segments) - 1)])


def sweep_paramset(dimension):
    """6 SM nuisance params + logLam; the logLam box is widened to include the null point -100."""
    b = _model.SCALE_BOUNDARIES[int(dimension)]
    return ParamSet(sm_paramset(with_mass=True) + [
        Param(name='logLam', value=float(np.mean(b)), ranges=[-101.0, float(b[1])], std=3, tag=ParamTag.SCALE)])


_STREAMS = {}
_MODELS = {}


def _sweep_model(dim, texture, src, inj, smearing, binning):
    """(LnProb, ParamSet, seed boxes) of one operator dimension, cached across sweeps."""
    key = (int(dim), str(texture), tuple(np.asarray(src, dtype=np.float64)), tuple(np.asarray(inj, dtype=np.float64)), float(smearing),
           np.asarray(binning, dtype=np.float64).tobytes())
    hit = _MODELS.get(key)
    if hit is None:
        pset = sweep_paramset(dim)
        args = Namespace(source_ratio=src / src.sum(), dimension=int(dim), texture=texture, binning=np.asarray(binning),
                         no_bsm=False, injected_ratio=inj / inj.sum(), smearing=float(smearing))
        hit = _MODELS[key] = (llh.LnProb(args, None, pset), pset, np.array(pset.seeds, dtype=np.float64))
    return hit



def _dim_stream(torch, dim):
    """One side stream per (device, dimension), created once: torch's caching allocator keeps a pool per
    stream, and a cold pool means a cudaMalloc -- which waits for every kernel already running and would
    serialise the dimensions."""
    key = (torch.cuda.current_device(), int(dim))
    if key not in _STREAMS:
        _STREAMS[key] = torch.cuda.Stream()
    return _STREAMS[key]


def sweep(dimensions=(3, 4, 5, 6, 7, 8), segments=100, texture=Texture.OET, source_ratio=(1, 2, 0),
          injected_ratio=(1, 1, 1), smearing=0.02, nwalkers=60, burnin=200, nsteps=1000, seed=25,
          binning=DEFAULT_BINNING, distributed=True):
    """Run one chain per (dimension, scale) grid point.

    Returns a dict of arrays over all grid points (identical on every rank):
    ``dimension``, ``scale``, ``mean_lnprob`` (posterior mean of ln_prob), ``max_lnprob``,
    ``acceptance`` (mean acceptance fraction), ``mean_fr`` [n, 3] (posterior-mean measured composition).
    """
    torch = _lib.torch_cuda()
    dist = _dist() if distributed else None
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    grid = [(int(d), float(s)) for d in dimensions for s in scale_grid(d, segments)]
    start, count = shard_range(len(grid), rank, world)
    mine = grid[start:start + count]
    rows = torch.zeros((len(grid), 8), dtype=torch.float64, device='cuda')
    src = np.asarray(source_ratio, dtype=np.float64)
    inj = np.asarray(injected_ratio, dtype=np.float64)
    # one CUDA stream per dimension: the launches of different dimensions (different models, hence different
    # kernel launches) are latency-bound single-warp clusters and run side by side on the SMs
    pending = []
    for dim in sorted({d for d, _ in mine}):
        idx = [start + i for i, (d, _) in enumerate(mine) if d == dim]
        scales = np.array([grid[i][1] for i in idx])
        # the host side of a dimension costs as much as its share of the kernel time if done naively (the launches of the
        # LAST dimension wait for the preparation of all the others): flattened models are cached, seeds drawn in one call
        fn, pset, seeds = _sweep_model(dim, texture, src, inj, smearing, binning)
        nchains, ndim = len(idx), len(pset)
        # == np.stack([flat_seed(pset, nwalkers) for every chain of the dimension]) with np.random seeded per dimension:
        # one C-ordered draw consumes the stream exactly like consecutive per-chain calls of mcmc.flat_seed
        # (mcmc.py:88-96).  The stream is a function of (seed, dimension) and is drawn for ALL chains of the dimension,
        # of which this rank keeps its own: the sweep is identical however the grid is sharded over ranks.
        sub = np.random.RandomState((int(seed) * 1000003 + dim) % (2 ** 31 - 1))
        first = [i for i, (d, _) in enumerate(grid) if d == dim][0]
        p0 = sub.uniform(low=seeds[:, 0], high=seeds[:, 1], size=(int(segments), nwalkers, ndim))[[i - first for i in idx]]
        p0[:, :, ndim - 1] = scales[:, None]                      # frozen column: identical in all walkers
        stream = _dim_stream(torch, dim)
        stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(stream):
            sampler = DeviceEnsembleSampler(nwalkers, ndim, fn, nchains=nchains, seed=seed + 1000 * dim, nfree=ndim - 1,
                                            chain0=idx[0])
            sampler.run_mcmc(p0, burnin, store=False, return_tensor=True, check_nan=False)   # seeds lie inside the prior box
            sampler.reset()
            pos, lnp, _ = sampler.run_mcmc(None, nsteps, store=False, return_tensor=True)
            # summaries from the final ensemble + the acceptance counters (no chain leaves the device)
            _, fr, _ = fn.evaluate(pos.reshape(-1, ndim), want_fr=True, want_status=True)
        pending.append((stream, dim, idx, scales, sampler, lnp, fr, nchains))
    for stream, dim, idx, scales, sampler, lnp, fr, nchains in pending:
        stream.synchronize()
        fr = fr.reshape(nchains, nwalkers, 3)
        acc = torch.as_tensor(np.atleast_2d(sampler.acceptance_fraction), device='cuda').reshape(nchains, nwalkers)
        ii = torch.as_tensor(idx, device='cuda')
        rows[ii, 0] = float(dim)
        rows[ii, 1] = torch.as_tensor(scales, device='cuda')
        rows[ii, 2] = lnp.mean(dim=1)
        rows[ii, 3] = lnp.max(dim=1).values
        rows[ii, 4] = acc.mean(dim=1)
        rows[ii, 5:8] = fr.mean(dim=1)
    if dist and world > 1:
        dist.all_reduce(rows, op=dist.ReduceOp.SUM)              # disjoint rows: sum == gather
    out = rows.cpu().numpy()
    return {'dimension': out[:, 0].astype(int), 'scale': out[:, 1], 'mean_lnprob': out[:, 2], 'max_lnprob': out[:, 3],
            'acceptance': out[:, 4], 'mean_fr': out[:, 5:8]}


def evidence_grid(dimensions=(3, 4, 5, 6, 7, 8), segments=100, texture=Texture.OET, source_ratio=(1, 2, 0),
                  injected_ratio=(1, 1, 1), smearing=0.02, samples=1_000_000, seed=26, binning=DEFAULT_BINNING, return_maxllh=False,
                  groups=None):
    """Monte-Carlo evidence per (dimension, scale) grid point (``scripts/sens.py:289-294`` stores
    ``(scale, lnZ)`` per point): the six SM nuisance parameters are drawn from their priors, the scale is
    frozen at the grid value, ``lnZ = ln mean(L)``.  Returns ``{dimension: array[segments, 2]}`` like the
    reference's ``evidence_arr`` (with ``return_maxllh`` also the ``maxllh_arr`` twin, ``sens.py:290-294``: the largest
    ln L among the samples); Bayes factors against the null point (scale -100) and the limit follow with
    ``get_limit`` (``plot.py:149-213``).

    With ``groups=R`` (a power of two in [2, 32], at most ``samples``) the same launches split the samples into R fixed groups,
    sample i in group i mod R, and the leave-one-group-out curves ``{dimension: array[R, segments, 2]}`` of (scale, lnZ without
    group r) are returned last: ``evidence_error`` gives the Monte-Carlo error of every lnZ from them, ``limit_table(..., loo=)``
    the error of the limit.  lnZ itself equals the ungrouped result up to rounding.

    ONE launch per dimension (``gf_scan_evidence_grid``, ``gf_scan_evidence_grid_groups`` with groups): every prior sample is
    drawn once, the scale-independent part of the physics is built once, and the sample is evaluated at all scales of the grid;
    samples are sharded over the ranks of the process group and the per-scale (max, sum-exp) pairs are merged with two
    all-reduces at the end."""
    import ctypes as C
    R = _check_groups(groups, samples)
    torch = _lib.torch_cuda()
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    src = np.asarray(source_ratio, dtype=np.float64)
    inj = np.asarray(injected_ratio, dtype=np.float64)
    dims = [int(d) for d in dimensions]
    grids = [scale_grid(d, segments) for d in dims]
    nsc = [len(g) for g in grids]
    offs = np.concatenate([[0], np.cumsum(nsc)])
    scales = torch.as_tensor(np.concatenate(grids)).cuda()
    lse = torch.empty((int(offs[-1]), 2) if R is None else (int(offs[-1]), R, 2), dtype=torch.float64, device='cuda')
    lse[..., 0] = -np.inf
    lse[..., 1] = 0.0
    start, n = shard_range(samples, rank, world)
    cfg = _lib.ScanConfig(seed=int(seed), first_index=int(start), count=int(n), nb=0)
    lib, stream = _lib.load(), _lib.stream_ptr(torch)
    if R is None:
        work_bytes = int(lib.gf_scan_evidence_grid_workspace(max(nsc)))
    else:
        work_bytes = int(lib.gf_scan_evidence_grid_groups_workspace(max(nsc), R))
    work = _workspace(torch, work_bytes)
    for k, dim in enumerate(dims):
        fm = _grid_model(dim, texture, src, inj, smearing, binning)
        sc, out = C.c_void_p(scales.data_ptr() + 8 * int(offs[k])), C.c_void_p(lse.data_ptr() + 16 * (R or 1) * int(offs[k]))
        if R is None:
            _lib.check(lib.gf_scan_evidence_grid(fm.ref, C.byref(cfg), sc, nsc[k], out, _lib.ptr(work), work_bytes, stream))
        else:
            _lib.check(lib.gf_scan_evidence_grid_groups(fm.ref, C.byref(cfg), sc, nsc[k], R, out, _lib.ptr(work), work_bytes, stream))
    if dist and world > 1:
        lse = _lse_allreduce(dist, lse)
    h = lse.cpu().numpy()
    allsc = np.concatenate(grids)
    if R is None:
        lnz, maxllh = _lnz(h, samples), h[:, 0]
    else:
        (lnz, loo), maxllh = _group_lnz(h, samples), h[..., 0].max(axis=-1)
    ev = {d: np.column_stack([allsc[offs[k]:offs[k + 1]], lnz[offs[k]:offs[k + 1]]]) for k, d in enumerate(dims)}
    out = (ev,)
    if return_maxllh:
        out += ({d: np.column_stack([allsc[offs[k]:offs[k + 1]], maxllh[offs[k]:offs[k + 1]]]) for k, d in enumerate(dims)},)
    if R is not None:
        out += ({d: np.stack([np.broadcast_to(grids[k], (R, nsc[k])), loo[:, offs[k]:offs[k + 1]]], axis=-1) for k, d in enumerate(dims)},)
    return out[0] if len(out) == 1 else out


def _grid_model(dim, texture, src, inj, smearing, binning):
    """The six SM nuisance parameters with the scale frozen (``sens.py:261-266``), the model of every sensitivity grid; the
    kernels substitute each grid scale."""
    args = Namespace(source_ratio=src / src.sum(), dimension=int(dim), texture=texture, binning=np.asarray(binning),
                     no_bsm=False, injected_ratio=inj / inj.sum(), smearing=float(smearing), fixed_scale=-100.0)
    return _model.flatten(args, None, ParamSet(sm_paramset(with_mass=True)))


def evidence_source_grid(sources, dimensions=(3, 4, 5, 6, 7, 8), segments=100, texture=Texture.OET, injected_ratio=(1, 1, 1),
                         smearing=0.02, samples=1_000_000, seed=26, binning=DEFAULT_BINNING, groups=None):
    """``evidence_grid`` for every source composition of ``sources`` ([nsrc, 3], or one [3]) at once: the reference's
    submitter runs ``scripts/sens.py`` once per (dimension, texture, source composition, Lambda segment), 30 compositions per
    texture (``submitter/sens_dag.py:8-16, 38-61, 76-95``).  ``injected_ratio`` is one composition shared by all sources or
    one per source.  Returns ``{dimension: array[nsrc, segments, 2]}``; ``ev[d][j]`` has exactly the layout of
    ``evidence_grid(source_ratio=sources[j], injected_ratio=...)[d]`` (the null point -100 and the same scale grid) and the
    same samples.  ``limit_table`` turns the result into limits.

    With ``groups=R`` also the leave-one-group-out curves ``{dimension: array[nsrc, R, segments, 2]}`` (see ``evidence_grid``):
    ``evidence_error`` and ``limit_table(ev, loo=...)`` turn them into errors of lnZ and of the limits.

    ONE launch per dimension (``gf_scan_evidence_sources``; per 256 sources beyond that, and with groups per ``min(256, 4096 / R)``):
    the eigen stage of each prior sample runs once per scale, and every source is then scored from its transition sums.  The
    model of a dimension is built like ``evidence_grid``'s (``_grid_model``); samples are sharded over the ranks of the
    process group and merged with two all-reduces."""
    src, inj = source_rows(sources, injected_ratio)
    R = _check_groups(groups, samples)
    torch = _lib.torch_cuda()
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    dims = [int(d) for d in dimensions]
    grids = [scale_grid(d, segments) for d in dims]
    nsc = len(grids[0])
    lse = torch.empty((len(dims), src.shape[0], nsc, 2) if R is None else (len(dims), src.shape[0], nsc, R, 2), dtype=torch.float64, device='cuda')
    lse[..., 0] = -np.inf
    lse[..., 1] = 0.0
    start, n = shard_range(samples, rank, world)
    cfg = _lib.ScanConfig(seed=int(seed), first_index=int(start), count=int(n), nb=0)
    lib, stream = _lib.load(), _lib.stream_ptr(torch)
    scales = torch.as_tensor(np.stack(grids)).cuda()
    # the model's own source and injected composition are ignored by the kernel: the first row stands in
    for k, dim in enumerate(dims):
        fm = _grid_model(dim, texture, src[0], inj[0], smearing, binning)
        _sources_launch(lib, fm, cfg, scales[k], nsc, src, inj, lse[k], stream, groups=R)
    if dist and world > 1:
        lse = _lse_allreduce(dist, lse)
    if R is None:
        lnz = _lnz(lse.cpu().numpy(), samples)
    else:
        lnz, loo = _group_lnz(lse.cpu().numpy(), samples)
    ev = {d: np.stack([np.broadcast_to(grids[k], lnz[k].shape), lnz[k]], axis=-1) for k, d in enumerate(dims)}
    if R is None:
        return ev
    return ev, {d: np.stack([np.broadcast_to(grids[k], loo[k].shape), loo[k]], axis=-1) for k, d in enumerate(dims)}


def _jackknife_sigma(full, loo):
    """Delete-one-group jackknife error of the estimates ``full`` [...] from their leave-one-out values ``loo`` [..., R]:
    sqrt((R - 1) / R * sum_r (loo_r - mean_r loo_r)^2).  NaN where ``full`` is not finite; +inf where it is but some
    leave-one-out value is not (all the information sits in the groups that were left out)."""
    full, loo = np.asarray(full, dtype=np.float64), np.asarray(loo, dtype=np.float64)
    R = loo.shape[-1]
    if R == 0:                                                   # no leave-one-out values (an empty table): nothing to estimate
        return np.full(full.shape, np.nan)
    ok = np.all(np.isfinite(loo), axis=-1)
    with np.errstate(invalid='ignore'):
        d = loo - loo.mean(axis=-1, keepdims=True)
        sigma = np.sqrt((R - 1) / R * np.sum(d * d, axis=-1))
    return np.where(~np.isfinite(full), np.nan, np.where(ok, sigma, np.inf))


def evidence_error(evidence, loo):
    """Monte-Carlo standard error of every lnZ of a grouped ``evidence_grid`` / ``evidence_source_grid`` result: the
    delete-one-group jackknife sigma = sqrt((R - 1) / R * sum_r (lnZ_(-r) - mean_r lnZ_(-r))^2) over the R leave-one-group-out
    curves.  ``evidence`` ``{d: [segments, 2]}`` with ``loo`` ``{d: [R, segments, 2]}``, or ``{d: [nsrc, segments, 2]}`` with
    ``{d: [nsrc, R, segments, 2]}``; returns ``{d: [segments]}`` or ``{d: [nsrc, segments]}``.  sigma is NaN where lnZ is -inf
    (no sample carried weight) and +inf where lnZ is finite but some lnZ_(-r) is -inf (all the weight sits in one group)."""
    if set(loo) != set(evidence):
        raise ValueError('evidence_error: the leave-one-out curves have dimensions %s, the evidence %s' % (sorted(loo), sorted(evidence)))
    out = {}
    for d, ev in evidence.items():
        ev, lo = np.asarray(ev, dtype=np.float64), np.asarray(loo[d], dtype=np.float64)
        if lo.ndim != ev.ndim + 1 or lo.shape[:-3] != ev.shape[:-2] or lo.shape[-2:] != ev.shape[-2:]:
            raise ValueError('evidence_error: dimension %s: leave-one-out curves of shape %s do not match the evidence %s' % (d, lo.shape, ev.shape))
        out[d] = _jackknife_sigma(ev[..., 1], np.moveaxis(lo[..., 1], -2, -1))
    return out


def profile_grid(dimensions=(3, 4, 5, 6, 7, 8), segments=100, texture=Texture.OET, source_ratio=(1, 2, 0),
                 injected_ratio=(1, 1, 1), smearing=0.02, nstarts=PROFILE_NSTARTS, seed=27, binning=DEFAULT_BINNING,
                 distributed=True, return_argmax=False):
    """Profile likelihood per (dimension, scale) grid point: the frequentist statistic of ``scripts/sens.py``
    (``StatCateg.FREQUENTIST``, which the reference takes from GolemFit's profiled fit, ``gf.get_llh_freq``).  With the Gaussian
    flavor-ratio likelihood it is the maximum of ``ln_prob`` over the six SM nuisance parameters inside their prior box, the
    scale frozen at the grid value; the Gaussian priors act as penalty terms.  Returns ``{dimension: array[segments, 2]}`` of
    (scale, profile ln_prob), the layout of ``evidence_grid``; ``get_limit(..., args=Namespace(stat_method=FREQUENTIST))``
    turns it into a limit.  With ``return_argmax`` also ``{dimension: array[segments, 6]}`` of the maximising parameters.

    ONE launch per dimension (``gf_profile_grid``: one block per scale, one thread per start), on one stream per dimension.
    The grid points are sharded over the ranks of the process group (``task0`` = index of the scale in its dimension's grid)
    and the disjoint rows are merged with one all-reduce: the result is the same for any number of ranks."""
    torch = _lib.torch_cuda()
    src = np.asarray(source_ratio, dtype=np.float64)
    inj = np.asarray(injected_ratio, dtype=np.float64)
    dims = [int(d) for d in dimensions]
    segments = int(segments)

    def launch(dim, scales, task0):
        fm = _grid_model(dim, texture, src, inj, smearing, binning)
        best, argmax = _profile_launch(torch, fm, scales, nstarts, seed, task0)[:2]
        return best[None], argmax[None]

    rows = _profile_rows(dims, segments, 1, distributed, launch)[:, 0]
    prof = {d: np.column_stack([scale_grid(d, segments), rows[k * segments:(k + 1) * segments, 0]]) for k, d in enumerate(dims)}
    if return_argmax:
        return prof, {d: rows[k * segments:(k + 1) * segments, 1:].copy() for k, d in enumerate(dims)}
    return prof


def profile_source_grid(sources, dimensions=(3, 4, 5, 6, 7, 8), segments=100, texture=Texture.OET, injected_ratio=(1, 1, 1), smearing=0.02,
                        nstarts=PROFILE_NSTARTS, seed=27, binning=DEFAULT_BINNING, distributed=True, return_argmax=False):
    """``profile_grid`` for every source composition of ``sources`` ([nsrc, 3], or one [3]) at once: the frequentist column of the
    reference's sensitivity table, whose submitter runs ``scripts/sens.py`` once per (dimension, texture, source composition,
    Lambda segment), 30 compositions per texture (``submitter/sens_dag.py``).  ``injected_ratio`` is one composition shared by
    all sources or one per source.  Returns ``{dimension: array[nsrc, segments, 2]}`` of (scale, profile ln_prob), the layout
    of ``evidence_source_grid``: ``limit_table(result, args=Namespace(stat_method=StatCateg.FREQUENTIST))`` gives the frequentist
    table.  Every source starts from the points ``profile_grid`` uses at each scale.  With ``return_argmax`` also
    ``{dimension: array[nsrc, segments, 6]}`` of the maximising parameters.

    ONE launch per dimension (per 256 sources beyond that; ``gf_profile_sources``: one block per (scale, source), one thread per
    start), on one stream per dimension, with the model of ``_grid_model``.  The (dimension, scale) rows are sharded over the
    ranks of the process group exactly as ``profile_grid`` shards them, and the disjoint rows are merged with one all-reduce:
    the result is the same for any number of ranks."""
    src, inj = source_rows(sources, injected_ratio)
    torch = _lib.torch_cuda()
    dims = [int(d) for d in dimensions]
    segments = int(segments)

    def launch(dim, scales, task0):
        # the model's own source and injected composition are ignored by the kernel: the first row stands in
        fm = _grid_model(dim, texture, src[0], inj[0], smearing, binning)
        return _profile_sources_launch(torch, fm, scales, src, inj, nstarts, seed, task0)[:2]

    rows = _profile_rows(dims, segments, src.shape[0], distributed, launch)
    prof = {}
    for k, d in enumerate(dims):
        r = rows[k * segments:(k + 1) * segments].transpose(1, 0, 2)          # [nsrc, segments, 1 + ndim]
        prof[d] = np.stack([np.broadcast_to(scale_grid(d, segments), r.shape[:2]), r[..., 0]], axis=-1)
    if return_argmax:
        return prof, {d: rows[k * segments:(k + 1) * segments, :, 1:].transpose(1, 0, 2).copy() for k, d in enumerate(dims)}
    return prof


def _profile_rows(dims, segments, nsrc, distributed, launch):
    """The rows [len(dims) * segments, nsrc, 1 + 6] of (profile, argmax) of a profile grid.  The (dimension, scale) rows are
    sharded over the ranks of the process group; this rank's rows of a dimension run as ``launch(dim, scales, task0)`` -> (best
    [nsrc, n], argmax [nsrc, n, 6]) CUDA tensors on the dimension's stream, ``task0`` the index of ``scales[0]`` in the
    dimension's grid.  The disjoint rows of the ranks are merged with one all-reduce."""
    torch = _lib.torch_cuda()
    dist = _dist() if distributed else None
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    grid = [(k, s) for k in range(len(dims)) for s in range(segments)]
    start, count = shard_range(len(grid), rank, world)
    ndim = len(sm_paramset(with_mass=True))
    rows = np.zeros((len(grid), nsrc, 1 + ndim))
    cur = torch.cuda.current_stream()
    pending = []
    for k, dim in enumerate(dims):
        mine = [s for kk, s in grid[start:start + count] if kk == k]
        if not mine:
            continue
        stream = _dim_stream(torch, dim)
        stream.wait_stream(cur)
        with torch.cuda.stream(stream):
            out = launch(dim, scale_grid(dim, segments)[mine[0]:mine[-1] + 1], mine[0])
        pending.append((stream, k * segments + mine[0], out))
    for stream, row0, (best, argmax) in pending:
        stream.synchronize()
        n = best.shape[1]
        rows[row0:row0 + n, :, 0] = best.cpu().numpy().T
        rows[row0:row0 + n, :, 1:] = argmax.cpu().numpy().transpose(1, 0, 2)
    if dist and world > 1:
        t = torch.as_tensor(rows).cuda()
        dist.all_reduce(t, op=dist.ReduceOp.SUM)                   # disjoint rows: sum == gather
        rows = t.cpu().numpy()
    return rows


BAYES_K = 1.   # golemflavor/plot.py:82: "Strong degree of belief"
FREQ_CL = 0.90  # confidence level of the frequentist limit


def get_limit(scales, statistic, args=None, mask_initial=False, return_interp=False, bayes_k=BAYES_K, verbose=False, cl=FREQ_CL):
    """Limit on the new-physics scale from the evidence curve of one operator dimension (``plot.get_limit``,
    ``plot.py:149-213``; the consumer of the ``(scale, lnZ)`` pairs ``scripts/sens.py:289-294`` stores).

    ``scales[0]`` is the null point (-100), ``statistic`` = lnZ per scale.  A parametric cubic spline through
    ``(scale, lnZ)`` (SciPy ``splprep(s=0)`` / ``splev`` on 1000 points, as the reference) gives the reduced evidence
    ``-(lnZ - lnZ_null)``; the limit is the first splined scale where it exceeds ``ln 10^BAYES_K``, minus ``log10 2``
    (conversion to the standard SME coefficient, ``plot.py:208-210``).  Same outcomes as the reference: ``AssertionError``
    ('Discovered LV!') if the null point itself is disfavoured by more than the threshold, ``None`` when no splined point
    crosses it, when the contour is peaked (>= 2 grid points beyond the crossing fall 0.1 below the threshold) or when
    fewer than 2 grid points beyond the crossing reach it; ``return_interp`` returns ``(splined scales, reduced evidence)``.

    With ``args.stat_method == StatCateg.FREQUENTIST`` ``statistic`` is the profile ln_prob (``profile_grid``) and only the
    threshold changes: ``chi2.ppf(cl, 1) / 2`` in ln L, i.e. Wilks' -2 Delta ln L > chi^2 with one degree of freedom; the
    spline and every rule above are the same.  No fixture pins this branch against the reference: its frequentist value
    comes from GolemFit (``gf.get_llh_freq``).  The rule is this project's definition, and Wilks' theorem is an
    approximation where the scale sits at a bounded end of its range."""
    from scipy.interpolate import splev, splprep
    scales = np.asarray(scales, dtype=np.float64)
    statistic = np.asarray(statistic, dtype=np.float64)
    thr = np.log(10 ** bayes_k)
    if args is not None and getattr(args, 'stat_method', None) is not None:
        method = str(getattr(args.stat_method, 'name', args.stat_method)).upper()
        if method == 'FREQUENTIST':
            from scipy.stats import chi2
            thr = chi2.ppf(cl, 1) / 2.
        elif method != 'BAYESIAN':
            raise NotImplementedError
    if (statistic[0] - np.max(statistic)) > thr:
        raise AssertionError('Discovered LV!')
    tck, _ = splprep([scales, statistic], s=0)
    sc, st = splev(np.linspace(0, 1, 1000), tck)
    if mask_initial:
        keep = sc >= scales[1]
        sc, st = sc[keep], st[keep]
    null = statistic[np.argmin(scales)]
    reduced_ev = -(st - null)
    al = sc[reduced_ev > thr]
    if len(al) == 0:
        if verbose:
            print('No points above the threshold')
        return None
    re = -(statistic - null)[scales > al[0]]
    if np.sum(re < thr - 0.1) >= 2:
        if verbose:
            print('Warning, peaked contour does not exclude large scales!')
        return None
    if np.sum(re >= thr + 0.0) < 2:
        if verbose:
            print('Warning, only single point above threshold!')
        return None
    if return_interp:
        return sc, reduced_ev
    return al[0] - np.log10(2.)


def limits(evidence, **kwargs):
    """``get_limit`` for every dimension of an ``evidence_grid`` result: ``{dimension: limit or None}``."""
    return {d: get_limit(ev[:, 0], ev[:, 1], **kwargs) for d, ev in evidence.items()}


def limit_table(evidence_by_source, loo=None, **kwargs):
    """``get_limit`` for every (dimension, source) of an ``evidence_source_grid`` result -- or of any
    ``{dimension: array[nsrc, segments, 2]}`` of (scale, statistic) curves, e.g. of ``profile_source_grid`` with
    ``args=Namespace(stat_method=StatCateg.FREQUENTIST)``: the tabulation of the reference's sensitivities
    (``plot.plot_table_sens``).  ``kwargs`` go to ``get_limit`` unchanged.  Returns ``(limits[ndims, nsrc],
    discovered[ndims, nsrc])`` with the dimensions in the dict's order: a limit is NaN where ``get_limit`` returns None or
    raises 'Discovered LV!', and ``discovered`` is True exactly where it raises 'Discovered LV!'.

    With ``loo``, the leave-one-group-out curves ``{dimension: array[nsrc, R, segments, 2]}`` of a grouped
    ``evidence_source_grid`` (for one ``evidence_grid(..., groups=R)`` result wrap both: ``limit_table({d: ev[d][None] for d in
    ev}, loo={d: loo[d][None] for d in loo})``), every leave-one-out curve gets its limit L_(-r) the same way, and the
    return is ``(limits, discovered, limit_err, n_undefined)``: ``limit_err[ndims, nsrc]`` is the jackknife error
    sqrt((R - 1) / R * sum_r (L_(-r) - mean_r L_(-r))^2) of the limit.  All scales share the samples, so it accounts for the
    correlation between the points of a curve.  It is NaN where the limit is NaN, +inf where the limit is defined but some L_(-r)
    is not, and ``n_undefined[ndims, nsrc]`` counts the r whose L_(-r) is not defined (no limit or 'Discovered LV!').
    ``get_limit`` reads the crossing off 1000 spline points, so limits are quantised to that resolution: an error of 0 means
    that the leave-one-out limits fall on the same spline point, not that the limit is exact."""
    dims = list(evidence_by_source)
    nsrc = {len(evidence_by_source[d]) for d in dims}
    if len(nsrc) > 1:
        raise ValueError('limit_table: the dimensions have different numbers of sources: %s' % sorted(nsrc))
    nsrc = nsrc.pop() if nsrc else 0
    R = 0
    if loo is not None:
        if set(loo) != set(dims):
            raise ValueError('limit_table: the leave-one-out curves have dimensions %s, the evidence %s' % (sorted(loo), sorted(dims)))
        R = np.shape(loo[dims[0]])[1] if dims and np.ndim(loo[dims[0]]) == 4 else 0
        for d in dims:
            ev_shape, lo_shape = np.shape(evidence_by_source[d]), np.shape(loo[d])
            if len(lo_shape) != 4 or lo_shape[0] != ev_shape[0] or lo_shape[1] != R or R < 2 or lo_shape[2:] != tuple(ev_shape[1:]):
                raise ValueError('limit_table: dimension %s: leave-one-out curves of shape %s do not match the evidence %s (expected [%d, R >= 2, %s])'
                                 % (d, lo_shape, ev_shape, ev_shape[0], ', '.join(map(str, ev_shape[1:]))))
    # curve 0 of a (dimension, source) is its evidence, curves 1 .. R its leave-one-out curves
    lim = np.full((len(dims), nsrc, 1 + R), np.nan)
    disc = np.zeros((len(dims), nsrc), dtype=bool)
    for i, d in enumerate(dims):
        for j, ev in enumerate(evidence_by_source[d]):
            curves = [ev] if loo is None else [ev] + list(loo[d][j])
            for c, curve in enumerate(curves):
                curve = np.asarray(curve, dtype=np.float64)
                try:
                    v = get_limit(curve[:, 0], curve[:, 1], **kwargs)
                except AssertionError as e:
                    if str(e) != 'Discovered LV!':
                        raise
                    if c == 0:
                        disc[i, j] = True
                    continue
                if v is not None:
                    lim[i, j, c] = v
    if loo is None:
        return lim[..., 0], disc
    return lim[..., 0], disc, _jackknife_sigma(lim[..., 0], lim[..., 1:]), np.sum(np.isnan(lim[..., 1:]), axis=-1)
