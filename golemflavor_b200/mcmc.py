"""emcee driver for the flavor-ratio analysis (drop-in for ``golemflavor/mcmc.py``).

The reference hands ``ln_prob`` to ``emcee.EnsembleSampler(nwalkers, ndim, ln_prob, threads=N)``
(``mcmc.py:29-31``), which scores one walker per Python call in a multiprocessing pool.  emcee is an
un-vendored, unpinned dependency of the reference and is not needed here: ``EnsembleSampler`` below
implements the same affine-invariant stretch move (Goodman & Weare 2010; red/blue half-ensembles,
a = 2) with the emcee-2 attributes the reference driver touches, and calls the log-posterior
*vectorised* -- each half-ensemble is ONE call ``ln_prob(theta[nwalkers/2, ndim]) -> [nwalkers/2]``,
i.e. one CUDA kernel launch.  Only the proposal bookkeeping (a few vector operations on
``nwalkers x ndim`` numbers) runs in NumPy; every log-posterior value comes from the GPU.

The convergence diagnostic, the integrated autocorrelation time tau that ``sampler.acor`` prints, is computed where the
chain lives: ``autocorr_time`` runs the estimator of ``integrated_time`` on a device chain for every chain and parameter
in one call (C ABI ``gf_autocorr_time``), and ``DeviceEnsembleSampler.get_autocorr_time`` uses it.  ``integrated_time``
stays the host reference.
"""

import os
import sys

import numpy as np

__all__ = ['EnsembleSampler', 'DeviceEnsembleSampler', 'mcmc', 'flat_seed', 'gaussian_seed', 'save_chains', 'integrated_time',
           'autocorr_time']


def _progress(iterable, total):
    if os.environ.get('GOLEMFLAVOR_PROGRESS', '0') != '1':
        return iterable
    try:
        from tqdm import tqdm
    except ImportError:
        return iterable
    return tqdm(iterable, total=total)


def integrated_time(x, c=5.0):
    """Integrated autocorrelation time per dimension of a chain ``x[nsteps, nwalkers, ndim]``
    (FFT autocorrelation averaged over walkers, Sokal's automatic window M >= c tau)."""
    x = np.asarray(x, dtype=np.float64)
    nsteps, nwalkers, ndim = x.shape
    n = 1 << int(np.ceil(np.log2(max(2 * nsteps, 2))))
    tau = np.empty(ndim)
    for d in range(ndim):
        acf = np.zeros(nsteps)
        for w in range(nwalkers):
            y = x[:, w, d] - x[:, w, d].mean()
            f = np.fft.rfft(y, n=n)
            a = np.fft.irfft(f * np.conjugate(f), n=n)[:nsteps]
            acf += a / a[0] if a[0] > 0 else 0.0
        acf /= nwalkers
        taus = 2.0 * np.cumsum(acf) - 1.0
        window = np.arange(nsteps) >= c * taus
        m = int(np.argmax(window)) if window.any() else nsteps - 1
        tau[d] = taus[m]
    return tau


def _autocorr_device(chain, c=5.0):
    """(tau [C, D], window [C, D]) CUDA tensors of a contiguous float64 CUDA chain [C, W, N, D], enqueued on the current
    stream (``gf_autocorr_time``)."""
    from . import _lib
    torch = _lib.torch_cuda()
    nchains, nwalkers, nsteps, ndim = (int(v) for v in chain.shape)
    lib = _lib.load()
    nbytes = lib.gf_autocorr_time_workspace(nchains, nwalkers, nsteps, ndim)
    tau = torch.empty((nchains, ndim), dtype=torch.float64, device=chain.device)
    window = torch.empty((nchains, ndim), dtype=torch.int64, device=chain.device)
    work = torch.empty((max(int(nbytes), 1),), dtype=torch.uint8, device=chain.device)
    _lib.check(lib.gf_autocorr_time(_lib.ptr(chain), nchains, nwalkers, nsteps, ndim, float(c), _lib.ptr(tau), _lib.ptr(window),
                                    _lib.ptr(work), int(nbytes), _lib.stream_ptr(torch)))
    return tau, window


def autocorr_time(chain, c=5.0, return_window=False):
    """Integrated autocorrelation time of a device chain: ``integrated_time`` (same definition, same window rule) for
    every chain and parameter in one device call.

    ``chain`` is a float64 CUDA tensor ``[C, W, N, D]`` (``DeviceEnsembleSampler``'s layout: chain, walker, step,
    parameter) or ``[W, N, D]``; it is made contiguous and processed on the current stream.  Returns tau as a NumPy array
    ``[C, D]`` (``[D]`` for a 3-D chain), with ``return_window`` also the windows m (int64, same shape): tau = tau(m).
    Only the lags up to the window are computed.  A walker whose values are bitwise equal contributes an autocorrelation
    of 0, so a parameter that is constant in every walker (a frozen column) gets tau = -1 at m = 0."""
    from . import _lib
    torch = _lib.torch_cuda()
    if not isinstance(chain, torch.Tensor) or not chain.is_cuda or chain.dtype != torch.float64 or chain.ndim not in (3, 4):
        raise ValueError('autocorr_time needs a float64 CUDA tensor [C, W, N, D] or [W, N, D]')
    one = chain.ndim == 3
    tau, window = _autocorr_device((chain.unsqueeze(0) if one else chain).contiguous(), c=c)
    tau, window = tau.cpu().numpy(), window.cpu().numpy()
    if one:
        tau, window = tau[0], window[0]
    return (tau, window) if return_window else tau


class EnsembleSampler(object):
    """Affine-invariant ensemble sampler with the emcee-2 surface used by the reference
    (``mcmc.py:29-49``): ``sample(p0, iterations=)``, ``reset()``, ``chain``, ``lnprobability``,
    ``acceptance_fraction``, ``acor``, ``flatchain``, ``run_mcmc``.

    ``lnpostfn`` must accept ``theta[n, ndim]`` and return ``[n]`` (``vectorize=True``, the
    default here); with ``vectorize=False`` it is mapped over walkers like emcee-2 does.
    ``threads`` is accepted and ignored: the parallelism is inside the kernel."""

    def __init__(self, nwalkers, ndim, lnpostfn, a=2.0, args=(), kwargs=None, threads=1, vectorize=True, seed=None):
        if nwalkers % 2 != 0:
            raise ValueError('The number of walkers must be even.')
        if nwalkers < 2 * ndim:
            raise ValueError('The number of walkers needs to be more than twice the dimension of your parameter space.')
        self.k, self.dim, self.a = int(nwalkers), int(ndim), float(a)
        self.lnpostfn, self.args, self.kwargs = lnpostfn, tuple(args), dict(kwargs or {})
        self.vectorize = bool(vectorize)
        self.threads = threads
        self._random = np.random.RandomState(seed)
        self.ncalls = 0  # number of log-posterior (kernel) calls
        self.reset()

    # -- bookkeeping ---------------------------------------------------------------------------
    def reset(self):
        self._chain = np.empty((self.k, 0, self.dim))
        self._lnprob = np.empty((self.k, 0))
        self.naccepted = np.zeros(self.k)
        self.iterations = 0
        self._last_run_mcmc_result = None

    chain = property(lambda self: self._chain)
    lnprobability = property(lambda self: self._lnprob)
    flatchain = property(lambda self: self._chain.reshape((-1, self.dim)))
    random_state = property(lambda self: self._random.get_state())

    @property
    def acceptance_fraction(self):
        return self.naccepted / max(self.iterations, 1)

    @property
    def acor(self):
        return self.get_autocorr_time()

    def get_autocorr_time(self, c=5.0):
        if self._chain.shape[1] < 50:
            raise RuntimeError('The chain is too short to reliably estimate the autocorrelation time')
        return integrated_time(np.swapaxes(self._chain, 0, 1), c=c)

    def _lnprob_of(self, p):
        self.ncalls += 1
        if self.vectorize:
            lp = self.lnpostfn(p, *self.args, **self.kwargs)
            lp = lp.detach().cpu().numpy() if hasattr(lp, 'detach') else np.asarray(lp, dtype=np.float64)
        else:
            lp = np.array([self.lnpostfn(row, *self.args, **self.kwargs) for row in p], dtype=np.float64)
        lp = lp.reshape(-1)
        if lp.shape[0] != p.shape[0]:
            raise ValueError('lnpostfn returned {0} values for {1} walkers'.format(lp.shape[0], p.shape[0]))
        if np.any(np.isnan(lp)):
            raise ValueError('lnprob returned NaN.')  # emcee raises on NaN log-probabilities
        return lp

    # -- sampling ------------------------------------------------------------------------------
    def sample(self, p0, lnprob0=None, rstate0=None, iterations=1, thin=1, storechain=True):
        """Advance the ensemble; yields ``(pos, lnprob, rstate)`` after every step."""
        if rstate0 is not None:
            self._random.set_state(rstate0)
        p = np.array(p0, dtype=np.float64)
        if p.shape != (self.k, self.dim):
            raise ValueError('p0 must have shape (nwalkers, ndim) = {0}, got {1}'.format((self.k, self.dim), p.shape))
        lnprob = self._lnprob_of(p) if lnprob0 is None else np.array(lnprob0, dtype=np.float64)
        n_store = iterations // thin if storechain else 0
        base = self._chain.shape[1]
        if storechain:
            self._chain = np.concatenate((self._chain, np.zeros((self.k, n_store, self.dim))), axis=1)
            self._lnprob = np.concatenate((self._lnprob, np.zeros((self.k, n_store))), axis=1)
        half = self.k // 2
        first, second = slice(0, half), slice(half, self.k)
        for i in range(int(iterations)):
            self.iterations += 1
            for S0, S1 in ((first, second), (second, first)):
                s, c = p[S0], p[S1]
                ns, nc = s.shape[0], c.shape[0]
                zz = ((self.a - 1.0) * self._random.rand(ns) + 1.0) ** 2 / self.a
                partner = c[self._random.randint(nc, size=ns)]
                q = partner - zz[:, None] * (partner - s)
                newlnprob = self._lnprob_of(q)
                with np.errstate(invalid='ignore'):
                    lnpdiff = (self.dim - 1.0) * np.log(zz) + newlnprob - lnprob[S0]
                accept = lnpdiff > np.log(self._random.rand(ns))
                idx = np.arange(S0.start, S0.stop)[accept]
                p[idx] = q[accept]
                lnprob[idx] = newlnprob[accept]
                self.naccepted[idx] += 1
            if storechain and (i + 1) % thin == 0 and (i + 1) // thin <= n_store:
                ind = base + (i + 1) // thin - 1
                self._chain[:, ind, :] = p
                self._lnprob[:, ind] = lnprob
            yield p, lnprob, self.random_state

    def run_mcmc(self, pos0, N, rstate0=None, lnprob0=None, **kwargs):
        if pos0 is None:
            if self._last_run_mcmc_result is None:
                raise ValueError('Cannot have pos0=None if run_mcmc has never been called.')
            pos0, lnprob0, rstate0 = self._last_run_mcmc_result
        results = None
        for results in self.sample(pos0, lnprob0, rstate0, iterations=N, **kwargs):
            pass
        self._last_run_mcmc_result = results
        return results


class DeviceEnsembleSampler(object):
    """Device-resident stretch-move sampler (C ABI ``gf_ensemble_run``): proposal, log-posterior and
    accept/reject of every half-step run inside one kernel, for ``nchains`` independent ensembles at
    once; the whole ``run_mcmc`` call is a single launch (one block per chain for ensembles of up to
    512 walkers, a cooperative grid otherwise).

    Same emcee-2 surface as ``EnsembleSampler`` (``chain``, ``lnprobability``, ``acceptance_fraction``,
    ``acor``, ``flatchain``, ``reset``, ``run_mcmc``, ``sample``); with ``nchains > 1`` the arrays gain
    a leading chain axis.  ``lnprob`` must be an ``llh.LnProb`` (the flattened model).  Columns that are
    identical in all walkers of a chain stay frozen; pass ``nfree`` = number of sampled dimensions.
    """

    def __init__(self, nwalkers, ndim, lnprob, nchains=1, a=2.0, seed=0, nfree=None, store_lnprob=True, chain0=0, mode=0, cluster_blocks=0):
        from . import _lib
        if nwalkers % 2 != 0:
            raise ValueError('The number of walkers must be even.')
        if not hasattr(lnprob, 'model') or lnprob.ndim != ndim:
            raise ValueError('DeviceEnsembleSampler needs an llh.LnProb with ndim = {0}'.format(ndim))
        self._lib = _lib
        self.k, self.dim, self.a, self.nchains = int(nwalkers), int(ndim), float(a), int(nchains)
        self.nfree = int(nfree) if nfree is not None else int(ndim)
        if self.k < 2 * self.nfree:
            raise ValueError('The number of walkers needs to be more than twice the dimension of your parameter space.')
        self.lnprob, self.seed, self.store_lnprob, self.chain0 = lnprob, int(seed), bool(store_lnprob), int(chain0)
        self.mode = int(mode)   # 0 auto, 1 grid barrier, 2 block per chain, 3 cluster per chain (gf_ensemble_config.mode)
        self.cluster_blocks = int(cluster_blocks)   # CTAs per cluster, 0 = auto
        self.total_steps = 0   # global step counter = RNG counter offset: continuing a run never reuses draws
        self._last = None
        self.reset()

    def reset(self):
        """Forget the stored chain and the acceptance counters (``mcmc.py:36``); the current ensemble
        stays on the device so that ``run_mcmc(None, n)`` continues from it."""
        self._chains, self._lnps = [], []
        self._naccept = None
        self.iterations = 0

    def _cat(self, parts, tail):
        import torch
        if not parts:
            return np.empty((self.nchains, self.k, 0) + tail)
        return torch.cat(parts, dim=2).cpu().numpy()

    def _squeeze(self, arr):
        return arr[0] if self.nchains == 1 else arr

    chain = property(lambda self: self._squeeze(self._cat(self._chains, (self.dim,))))
    lnprobability = property(lambda self: self._squeeze(self._cat(self._lnps, ())))
    flatchain = property(lambda self: self.chain.reshape((-1, self.dim)) if self.nchains == 1
                         else self.chain.reshape((self.nchains, -1, self.dim)))

    @property
    def acceptance_fraction(self):
        if self._naccept is None:
            return self._squeeze(np.zeros((self.nchains, self.k)))
        return self._squeeze(self._naccept.cpu().numpy().astype(np.float64) / max(self.iterations, 1))

    @property
    def acor(self):
        return self.get_autocorr_time()

    def get_autocorr_time(self, c=5.0):
        """tau per chain and parameter (``autocorr_time`` on the device chain: the parts of several ``run_mcmc`` calls are
        joined on the device, nothing is copied to the host but the result)."""
        if sum(int(x.shape[2]) for x in self._chains) < 50:
            raise RuntimeError('The chain is too short to reliably estimate the autocorrelation time')
        import torch
        ch = self._chains[0] if len(self._chains) == 1 else torch.cat(self._chains, dim=2)
        return self._squeeze(autocorr_time(ch, c=c))

    def run_mcmc(self, pos0, N, lnprob0=None, thin=1, store=True, return_tensor=False, check_nan=True):
        """Advance all chains by N steps.  pos0 [nwalkers, ndim] or [nchains, nwalkers, ndim]
        (None: continue).  Returns (pos, lnprob, None) like emcee.  ``check_nan=False`` skips emcee's NaN check of
        the initial log-posteriors (it needs a device synchronisation) for callers that seed inside the prior box."""
        import ctypes as C
        _lib = self._lib
        torch = _lib.torch_cuda()
        if pos0 is None:
            if self._last is None:
                raise ValueError('Cannot have pos0=None if run_mcmc has never been called.')
            pos, lnp = self._last
        else:
            pos = _lib.to_device(pos0, torch, self.dim).reshape(self.nchains, self.k, self.dim).clone()
            lnp = None if lnprob0 is None else _lib.to_device(lnprob0, torch).reshape(self.nchains, self.k).clone()
        if lnp is None:
            lnp = self.lnprob.evaluate(pos.reshape(-1, self.dim)).reshape(self.nchains, self.k)
        # emcee raises on a NaN log-probability; only freshly supplied positions can carry one (the move
        # rejects NaN proposals), and skipping the check on continuation keeps run_mcmc asynchronous
        if check_nan and pos0 is not None and bool(torch.isnan(lnp).any()):
            raise ValueError('lnprob returned NaN.')
        nstore = int(N) // int(thin) if store else 0
        chain = torch.empty((self.nchains, self.k, nstore, self.dim), dtype=torch.float64, device='cuda') if nstore else None
        lchain = torch.empty((self.nchains, self.k, nstore), dtype=torch.float64, device='cuda') \
            if nstore and self.store_lnprob else None
        if self._naccept is None:
            self._naccept = torch.zeros((self.nchains, self.k), dtype=torch.int64, device='cuda')
        cfg = _lib.EnsembleConfig(nchains=self.nchains, nwalkers=self.k, nfree=self.nfree, nsteps=int(N),
                                  step0=self.total_steps, thin=int(thin), a=self.a, seed=self.seed, chain0=self.chain0, mode=self.mode, cluster_blocks=self.cluster_blocks)
        _lib.check(_lib.load().gf_ensemble_run(self.lnprob.model.ref, C.byref(cfg), _lib.ptr(pos), _lib.ptr(lnp),
                                               _lib.ptr(chain), _lib.ptr(lchain), _lib.ptr(self._naccept),
                                               _lib.stream_ptr(torch)))
        self.total_steps += int(N)
        self.iterations += int(N)
        if chain is not None:
            self._chains.append(chain)
        if lchain is not None:
            self._lnps.append(lchain)
        self._last = (pos, lnp)
        if return_tensor:
            return pos, lnp, None
        return self._squeeze(pos.cpu().numpy()), self._squeeze(lnp.cpu().numpy()), None

    def sample(self, p0, lnprob0=None, rstate0=None, iterations=1, thin=1, storechain=True):
        """emcee-2 generator interface (``mcmc.py:34-41``).  The device sampler advances all
        ``iterations`` in one launch and yields once."""
        yield self.run_mcmc(p0, iterations, lnprob0=lnprob0, thin=thin, store=storechain)


def _as_lnprob_object(ln_prob):
    """``LnProb`` behind ``ln_prob`` if it is one, or a ``functools.partial`` of ``llh.ln_prob``
    with its three closure arguments bound (the reference's calling pattern, ``scripts/fr.py:182-187``)."""
    from . import llh
    if isinstance(ln_prob, llh.LnProb):
        return ln_prob
    func = getattr(ln_prob, 'func', None)
    if func is llh.ln_prob:
        kw = dict(ln_prob.keywords or {})
        names = ['args', 'asimov_paramset', 'llh_paramset']
        pos = list(ln_prob.args or ())
        try:
            bound = [kw[n] if n in kw else pos.pop(0) for n in names]
        except IndexError:
            return None
        return llh.LnProb(*bound)
    return None


def _accepts_batches(ln_prob, p0):
    """Probe a foreign callable once with a 2-row (3-row for ndim = 2) batch: a reference-style scalar ``ln_prob(theta[ndim])`` raises or
    returns something that is not ``[2]`` -- it is then mapped over the walkers like emcee-2 does."""
    rows = 3 if p0.shape[-1] == 2 else 2     # a row count different from ndim: `x, y = theta` must not unpack rows
    try:
        out = ln_prob(p0[:rows])
        out = out.detach().cpu().numpy() if hasattr(out, 'detach') else np.asarray(out, dtype=np.float64)
        return out.shape == (rows,)
    except Exception:  # noqa: BLE001
        return False


def mcmc(p0, ln_prob, ndim, nwalkers, burnin, nsteps, threads=1, vectorize=None, seed=None, device=None):
    """Run burn-in, reset, run, flatten walker-major (``mcmc.py:27-53``).  Returns ``samples[nwalkers*nsteps, ndim]``.

    ``ln_prob`` = an ``llh.LnProb`` or a ``functools.partial`` of ``llh.ln_prob`` runs on the device-resident sampler
    (``seed=None`` draws a fresh 63-bit seed and prints it); any other callable runs on the bundled host sampler,
    batched if it accepts ``theta[n, ndim]`` (``vectorize=None`` probes it once), else one walker per call."""
    fn = _as_lnprob_object(ln_prob) if device in (None, True) else None
    if device is True and fn is None:
        raise ValueError('device=True needs an llh.LnProb or a partial of llh.ln_prob')
    if fn is not None:
        # device-resident sampler: proposal + log-posterior + accept in one kernel, no host loop
        if seed is None:
            # the reference never seeds emcee (mcmc.py:29-31): independent runs must use independent streams
            seed = int.from_bytes(os.urandom(8), 'little') >> 1
            print('device sampler seed', seed)
        sampler = DeviceEnsembleSampler(nwalkers, ndim, fn, seed=seed)
    else:
        if vectorize is None:   # the package's own callables are batched; foreign ones are probed once
            vectorize = True if _as_lnprob_object(ln_prob) is not None else _accepts_batches(ln_prob, np.asarray(p0, dtype=np.float64))
        sampler = EnsembleSampler(nwalkers, ndim, ln_prob, threads=threads, vectorize=vectorize, seed=seed)
    print("Running burn-in")
    pos = np.asarray(p0)
    for pos, _, _ in _progress(sampler.sample(p0, iterations=burnin), burnin):
        pass
    sampler.reset()
    print("Finished burn-in")
    print("Running")
    for _ in _progress(sampler.sample(pos, iterations=nsteps), nsteps):
        pass
    print("Finished")
    samples = sampler.chain.reshape((-1, ndim))
    print('acceptance fraction', sampler.acceptance_fraction)
    print('sum of acceptance fraction', np.sum(sampler.acceptance_fraction))
    print('np.unique(samples[:,0]).shape', np.unique(samples[:, 0]).shape)
    try:
        print('autocorrelation', sampler.acor)
    except Exception:
        print('WARNING : NEED TO RUN MORE SAMPLES')
    mcmc.last_sampler = sampler
    return samples


def flat_seed(paramset, nwalkers):
    """Uniform starting positions inside the ``Param.seed`` boxes (``mcmc.py:88-96``)."""
    seeds = np.array(paramset.seeds, dtype=np.float64)
    return np.random.uniform(low=seeds[:, 0], high=seeds[:, 1], size=[nwalkers, len(paramset)])


def gaussian_seed(paramset, nwalkers):
    """Gaussian starting positions around the current values (``mcmc.py:99-105``)."""
    return np.random.normal(paramset.values, paramset.stds, size=[nwalkers, len(paramset)])


def save_chains(chains, outfile):
    """``np.save`` of the chains; like the reference (``mcmc.py:108-126``) ``.npy`` is always appended."""
    directory = os.path.dirname(outfile)
    if directory and not os.path.isdir(directory):
        os.makedirs(directory, exist_ok=True)
    print('Saving chains to location {0}'.format(outfile + '.npy'))
    np.save(outfile + '.npy', chains)
