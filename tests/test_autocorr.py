"""Integrated autocorrelation time on the device (``gf_autocorr_time``, ``mcmc.autocorr_time``).

The host ``mcmc.integrated_time`` (FFT autocorrelation, Sokal's window) is the reference.  The CPU tests pin a NumPy
direct-sum restatement of its definition, the one the device implements; the GPU tests compare the device with
``integrated_time`` on host copies of synthetic and sampled chains."""

import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from golemflavor_b200 import _lib, llh, mcmc  # noqa: E402

import models  # noqa: E402

TILE = 256   # lags per device tile (csrc/gf_autocorr.cu)


def ar1(nsteps, nwalkers, rho, seed):
    """AR(1) chains x[nsteps, nwalkers, ndim] with unit stationary variance; parameter d has coefficient rho[d], so its
    true tau is (1 + rho) / (1 - rho)."""
    rng = np.random.default_rng(seed)
    rho = np.asarray(rho, dtype=np.float64)
    x = np.empty((nsteps, nwalkers, rho.size))
    x[0] = rng.standard_normal((nwalkers, rho.size))
    s = np.sqrt(1.0 - rho ** 2)
    for i in range(1, nsteps):
        x[i] = rho * x[i - 1] + s * rng.standard_normal((nwalkers, rho.size))
    return x


def host_window(x, c=5.0):
    """``integrated_time`` with its window and its whole tau(t) curve (the same statements, in the same order)."""
    nsteps, nwalkers, ndim = x.shape
    n = 1 << int(np.ceil(np.log2(max(2 * nsteps, 2))))
    tau, win, curves = np.empty(ndim), np.empty(ndim, dtype=np.int64), []
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
        tau[d], win[d] = taus[m], m
        curves.append(taus)
    return tau, win, curves


def direct_tau(x, c=5.0):
    """The definition of the device estimator as a direct lag sum: a_w(t) = sum_i y_i y_{i+t} with y = x_w - mean(x_w);
    a walker whose values are bitwise equal contributes 0; acf = the walker mean of a_w(t) / a_w(0); tau(t) =
    2 cumsum(acf) - 1; the window is the first t >= c tau(t), else N - 1."""
    nsteps, nwalkers, ndim = x.shape
    tau, win = np.empty(ndim), np.empty(ndim, dtype=np.int64)
    for d in range(ndim):
        acf = np.zeros(nsteps)
        for w in range(nwalkers):
            v = np.ascontiguousarray(x[:, w, d])
            if np.all(v.view(np.int64) == v.view(np.int64)[0]):
                continue
            y = v - v.mean()
            a = np.correlate(y, y, 'full')[nsteps - 1:]
            if a[0] > 0:
                acf += a / a[0]
        acf /= nwalkers
        taus = 2.0 * np.cumsum(acf) - 1.0
        window = np.arange(nsteps) >= c * taus
        m = int(np.argmax(window)) if window.any() else nsteps - 1
        tau[d], win[d] = taus[m], m
    return tau, win


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b)) / np.maximum(np.abs(np.asarray(b)), 1e-300)))


# ---------------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize('nsteps', [50, 1000, 2001])
def test_direct_sum_restates_integrated_time(nsteps):
    x = ar1(nsteps, 6, [0.0, 0.3, 0.7, 0.9, 0.97], seed=nsteps)
    ref = mcmc.integrated_time(x)
    tau_h, win_h, _ = host_window(x)
    assert np.array_equal(tau_h, ref)                     # host_window is integrated_time with its window
    tau, win = direct_tau(x)
    assert rel(tau, ref) < 1e-10
    assert np.array_equal(win, win_h)


def test_direct_sum_constant_walkers():
    x = ar1(400, 5, [0.5, 0.8], seed=3)
    x[:, 2, 0] = 0.375                                    # one bitwise-constant walker: contributes rho = 0
    tau, win = direct_tau(x)
    # the same acf from the four moving walkers alone, still divided by all five
    alone, _ = direct_tau(x[:, [0, 1, 3, 4], :1])
    acf_sum = None
    for w in (0, 1, 3, 4):
        y = x[:, w, 0] - x[:, w, 0].mean()
        a = np.correlate(y, y, 'full')[399:]
        acf_sum = a / a[0] if acf_sum is None else acf_sum + a / a[0]
    taus = 2.0 * np.cumsum(acf_sum / 5.0) - 1.0
    m = int(np.argmax(np.arange(400) >= 5.0 * taus))
    assert win[0] == m and tau[0] == taus[m] and tau[0] != alone[0]
    # a dyadic constant has an exact NumPy mean, so integrated_time takes its a[0] > 0 branch the same way
    assert rel(tau, mcmc.integrated_time(x)) < 1e-10
    x[:, :, 1] = 0.1                                      # constant in every walker: tau = -1 at m = 0
    tau, win = direct_tau(x)
    assert tau[1] == -1.0 and win[1] == 0


def test_workspace_size_and_refused_shapes():
    lib = _lib.load()
    assert lib.gf_autocorr_time_workspace(1, 2, 50, 1) > 0
    big = lib.gf_autocorr_time_workspace(7, 1024, 10007, 16)
    assert big >= 7 * 16 * 1024 * TILE * 8                 # the per-walker lag tile dominates
    for shape in ((0, 2, 50, 1), (1, 0, 50, 1), (1, 2, 1, 1), (1, 2, 50, 0), (1, 2, 50, 17), (1 << 22, 1 << 10, 50, 1)):
        assert lib.gf_autocorr_time_workspace(*shape) == 0, shape


# ---------------------------------------------------------------------------------------------------------------- GPU


@pytest.fixture(scope='module')
def torch():
    import torch
    assert torch.cuda.is_available(), 'these tests need a CUDA device'
    return torch


def device_chain(torch, x):
    """x[C][N, W, D] host chains -> the sampler's layout [C, W, N, D] on the device."""
    return torch.as_tensor(np.ascontiguousarray(np.stack([np.swapaxes(v, 0, 1) for v in x]))).cuda()


def check_against_host(tau, win, xs, c=5.0):
    for j, x in enumerate(xs):
        ref = mcmc.integrated_time(x, c=c)
        tau_h, win_h, curves = host_window(x, c=c)
        assert np.array_equal(tau_h, ref)
        assert np.array_equal(win[j], win_h), (j, win[j], win_h)
        assert rel(tau[j], ref) < 1e-9, (j, tau[j], ref)
        for d, m in enumerate(win_h):    # no tie at the crossing that rounding could flip
            for t in range(max(m - 1, 0), m + 1):
                assert abs(t - c * curves[d][t]) > 1e-6, (j, d, t)


SHAPES = [  # (C, W, N, rho per parameter)
    (1, 1024, 10007, [0.0, 0.5, 0.9, 0.95, 0.98, 0.99]),
    (7, 33, 1000, list(np.linspace(0.0, 0.97, 16))),
    (7, 2, 50, [0.6]),
    (1, 2, 10007, list(np.linspace(0.1, 0.995, 16))),
]


@pytest.mark.gpu
@pytest.mark.parametrize('shape', SHAPES, ids=lambda s: 'C{0}_W{1}_N{2}_D{3}'.format(s[0], s[1], s[2], len(s[3])))
def test_shapes_match_integrated_time(torch, shape):
    C_, W, N, rho = shape
    xs = [ar1(N, W, rho, seed=100 * j + N + W) for j in range(C_)]
    tau, win = mcmc.autocorr_time(device_chain(torch, xs), return_window=True)
    assert tau.shape == win.shape == (C_, len(rho)) and win.dtype == np.int64
    check_against_host(tau, win, xs)
    if C_ == 1:   # a 3-D chain gives [D]
        t1 = mcmc.autocorr_time(device_chain(torch, xs)[0])
        assert t1.shape == (len(rho),) and np.array_equal(t1, tau[0])


@pytest.mark.gpu
def test_window_at_the_last_lag(torch):
    """A mean-subtracted series has sum_t a(t) = a(0) / 2, so tau(N - 1) = 0 up to rounding and every window closes by
    N - 1.  Strongly correlated short chains (rho = 0.999, N = 200) close late, in the middle of the chain; a large c
    keeps the window open until the last lag, where host and device both stop with tau ~ 0."""
    x = ar1(200, 8, [0.999, 0.999], seed=11)
    tau, win = mcmc.autocorr_time(device_chain(torch, [x]), return_window=True)
    check_against_host(tau, win, [x])
    _, win_h, _ = host_window(x, c=1e6)
    assert np.all(win_h == 199)
    tau, win = mcmc.autocorr_time(device_chain(torch, [x]), c=1e6, return_window=True)
    assert np.all(win == 199)
    assert np.max(np.abs(tau[0] - mcmc.integrated_time(x, c=1e6))) < 1e-12


@pytest.mark.gpu
def test_constant_walkers(torch):
    x = ar1(700, 9, [0.4, 0.8, 0.9], seed=5)
    x[:, 4, 0] = 0.1                          # one bitwise-constant walker (its NumPy mean is not exact)
    x[:, :, 2] = -3.7                         # a column constant in every walker (the sweep's frozen scale)
    tau, win = mcmc.autocorr_time(device_chain(torch, [x]), return_window=True)
    ref, ref_win = direct_tau(x)
    assert np.array_equal(win[0], ref_win)
    assert rel(tau[0, :2], ref[:2]) < 1e-9
    assert tau[0, 2] == -1.0 and win[0, 2] == 0


def notebook_sampler(golden, nwalkers, nchains, seed):
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    np.random.seed(seed)
    p0 = np.stack([mcmc.flat_seed(pset, nwalkers) for _ in range(nchains)])
    smp = mcmc.DeviceEnsembleSampler(nwalkers, fn.ndim, fn, nchains=nchains, seed=seed)
    return smp, p0 if nchains > 1 else p0[0]


@pytest.mark.gpu
def test_sampler_autocorr_time_two_parts(torch, golden):
    smp, p0 = notebook_sampler(golden, 256, 1, seed=41)
    smp.run_mcmc(p0, 300)
    smp.reset()
    with pytest.raises(RuntimeError, match='too short'):
        smp.get_autocorr_time()
    smp.run_mcmc(None, 1000)
    smp.run_mcmc(None, 1000)
    got = smp.get_autocorr_time()
    chain = smp.chain
    assert chain.shape == (256, 2000, 6) and got.shape == (6,)
    ref = mcmc.integrated_time(np.swapaxes(chain, 0, 1))
    assert rel(got, ref) < 1e-9
    assert np.array_equal(smp.acor, got)
    _, win_h, _ = host_window(np.swapaxes(chain, 0, 1))
    _, win = mcmc.autocorr_time(torch.cat(smp._chains, dim=2), return_window=True)
    assert np.array_equal(win[0], win_h)


@pytest.mark.gpu
def test_sampler_autocorr_time_per_chain(torch, golden):
    smp, p0 = notebook_sampler(golden, 64, 5, seed=42)
    smp.run_mcmc(p0, 200)
    smp.reset()
    smp.run_mcmc(None, 1500)
    got = smp.get_autocorr_time()
    chain = smp.chain
    assert got.shape == (5, 6)
    for j in range(5):
        assert rel(got[j], mcmc.integrated_time(np.swapaxes(chain[j], 0, 1))) < 1e-9, j


@pytest.mark.gpu
def test_bit_identical_and_independent_of_batch(torch):
    xs = [ar1(1500, 40, [0.2, 0.9, 0.97], seed=60 + j) for j in range(6)]
    ch = device_chain(torch, xs)
    tau, win = mcmc.autocorr_time(ch, return_window=True)
    for _ in range(2):
        t2, w2 = mcmc.autocorr_time(ch, return_window=True)
        assert np.array_equal(t2, tau) and np.array_equal(w2, win)
    for j in range(6):
        tj, wj = mcmc.autocorr_time(ch[j], return_window=True)
        assert np.array_equal(tj, tau[j]) and np.array_equal(wj, win[j])
    # the same chain beside chains whose windows are far longer (more tiles run for them)
    mixed = torch.cat([ch[2:3], device_chain(torch, [ar1(1500, 40, [0.999] * 3, seed=9)])])
    tm, wm = mcmc.autocorr_time(mixed, return_window=True)
    assert np.array_equal(tm[0], tau[2]) and np.array_equal(wm[0], win[2]) and np.all(wm[1] > win[2])


@pytest.mark.gpu
def test_launch_count(torch):
    lib = _lib.load()
    ch = device_chain(torch, [ar1(1000, 8, [0.5], seed=1)])
    before = lib.gf_launch_count()
    mcmc.autocorr_time(ch)
    assert lib.gf_launch_count() - before == 1 + 2 * -(-1000 // TILE)


@pytest.mark.gpu
def test_c_abi_refusals(torch):
    lib = _lib.load()
    C_, W, N, D = 2, 4, 100, 3
    ch = torch.zeros((C_, W, N, D), dtype=torch.float64, device='cuda')
    tau = torch.full((C_, D), 7.0, dtype=torch.float64, device='cuda')
    win = torch.full((C_, D), 7, dtype=torch.int64, device='cuda')
    nb = int(lib.gf_autocorr_time_workspace(C_, W, N, D))
    work = torch.empty(nb, dtype=torch.uint8, device='cuda')
    P = _lib.ptr
    good = dict(chain=P(ch), nchains=C_, nwalkers=W, nsteps=N, ndim=D, c=5.0, tau=P(tau), window=P(win), work=P(work), nbytes=nb)
    cases = [('chain', None), ('tau', None), ('window', None), ('work', None), ('nchains', 0), ('nchains', -1), ('nwalkers', 0),
             ('nsteps', 1), ('nsteps', 0), ('ndim', 0), ('ndim', 17), ('nwalkers', 1 << 30), ('c', 0.0), ('c', -5.0), ('c', float('inf')), ('c', float('nan')),
             ('nbytes', nb - 1), ('nbytes', 0)]
    stream = _lib.stream_ptr(torch)
    for key, bad in cases:
        a = dict(good, **{key: bad})
        before = lib.gf_launch_count()
        rc = lib.gf_autocorr_time(a['chain'], a['nchains'], a['nwalkers'], a['nsteps'], a['ndim'], a['c'], a['tau'], a['window'],
                                  a['work'], a['nbytes'], stream)
        assert rc == _lib.GF_ERR_ARG, (key, bad)
        assert lib.gf_last_error().decode().startswith('gf_autocorr_time:'), (key, bad)
        assert lib.gf_launch_count() == before, (key, bad)
    torch.cuda.synchronize()
    assert bool((tau == 7.0).all()) and bool((win == 7).all())
    a = good
    assert lib.gf_autocorr_time(a['chain'], C_, W, N, D, 5.0, a['tau'], a['window'], a['work'], nb, stream) == _lib.GF_OK
    assert bool((tau.cpu() == -1.0).all()) and bool((win.cpu() == 0).all())     # all-zero chains: every column constant
    with pytest.raises(ValueError):
        mcmc.autocorr_time(ch.float())
    with pytest.raises(ValueError):
        mcmc.autocorr_time(ch.cpu())
    with pytest.raises(ValueError, match='gf_autocorr_time: c'):
        mcmc.autocorr_time(ch, c=0.0)


@pytest.mark.gpu
def test_sweep_autocorr(torch):
    from golemflavor_b200 import sens
    from golemflavor_b200.enums import Texture
    from golemflavor_b200.scan import DEFAULT_BINNING
    kw = dict(dimensions=(3, 6), segments=5, nwalkers=60, burnin=200, nsteps=1000, seed=25, distributed=False)
    on = sens.sweep(autocorr=True, **kw)
    off = sens.sweep(**kw)
    assert set(on) == set(off) | {'tau'}
    for k in off:
        assert np.array_equal(on[k], off[k]), k
    assert on['tau'].shape == (10, 6) and np.all(np.isfinite(on['tau'])) and np.all(on['tau'] > 0)
    # rebuild grid point 7 (dimension 6, third scale) as the sweep seeds it: chain0 = its grid index
    gi, dim, first = 7, 6, 5
    fn, pset, seeds = sens._sweep_model(dim, Texture.OET, np.array([1.0, 2.0, 0.0]), np.array([1.0, 1.0, 1.0]), 0.02, DEFAULT_BINNING)
    sub = np.random.RandomState((25 * 1000003 + dim) % (2 ** 31 - 1))
    p0 = sub.uniform(low=seeds[:, 0], high=seeds[:, 1], size=(5, 60, 7))[gi - first]
    p0[:, 6] = sens.scale_grid(dim, 5)[gi - first]
    smp = mcmc.DeviceEnsembleSampler(60, 7, fn, seed=25 + 1000 * dim, nfree=6, chain0=gi)
    smp.run_mcmc(p0, 200, store=False, return_tensor=True, check_nan=False)
    smp.reset()
    smp.run_mcmc(None, 1000, return_tensor=True)
    assert abs(smp.acceptance_fraction.mean() - on['acceptance'][gi]) < 1e-12
    ref = mcmc.integrated_time(np.swapaxes(smp.chain, 0, 1))[:6]
    assert rel(on['tau'][gi], ref) < 1e-9
