"""Developer timing of the device autocorrelation time (``gf_autocorr_time``) against the host ``integrated_time``.

1. The README quick-start chain, 1 x 1024 walkers x 10^4 steps x 6 parameters from a device-sampler run: device
   ``get_autocorr_time`` (CUDA events, median of 10 after a warm-up), host ``integrated_time`` on the copied chain, max
   relative tau difference.
2. Kernel rate: fp64 FMAs of the lag tiles actually computed (W * sum over computed lags t of (N - t), per parameter),
   over the summed ``k_acor_tile`` time from torch.profiler, as a fraction of ``gf_fp64_peak_probe`` mode 0 in the same run.
3. ``sens.sweep`` at bench.py's shape (600 grid points x 60 walkers x 200 + 1000 steps) with ``autocorr=True`` and
   ``False``, alternated twice each after a warm-up; the tau range and the share of points with nsteps < 50 tau.

``python scratch/autocorr_bench.py [out.json]``; prints the card name and power limit of the same run.
"""
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from golemflavor_b200 import _lib, llh, mcmc, sens
from golemflavor_b200.enums import ParamTag, PriorsCateg
from golemflavor_b200.param import Param, ParamSet
from golemflavor_b200 import fr

TILE = 256


def card():
    q = 'name,power.limit,clocks.max.sm'
    out = subprocess.run(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
    return out.splitlines()[torch.cuda.current_device()] if out else 'unknown'


def quickstart_lnprob():
    from argparse import Namespace
    measured = fr.u_to_fr(fr.normalize_fr((1, 0, 0)), fr.NUFIT_U)
    a1, a2 = fr.fr_to_angles(measured)
    asimov = ParamSet([Param('measured_angle1', a1, [0., 1.], std=0.02, tag=ParamTag.BESTFIT),
                       Param('measured_angle2', a2, [-1., 1.], std=0.02, tag=ParamTag.BESTFIT)])
    lg, t = PriorsCateg.LIMITEDGAUSS, ParamTag.SM_ANGLES
    pset = ParamSet([Param('s_12_2', 0.307, [0., 1.], seed=[0.26, 0.35], std=0.013, prior=lg, tag=t),
                     Param('c_13_4', (1 - 0.02206) ** 2, [0., 1.], seed=[0.950, 0.961], std=0.00147, prior=lg, tag=t),
                     Param('s_23_2', 0.538, [0., 1.], seed=[0.31, 0.75], std=0.069, prior=lg, tag=t),
                     Param('dcp', 4.08404, [0., 2 * np.pi], std=2.0, tag=t),
                     Param('source_angle1', 0, [0., 1.], tag=ParamTag.SRCANGLES),
                     Param('source_angle2', 0, [-1., 1.], tag=ParamTag.SRCANGLES)])
    return llh.LnProb(Namespace(source_ratio=[1, 2, 0], no_bsm=True), asimov, pset), pset


def event_time(fn, reps):
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) * 1e-3)
    return float(np.median(out))


def computed_fmas(W, N, D_windows):
    """FMAs of the lag tiles run: every pair computes whole tiles up to the one holding its window."""
    total = 0
    for m in D_windows:
        lags = min(N, TILE * (int(m) // TILE + 1))
        total += W * (lags * N - lags * (lags - 1) // 2)
    return total


def main():
    res = {'card': card()}
    print('card:', res['card'])
    lib = _lib.load()

    # -- 1. quick-start chain
    fn, pset = quickstart_lnprob()
    np.random.seed(7)
    smp = mcmc.DeviceEnsembleSampler(1024, 6, fn, seed=7)
    smp.run_mcmc(mcmc.flat_seed(pset, 1024), 100)
    smp.reset()
    smp.run_mcmc(None, 10000)
    torch.cuda.synchronize()
    tau_dev = smp.get_autocorr_time()
    dev_s = event_time(lambda: smp.get_autocorr_time(), 10)
    t0 = time.perf_counter()
    chain = smp.chain
    copy_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    tau_host = mcmc.integrated_time(np.swapaxes(chain, 0, 1))
    host_s = time.perf_counter() - t0
    _, win = mcmc.autocorr_time(smp._chains[0], return_window=True)
    res['quickstart'] = dict(shape=[1, 1024, 10000, 6], device_seconds=dev_s, host_integrated_time_seconds=host_s, host_copy_seconds=copy_s,
                             ratio_device_over_host=dev_s / host_s, tau=tau_dev.tolist(), window=win[0].tolist(),
                             max_rel_tau_diff=float(np.max(np.abs(tau_dev - tau_host) / np.abs(tau_host))))
    print('quick start: device %.5f s, host %.3f s (copy %.3f s), ratio %.5f, tau %s, max rel diff %.2e' % (
        dev_s, host_s, copy_s, dev_s / host_s, np.array2string(tau_dev, precision=2), res['quickstart']['max_rel_tau_diff']))

    # -- 2. kernel rate against the fp64 probe
    sink = torch.zeros(8, dtype=torch.float64, device='cuda')
    flops = C.c_double()
    probe = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(lib.gf_fp64_peak_probe(0, 100000, _lib.ptr(sink), C.byref(flops), None))
        e1.record()
        torch.cuda.synchronize()
        probe.append(flops.value / 2 / (e0.elapsed_time(e1) * 1e-3))
    peak_fma = max(probe)
    cases = [('quickstart', smp._chains[0])]
    g = torch.Generator(device='cuda').manual_seed(3)
    # a long-window case: AR(1) rho = 0.995 (tau ~ 400), 1 x 1024 x 10^4 x 6
    x = torch.empty((1, 1024, 10000, 6), dtype=torch.float64, device='cuda')
    eps = torch.randn((1, 1024, 10000, 6), dtype=torch.float64, device='cuda', generator=g)
    x[:, :, 0] = eps[:, :, 0]
    for i in range(1, 10000):
        x[:, :, i] = 0.995 * x[:, :, i - 1] + 0.0999 * eps[:, :, i]
    cases.append(('ar1_rho0.995', x))
    res['kernel'] = {'fp64_probe_fma_per_s': peak_fma}
    for name, ch in cases:
        _, w = mcmc.autocorr_time(ch, return_window=True)
        fmas = computed_fmas(ch.shape[1], ch.shape[2], w[0]) * 1
        reps = 5
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                mcmc.autocorr_time(ch)
            torch.cuda.synchronize()
        kt = {}
        for e in prof.key_averages():
            if e.key.startswith('k_acor') or 'k_acor' in e.key:
                us = getattr(e, 'device_time_total', None)
                if us is None:
                    us = e.cuda_time_total
                kt[e.key.split('(')[0]] = us * 1e-6 / reps
        tile_s = sum(v for k, v in kt.items() if 'tile' in k)
        call_s = event_time(lambda: mcmc.autocorr_time(ch), 5)
        rate = fmas / tile_s if tile_s else float('nan')
        res['kernel'][name] = dict(windows=w[0].tolist(), fmas=fmas, kernel_seconds=kt, call_seconds=call_s, fma_per_s=rate,
                                   fraction_of_probe=rate / peak_fma)
        print('%s: windows %s, %.3e FMAs, tile kernels %.5f s (%s), call %.5f s, %.3e FMA/s = %.3f of the fp64 probe (%.3e FMA/s)' % (
            name, w[0].tolist(), fmas, tile_s, {k: round(v, 6) for k, v in kt.items()}, call_s, rate, rate / peak_fma, peak_fma))
    del x, eps

    # -- 3. sweep
    kw = dict(segments=100, nwalkers=60, burnin=200, nsteps=1000, distributed=False)
    sens.sweep(segments=100, nwalkers=60, burnin=5, nsteps=5, distributed=False)
    sens.sweep(segments=100, nwalkers=60, burnin=5, nsteps=60, distributed=False, autocorr=True)
    times = {False: [], True: []}
    out = {}
    for _ in range(2):
        for ac in (False, True):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out[ac] = sens.sweep(autocorr=ac, **kw)
            times[ac].append(time.perf_counter() - t0)
    same = all(np.array_equal(out[True][k], out[False][k]) for k in out[False])
    tau = out[True]['tau']
    res['sweep'] = dict(seconds_off=times[False], seconds_on=times[True], outputs_identical=bool(same), tau_min=float(tau.min()),
                        tau_max=float(tau.max()), share_nsteps_below_50tau=float(np.mean(np.any(1000 < 50 * tau, axis=1))),
                        share_pairs_below_50tau=float(np.mean(1000 < 50 * tau)))
    print('sweep: off %s s, on %s s, outputs identical %s, tau in [%.2f, %.2f], grid points with 1000 < 50 tau (any parameter): %.3f, '
          '(point, parameter) pairs: %.3f' % (times[False], times[True], same, tau.min(), tau.max(), res['sweep']['share_nsteps_below_50tau'],
                                               res['sweep']['share_pairs_below_50tau']))
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
