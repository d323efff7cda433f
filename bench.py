#!/usr/bin/env python
"""Benchmark of the log-posterior hot path (driver contract: one JSON line on stdout).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json config 3, the BSM fit the north star's roofline target names): the batched
BSM dim-6 / texture-OET log-posterior -- 6 SM parameters + log10(Lambda) per point, 20 energy bins,
Gaussian flavor-ratio likelihood + (truncated-)Gaussian priors -- on a synthetic batch of
4096 walkers x 1024 independent chains = 2^22 parameter points per step and per GPU (theta is
235 MB, larger than the 126 MB L2, so every step streams its input from HBM).  One step = one pass of
the hot path over that batch = ONE kernel launch.

  value    : log-posterior evaluations / s over all ranks, theta resident in HBM (CUDA events on the
             launching stream, barrier + synchronize on both sides, max over ranks)
  e2e      : same metric through the public host API (`llh.LnProb.evaluate_host` -> C ABI
             `gf_lnprob_host`): pinned host theta -> chunked H2D -> kernel -> D2H of the results
  roofline : EXECUTED fp64 instructions of the kernel (per point: counted by ncu for this very build,
             profiles/roofline_traffic.json, "ncu, offline") x evaluations / kernel time, as FMA-issue
             equivalents (2 FLOP per issue slot), against the fp64 FMA peak MEASURED in the same run by a
             DFMA microbenchmark (MEASURED_PEAKS.json carries no fp64 figure): `frac` is the share of
             the fp64 pipe's issue slots the kernel uses, <= 1 by construction.  The throughput in
             ALGORITHMIC FLOPs (SURVEY.md 8d: 9252 per evaluation of the reference's formulas; the
             kernel's own algebra needs fewer) is reported beside it as `algorithmic_tflops` /
             `algorithmic_ratio`; `sustained_*` repeats the measurement over >= 1 s of launches
  config   : besides the workload, the secondary sections the driver must keep: the sharded
             Monte-Carlo scan (config 4, `scan_*`: whole-job seconds incl. the NCCL all-reduce of the
             histograms, checksum) and the sampler-shaped configs C1/C2/C3/C5 and K1 (`c*_`, `k1_*`)
  cpu_baseline : the reference's scalar float128 ln_prob (baseline/_ref; the oracle port if that is absent) on
             1 host core for the headline model, plus the config-2 notebook model and config 1 end to end on
             the CPU (both: the oracle port)

`--impl reference` times the reference's own CPU implementation -- the UNMODIFIED package installed in
baseline/_ref (git-ignored, travels with the snapshot; `kind: "reference"`), else the oracle port
(`kind: "port"`) -- on all host cores for the same metric and config: exactly K steps after W warm-up
steps, each step a bounded sample of the workload.

`--dump-outputs DIR` writes what the last of the K timed GPU steps computed, the log-posterior of the batch, as
float64: DIR/lnprob.npy holds every point (32 MiB).  With N > 1 ranks, rank r writes DIR/lnprob_rank<r>.npy holding
every N-th point of its batch (rows 0, N, 2N, ...), so the files total 32 MiB whatever N is.  theta is drawn from a
fixed seed per rank, so two builds run with the same arguments can be compared output for output.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

FLOP_PER_EVAL = 9252          # SURVEY.md 8(d): F_BSM for D=7, G=5, 20 bins
BYTES_PER_EVAL = 64           # 7 doubles in, 1 out
WALKERS, CHAINS = 4096, 1024
METRIC = 'log-posterior evals/sec'
WORKLOAD = ('C3: BSM dim-6 operator, texture OET, 6 SM params + logLambda, 20 energy bins, Gaussian flavor-ratio LLH '
            '+ priors; 4096 walkers x 1024 chains = 4194304 points per step per GPU')


def build_problem():
    import models
    from golemflavor_b200.enums import Texture
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_llh.npz'))
    return models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OET), models


def synth_theta(pset, n, seed, models):
    """Uniform inside Param.ranges for the SM block (SURVEY 8d 'throughput batches'), logLam across
    the dim-6 scale boundaries."""
    rng = np.random.default_rng(seed)
    return models.draw_in_ranges(pset, n, rng)


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """Samples SM clock, power and throttle reasons of one GPU through NVML every 5 ms from a
    background thread while the timed region runs (the main thread sits in a CUDA synchronize,
    which releases the GIL)."""
    BAD = {'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20, 'sw_power_cap': 0x4,
           'hw_power_brake_slowdown': 0x80}

    def __init__(self, index):
        self.index, self.rows, self._stop, self.thread, self.err = index, [], threading.Event(), None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(visible.split(',')[index]) if visible and visible.split(',')[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception as exc:  # noqa: BLE001
            self.nv, self.err = None, repr(exc)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.rows.append((sm, pw, rs))
            except Exception as exc:  # noqa: BLE001
                self.err = repr(exc)
                break
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        if self.thread is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['clock sampling unavailable: %s' % self.err]}
        self._stop.set()
        self.thread.join()
        sm = [r[0] for r in self.rows]
        power = [r[1] for r in self.rows]
        reasons = sorted(name for name, bit in self.BAD.items() if any(r[2] & bit for r in self.rows))
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_min_mhz': min(sm) if sm else None, 'sm_max_mhz': self.max_sm,
                'power_w_max': max(power) if power else None, 'samples': len(sm), 'reasons': reasons}


# ---------------------------------------------------------------------------------------------- CPU arm
_CPU_STATE = {}


def _cpu_problem():
    """Model + oracle of the headline workload, built once per process (fork pool workers inherit it)."""
    if 'problem' not in _CPU_STATE:
        import models  # noqa: F401  (sys.path set at import)
        from oracle import golem_oracle as go
        (args, asimov, pset), _ = build_problem()
        _CPU_STATE['problem'] = (go, args, asimov, pset)
    return _CPU_STATE['problem']


def _cpu_eval_chunk(job):
    """Scalar float128 ln_prob of the oracle (restatement of llh.py:121-130 + fr.py) on a chunk."""
    seed, count = job
    go, args, asimov, pset = _cpu_problem()
    theta = synth_theta(pset, count, seed, sys.modules['models'])
    t0 = time.perf_counter()
    out = []
    for t in theta:
        try:
            out.append(go.ln_prob(list(t), args, asimov, pset))
        except AssertionError:   # the reference's unitarity assertion (fr.py:493-498): same work was done
            out.append(np.nan)
    return time.perf_counter() - t0, count, float(np.sum(np.isfinite(out)))


# ---------------------------------------------------------------------------------------------- the reference itself
REF_DIR = os.path.join(ROOT, 'baseline', '_ref')
TEXTURE_OET = (0. + 1e-9, 0.25, 0. + 1e-9, 0. + 1e-9)      # fr.py:370-376, the OET angle tuple


KIND_NOTE = {
    'reference': "the UNMODIFIED reference package (baseline/_ref): llh.lnprior + fr.flux_averaged_BSMu + llh.multi_gaussian composed "
                 "as llh.ln_prob / examples/inference.ipynb (GolemFit absent)",
    'port': 'the oracle restatement of the same functions (baseline/_ref not installed)'}


def _reference_problem():
    """The UNMODIFIED reference package (`pip install --target baseline/_ref /root/reference`, git-ignored, travels to
    the GPU box with the snapshot) set up for the headline workload, or None when it is not installed / importable.
    Imported behind the two-line Python-3.12 shim of tests/golden/make_golden.py; nothing else is patched.  GolemFit is
    proprietary and absent, so the likelihood is the Gaussian stand-in the reference documents
    (examples/inference.ipynb:307-366, README.md:76-77): `llh.ln_prob` (llh.py:121-130: deep copies, `lnprior`, early
    -inf) with `multi_gaussian(flux_averaged_BSMu(theta), injected, smearing)` in place of `gf_utils.get_llh`.  The
    fixed texture is passed as Texture.NONE with the explicit OET angle tuple (fr.py:370-376) because the texture branch
    builds a ragged array under NumPy >= 1.24 (same work-around as the golden fixtures): identical arithmetic."""
    if 'ref' in _CPU_STATE:
        return _CPU_STATE['ref']
    _CPU_STATE['ref'] = None
    if not os.path.isdir(os.path.join(REF_DIR, 'golemflavor')):
        return None
    try:
        import collections
        import collections.abc
        import fractions
        import math
        from argparse import Namespace
        if not hasattr(fractions, 'gcd'):
            fractions.gcd = math.gcd                           # golemflavor/misc.py:15
        if not hasattr(collections, 'Sequence'):
            collections.Sequence = collections.abc.Sequence    # golemflavor/param.py:15
        if REF_DIR not in sys.path:
            sys.path.insert(0, REF_DIR)
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):        # "Running without GolemFit"
            import golemflavor.fr as rfr
            import golemflavor.llh as rllh
            from golemflavor import enums as renums
            from golemflavor.param import Param as RParam, ParamSet as RParamSet
    except Exception as exc:  # noqa: BLE001
        _note('reference package in baseline/_ref not importable:', repr(exc))
        return None
    import models  # noqa: F401
    (args, asimov, pset), _ = build_problem()

    def conv(p, tag=None):
        prior = getattr(renums.PriorsCateg, p.prior.name) if p.prior is not None else None
        return RParam(name=p.name, value=p.nominal_value, seed=list(p.seed), ranges=list(p.ranges), std=p.std, prior=prior,
                      tag=getattr(renums.ParamTag, (tag or p.tag).name))

    plist = [conv(p) for p in pset]
    scale_at = [k for k, p in enumerate(plist) if p.tag is renums.ParamTag.SCALE][0]
    mm = [RParam(name=nm, value=v, ranges=[0., 2 * np.pi], std=0.2, tag=renums.ParamTag.MMANGLES)
          for nm, v in zip(['np_s12', 'np_c13', 'np_s23', 'np_dcp'], TEXTURE_OET)]
    rpset = RParamSet(plist[:scale_at] + mm + plist[scale_at:])
    rasimov = RParamSet([conv(p) for p in asimov])
    rargs = Namespace(binning=np.asarray(args.binning), source_ratio=rfr.normalize_fr(args.source_ratio), dimension=args.dimension,
                      texture=renums.Texture.NONE, no_bsm=False)
    smearing = rasimov[0].std
    injected = rfr.angles_to_fr(rasimov.from_tag(renums.ParamTag.BESTFIT, values=True))
    from copy import deepcopy

    def ln_prob(theta7):
        theta = list(theta7[:scale_at]) + list(TEXTURE_OET) + list(theta7[scale_at:])
        dc_pset = deepcopy(rpset)                    # llh.py:122-123
        deepcopy(rasimov)
        lp = rllh.lnprior(theta, paramset=dc_pset)
        if not np.isfinite(lp):
            return -np.inf
        fr = rfr.flux_averaged_BSMu(theta, rargs, -2.0, dc_pset)
        return lp + rllh.multi_gaussian(fr, injected, smearing)

    _CPU_STATE['ref'] = (ln_prob, pset)
    return _CPU_STATE['ref']


def _ref_eval_chunk(job):
    """The reference's own ln_prob composition on a chunk of the synthetic theta distribution."""
    seed, count = job
    ln_prob, pset = _reference_problem()
    theta = synth_theta(pset, count, seed, sys.modules['models'])
    t0 = time.perf_counter()
    out = []
    with np.errstate(all='ignore'):
        for t in theta:
            try:
                out.append(float(ln_prob(t)))
            except AssertionError:   # the reference's unitarity assertion (fr.py:493-498): same work was done
                out.append(np.nan)
    return time.perf_counter() - t0, count, float(np.sum(np.isfinite(out)))


def cpu_baseline(per_core, cores, pool=None, seed0=1000, kind='port'):
    chunk = _ref_eval_chunk if kind == 'reference' else _cpu_eval_chunk
    jobs = [(seed0 + c, per_core) for c in range(cores)]
    t0 = time.perf_counter()
    if cores == 1:
        res = [chunk(jobs[0])]
    elif pool is not None:
        res = pool.map(chunk, jobs, chunksize=1)
    else:
        import multiprocessing as mp
        with mp.get_context('fork').Pool(cores) as p:
            res = p.map(chunk, jobs, chunksize=1)
    wall = time.perf_counter() - t0
    total = sum(r[1] for r in res)
    compute = max(r[0] for r in res)
    return total / compute, total, wall


def cpu_baseline_c2(count):
    """Config-2 model (examples/inference.ipynb:307-366: 4 PMNS coordinates with LIMITEDGAUSS priors + 2 source
    angles, Gaussian LLH): the oracle's scalar float128 ln_prob on one core (BASELINE.md section 2: ~252 evals/s/core
    for the unmodified reference)."""
    import models as _m
    from oracle import golem_oracle as go
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_llh.npz'))
    args, asimov, pset = _m.notebook_model(g['asimov_angles'])
    theta = _m.draw_in_ranges(pset, count, np.random.default_rng(25), seeds=True)
    t0 = time.perf_counter()
    with np.errstate(divide='ignore'):
        for t in theta:
            go.ln_prob(list(t), args, asimov, pset)
    sec = time.perf_counter() - t0
    return {'value': count / sec, 'unit': 'evals/s', 'cores': 1, 'kind': 'port',
            'sample': '%d scalar float128 ln_prob evaluations of the 6-D notebook model (%.1f s)' % (count, sec)}


def cpu_baseline_c1(nsteps):
    """Config 1 END TO END on the CPU (BASELINE.md section 3): 100 walkers, 3 raw source ratios, PMNS fixed at NUFIT_U,
    the bundled NumPy stretch-move sampler (emcee is absent) scoring one walker per call with the oracle's scalar
    ln_prob, like emcee-2 with threads=1.  A bounded number of steps of the 1000-step chain."""
    import models as _m
    from golemflavor_b200 import mcmc
    from oracle import golem_oracle as go
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_llh.npz'))
    args, asimov, pset = _m.sm_fit_c1(g['asimov_angles'])
    np.random.seed(25)
    p0 = mcmc.flat_seed(pset, 100)

    def lnp(t):
        with np.errstate(divide='ignore'):
            v = go.ln_prob(list(t), args, asimov, pset)
        return v if v == v else -np.inf

    smp = mcmc.EnsembleSampler(100, 3, lnp, vectorize=False, seed=25)
    t0 = time.perf_counter()
    smp.run_mcmc(p0, nsteps)
    sec = time.perf_counter() - t0
    evals = 100 * (nsteps + 1)
    return {'value': evals / sec, 'unit': 'evals/s', 'cores': 1, 'kind': 'port', 'seconds_per_1000_steps': sec * 1000.0 / nsteps,
            'sample': '%d of the 1000 steps of the 100-walker chain, end to end on 1 core (%.1f s)' % (nsteps, sec)}


def run_reference(opts):
    """The reference arm: the oracle port on all host cores (emcee-2 `threads=N` style fork pool), EXACTLY K timed
    steps after W warm-up steps; a step is a bounded sample of the workload (the same synthetic theta distribution)
    sized so that the whole run takes about half a minute whatever K and W are."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    steps, warmup = opts.steps, max(0, opts.warmup)
    per_core = int(min(150, max(4, round(30.0 * 90.0 / (steps + warmup)))))   # ~90 evals/s/core
    kind = 'reference' if _reference_problem() is not None else 'port'         # set up before the fork: workers inherit it
    if kind == 'port':
        _cpu_problem()
    with mp.get_context('fork').Pool(cores) as pool:
        for w in range(warmup):
            cpu_baseline(per_core, cores, pool, seed0=500000 + 1000 * w, kind=kind)
        t0 = time.perf_counter()
        total = 0
        for k in range(steps):
            _, n, _ = cpu_baseline(per_core, cores, pool, seed0=1000 * (k + 1), kind=kind)
            total += n
        elapsed = time.perf_counter() - t0
    value = total / elapsed
    sample = '{0} scalar float128 ln_prob evaluations per step ({1} per process x {2} processes), same model and synthetic theta ' \
             'distribution as the GPU arm; {3}'.format(per_core * cores, per_core, cores, KIND_NOTE[kind])
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'evals/s', 'n_gpus': opts.gpus, 'steps': steps,
        'warmup': warmup, 'ms_per_step': 1e3 * elapsed / steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f80 (x87 long double, as the reference)', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'sample': sample},
        'cpu_baseline': {'value': value, 'unit': 'evals/s', 'cores': cores, 'kind': kind, 'sample': sample},
        'e2e': {'value': value, 'unit': 'evals/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------- GPU arm
def _note(*a):
    """Details that do not belong into the one JSON line go to stderr."""
    sys.stderr.write(' '.join(str(x) for x in a) + '\n')
    sys.stderr.flush()


def run_gpu(opts):
    import ctypes as C

    import torch
    import torch.distributed as dist
    from golemflavor_b200 import _lib, llh, scan

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- the GPU arm has no CPU fallback (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    numa = None
    try:  # keep this rank (and the pinned buffers it first-touches) on the CPUs / NUMA node next to its GPU
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get('CUDA_VISIBLE_DEVICES')
        phys = int(visible.split(',')[local]) if visible and visible.split(',')[local].isdigit() else local
        handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        try:
            numa = int(pynvml.nvmlDeviceGetNumaNodeId(handle))
        except Exception:  # noqa: BLE001
            numa = None
    except Exception:  # noqa: BLE001  (affinity is an optimisation, never a requirement)
        pass
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    lib = _lib.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def over_ranks(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(x):
        return over_ranks(x, dist.ReduceOp.MAX)

    def min_over_ranks(x):
        return over_ranks(x, dist.ReduceOp.MIN)

    (args, asimov, pset), models = build_problem()
    fn = llh.LnProb(args, asimov, pset)
    n = WALKERS * CHAINS
    theta_host = torch.as_tensor(synth_theta(pset, n, 25 + rank, models)).pin_memory()
    theta = theta_host.cuda()
    out = torch.empty(n, dtype=torch.float64, device='cuda')
    stream = _lib.stream_ptr(torch)

    def step():
        _lib.check(lib.gf_lnprob(fn.model.ref, _lib.ptr(theta), n, fn.ndim, 1, _lib.ptr(out), None, None, stream))

    # -- fp64 peak probe (same run, same clocks)
    sink = torch.zeros(8, dtype=torch.float64, device='cuda')
    flops = C.c_double()
    peak = 0.0
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(lib.gf_fp64_peak_probe(0, 200000, _lib.ptr(sink), C.byref(flops), stream))
        e1.record()
        torch.cuda.synchronize()
        peak = max(peak, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)

    # -- warm-up, then the same launch repeated for >= 1 s (sustained clocks and rate under a long load), then EXACTLY K timed steps
    for _ in range(opts.warmup):
        step()
    sus_steps = int(max(opts.steps, np.ceil(opts.sustain_s * 1e3 / 0.55))) if opts.sustain_s > 0 else 0
    sustained = None
    if sus_steps:
        clocks2 = ClockSampler(local)
        barrier()
        if rank == 0:
            clocks2.start()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(sus_steps):
            step()
        s1.record()
        barrier()
        sus_ms = max_over_ranks(s0.elapsed_time(s1))
        c2 = clocks2.stop() if rank == 0 else None
        sustained = {'steps': sus_steps, 'seconds': sus_ms * 1e-3, 'ms_per_step': sus_ms / sus_steps,
                     'value': world * n * sus_steps / (sus_ms * 1e-3), 'clocks': c2}

    # -- device-resident throughput: exactly K steps
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    launches0 = lib.gf_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(opts.steps):
        step()
    e1.record()
    barrier()
    launches = lib.gf_launch_count() - launches0
    ms = max_over_ranks(e0.elapsed_time(e1))
    clock_info = clocks.stop() if rank == 0 else None
    value = world * n * opts.steps / (ms * 1e-3)
    kernel_ms = ms / opts.steps
    if opts.dump_outputs:
        name = 'lnprob.npy' if world == 1 else 'lnprob_rank%d.npy' % rank
        np.save(os.path.join(opts.dump_outputs, name), out[::world].cpu().numpy())   # one world-th of each rank's rows

    # -- end to end through the host API
    out_host = torch.empty(n, dtype=torch.float64).pin_memory()
    th_np, out_np = theta_host.numpy(), out_host.numpy()
    e2e_steps = max(3, min(opts.steps, 10))
    for _ in range(2):
        fn.evaluate_host(th_np, out=out_np)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        fn.evaluate_host(th_np, out=out_np)     # returns after the results are in host memory
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * n * e2e_steps / e2e_s
    assert np.array_equal(out_np, out.cpu().numpy()), 'host pipeline and device path disagree'
    # context for e2e: the plain pinned-host -> device copy rate of the same theta buffer, measured on ALL ranks AT THE
    # SAME TIME (barrier first): the contended link ceiling of this box, which the pipeline cannot exceed
    link = 0.0
    for _ in range(3):
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        theta.copy_(theta_host, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        link = max(link, theta_host.numel() * 8 / (c0.elapsed_time(c1) * 1e-3) / 1e9)
    link_min = min_over_ranks(link)
    # ... and the same input copy while the step's results stream back on a second stream, as they do inside the pipeline
    # (H2D 56 B + D2H 8 B per point): the ceiling the pipeline itself can reach on this host
    link_bidir, side = 0.0, torch.cuda.Stream()
    for _ in range(3):
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            out_host.copy_(out, non_blocking=True)
        theta.copy_(theta_host, non_blocking=True)
        torch.cuda.current_stream().wait_stream(side)
        c1.record()
        torch.cuda.synchronize()
        link_bidir = max(link_bidir, theta_host.numel() * 8 / (c0.elapsed_time(c1) * 1e-3) / 1e9)
    link_bidir_min = min_over_ranks(link_bidir)
    finite_frac = float(np.isfinite(out_np).mean())

    # -- secondary: sharded Monte-Carlo scan with the histogram all-reduce (config 4)
    def _scan_section():
        if opts.scan_samples <= 0:
            return {}
        fm = scan.scan_model(opts.scan_mode, dimension=6)
        scan.scan_histogram(fm, 10 ** 7, nb=25, seed=26)      # warm-up (also NCCL channel set-up)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        hist, kept = scan.scan_histogram(fm, opts.scan_samples, nb=25, seed=26, return_tensor=True)
        s1.record()
        barrier()
        scan_ms = max_over_ranks(s0.elapsed_time(s1))
        checksum = int((hist.flatten() * torch.arange(hist.numel(), device='cuda') % 1000003).sum().item())
        return {'scan_mode': opts.scan_mode, 'scan_samples': opts.scan_samples, 'scan_nb': 25, 'scan_seconds': scan_ms * 1e-3,
                'scan_samples_per_s': opts.scan_samples / (scan_ms * 1e-3), 'scan_scaling': 'strong', 'scan_kept': int(kept.item()),
                'scan_hist_checksum': checksum,
                'scan_collective': 'one NCCL all-reduce (sum, int64) of the 26^3 histogram' if world > 1 else 'none (1 GPU)'}

    try:
        scan_info = _scan_section()
    except Exception as exc:  # noqa: BLE001  (a secondary section must never cost the headline line)
        scan_info = {'scan_error': repr(exc)}

    # -- secondary: the sampler-shaped configs of BASELINE.json (latency-bound by design: 50 / 512 / 2048 /
    #    18000 points per half-step), run on the device-resident ensemble sampler, and K1 against HBM
    def _configs_section():
        if not opts.configs:
            return {}
        import models as _m
        from golemflavor_b200 import mcmc, sens
        g = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_llh.npz'))
        info = {}

        def timed(fn_):
            barrier()
            t0_ = time.perf_counter()
            r_ = fn_()
            torch.cuda.synchronize()
            return max_over_ranks(time.perf_counter() - t0_), r_

        a2, as2, ps2 = _m.notebook_model(g['asimov_angles'])
        f2 = llh.LnProb(a2, as2, ps2)
        np.random.seed(25)
        p0 = mcmc.flat_seed(ps2, 1024)
        p0[:, 4], p0[:, 5] = np.random.uniform(.9, 1, 1024), np.random.uniform(.8, 1, 1024)
        # K1: the SM-only log-posterior (161 algorithmic FLOP / 56 B per point) is HBM-bound: report it against HBM
        n1 = 1 << 24
        th1 = torch.as_tensor(_m.draw_in_ranges(ps2, 1 << 20, np.random.default_rng(3))).cuda().repeat(16, 1)
        o1 = torch.empty(n1, dtype=torch.float64, device='cuda')
        k1 = lambda: _lib.check(lib.gf_lnprob(f2.model.ref, _lib.ptr(th1), n1, 6, 1, _lib.ptr(o1), None, None, stream))  # noqa: E731
        for _ in range(3):
            k1()
        torch.cuda.synchronize()
        k0e, k1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0e.record()
        for _ in range(20):
            k1()
        k1e.record()
        torch.cuda.synchronize()
        k1ms = k0e.elapsed_time(k1e) / 20
        info['k1_sm_lnprob_evals_per_s'] = n1 / (k1ms * 1e-3)
        info['k1_sm_lnprob_gbs'] = 56.0 * n1 / (k1ms * 1e-3) / 1e9      # 6-D notebook model, theta 805 MB > L2, 56 B / point
        del th1, o1
        smp = mcmc.DeviceEnsembleSampler(1024, 6, f2, seed=25)
        smp.run_mcmc(p0, 200, store=False)
        sec, _ = timed(lambda: smp.run_mcmc(None, 10000, store=True, return_tensor=True))
        info['c2_emcee_1024x10000_seconds'] = sec
        info['c2_acceptance'] = float(np.mean(smp.acceptance_fraction))
        # C1: the reference's own CPU-sized case (3 raw source ratios, fixed NuFIT PMNS), here on the device sampler
        a1, as1, ps1 = _m.sm_fit_c1(g['asimov_angles'])
        f1 = llh.LnProb(a1, as1, ps1)
        p1 = mcmc.flat_seed(ps1, 100)
        smp1 = mcmc.DeviceEnsembleSampler(100, 3, f1, seed=25)
        smp1.run_mcmc(p1, 100, store=False)
        sec, _ = timed(lambda: smp1.run_mcmc(None, 1000, store=True, return_tensor=True))
        info['c1_emcee_100x1000_seconds'] = sec
        p3 = mcmc.flat_seed(pset, 4096)
        smp3 = mcmc.DeviceEnsembleSampler(4096, fn.ndim, fn, seed=25)
        smp3.run_mcmc(p3, 100, store=False)
        sec = min(timed(lambda: smp3.run_mcmc(None, 2000, store=False, return_tensor=True))[0] for _ in range(2))   # best of two launches
        info['c3_bsm_4096_walkers_us_per_step'] = sec / 2000 * 1e6
        info['c3_acceptance'] = float(np.mean(smp3.acceptance_fraction))
        sens.sweep(segments=100, nwalkers=60, burnin=5, nsteps=5)   # warm-up (first launches, NCCL float64 path)
        sec, sw = timed(lambda: sens.sweep(segments=100, nwalkers=60, burnin=200, nsteps=1000))
        info['c5_sweep_600x60x1200_seconds'] = sec      # grid points split over the ranks, one all-reduce of the summaries
        info['c5_sweep_acceptance'] = float(sw['acceptance'].mean())
        sens.evidence_grid(dimensions=(6,), segments=4, samples=10000)                 # warm-up
        sec, ev = timed(lambda: sens.evidence_grid(segments=100, samples=1000000))
        info['c5_evidence_600x1e6_seconds'] = sec       # Monte-Carlo evidence per (dimension, scale); samples sharded over the ranks
        info['c5_evidence_samples_per_s'] = 6e8 / sec
        return info

    try:
        cfg_info = _configs_section()
    except Exception as exc:  # noqa: BLE001  (a secondary section must never cost the headline line)
        cfg_info = {'configs_error': repr(exc)}

    if rank == 0:
        base = None
        if world == 1 and opts.cpu_evals > 0:
            kind = 'reference' if _reference_problem() is not None else 'port'
            v, total, wall = cpu_baseline(opts.cpu_evals, 1, kind=kind)
            base = {'value': v, 'unit': 'evals/s', 'cores': 1, 'kind': kind,
                    'sample': '{0} scalar float128 ln_prob evaluations of the same model ({1:.1f} s); {2}'.format(total, wall, KIND_NOTE[kind])}
            try:
                base['c2_notebook_model'] = cpu_baseline_c2(max(50, opts.cpu_evals // 3))
                base['c1_end_to_end'] = cpu_baseline_c1(max(10, opts.cpu_evals // 8))
            except Exception as exc:  # noqa: BLE001
                base['secondary_error'] = repr(exc)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except (OSError, ValueError):
            pass
        hbm_peak = peaks.get('hbm_gbs', 6650.0)
        prof = {}
        try:
            prof = json.load(open(os.path.join(ROOT, 'profiles', 'roofline_traffic.json')))
        except (OSError, ValueError):
            pass
        inst = prof.get('k_lnprob_fp64_thread_inst_per_point')      # ncu count for this build (dfma + dmul + dadd + other fp64-pipe)
        evals_per_s_gpu = n / (kernel_ms * 1e-3)
        executed = 2.0 * inst * evals_per_s_gpu / 1e12 if inst else None   # TFLOP/s in FMA-issue equivalents (2 per issue slot)
        algorithmic = FLOP_PER_EVAL * evals_per_s_gpu / 1e12
        hbm_gbs = BYTES_PER_EVAL * evals_per_s_gpu / 1e9
        roof = {'bound': 'fp64', 'achieved': executed, 'peak': peak, 'unit': 'TFLOP/s (FMA-issue equivalents: 2 per fp64 instruction)',
                'frac': executed / peak if executed and peak else None,
                'traffic': prof.get('k_lnprob_bytes_per_launch'), 'traffic_source': 'ncu --set full, offline (%s)' % prof.get('k_lnprob_bytes_per_launch_source'),
                'kernel': 'k_lnprob<0,5,1>', 'fp64_inst_per_eval': inst, 'fp64_inst_source': 'ncu, offline (%s)' % prof.get('k_lnprob_fp64_inst_source'),
                'fp64_pipe_active_pct_ncu': prof.get('k_lnprob_fp64_pipe_pct'),
                'algorithmic_flop_per_eval': FLOP_PER_EVAL, 'algorithmic_tflops': algorithmic, 'algorithmic_ratio': algorithmic / peak if peak else None,
                'peak_source': 'DFMA microbenchmark (gf_fp64_peak_probe) in this run; nominal 148 SM x 64 FMA/clk x 2 x 1.965 GHz = 37.2',
                'hbm_gbs': hbm_gbs, 'hbm_frac': hbm_gbs / hbm_peak, 'hbm_peak_source': 'MEASURED_PEAKS.json' if peaks else 'fallback'}
        # dispatch bound: a sub-partition dispatches one warp instruction per cycle and an fp64 instruction holds the port for
        # two, so a warp needs >= N_fp64 + N_all cycles per point (DESIGN.md, K2); measured = kernel time x SM clock / warps per sub-partition
        winst = prof.get('k_lnprob_warp_inst_per_point')
        sm_mhz = (clock_info or {}).get('sm_mhz') or _lib.device_info()['clock_khz'] / 1e3
        if inst and winst and sm_mhz:
            warps_per_subpartition = n / 32.0 / (_lib.device_info()['sm_count'] * 4)
            measured_cycles = kernel_ms * 1e-3 * sm_mhz * 1e6 / warps_per_subpartition
            roof['dispatch_bound'] = {'cycles_per_warp_point_min': inst + winst, 'cycles_per_warp_point_measured': measured_cycles,
                                      'frac': (inst + winst) / measured_cycles, 'warp_inst_per_eval': winst,
                                      'note': '2 x fp64 + other warp instructions (ncu, offline) against kernel time x SM clock'}
        if sustained:
            roof['sustained_seconds'] = sustained['seconds']
            roof['sustained_ms_per_step'] = sustained['ms_per_step']
            roof['sustained_value'] = sustained['value']
            roof['sustained_frac'] = (2.0 * inst * (n / (sustained['ms_per_step'] * 1e-3)) / 1e12 / peak) if inst and peak else None
            if clock_info is not None and sustained['clocks']:
                clock_info['sustained'] = {k: sustained['clocks'].get(k) for k in ('sm_mhz', 'sm_min_mhz', 'power_w_max', 'samples', 'reasons')}
        config = {'workload': WORKLOAD, 'points_per_step_per_gpu': n, 'ndim': fn.ndim, 'nbins': 20,
                  'parallelism': 'dp%d (independent shards, no data-path collective)' % world,
                  'l2': 'inputs (235 MB theta per step) larger than the 126 MB L2', 'finite_fraction': finite_frac}
        config.update(scan_info)
        config.update(cfg_info)
        if 'k1_sm_lnprob_gbs' in config:
            config['k1_hbm_frac'] = config['k1_sm_lnprob_gbs'] / hbm_peak
        line = {
            'metric': METRIC, 'value': value, 'unit': 'evals/s', 'n_gpus': world, 'steps': opts.steps, 'warmup': opts.warmup,
            'ms_per_step': kernel_ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic',
            'config': config,
            'roofline': roof,
            'cpu_baseline': base,
            'e2e': {'value': e2e_value, 'unit': 'evals/s', 'h2d_bytes_per_step': n * fn.ndim * 8, 'd2h_bytes_per_step': n * 8,
                    'steps': e2e_steps, 'api': 'llh.LnProb.evaluate_host -> gf_lnprob_host (pinned host buffers)',
                    'h2d_gbs': e2e_value / world * fn.ndim * 8 / 1e9, 'h2d_link_gbs': link, 'h2d_link_gbs_min_over_ranks': link_min,
                    'h2d_link_gbs_with_d2h': link_bidir, 'h2d_link_gbs_with_d2h_min_over_ranks': link_bidir_min,
                    'link_note': 'plain pinned copies of the same buffers, all ranks at the same time after a barrier',
                    'numa_node': numa},
            'gpu_launches': int(launches),
            'clocks': clock_info,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def _claim_stdout():
    """The driver parses ONE JSON line from stdout, but libraries write there too (NCCL prints its
    version banner to fd 1 on communicator creation).  Keep a private duplicate of the real stdout
    for the result line and point fd 1 at stderr for everybody else."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=400)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--cpu-evals', type=int, default=1500, help='size of the bounded CPU-baseline sample (0 = skip)')
    ap.add_argument('--scan-samples', type=int, default=10 ** 10, help='samples of the secondary scan section (0 = skip)')
    ap.add_argument('--configs', type=int, default=1, help='1: also time the sampler-shaped configs C2/C3/C5 (secondary section)')
    ap.add_argument('--scan-mode', default='anarchic', choices=['unitary', 'x', 'texture', 'anarchic'])
    ap.add_argument('--sustain-s', type=float, default=1.2, help='length of the sustained k_lnprob loop after the K timed steps (0 = skip)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the log-posterior of the last timed step to DIR (GPU arm; 32 MiB in all)')
    opts = ap.parse_args()
    if opts.steps < 1:
        ap.error('--steps must be at least 1')
    if opts.dump_outputs:
        if opts.impl == 'reference':
            ap.error('--dump-outputs writes the outputs of the GPU arm; the reference arm keeps none')
        os.makedirs(opts.dump_outputs, exist_ok=True)
    opts.warmup = max(opts.warmup, 3) if opts.impl == 'b200' else opts.warmup
    if opts.impl == 'reference':
        run_reference(opts)
    else:
        run_gpu(opts)


if __name__ == '__main__':
    main()
