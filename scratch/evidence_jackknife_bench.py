"""Cost of the jackknife groups: sens.evidence_grid and sens.evidence_source_grid (30 sources) with and without groups=16,
timed alternately in one run.

python scratch/evidence_jackknife_bench.py [output.json]

Prints the card's name, power limit and SM clocks, then for dims 3-8 x 100 scales x 10^6 samples: seconds of each of the four
calls (median of three rounds, the four calls alternating within a round, each call bracketed by CUDA events after a device
synchronise, every shape warmed up first), the grouped / ungrouped ratios, the largest |lnZ| difference between the grouped
and the ungrouped results (the same samples, merged in another order), the errors of the 30-source table at R = 16, and at every
R = 2 ... 32 the two parts of a call timed apart: the kernel launches of all dimensions (CUDA events around the launches only,
the same alternating rounds) and the host leave-one-out (scan._group_lnz on the copied-back pairs, host clock)."""

import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from golemflavor_b200 import _lib, scan, sens  # noqa: E402
from golemflavor_b200.enums import Texture  # noqa: E402

DIMS, SEG, N, R = (3, 4, 5, 6, 7, 8), 100, 1_000_000, 16


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3, out


def launches(sources, groups):
    """fn() enqueuing exactly the kernel launches of sens.evidence_grid (sources None) or sens.evidence_source_grid for all
    dimensions into preallocated outputs -- no host post-processing -- and the output tensor."""
    lib, stream = _lib.load(), _lib.stream_ptr(torch)
    grids = [sens.scale_grid(d, SEG) for d in DIMS]
    scales = torch.as_tensor(np.stack(grids)).cuda()
    cfg = _lib.ScanConfig(seed=26, first_index=0, count=N, nb=0)
    R = groups or 1
    one, inj = np.array([1., 2., 0.]), np.array([1., 1., 1.])
    fms = [sens._grid_model(d, Texture.OET, one, inj, 0.02, scan.DEFAULT_BINNING) for d in DIMS]
    if sources is None:
        lse = torch.empty((len(DIMS), SEG, R, 2), dtype=torch.float64, device='cuda')
        wb = int(lib.gf_scan_evidence_grid_groups_workspace(SEG, R) if groups else lib.gf_scan_evidence_grid_workspace(SEG))
        work = torch.empty(wb, dtype=torch.uint8, device='cuda')

        def fn():
            for k, fm in enumerate(fms):
                sc, out = C.c_void_p(scales[k].data_ptr()), C.c_void_p(lse[k].data_ptr())
                if groups:
                    _lib.check(lib.gf_scan_evidence_grid_groups(fm.ref, C.byref(cfg), sc, SEG, R, out, _lib.ptr(work), wb, stream))
                else:
                    _lib.check(lib.gf_scan_evidence_grid(fm.ref, C.byref(cfg), sc, SEG, out, _lib.ptr(work), wb, stream))
    else:
        src, injs = scan.source_rows(sources, inj)
        lse = torch.empty((len(DIMS), len(src), SEG, R, 2), dtype=torch.float64, device='cuda')

        def fn():
            for k, fm in enumerate(fms):
                scan._sources_launch(lib, fm, cfg, scales[k], SEG, src, injs, lse[k], stream, groups=groups)
    return fn, lse


def timed_launches(fn, lse):
    lse[..., 0], lse[..., 1] = -np.inf, 0.0
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3


def max_dlnz(a, b):
    out = 0.0
    for d in a:
        x, y = a[d][..., 1], b[d][..., 1]
        assert np.array_equal(np.isfinite(x), np.isfinite(y)), d
        f = np.isfinite(x)
        out = max(out, float(np.abs(x[f] - y[f]).max(initial=0.0)))
    return out


def main():
    card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader'],
                          capture_output=True, text=True).stdout.strip()
    print('card (name, power limit, SM clock, max SM clock):', card)
    rng = np.random.default_rng(26)
    sources = np.concatenate([[(1., 2., 0.), (1., 0., 0.), (0., 1., 0.)], rng.uniform(size=(27, 3))])
    runs = {
        'grid': lambda: sens.evidence_grid(dimensions=DIMS, segments=SEG, samples=N),
        'grid_groups16': lambda: sens.evidence_grid(dimensions=DIMS, segments=SEG, samples=N, groups=R),
        'sources30': lambda: sens.evidence_source_grid(sources, dimensions=DIMS, segments=SEG, samples=N),
        'sources30_groups16': lambda: sens.evidence_source_grid(sources, dimensions=DIMS, segments=SEG, samples=N, groups=R),
    }
    for fn in runs.values():                                                  # warm-up of every shape
        fn()
    times, outs = {k: [] for k in runs}, {}
    for _ in range(3):
        for k, fn in runs.items():
            t, outs[k] = timed(fn)
            times[k].append(t)
    sec = {k: float(np.median(v)) for k, v in times.items()}
    res = {'card': card, 'grid': '%d dims x %d scales x %d samples, groups %d' % (len(DIMS), SEG, N, R), 'seconds': sec, 'all_seconds': times,
           'ratio_grid': sec['grid_groups16'] / sec['grid'], 'ratio_sources30': sec['sources30_groups16'] / sec['sources30'],
           'max_abs_dlnz_grid': max_dlnz(outs['grid_groups16'][0], outs['grid']),
           'max_abs_dlnz_sources30': max_dlnz(outs['sources30_groups16'][0], outs['sources30'])}
    for k in runs:
        print('%-20s %.4f s  (rounds %s)' % (k, sec[k], ' '.join('%.4f' % t for t in times[k])))
    print('grouped / ungrouped: evidence_grid %.4f, evidence_source_grid (30 sources) %.4f' % (res['ratio_grid'], res['ratio_sources30']))
    print('max |dlnZ| grouped vs ungrouped: grid %.2e, sources %.2e' % (res['max_abs_dlnz_grid'], res['max_abs_dlnz_sources30']))
    # the two parts of a call apart: kernel launches only (events around the launches, alternating rounds) and the host
    # leave-one-out of the copied-back pairs
    res['parts'] = {}
    for what, srcs in (('grid', None), ('sources30', sources)):
        shapes = {g: launches(srcs, g) for g in (None, 2, 4, 8, 16, 32)}
        for fn, lse in shapes.values():                                       # warm-up
            timed_launches(fn, lse)
        kt = {g: [] for g in shapes}
        for _ in range(3):
            for g, (fn, lse) in shapes.items():
                kt[g].append(timed_launches(fn, lse))
        base = float(np.median(kt[None]))
        res['parts'][what] = {'kernels_ungrouped_seconds': base}
        print('%s kernels only, ungrouped: %.4f s' % (what, base))
        for g in (2, 4, 8, 16, 32):
            k = float(np.median(kt[g]))
            h = shapes[g][1].cpu().numpy()
            if srcs is None:
                h = h.reshape(-1, SEG, g, 2)
            ht = []
            for _ in range(3):
                t0 = time.perf_counter()
                scan._group_lnz(h, N)
                ht.append(time.perf_counter() - t0)
            hs = float(np.median(ht))
            res['parts'][what][g] = dict(kernels_seconds=k, kernels_ratio=k / base, host_loo_seconds=hs)
            print('%s groups=%2d: kernels %.4f s (%.4f of ungrouped), host leave-one-out %.4f s' % (what, g, k, k / base, hs))
    ev, loo = outs['sources30_groups16']
    sig = sens.evidence_error(ev, loo)
    L, disc, err, nund = sens.limit_table(ev, loo=loo)
    fin = np.concatenate([s[np.isfinite(s)] for s in sig.values()])
    res['sigma_lnz_median'], res['sigma_lnz_max_finite'] = float(np.median(fin)), float(fin.max())
    res['limits_defined'], res['limit_err_finite'] = int(np.sum(~np.isnan(L))), int(np.sum(np.isfinite(err)))
    res['limit_err_median'] = float(np.median(err[np.isfinite(err)])) if np.isfinite(err).any() else None
    print('30-source table: sigma(lnZ) median %.3g (max finite %.3g); %d limits, %d with a finite error (median %s), %d with +inf'
          % (res['sigma_lnz_median'], res['sigma_lnz_max_finite'], res['limits_defined'], res['limit_err_finite'], res['limit_err_median'],
             int(np.sum(np.isposinf(err)))))
    if len(sys.argv) > 1:
        with open(sys.argv[1], 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
