"""Profile likelihood over many source compositions (sens.profile_source_grid) timed against a loop of single-source profile
grids in one run.

python scratch/profile_source_bench.py [output.json]

Prints the card's name, power limit and SM clocks, then for dims 3-8 x 100 scales x 64 starts with J = 1, 3 and 30 sources
(the 30 of scratch/source_grid_bench.py): seconds (median of three calls bracketed by CUDA events after a warm-up call of every
shape), objective evaluations per second (from the kernels' counts) and the ratio to the loop of J single-source
sens.profile_grid calls.  The loop of 30 is timed the same way in the same run; the loops of 1 and 3 are its 1/30 and 3/30
shares.  Also the largest |profile| difference between the source grid and the loop (the transition sums and the per-bin mix
differ in the last bits, so Nelder-Mead paths may part)."""

import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from golemflavor_b200 import scan, sens  # noqa: E402

DIMS, SEG, NSTARTS = (3, 4, 5, 6, 7, 8), 100, 64


def timed(fn, reps=3):
    """median seconds of `reps` calls, each bracketed by CUDA events after a device synchronise"""
    out, ts = None, []
    for _ in range(reps):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    return float(np.median(ts)), out


def evaluations(sources):
    """objective evaluations of one profile_source_grid call (the kernels' counts, one extra launch per dimension)"""
    n = 0
    for d in DIMS:
        fm = sens._grid_model(d, sens.Texture.OET, sources[0], np.ones(3), 0.02, scan.DEFAULT_BINNING)
        n += int(scan.scan_profile_sources(fm, sens.scale_grid(d, SEG), sources, (1, 1, 1), nstarts=NSTARTS)['nevals'].sum())
    return n


def main():
    card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader'],
                          capture_output=True, text=True).stdout.strip()
    print('card (name, power limit, SM clock, max SM clock):', card)
    print('library:', os.environ.get('GOLEMFLAVOR_B200_LIB', 'default'), 'GF_PROFILE_SPEC:', os.environ.get('GF_PROFILE_SPEC', 'default'))
    rng = np.random.default_rng(26)
    sources = np.concatenate([[(1., 2., 0.), (1., 0., 0.), (0., 1., 0.)], rng.uniform(size=(27, 3))])
    res = {'card': card, 'grid': '%d dims x %d scales x %d starts' % (len(DIMS), SEG, NSTARTS), 'sources': {}}

    def loop(j):
        return [sens.profile_grid(dimensions=DIMS, segments=SEG, source_ratio=s, nstarts=NSTARTS, distributed=False) for s in sources[:j]]

    loop(1)                                                                  # warm-up
    loop_sec, loop_pr = timed(lambda: loop(30))
    res['loop30_seconds'] = loop_sec
    print('loop of 30 profile_grid calls: %.4f s (%.4f s per source)' % (loop_sec, loop_sec / 30))
    for j in (1, 3, 30):
        run = lambda: sens.profile_source_grid(sources[:j], dimensions=DIMS, segments=SEG, nstarts=NSTARTS, distributed=False)  # noqa: E731
        run()                                                                # warm-up
        sec, pr = timed(run)
        evals = evaluations(sources[:j])
        diff = max(float(np.nan_to_num(np.abs(pr[d][k][:, 1] - loop_pr[k][d][:, 1]), nan=0.0).max()) for d in DIMS for k in range(j))
        ref = loop_sec * j / 30
        res['sources'][j] = dict(seconds=sec, evals=evals, evals_per_s=evals / sec, loop_seconds=ref, ratio_to_loop=sec / ref, max_abs_dprofile=diff)
        print('profile_source_grid J=%2d: %.4f s, %.3e evaluations (%.3e/s), %.3f of the loop of %d (%.4f s), max |d profile| %.2e'
              % (j, sec, evals, evals / sec, sec / ref, j, ref, diff))
    if len(sys.argv) > 1:
        with open(sys.argv[1], 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
