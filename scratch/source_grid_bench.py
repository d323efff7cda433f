"""Evidence grid over many source compositions (sens.evidence_source_grid) timed against a loop of single-source evidence grids
in one run.

python scratch/source_grid_bench.py [output.json]

Prints the card's name, power limit and SM clocks, then for dims 3-8 x 100 scales x 10^6 samples with J = 1, 3 and 30 sources:
seconds (median of three calls bracketed by CUDA events after a warm-up call of every shape), (sample, scale, source)
evaluations per second and the ratio to the loop of J single-source sens.evidence_grid calls.  The loop of 30 is timed the same
way in the same run; the loops of 1 and 3 are its 1/30 and 3/30 shares.  Also the largest |lnZ| difference between the source
grid and the loop (the two compute the same samples)."""

import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from golemflavor_b200 import sens  # noqa: E402

DIMS, SEG, N = (3, 4, 5, 6, 7, 8), 100, 1_000_000


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


def main():
    card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader'],
                          capture_output=True, text=True).stdout.strip()
    print('card (name, power limit, SM clock, max SM clock):', card)
    rng = np.random.default_rng(26)
    sources = np.concatenate([[(1., 2., 0.), (1., 0., 0.), (0., 1., 0.)], rng.uniform(size=(27, 3))])
    res = {'card': card, 'grid': '%d dims x %d scales x %d samples' % (len(DIMS), SEG, N), 'sources': {}}

    def loop(j):
        return [sens.evidence_grid(dimensions=DIMS, segments=SEG, source_ratio=s, samples=N) for s in sources[:j]]

    loop(1)                                                                  # warm-up
    loop_sec, loop_ev = timed(lambda: loop(30))
    res['loop30_seconds'] = loop_sec
    print('loop of 30 evidence_grid calls: %.4f s (%.4f s per source)' % (loop_sec, loop_sec / 30))
    for j in (1, 3, 30):
        run = lambda: sens.evidence_source_grid(sources[:j], dimensions=DIMS, segments=SEG, samples=N)  # noqa: E731
        run()                                                                # warm-up
        sec, ev = timed(run)
        evals = len(DIMS) * SEG * N * j
        diff = 0.0
        for d in DIMS:
            for k in range(j):
                a, b = ev[d][k][:, 1], loop_ev[k][d][:, 1]
                f = np.isfinite(a) & np.isfinite(b)
                assert np.array_equal(np.isfinite(a), np.isfinite(b)), (d, k)
                diff = max(diff, float(np.abs(a[f] - b[f]).max(initial=0.0)))
        ref = loop_sec * j / 30
        res['sources'][j] = dict(seconds=sec, evals_per_s=evals / sec, loop_seconds=ref, ratio_to_loop=sec / ref, max_abs_dlnz=diff)
        print('evidence_source_grid J=%2d: %.4f s, %.3e (sample, scale, source)/s, %.3f of the loop of %d (%.4f s), max |dlnZ| %.2e'
              % (j, sec, evals / sec, sec / ref, j, ref, diff))
    if len(sys.argv) > 1:
        with open(sys.argv[1], 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
