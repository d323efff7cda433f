"""Profile-likelihood grid (gf_profile_grid via sens.profile_grid) timed against K2 and the evidence grid in one run.

python scratch/profile_bench.py [output.json]

Prints the card's name and power limit, then for dims 3-8 x 100 scales at 32, 64 and 128 starts: seconds (CUDA events around
synchronised work, after a warm-up call of every shape), total optimiser evaluations, evaluations/s, the share of starts
that converged before max_evals and the largest change of the profile between start counts.  K2 (LnProb.evaluate on 2^22
points) and sens.evidence_grid (10^6 samples per scale) are timed the same way."""

import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import models  # noqa: E402
from golemflavor_b200 import scan, sens  # noqa: E402
from golemflavor_b200.enums import Texture  # noqa: E402
from golemflavor_b200.llh import LnProb  # noqa: E402

DIMS, SEG = (3, 4, 5, 6, 7, 8), 100


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


def counts(nstarts):
    """evaluations and converged starts of the same grid, from scan_profile_grid (same seed and task indices)"""
    nev, conv = 0, 0
    for d in DIMS:
        fm = sens._grid_model(d, Texture.OET, np.array([1., 2, 0]), np.array([1., 1, 1]), 0.02, scan.DEFAULT_BINNING)
        r = scan.scan_profile_grid(fm, sens.scale_grid(d, SEG), nstarts=nstarts, seed=27)
        nev += int(r['nevals'].sum())
        conv += int(r['nconverged'].sum())
    return nev, conv / (len(DIMS) * SEG * nstarts)


def main():
    card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                          capture_output=True, text=True).stdout.strip()
    print('card:', card)
    res = {'card': card, 'profile': {}}
    prev = None
    for ns in (32, 64, 128):
        run = lambda: sens.profile_grid(dimensions=DIMS, segments=SEG, nstarts=ns, distributed=False)  # noqa: E731
        run()                                                                                              # warm-up
        sec, prof = timed(run)
        nev, conv = counts(ns)
        cur = np.concatenate([prof[d][:, 1] for d in DIMS])
        delta = None if prev is None else float(np.max(np.abs(cur - prev)))
        prev = cur
        res['profile'][ns] = dict(seconds=sec, evaluations=nev, evals_per_s=nev / sec, converged_share=conv, max_change_vs_previous=delta)
        print('profile_grid dims 3-8 x %d scales, %3d starts: %.4f s, %.3e evaluations, %.3e evals/s, converged %.4f, max |change| vs '
              'previous start count %s' % (SEG, ns, sec, nev, nev / sec, conv, delta))
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_llh.npz'))
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OET)
    fn = LnProb(args, asimov, pset)
    theta = torch.as_tensor(models.draw_in_ranges(pset, 1 << 22, np.random.default_rng(3), seeds=True)).cuda()
    fn.evaluate(theta)
    sec, _ = timed(lambda: fn.evaluate(theta), reps=10)
    res['k2'] = dict(points=1 << 22, seconds=sec, evals_per_s=(1 << 22) / sec)
    print('K2 LnProb.evaluate 2^22 points: %.5f s, %.3e evals/s' % (sec, (1 << 22) / sec))
    sens.evidence_grid(dimensions=DIMS, segments=SEG, samples=1_000_000)
    sec, _ = timed(lambda: sens.evidence_grid(dimensions=DIMS, segments=SEG, samples=1_000_000))
    ev = len(DIMS) * SEG * 1_000_000
    res['evidence_grid'] = dict(evaluations=ev, seconds=sec, evals_per_s=ev / sec)
    print('evidence_grid dims 3-8 x %d scales x 1e6 samples: %.4f s, %.3e evals/s' % (SEG, sec, ev / sec))
    if len(sys.argv) > 1:
        with open(sys.argv[1], 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
