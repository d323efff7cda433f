"""Cost of the fast-path cut (GFP_FAST_MIN_SIN2) for the library named by GOLEMFLAVOR_B200_LIB: K2 log-posterior on 2^22
points (dim-6 OET, the bench workload), the texture and anarchic scans (2^28 samples, nb = 25), the dim-6 sampler step
(4096 walkers, cluster launch), and the share of points / samples whose bin loop took the refinement.
Run by scratch/cut_cost.sh, which alternates the two builds in one call."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np, torch, models
from golemflavor_b200 import _lib, llh, mcmc, scan
from golemflavor_b200.enums import Texture


def events(fn, reps):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


g = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_llh.npz'))
args, asimov, pset = models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OET)
f3 = llh.LnProb(args, asimov, pset)
lib = _lib.load()
n = 1 << 22
th = torch.as_tensor(models.draw_in_ranges(pset, n, np.random.default_rng(25))).cuda()
out = torch.empty(n, dtype=torch.float64, device='cuda')
k2 = min(events(lambda: _lib.check(lib.gf_lnprob(f3.model.ref, _lib.ptr(th), n, f3.ndim, 1, _lib.ptr(out), None, None, None)), 200)
         for _ in range(3))
st = f3.evaluate(th, want_status=True)[2].cpu().numpy()
line = ['%s' % os.path.basename(_lib.LIB_PATH), 'K2 %.4f ms refined %.4f%%' % (k2, 100 * np.mean((st & _lib.ST_REFINED) > 0))]
for mode in ('texture', 'anarchic'):
    fm = scan.scan_model(mode)
    hist = torch.zeros(26 ** 3, dtype=torch.int64, device='cuda')
    t = min(events(lambda: scan.scan_histogram(fm, 1 << 28, nb=25, distributed=False, out=hist, return_tensor=True), 3) for _ in range(2))
    _, _, sst = scan.scan_samples(fm, 1 << 22, seed=26)
    line.append('%s %.2f ms/2^28 (%.3g samples/s) refined %.4f%%' % (mode, t, (1 << 28) / t * 1e3, 100 * np.mean((sst & _lib.ST_REFINED) > 0)))
np.random.seed(25)
p3 = mcmc.flat_seed(pset, 4096)
s = mcmc.DeviceEnsembleSampler(4096, f3.ndim, f3, seed=25, mode=3)
s.run_mcmc(p3, 100, store=False)
torch.cuda.synchronize()
t0 = time.perf_counter()
s.run_mcmc(None, 2000, store=False, return_tensor=True)
torch.cuda.synchronize()
line.append('C3 sampler %.2f us/step' % ((time.perf_counter() - t0) / 2000 * 1e6))
print(' | '.join(line), flush=True)
