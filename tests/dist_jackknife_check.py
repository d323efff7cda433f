"""Multi-GPU check of the grouped evidence grids run under torchrun (not collected by pytest): every rank computes the
sharded scan.scan_evidence_grid / scan_evidence_sources with groups (per-group NCCL all-reduces) and compares lnZ and the
leave-one-group-out lnZ with the single-rank result it computes itself.
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/dist_jackknife_check.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import torch.distributed as dist
from golemflavor_b200 import scan, sens
from golemflavor_b200.enums import Texture


def close(a, b):
    f = np.isfinite(b)
    return bool(np.array_equal(np.isfinite(a), f)) and float(np.max(np.abs(a[f] - b[f]) / np.maximum(1, np.abs(b[f])), initial=0.0)) < 1e-12


local = int(os.environ.get('LOCAL_RANK', '0'))
torch.cuda.set_device(local)
dist.init_process_group('nccl', device_id=torch.device('cuda', local))
fm = sens._grid_model(6, Texture.OET, np.array([1., 2., 0.]), np.array([1., 1., 1.]), 0.02, scan.DEFAULT_BINNING)
scales = sens.scale_grid(6, 30)
src = np.array([(1., 2., 0.), (1., 0., 0.), (0., 1., 0.), (0., 0., 1.), (0.3, 0.5, 0.2)])
ok = True
for R in (2, 16):
    for a, b in zip(scan.scan_evidence_grid(fm, scales, 400_003, seed=26, first_index=7, groups=R),
                    scan.scan_evidence_grid(fm, scales, 400_003, seed=26, first_index=7, distributed=False, groups=R)):
        ok = ok and close(a, b)
    for a, b in zip(scan.scan_evidence_sources(fm, scales, src, (1, 1, 1), 400_003, seed=26, groups=R),
                    scan.scan_evidence_sources(fm, scales, src, (1, 1, 1), 400_003, seed=26, distributed=False, groups=R)):
        ok = ok and close(a, b)
ev, loo = sens.evidence_source_grid(src, dimensions=(3, 6), segments=10, samples=100_001, groups=16)
ok = ok and all(loo[d].shape == (5, 16, 10, 2) for d in loo)
if dist.get_rank() == 0:
    print('grouped grids: 5 sources x 30 scales x 400003 samples, groups 2 and 16, world=%d ok=%s' % (dist.get_world_size(), ok))
flag = torch.tensor([int(ok)], device='cuda')
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag) else 1)
