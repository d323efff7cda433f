"""Multi-GPU check of the source-grid evidence run under torchrun (not collected by pytest): every rank computes the
sharded scan.scan_evidence_sources with the NCCL all-reduces and compares it with the single-rank result it computes itself.
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/dist_source_check.py
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

local = int(os.environ.get('LOCAL_RANK', '0'))
torch.cuda.set_device(local)
dist.init_process_group('nccl', device_id=torch.device('cuda', local))
fm = sens._grid_model(6, Texture.OET, np.array([1., 2., 0.]), np.array([1., 1., 1.]), 0.02, scan.DEFAULT_BINNING)
scales = sens.scale_grid(6, 30)
src = np.array([(1., 2., 0.), (1., 0., 0.), (0., 1., 0.), (0., 0., 1.), (0.3, 0.5, 0.2)])
sharded = scan.scan_evidence_sources(fm, scales, src, (1, 1, 1), 400_003, seed=26)
single = scan.scan_evidence_sources(fm, scales, src, (1, 1, 1), 400_003, seed=26, distributed=False)
f = np.isfinite(single)
ok = bool(np.array_equal(np.isfinite(sharded), f)) and float(np.max(np.abs(sharded[f] - single[f]) / np.maximum(1, np.abs(single[f])))) < 1e-12
ev = sens.evidence_source_grid(src, dimensions=(3, 6), segments=10, samples=100_001)
ok = ok and all(np.isfinite(ev[d][:, :, 0]).all() for d in ev)
if dist.get_rank() == 0:
    print('source grid: 5 sources x 30 scales x 400003 samples world=%d ok=%s' % (dist.get_world_size(), ok))
flag = torch.tensor([int(ok)], device='cuda')
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag) else 1)
