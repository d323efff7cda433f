"""Multi-GPU check of the profile source grid run under torchrun (not collected by pytest): every rank computes the sharded
sens.profile_source_grid with the NCCL all-reduce and compares it with the single-rank result it computes itself.
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/dist_profile_source_check.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import torch.distributed as dist
from golemflavor_b200 import sens

local = int(os.environ.get('LOCAL_RANK', '0'))
torch.cuda.set_device(local)
dist.init_process_group('nccl', device_id=torch.device('cuda', local))
src = np.array([(1., 2., 0.), (1., 0., 0.), (0., 1., 0.), (0., 0., 1.), (0.3, 0.5, 0.2)])
kw = dict(dimensions=(3, 6), segments=7, nstarts=32)
sharded, am = sens.profile_source_grid(src, return_argmax=True, **kw)
single, am1 = sens.profile_source_grid(src, return_argmax=True, distributed=False, **kw)
ok = all(np.array_equal(sharded[d], single[d]) and np.array_equal(am[d], am1[d]) for d in single)
if dist.get_rank() == 0:
    print('profile source grid: 5 sources x 2 dims x 7 scales world=%d ok=%s' % (dist.get_world_size(), ok))
flag = torch.tensor([int(ok)], device='cuda')
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag) else 1)
