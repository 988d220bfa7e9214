"""Worker of test_parity_gpu.py::test_peer_exchange_between_processes (launched with torch.distributed.run).
Every rank is its own process with its own CUDA context; all ranks use cuda:0, so the arenas are mapped through
CUDA IPC exactly as between GPUs and the ranks time-slice the device.  gloo carries the 128-byte arena
descriptions.  Prints one line 'rank R ok <max rel diff>' per rank."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests', 'golden'), os.path.join(ROOT, 'tests')):
    sys.path.insert(0, p)

import numpy as np
import torch
import torch.distributed as dist

import workloads
from oracle import mrgp_oracle as O
from cimrgp_b200.distributed import ShardedEngine
from cimrgp_b200.engine import Engine
from parity import compare

rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
mode = sys.argv[1]
torch.cuda.set_device(0)
dist.init_process_group('gloo')
n, res, M = 30000, 6, 30
x, y = workloads.workload1(n)
xs = (x - x.mean(0)) / x.std(0)
offsets = O.uniform_offsets(n, res, 2)
e = ShardedEngine(xs, y, offsets, M, rank, world, mode=mode, device=0)
e.sweep(1, use_graph=False)          # phase by phase through mrgp_exchange
e.sweep(2)                           # one captured CUDA graph per sweep, exchanges inside
e.synchronize()
ref = Engine(xs, y, offsets, M, mode=mode, device=0)
ref.sweep(3)
ref.synchronize()
a, b = e.state(), ref.state(latent=False)
try:
    compare(a, b, rtol=1e-9)       # the comparison rule of all parity tests (tests/parity.py)
    worst = 0.0
except AssertionError as ex:
    print('rank %d: %s' % (rank, str(ex)[:1500]), flush=True)
    worst = 1.0
# replicated state must be bit-identical on every rank: compare a digest
digest = float(sum(np.sum(a[k]) for k in sorted(a)))
out = [None] * world
dist.all_gather_object(out, digest)
same = all(v == out[0] for v in out)
print('rank %d %s %.3e identical=%s' % (rank, 'ok' if worst < 1e-9 and same else 'MISMATCH', worst, same), flush=True)
dist.barrier()
sys.stdout.flush()
os._exit(0)
