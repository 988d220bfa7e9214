"""In-process multi-rank check of the peer exchange (threads, one GPU). argv: world stages"""
import os, sys, time, threading
sys.path.insert(0, '/root/repo'); sys.path.insert(0, '/root/repo/tests/golden'); sys.path.insert(0, '/root/repo/tests')
import numpy as np, torch
import workloads
from oracle import mrgp_oracle as O
from cimrgp_b200.distributed import ShardedEngine
from cimrgp_b200.engine import Engine
world = int(sys.argv[1]); warm1 = int(sys.argv[2])
n, res, M = 30000, 6, 30
x, y = workloads.workload1(n); xs = (x - x.mean(0)) / x.std(0); offs = O.uniform_offsets(n, res, 2)
ref = Engine(xs, y, offs, M); ref.sweep(3); ref.synchronize()

class TC(object):
    def __init__(self, world):
        self.world, self.slots, self.barrier = world, [None] * world, threading.Barrier(world)
        self.local = threading.local()
    def all_gather_bytes(self, payload):
        self.slots[self.local.rank] = bytes(payload); self.barrier.wait(); out = list(self.slots); self.barrier.wait(); return out
    def sync(self):
        self.barrier.wait()

if warm1:
    c1 = TC(1); c1.local.rank = 0
    e1 = ShardedEngine(xs, y, offs, M, 0, 1, comm=c1); e1.sweep(2); e1.sweep(1, use_graph=False); e1.synchronize()
    a, b = e1.state(), ref.state(latent=False)
    print('world-1 sharded max rel diff %.2e' % max(float(np.max(np.abs(a[k]-b[k])/(np.abs(b[k])+1e-12*np.abs(b[k]).max()+1e-300))) for k in b), flush=True)
comm = TC(world); engines = [None] * world
def work(rank):
    comm.local.rank = rank
    t0 = time.time()
    try:
        e = ShardedEngine(xs, y, offs, M, rank, world, comm=comm)
        print(rank, 'built %.2fs' % (time.time() - t0), flush=True)
        if os.environ.get('GRAPH','1')=='1':
            e.sweep(2); e.synchronize(); print(rank, 'graph sweeps ok %.2fs' % (time.time() - t0), flush=True)
        else:
            e.sweep(2, use_graph=False); e.synchronize()
        e.sweep(1, use_graph=False); e.synchronize(); print(rank, 'stepwise ok %.2fs' % (time.time() - t0), flush=True)
        engines[rank] = e
    except Exception as ex:
        print(rank, 'FAILED after %.2fs' % (time.time() - t0), ex, flush=True); comm.barrier.abort()
ts = [threading.Thread(target=work, args=(r,)) for r in range(world)]
[t.start() for t in ts]; [t.join() for t in ts]
if all(e is not None for e in engines):
    b = ref.state(latent=False)
    for e in engines:
        a = e.state()
        print('max rel diff %.2e' % max(float(np.max(np.abs(a[k]-b[k])/(np.abs(b[k])+1e-12*np.abs(b[k]).max()+1e-300))) for k in b), flush=True)
os._exit(0)
