"""Multi-process check of the sharded path against the unsharded engine (run under torchrun).
env: MRGP_ONE_GPU=1 -> every rank uses cuda:0 and gloo (separate processes time-slice one device)."""
import os, sys, time
sys.path.insert(0,'/root/repo'); sys.path.insert(0,'/root/repo/tests/golden'); sys.path.insert(0,'/root/repo/tests')
import numpy as np, torch, torch.distributed as dist
rank=int(os.environ['RANK']); world=int(os.environ['WORLD_SIZE']); lr=int(os.environ['LOCAL_RANK'])
one=os.environ.get('MRGP_ONE_GPU','0')=='1'
if one: lr=0
torch.cuda.set_device(lr)
if one: dist.init_process_group('gloo')
else: dist.init_process_group('nccl', device_id=torch.device('cuda',lr))
import workloads
from oracle import mrgp_oracle as O
from cimrgp_b200.distributed import ShardedEngine
from cimrgp_b200.engine import Engine
n,res,M=int(os.environ.get('MRGP_N','200000')),7,30
x,y=workloads.workload1(n); xs=(x-x.mean(0))/x.std(0); offs=O.uniform_offsets(n,res,2)
t=time.time()
e=ShardedEngine(xs,y,offs,M,rank,world,device=lr)
print('rank',rank,'built %.2fs'%(time.time()-t),flush=True)
t=time.time(); e.sweep(2,use_graph=False); e.synchronize(); print('rank',rank,'2 stepwise sweeps ok %.2fs'%(time.time()-t),flush=True)
t=time.time(); e.sweep(3); e.synchronize(); print('rank',rank,'3 graph sweeps ok %.2fs'%(time.time()-t),flush=True)
ref=Engine(xs,y,offs,M,device=lr); ref.sweep(5); ref.synchronize()
a,b=e.state(),ref.state(latent=False)
worst=max(float(np.max(np.abs(a[k]-b[k])/(np.abs(b[k])+1e-12*np.abs(b[k]).max()+1e-300))) for k in b)
print('rank',rank,'max rel diff vs unsharded %.2e'%worst,flush=True)
if not one:
    ev0,ev1=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
    e.sweep(5); e.synchronize(); dist.barrier()
    ev0.record(e.stream); e.sweep(20); ev1.record(e.stream); e.synchronize()
    print('rank',rank,'graph sweep %.1f us'%(ev0.elapsed_time(ev1)*1000/20),flush=True)
dist.barrier()
sys.stdout.flush()
os._exit(0)
