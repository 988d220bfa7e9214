"""Tail of the fused ci sweep at config 4 (N = 1e6, 10 layers, M = 30): %globaltimer stamps of one k_ci_sweep<30>, warm
L2 and L2 flushed (the 256 MB write of bench.py), in us from the kernel's first stamp.  Per layer j:
  chain   CTA 0: gather of the region sums of layer j, shared step and omega solve of layer j
  mid1    worker warps: P1-finish of layer j + 1 (earliest start over the warps -> latest end)
  finish  worker warps: S2 / P4 / P5 of layer j
and tail = last exit of a warp of the cluster - exit of CTA 0 (the finish of the finest layers runs after the chain).
Median over the repetitions of every stamp.  Usage: python scratch/sweep_tail.py [reps]"""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
import numpy as np
import torch

import bench

J = 10
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7
m = bench.make_model(1000000, J, 0)
e = m._engine
e.lib.mrgp_timeline_enable(e.handle, 1)
e.sweep(8)
e.synchronize()
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device='cuda')
print(torch.cuda.get_device_name(0), 'ci sweep, N = 1e6, %d layers, M = 30' % J)


def read(flushed):
    if flushed:
        with torch.cuda.stream(e.stream):
            flush.zero_()
    else:
        e.sweep(1)
    torch.cuda.synchronize()
    tags = (C.c_int32 * 256)()
    ms = (C.c_float * 512)()
    n = e.lib.mrgp_timeline_read(e.handle, tags, ms, 256)
    assert n > 0, n
    return np.array(ms[:2 * n], dtype=np.float64).reshape(n, 2) * 1e3      # (slot, begin / end) in us


for flushed in (False, True):
    st = np.median(np.stack([read(flushed) for _ in range(reps)]), axis=0)
    print('\n%s (median of %d sweeps), us' % ('L2 flushed' if flushed else 'warm L2', reps))
    print('%3s  %-22s %-22s %-22s' % ('j', 'chain (CTA 0)', 'mid1 of j+1', 'finish'))
    for j in range(J):
        cells = []
        for k in (3, 1, 0):
            b, en = st[j * 4 + k]
            cells.append('-' if en < 0 or (k == 1 and j == J - 1) else '%6.1f-%6.1f %5.1f' % (b, en, en - b))
        print('%3d  %-22s %-22s %-22s' % (j, cells[0], cells[1], cells[2]))
    cta0, last = st[2][1], st[6][1]
    print('CTA 0 exit %.1f, last warp exit %.1f: tail %.1f us' % (cta0, last, last - cta0))
