"""Same work, bit for bit: every state array, the ELBO and the launch counts of a set of sweep paths, written to one
.npz, so that two builds of the library can be compared exactly when a change must not alter what is enqueued.

    python scratch/same_work.py --root <tree whose cimrgp_b200 is imported> --out a.npz
    python scratch/same_work.py --compare a.npz b.npz

Run each build in its own process.  The paths: config 4 (fused ci sweep), the multi-kernel sweep (MRGP_FUSED=0) at
M = 30 and 24, shared noise and shared bias, adaptive intervals, M = 40, fi, the tripped guard of the fused sweep in its
streamed and its small form (MRGP_CHAIN_GUARD), prefetched observations (direct launches), a batched and a mixed group,
the per-phase sweep, and sample sharding over the peer exchange with two in-process ranks."""
import argparse
import ctypes as C
import os
import sys
import threading

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(root, out):
    for p in (os.path.join(root, 'tests', 'golden'), os.path.join(root, 'tests'), root):
        sys.path.insert(0, p)
    import workloads
    from oracle import mrgp_oracle as O
    import cimrgp_b200
    from cimrgp_b200 import _lib
    from cimrgp_b200.engine import Engine
    from cimrgp_b200.distributed import ShardedEngine
    print('package', cimrgp_b200.__file__, flush=True)
    lib = _lib.load()
    res = {}

    def normed(x):
        return (x - x.mean(0)) / x.std(0)

    def make(n, layers, m, env=None, seed=10, **kw):
        x, y = workloads.workload1(n, seed=seed)
        saved = {k: os.environ.get(k) for k in (env or {})}
        os.environ.update(env or {})
        try:
            return Engine(normed(x), y, O.uniform_offsets(n, layers - 1, 2), m, **kw)
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v

    def record(name, e, elbo=True):
        e.synchronize()
        for k, v in e.state(latent=False).items():
            res['%s/%s' % (name, k)] = v
        if elbo and e.mode == 'ci':   # the library defines the bound in ci mode only
            res[name + '/elbo'] = e.elbo()
        res[name + '/launches'] = np.array([e.launch_count()])
        print(name, 'launches', e.launch_count(), flush=True)

    def swept(name, e, steps=(1, 2)):
        """Launch counts after the first sweep (builds and statistics) and after the replays."""
        counts = []
        for k in steps:
            e.sweep(k)
            e.synchronize()
            counts.append(e.launch_count())
        res[name + '/launch_steps'] = np.array(counts)
        record(name, e)

    swept('config4', make(1000000, 10, 30))
    swept('multi_m30', make(20000, 7, 30, env={'MRGP_FUSED': '0'}))
    swept('multi_m24', make(20000, 7, 24, env={'MRGP_FUSED': '0'}))
    swept('shared_noise', make(20000, 6, 30, noise_region_specific=False))
    swept('shared_bias', make(20000, 6, 30, bias_region_specific=False))
    e = make(20000, 6, 30)
    e.set_adaptive_intervals(-1, use_prior=True)
    swept('adaptive', e)
    swept('m40', make(20000, 7, 40))
    swept('fi', make(20000, 7, 30, mode='fi'))
    swept('guard_streamed', make(150000, 3, 12, env={'MRGP_CHAIN_GUARD': '0.9'}), steps=(1, 3))
    swept('guard_small', make(6000, 3, 12, env={'MRGP_CHAIN_GUARD': '0.9'}), steps=(1, 3))

    # prefetched observations: the fused sweep launched on the stream, not through a graph
    e = make(60000, 6, 30)
    e.sweep(2)
    rng = np.random.default_rng(5)
    _, y = workloads.workload1(60000)
    ys = [y + 0.05 * rng.standard_normal(y.shape) for _ in range(3)]
    e.prefetch_observations(ys[0])
    for k in range(3):
        e.refresh_statistics()
        if k + 1 < 3:
            e.prefetch_observations(ys[k + 1])
        e.sweep(2)
    record('prefetched', e)

    def group(name, engines, k=3):
        arr = (C.c_void_p * len(engines))(*[x.handle for x in engines])
        g = C.c_void_p()
        assert lib.mrgp_group_create(arr, len(engines), None, C.byref(g)) == 0, lib.mrgp_last_error(None)
        try:
            for _ in range(2):
                assert lib.mrgp_group_sweep(g, k) == 0
                assert lib.mrgp_group_synchronize(g) == 0
            res[name + '/group_launches'] = np.array([lib.mrgp_group_launch_count(g)])
            print(name, 'group launches', lib.mrgp_group_launch_count(g), flush=True)
        finally:
            lib.mrgp_group_destroy(g)
        for i, x in enumerate(engines):
            record('%s/%d' % (name, i), x)

    def series(n, layers, m, seed, **kw):
        return make(n, layers, m, seed=seed, n_ctas=max(1, min(64, n // 1024)), **kw)

    group('group_batched', [series(n, layers, m, 30 + i) for i, (n, layers, m) in
                            enumerate([(1500, 4, 17), (5000, 5, 20), (32768, 6, 24), (9000, 6, 17)])])
    group('group_mixed', [series(3000, 5, 20, 50), series(2500, 5, 33, 51), series(2500, 5, 20, 52, mode='fi'),
                          series(2500, 5, 20, 53, noise_region_specific=False)])

    for mode in ('ci', 'fi'):
        e = make(20000, 6, 30, mode=mode)
        for _ in range(3):
            e.sweep_stepwise()
        record('stepwise_' + mode, e)

    # two ranks as threads of this process, each with its own handle on the one device
    class Comm(object):
        def __init__(self, world):
            self.world, self.slots, self.barrier = world, [None] * world, threading.Barrier(world)
            self.local = threading.local()

        def all_gather_bytes(self, payload):
            self.slots[self.local.rank] = bytes(payload)
            self.barrier.wait()
            got = list(self.slots)
            self.barrier.wait()
            return got

        def sync(self):
            self.barrier.wait()

    n = 30000
    x, y = workloads.workload1(n)
    offs = O.uniform_offsets(n, 5, 2)
    for mode in ('ci', 'fi'):
        comm, engines, errors = Comm(2), [None, None], []

        def work(rank):
            comm.local.rank = rank
            try:
                e = ShardedEngine(normed(x), y, offs, 30, rank, 2, comm=comm, mode=mode)
                # phase by phase, as in test_sample_sharding_matches_single_handle: with both ranks in one process on
                # one device the captured sweep's exchanges time out; the captured form is checked between processes
                e.sweep(3, use_graph=False)
                e.synchronize()
                engines[rank] = e
            except Exception as ex:
                errors.append(ex)
                comm.barrier.abort()

        threads = [threading.Thread(target=work, args=(r,)) for r in range(2)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        assert not errors, errors
        for r, e in enumerate(engines):
            record('sharded_%s/%d' % (mode, r), e, elbo=False)
    np.savez(out, **res)
    print('wrote', out, len(res), 'arrays', flush=True)


def compare(a, b):
    A, B = np.load(a), np.load(b)
    keys = sorted(set(A.files) | set(B.files))
    bad = [k for k in keys if k not in A.files or k not in B.files or A[k].shape != B[k].shape
           or not np.array_equal(A[k], B[k], equal_nan=True)]
    for k in bad[:40]:
        print('DIFFERS', k)
    print('%d arrays, %d differ' % (len(keys), len(bad)))
    return 1 if bad else 0


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--root', default=HERE)
    ap.add_argument('--out')
    ap.add_argument('--compare', nargs=2)
    args = ap.parse_args()
    if args.compare:
        sys.exit(compare(*args.compare))
    run(os.path.abspath(args.root), args.out)
    os._exit(0)
