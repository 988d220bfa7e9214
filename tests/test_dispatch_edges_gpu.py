"""The size-dispatched paths of the library on both sides of every boundary, against the NumPy oracle.

The library picks a compiled instantiation, a work split or a whole code path by size: the solver size of the fused
sweep and the width of the streaming kernels by n_basis, the worker tier of the fused sweep by the regions per worker
warp and the cluster size, the form of the layer-0 statistics by the longest layer-0 region and the number of regions,
the tile pipeline of the streaming kernels by the samples of a CTA, batched or graph form of a group by its members,
one thread or one warp per matrix in the batched Cholesky.  Every case here states which side it is on through
something the host observes (launch counts, the plan hooks, the offsets, a group's launch count) and compares every
state array, including the per-sample latent functions, with the oracle at the rule of parity.compare."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import mrgp_oracle as O
from parity import compare
import workloads
from mrgp_helpers import Oracle, dropin, engine, ragged

pytestmark = pytest.mark.gpu

# ---- restated dispatch rules (the source of each is named; the tests assert the observable side of each) ------------
def chain_solver_size(m):
    """mrgp_chain.h, chain_solver_size: the compiled omega solver of the fused sweep (0: multi-kernel sweep)."""
    return 30 if m == 30 else 8 if m <= 8 else 16 if m <= 16 else 24 if m <= 24 else 32 if m <= 32 else 0


def padded_basis(m):
    """cimrgp.cu, padded_basis: the instantiation of the streaming kernels."""
    return 8 if m <= 8 else 20 if m <= 20 else 30 if m <= 30 else 40 if m <= 40 else 48


K_YSTATS_SMALL_MAX_REGION = 32768      # mrgp_chain.h, kYstatsSmallMaxRegion
K_YSTATS_FUSED_TAIL_MAX_REGIONS = 64   # cimrgp.cu, do_ystats: the statistics pass sums its own partials up to here
K_MAX_LAYERS = 24                      # cimrgp.cu kMaxLayers, mrgp_chain.h kChainMaxLayers
K_TILE = 1024                          # mrgp_kernels.cuh, kTile


def worker_warps(cluster):
    """chain.cu, k_ci_sweep: 7 worker warps for a cluster of one CTA (warp 0 solves), 8 per worker CTA otherwise."""
    return 7 if cluster == 1 else 8 * (cluster - 1)


def worker_tiers(r, n_w):
    """chain.cu, layer_mid1 / layer_finish for a layer above the first: regions per warp of each step (8 and 4 are
    the strided loops of the last tier)."""
    mid1 = 1 if r <= n_w else 2 if r <= 2 * n_w else 4 if r <= 4 * n_w else 8
    finish = 1 if r <= n_w else 2 if r <= 2 * n_w else 4
    return mid1, finish


# ---- helpers ----------------------------------------------------------------------------------------------------------
def sweep(eng, k):
    eng.sweep(k)
    eng.synchronize()


def launches_per_sweep(eng):
    """Launches of one sweep once the sweep is captured (the first sweep also builds invariants and statistics)."""
    a = eng.launch_count()
    sweep(eng, 2)
    return (eng.launch_count() - a) / 2


def fused_launches(x, y, offsets):
    """Per-sweep launch count of the fused sweep on this data: an M = 30 ci model, which always takes it."""
    e = engine(x, y, offsets, 30)
    sweep(e, 1)
    return launches_per_sweep(e)


def per_cta_samples(eng, layer=0):
    lib = eng.lib
    n_ctas, n_seg, n_runs = C.c_int32(), C.c_int32(), C.c_int32()
    assert lib.mrgp_plan_info(eng.handle, layer, C.byref(n_ctas), C.byref(n_seg), C.byref(n_runs)) == 0
    seg = np.zeros((n_seg.value, 6), dtype=np.int64)
    assert lib.mrgp_plan_segments(eng.handle, layer, seg.ctypes.data_as(C.POINTER(C.c_int64))) == 0
    return np.bincount(seg[:, 5], weights=seg[:, 1] - seg[:, 0], minlength=n_ctas.value).astype(np.int64)


def run_against_oracle(eng, ora, elbo=True, predict=True):
    """Sweeps 1 and 3 against the oracle; the engine must not have swept yet."""
    sweep(eng, 1)
    ora.sweep(1)
    ora.check(eng)
    sweep(eng, 2)
    ora.sweep(2)
    ora.check(eng)
    if elbo and ora.ora.mode == 'ci':
        ora.check_elbo(eng)
    if predict:
        ora.check_predictions(eng)


# ---------------------------------------------------------------------------------------------------------------------
# 1. basis sizes: solver sizes 8 / 16 / 24 / 30 / 32 of the fused sweep, widths 8 / 20 / 30 / 40 / 48 of the streaming
#    kernels, fused (M <= 32) or multi-kernel sweep (M > 32)
# ---------------------------------------------------------------------------------------------------------------------
BASIS_SIZES = [9, 16, 17, 21, 24, 31, 32, 33, 41, 48]
for _s in (16, 24, 32):                              # each solver size exact (unpadded branch) and padded
    assert _s in BASIS_SIZES and any(chain_solver_size(m) == _s and m != _s for m in BASIS_SIZES)
for _w, _prev in ((20, 8), (30, 20), (40, 30), (48, 40)):  # each streaming width at its first padded M
    assert _prev + 1 in BASIS_SIZES and padded_basis(_prev + 1) == _w
assert 48 in BASIS_SIZES and 33 in BASIS_SIZES and chain_solver_size(33) == 0


def _basis_case(m, fi, n, resolution):
    x, y = workloads.workload1(n)
    model = dropin(x, y, m, resolution, fi)
    eng = model._engine
    ora = Oracle(x, y, m, O.uniform_offsets(n, resolution, 2), mode='fi' if fi else 'ci')
    run_against_oracle(eng, ora)
    if not fi:
        fused = chain_solver_size(m) != 0
        got = launches_per_sweep(eng)
        want = fused_launches(x, y, O.uniform_offsets(n, resolution, 2))
        assert (got == want) == fused, (m, got, want)


@pytest.mark.parametrize('fi', [False, True])
@pytest.mark.parametrize('m', BASIS_SIZES)
def test_basis_size_edges_against_oracle(m, fi):
    _basis_case(m, fi, 3000, 4)


@pytest.mark.parametrize('m', [32, 48])
def test_basis_size_edges_at_mid_size(m):
    """8 layers, N = 40000: M = 32 fills every lane of the fused sweep, M = 48 is the widest streaming instantiation."""
    _basis_case(m, False, 40000, 7)


@pytest.mark.parametrize('m', [24, 32])
def test_multi_kernel_sweep_with_the_block_omega_solver(m, monkeypatch):
    """MRGP_FUSED=0 at M = 24 and 32: the multi-kernel sweep takes the one-CTA omega solve (k_scale), because the
    single-warp solver (k_scale_warp) is instantiated only for M = 8, 20 and 30."""
    n, resolution = 3000, 4
    x, y = workloads.workload1(n)
    offsets = O.uniform_offsets(n, resolution, 2)
    want = fused_launches(x, y, offsets)
    monkeypatch.setenv('MRGP_FUSED', '0')
    eng = engine(x, y, offsets, m)
    run_against_oracle(eng, Oracle(x, y, m, offsets))
    assert launches_per_sweep(eng) > want


# ---------------------------------------------------------------------------------------------------------------------
# 2. worker tiers and cluster sizes of the fused sweep
# ---------------------------------------------------------------------------------------------------------------------
CLUSTERS = [1, 2, 4, 8, 16]


def tier_counts(cluster):
    """Regions per layer, non-decreasing from one: n_w - 1, n_w, n_w + 1, 2 n_w, 2 n_w + 1, 4 n_w + 1, 8 n_w + 1."""
    w = worker_warps(cluster)
    return [1, w - 1, w, w + 1, 2 * w, 2 * w + 1, 4 * w + 1, 8 * w + 1]


for _c in CLUSTERS:   # every tier of both worker steps, and a partial last pass of each strided loop, for every cluster size
    _w = worker_warps(_c)
    _t = [worker_tiers(r, _w) for r in tier_counts(_c)[1:]]
    assert {t[0] for t in _t} == {1, 2, 4, 8} and {t[1] for t in _t} == {1, 2, 4}, _c
    assert any(r % (8 * _w) not in (0, r) for r in tier_counts(_c)) and any(r % (4 * _w) not in (0, r) for r in tier_counts(_c))
    assert any(r < _w for r in tier_counts(_c)[1:])


def _cluster_run(monkeypatch, x, y, offsets, cluster):
    monkeypatch.setenv('MRGP_CHAIN_CLUSTER', str(cluster))
    eng = engine(x, y, offsets, 30)
    monkeypatch.delenv('MRGP_CHAIN_CLUSTER')
    return eng


def omega_converged(eng):
    """The omega solve of every layer reached its tolerance in the last sweep (MultiResolutionGaussianProcess.
    omega_solve_report: 2040 evaluations mean the fused sweep's budget is used up)."""
    from cimrgp_b200 import _lib
    return bool(np.all(eng.get(-1, _lib.F_OMEGA_ITERS, (eng.J,)) < 2040))


@pytest.mark.parametrize('cluster', CLUSTERS)
def test_worker_tiers_of_every_cluster_size(cluster, monkeypatch):
    """One ragged model per cluster size whose layers reach every worker tier, against the oracle, and the same model
    under every other cluster size.  A region's sums are formed by one warp, but which warp a region goes to and the
    order in which warps and CTAs add their partial sums depend on the number of workers: the cluster sizes agree to
    roundoff (1e-12), not bit for bit.

    Every sweep runs every tier.  After the first sweep the models with hundreds of small regions per layer have tables
    log omega_hat that span 1e3 - 1e4; the fused sweep's omega solve then uses up its budget (48 accelerated and 2000
    plain Sinkhorn evaluations) and leaves the last iterate, 1e-5 - 1e-3 from the exact scaling; the drop-in class
    hands such a model to the multi-kernel sweep.  Sweeps 2 and 3 are compared (with the oracle and across cluster sizes)
    where the solve converged in every layer of both sweeps, the first sweep always."""
    n = 15000 if cluster == 16 else 8000
    x, y = workloads.workload1(n, seed=20 + cluster)
    offsets = ragged(n, tier_counts(cluster), seed=cluster)
    if cluster == 16:
        assert np.min(np.diff(offsets[-1])) < 32
    ora = Oracle(x, y, 30, offsets)
    engines = {c: _cluster_run(monkeypatch, x, y, offsets, c) for c in CLUSTERS}
    eng = engines[cluster]
    sweep(eng, 1)
    ora.sweep(1)
    ora.check(eng)
    want = eng.state()
    for c, e in engines.items():
        if c != cluster:
            sweep(e, 1)
            compare(e.state(), want, rtol=1e-12)
    converged = True
    for _ in range(2):
        sweep(eng, 1)
        converged = converged and omega_converged(eng)
    if not converged:
        return
    ora.sweep(2)
    ora.check(eng)
    ora.check_elbo(eng)
    want = eng.state()
    for c, e in engines.items():
        if c != cluster:
            sweep(e, 2)
            compare(e.state(), want, rtol=1e-12)


def test_fewer_regions_than_worker_warps_at_the_largest_cluster(monkeypatch):
    n = 4000
    x, y = workloads.workload1(n, seed=3)
    offsets = ragged(n, [1, 3, 10, 40, 100], seed=4)
    assert all(len(o) - 1 < worker_warps(16) for o in offsets)
    eng = _cluster_run(monkeypatch, x, y, offsets, 16)
    run_against_oracle(eng, Oracle(x, y, 30, offsets))


# ---------------------------------------------------------------------------------------------------------------------
# 3. layer-0 statistics: one CTA per region (every region <= 32768 samples), the streaming pass with its own tail sum
#    (R0 <= 64), the streaming pass and k_reduce_ystats (R0 > 64)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n', [32768, 32769])
@pytest.mark.parametrize('m', [8, 30])
def test_layer0_statistics_at_the_region_length_limit(m, n):
    x, y = workloads.workload1(n, seed=7)
    offsets = [np.array([0, n], dtype=np.int64)] + ragged(n, [3, 9, 30], seed=8)
    assert (np.max(np.diff(offsets[0])) <= K_YSTATS_SMALL_MAX_REGION) == (n == 32768)
    eng = engine(x, y, offsets, m)
    run_against_oracle(eng, Oracle(x, y, m, offsets))


@pytest.mark.parametrize('n_ctas', [1, 3])
def test_streamed_layer0_statistics_on_few_ctas(n_ctas):
    n = 32769
    x, y = workloads.workload1(n, seed=7)
    offsets = [np.array([0, n], dtype=np.int64)] + ragged(n, [3, 9, 30], seed=8)
    eng = engine(x, y, offsets, 30, n_ctas=n_ctas)
    assert len(per_cta_samples(eng)) == n_ctas
    run_against_oracle(eng, Oracle(x, y, 30, offsets), predict=False)


@pytest.mark.parametrize('r0', [64, 65])
def test_layer0_statistics_of_many_regions_one_of_them_long(r0):
    short = 150
    n = (r0 - 1) * short + K_YSTATS_SMALL_MAX_REGION + 500
    x, y = workloads.workload1(n, seed=9)
    layer0 = np.r_[np.arange(r0) * short, n].astype(np.int64)          # the last region is the long one
    offsets = [layer0] + ragged(n, [90, 200], seed=10)
    assert len(offsets[0]) - 1 == r0 and np.max(np.diff(layer0)) > K_YSTATS_SMALL_MAX_REGION
    assert (r0 > K_YSTATS_FUSED_TAIL_MAX_REGIONS) == (r0 == 65)
    eng = engine(x, y, offsets, 30)
    run_against_oracle(eng, Oracle(x, y, 30, offsets), predict=False)


# ---------------------------------------------------------------------------------------------------------------------
# 4. full tiles of the streaming kernels: per-CTA sample ranges k * 1024 + r
# ---------------------------------------------------------------------------------------------------------------------
TILE_REMAINDERS = [0, 1, 255, 256, 257, 1023]


def _cta_split(n, n_ctas):
    """mrgp_create's split of the samples (cimrgp.cu): used to choose N only; the tests read the plan itself."""
    want = min(n_ctas, max(1, -(-n // 1024)))
    q = -(-n // want)
    q = -(-q // 32) * 32
    return [min(q, n - c * q) for c in range(-(-n // q))]


def _n_for(n_ctas, r):
    base = 2 * K_TILE * n_ctas
    for n in range(base, base + 4 * K_TILE * n_ctas):
        s = _cta_split(n, n_ctas)
        if len(s) == n_ctas and s[-1] % K_TILE == r and min(s) >= K_TILE:
            return n
    raise AssertionError((n_ctas, r))


TILE_CASES = []
for _mode in ('fi', 'stream_all'):
    for _m in (30, 48):
        for _c in (1, 2, 3):
            TILE_CASES.append((_mode, _m, _c, TILE_REMAINDERS[len(TILE_CASES) % len(TILE_REMAINDERS)]))
for _mode in ('fi', 'stream_all'):
    assert {c[3] for c in TILE_CASES if c[0] == _mode} == set(TILE_REMAINDERS)


def _tile_offsets(n, seed):
    """Ragged regions (boundaries inside tiles) and one region of 20 samples, shorter than a warp."""
    offsets = [np.array([0, n], dtype=np.int64)] + ragged(n, [3, 7, 15], seed=seed, min_len=40)
    last = offsets[-1]
    offsets[-1] = np.unique(np.r_[last, last[5] + 20]).astype(np.int64)
    return offsets


@pytest.mark.parametrize('mode,m,n_ctas,r', TILE_CASES)
def test_full_tiles_of_the_streaming_kernels(mode, m, n_ctas, r, monkeypatch):
    n = _n_for(n_ctas, r)
    x, y = workloads.workload1(n, seed=n_ctas)
    offsets = _tile_offsets(n, seed=r)
    assert np.min(np.diff(offsets[-1])) == 20 and np.any(offsets[1][1:-1] % 32 != 0)
    if mode == 'stream_all':
        want = fused_launches(x, y, offsets)
        monkeypatch.setenv('MRGP_STREAM_ALL', '1')
    eng = engine(x, y, offsets, m, mode='fi' if mode == 'fi' else 'ci', n_ctas=n_ctas)
    per_cta = per_cta_samples(eng)
    assert len(per_cta) == n_ctas and np.all(per_cta >= K_TILE) and per_cta[-1] % K_TILE == r, per_cta
    run_against_oracle(eng, Oracle(x, y, m, offsets, mode='fi' if mode == 'fi' else 'ci'))
    if mode == 'stream_all':
        assert launches_per_sweep(eng) > want


# ---------------------------------------------------------------------------------------------------------------------
# 5. groups (mrgp_group_*, as cimrgp_b200/batch.py drives them)
# ---------------------------------------------------------------------------------------------------------------------
class Group(object):
    def __init__(self, engines):
        from cimrgp_b200 import _lib
        self.lib, self.engines = _lib.load(), engines
        arr = (C.c_void_p * len(engines))(*[e.handle for e in engines])
        self.g = C.c_void_p()
        rc = self.lib.mrgp_group_create(arr, len(engines), None, C.byref(self.g))
        assert rc == 0, self.lib.mrgp_last_error(None)

    def sweep(self, k):
        assert self.lib.mrgp_group_sweep(self.g, k) == 0
        assert self.lib.mrgp_group_synchronize(self.g) == 0

    def launches(self):
        return int(self.lib.mrgp_group_launch_count(self.g))

    def form(self, k=2):
        """'batched' (one fused launch plus the layer-0 fallback per iteration, nothing on the members' counts) or
        'graph' (the members' own sweeps); sweeps k times."""
        g0, m0 = self.launches(), [e.launch_count() for e in self.engines]
        self.sweep(k)
        dg, dm = self.launches() - g0, [e.launch_count() - a for e, a in zip(self.engines, m0)]
        if dg == 2 * k and not any(dm):
            return 'batched'
        assert all(d > 0 for d in dm) and dg == sum(dm), (dg, dm)
        return 'graph'

    def close(self):
        self.lib.mrgp_group_destroy(self.g)


def _series_engine(x, y, offsets, m, mode='ci', **kw):
    return engine(x, y, offsets, m, mode=mode, n_ctas=max(1, min(64, x.shape[0] // 1024)), **kw)


def _assert_same(a, b, what):
    sa, sb = a.state(), b.state()
    for k in sb:
        assert np.array_equal(sa[k], sb[k]), (what, k)


# N, resolution (J = resolution + 1), M: one solver size (24), different shapes
GROUP_SHAPES = [(1500, 3, 17), (5000, 4, 20), (32768, 5, 24), (9000, 5, 17)]


def test_batched_group_of_members_of_different_shapes():
    members, twins, data = [], [], []
    for i, (n, res, m) in enumerate(GROUP_SHAPES):
        x, y = workloads.workload1(n, seed=30 + i)
        offsets = O.uniform_offsets(n, res, 2)
        data.append((x, y, offsets, m))
        members.append(_series_engine(x, y, offsets, m))
        twins.append(_series_engine(x, y, offsets, m))
    assert {chain_solver_size(d[3]) for d in data} == {24}
    g = Group(members)
    try:
        g.sweep(1)
        assert g.form(2) == 'batched'
        for t in twins:
            sweep(t, 3)
        for i, (mem, t) in enumerate(zip(members, twins)):
            _assert_same(mem, t, i)
        for i in range(3):             # one member of each (N, J, M)
            x, y, offsets, m = data[i]
            ora = Oracle(x, y, m, offsets)
            ora.sweep(3)
            ora.check(members[i])
            ora.check_elbo(members[i])
    finally:
        g.close()


def test_series_batch_of_different_lengths():
    from cimrgp_b200 import IndexSetUniform, LaplacianEigenpairs, MaternKernel, SeriesBatch
    from cimrgp_b200.MRGP import MultiResolutionGaussianProcess
    sizes, res, m = [1500, 2048, 3001, 5000, 777], 4, 30
    xs, ys = zip(*[workloads.workload1(n, seed=40 + i) for i, n in enumerate(sizes)])
    batch = SeriesBatch(list(xs), list(ys), m, res, LaplacianEigenpairs(), MaternKernel(nu=1, l=1, sf=1), n_streams=3)
    batch.fit(3)
    assert len(batch.groups) == 1 and batch.launch_count() == 1 + 2 * 3     # batched: statistics once, then 2 per sweep
    for s, n in enumerate(sizes):
        one = MultiResolutionGaussianProcess([xs[s], ys[s]], m, IndexSetUniform(n, res, 2), LaplacianEigenpairs(),
                                             MaternKernel(nu=1, l=1, sf=1), n_ctas=max(1, min(64, n // 1024)))
        one.fit(3, None)
        _assert_same(batch[s]._engine, one._engine, s)
    x, y = xs[-1], ys[-1]
    ora = Oracle(x, y, m, O.uniform_offsets(sizes[-1], res, 2))
    ora.sweep(3)
    ora.check(batch[len(sizes) - 1]._engine)


@pytest.mark.parametrize('other', ['m33', 'fi', 'shared_noise'])
def test_mixed_group_takes_the_graph_form(other):
    n, res = 3000, 4
    x, y = workloads.workload1(n, seed=50)
    x2, y2 = workloads.workload1(2500, seed=51)
    off, off2 = O.uniform_offsets(n, res, 2), O.uniform_offsets(2500, res, 2)
    kw = dict(m33=dict(m=33), fi=dict(m=20, mode='fi'), shared_noise=dict(m=20, noise_region_specific=False))[other]
    make = lambda: [_series_engine(x, y, off, 20), _series_engine(x2, y2, off2, **kw)]
    members, twins = make(), make()
    g = Group(members)
    try:
        g.sweep(1)
        assert g.form(2) == 'graph'
        for i, (mem, t) in enumerate(zip(members, twins)):
            sweep(t, 3)
            _assert_same(mem, t, i)
    finally:
        g.close()


def test_guard_trips_in_one_member_of_a_batched_group(monkeypatch):
    from cimrgp_b200 import _lib
    data = [workloads.workload1(n, seed=60 + i) for i, n in enumerate((2000, 3000, 2500))]
    offs = [O.uniform_offsets(x.shape[0], 4, 2) for x, _ in data]

    def make():
        out = []
        for i, ((x, y), off) in enumerate(zip(data, offs)):
            if i == 1:
                monkeypatch.setenv('MRGP_CHAIN_GUARD', '0.9')
            out.append(_series_engine(x, y, off, 12))
            monkeypatch.delenv('MRGP_CHAIN_GUARD', raising=False)
        return out

    members, twins = make(), make()
    g = Group(members)
    try:
        g.sweep(1)
        assert g.form(2) == 'batched'
        for i, (mem, t) in enumerate(zip(members, twins)):
            sweep(t, 3)
            _assert_same(mem, t, i)
            guard = mem.get(-1, _lib.F_FUSED_GUARD, (2,))
            assert guard[1] == (1.0 if i == 1 else 0.0), (i, guard)
        (x, y), off = data[1], offs[1]
        ora = Oracle(x, y, 12, off)
        ora.sweep(3)
        ora.check(members[1])
    finally:
        g.close()


def test_new_observations_of_one_member_of_a_batched_group():
    data = [workloads.workload1(n, seed=70 + i) for i, n in enumerate((2000, 3000, 2500))]
    offs = [O.uniform_offsets(x.shape[0], 4, 2) for x, _ in data]
    make = lambda: [_series_engine(x, y, off, 30) for (x, y), off in zip(data, offs)]
    members, twins = make(), make()
    y_new = data[1][1] + 0.05 * np.random.RandomState(1).standard_normal(data[1][1].shape)
    g = Group(members)
    try:
        g.sweep(2)
        members[1].set_observations(y_new)
        g0 = g.launches()
        g.sweep(2)
        assert g.launches() - g0 == 1 + 2 * 2       # the statistics of layer 0 again, then two batched sweeps
        for i, t in enumerate(twins):
            sweep(t, 2)
            if i == 1:
                t.set_observations(y_new)
            sweep(t, 2)
            _assert_same(members[i], t, i)
    finally:
        g.close()


# ---------------------------------------------------------------------------------------------------------------------
# 6. depth: the largest number of layers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('fi', [False, True])
def test_deepest_model_against_oracle(fi):
    n = 6000
    x, y = workloads.workload1(n, seed=80)
    # (no second single-region layer: in fi mode its bias would be the mean of residuals that cancel, pure roundoff)
    offsets = [np.array([0, n], dtype=np.int64)] + ragged(n, [2 + j // 2 for j in range(K_MAX_LAYERS - 1)], seed=81)
    assert len(offsets) == K_MAX_LAYERS
    eng = engine(x, y, offsets, 30, mode='fi' if fi else 'ci')
    run_against_oracle(eng, Oracle(x, y, 30, offsets, mode='fi' if fi else 'ci'))
    if not fi:
        assert launches_per_sweep(eng) == fused_launches(x, y, offsets[:2])


# ---------------------------------------------------------------------------------------------------------------------
# 7. batched Cholesky: one thread per matrix (n <= 8), one warp per matrix (n > 8)
# ---------------------------------------------------------------------------------------------------------------------
def _chol_ld(a):
    """Cholesky in long double of a batch; columns from the first non-positive pivot on are left zero.  Returns the
    factor and the 1-based index of that pivot (0: none)."""
    a = np.asarray(a, dtype=np.longdouble)
    b, n, _ = a.shape
    L = np.zeros_like(a)
    info = np.zeros(b, dtype=np.int64)
    for k in range(n):
        piv = a[:, k, k] - np.sum(L[:, k, :k] ** 2, axis=1)
        bad = (piv <= 0) & (info == 0)
        info[bad] = k + 1
        ok = info == 0
        d = np.sqrt(np.where(ok, piv, 1))
        L[:, k, k] = np.where(ok, d, 0)
        col = (a[:, k + 1:, k] - np.einsum('bij,bj->bi', L[:, k + 1:, :k], L[:, k, :k])) / d[:, None]
        L[:, k + 1:, k] = np.where(ok[:, None], col, 0)
    return L, info


def _run_cholesky(a):
    import torch
    from cimrgp_b200 import _lib
    lib = _lib.load()
    batch, n, _ = a.shape
    t = torch.as_tensor(np.ascontiguousarray(a), device='cuda')
    info = torch.full((batch,), -7, dtype=torch.int32, device='cuda')
    torch.cuda.synchronize()
    assert lib.mrgp_batched_cholesky(None, C.c_void_p(t.data_ptr()), n, batch, C.c_void_p(info.data_ptr())) == 0
    torch.cuda.synchronize()
    return t.cpu().numpy(), info.cpu().numpy()


def _spd(rng, batch, n, cond):
    q, _ = np.linalg.qr(rng.standard_normal((batch, n, n)))
    lam = np.exp(rng.uniform(0, np.log(cond), (batch, n)))
    lam[:, 0], lam[:, -1] = 1.0, cond
    a = np.einsum('bij,bj,bkj->bik', q, lam, q)
    return 0.5 * (a + np.swapaxes(a, 1, 2))


CHOL_N = [1, 3, 7, 8, 9, 31, 32]
CHOL_BATCH = [1, 33, 257, 10007]


@pytest.mark.parametrize('n', CHOL_N)
def test_batched_cholesky_against_long_double(n):
    rng = np.random.RandomState(n)
    for batch in CHOL_BATCH:
        a = _spd(rng, batch, n, 1e3)
        iu = np.triu_indices(n, 1)
        a[:, iu[0], iu[1]] = rng.standard_normal((batch, len(iu[0])))   # the kernel reads the lower triangle only
        low = np.tril(a) + np.swapaxes(np.tril(a, -1), 1, 2)
        got, info = _run_cholesky(a)
        ref, rinfo = _chol_ld(low)
        assert not np.any(rinfo) and not np.any(info), (batch, np.flatnonzero(info)[:5])
        assert np.array_equal(got[:, iu[0], iu[1]].view(np.int64), a[:, iu[0], iu[1]].view(np.int64)), batch
        lo = np.tril(got)
        err = np.abs(lo - ref.astype(np.float64))
        assert np.all(err <= 1e-13 * np.abs(ref.astype(np.float64)) + 1e-13 * np.max(np.abs(ref.astype(np.float64)), axis=(1, 2), keepdims=True)), \
            (batch, float(np.max(err)))


@pytest.mark.parametrize('n', CHOL_N)
def test_batched_cholesky_of_graded_matrices_has_a_small_backward_error(n):
    """Condition 1e12 (scaled rows and columns): only the backward error is bounded, ||L L^T - A|| <= 4 n eps ||A||."""
    rng = np.random.RandomState(100 + n)
    batch = 257
    b = _spd(rng, batch, n, 10.0)
    s = np.logspace(0, -6, n)
    a = b * s[None, :, None] * s[None, None, :]
    got, info = _run_cholesky(a)
    assert not np.any(info)
    L = np.tril(got).astype(np.longdouble)
    res = np.einsum('bik,bjk->bij', L, L) - a.astype(np.longdouble)
    rel = np.linalg.norm(res.astype(np.float64), axis=(1, 2)) / np.linalg.norm(a, axis=(1, 2))
    assert np.all(rel <= 4 * n * np.finfo(np.float64).eps), float(np.max(rel))


@pytest.mark.parametrize('n', CHOL_N)
def test_batched_cholesky_reports_the_failing_pivot(n):
    """A = L0 D L0^T with D_k < 0 fails at pivot k: info = k, the first k - 1 columns are the factor's, the other
    matrices of the batch are untouched by the failure."""
    rng = np.random.RandomState(200 + n)
    for batch in (33, 257):
        pivots = sorted({1, math.ceil(n / 2), n})
        a = _spd(rng, batch, n, 1e2)
        iu = np.triu_indices(n, 1)
        fail_at = {}
        for i, k in enumerate(pivots):
            b = 3 + 7 * i
            l0 = np.eye(n) + np.tril(0.3 * rng.standard_normal((n, n)), -1)
            d = rng.uniform(0.5, 2.0, n)
            d[k - 1] = -1.0
            a[b] = (l0 * d) @ l0.T
            fail_at[b] = k
        a[:, iu[0], iu[1]] = 1e300                    # never read
        low = np.tril(a) + np.swapaxes(np.tril(a, -1), 1, 2)
        got, info = _run_cholesky(a)
        ref, rinfo = _chol_ld(low)
        want = np.zeros(batch, dtype=np.int64)
        for b, k in fail_at.items():
            want[b] = k
        assert np.array_equal(rinfo, want)             # the long-double reference fails where it should, too
        assert np.array_equal(info, want), (batch, info[list(fail_at)])
        assert np.all(got[:, iu[0], iu[1]] == 1e300)
        r64 = ref.astype(np.float64)
        for b in range(batch):
            k = want[b] - 1 if want[b] else n        # leading columns that are factor columns
            g, r = np.tril(got[b])[:, :k], r64[b][:, :k]
            assert np.all(np.abs(g - r) <= 1e-13 * np.max(np.abs(r64[b])) + 1e-13 * np.abs(r)), (b, want[b])
