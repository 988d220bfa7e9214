"""CPU checks of the C ABI library: it loads, exports every symbol include/cimrgp.h declares, builds
correct plans, refuses to compute without a GPU, and its host-compiled math matches the oracle / goldens.
No compute entry point is called."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from cimrgp_b200 import _lib
from oracle import mrgp_oracle as O
from parity import mismatch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, 'tests', 'golden')


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    header = open(os.path.join(ROOT, 'include', 'cimrgp.h')).read()
    header = re.sub(r'/\*.*?\*/', '', header, flags=re.S)
    declared = set(re.findall(r'\b(mrgp_[a-z0-9_]+)\s*\(', header))
    assert declared, 'no declarations parsed'
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.mrgp_abi_version() == _lib.ABI_VERSION


def _create(n, offsets, m=30, mode=_lib.MODE_CI, n_ctas=0, dy=2, dx=1, noise=1, bias=1):
    lib = _lib.load()
    cfg = _lib.Config(_lib.ABI_VERSION, mode, n, dx, dy, m, len(offsets), noise, bias, 0, n_ctas)
    ptrs, keep = _lib.offsets_arg(offsets)
    nreg = (C.c_int32 * len(offsets))(*[len(o) - 1 for o in offsets])
    h = C.c_void_p()
    rc = lib.mrgp_create(C.byref(cfg), ptrs, nreg, C.byref(h))
    return lib, rc, h


def _plan(lib, h, j):
    a, b, c = C.c_int32(), C.c_int32(), C.c_int32()
    assert lib.mrgp_plan_info(h, j, C.byref(a), C.byref(b), C.byref(c)) == 0
    seg = np.zeros((b.value, 6), dtype=np.int64)
    assert lib.mrgp_plan_segments(h, j, seg.ctypes.data_as(C.POINTER(C.c_int64))) == 0
    return a.value, c.value, seg


@pytest.mark.parametrize('n,res,div,ctas', [(32, 5, 2, 0), (1000, 3, 3, 4), (100000, 7, 2, 148), (1000000, 9, 2, 148),
                                             (2048, 5, 2, 3)])
def test_plan_partitions_samples(n, res, div, ctas):
    offsets = O.uniform_offsets(n, res, div)
    lib, rc, h = _create(n, offsets, n_ctas=ctas)
    assert rc == 0, lib.mrgp_last_error(None)
    try:
        for j, off in enumerate(offsets):
            n_ctas, n_runs, seg = _plan(lib, h, j)
            # segments tile [0, n) in order
            assert seg[0, 0] == 0 and seg[-1, 1] == n and np.array_equal(seg[1:, 0], seg[:-1, 1])
            assert np.all(seg[:, 1] > seg[:, 0])
            # each segment lies in one region of the layer, one region of the parent and one CTA
            reg = np.searchsorted(off, seg[:, 0], side='right') - 1
            assert np.array_equal(reg, seg[:, 2]) and np.all(seg[:, 1] <= off[reg + 1])
            if j > 0:
                par = np.searchsorted(offsets[j - 1], seg[:, 0], side='right') - 1
                assert np.array_equal(par, seg[:, 3]) and np.all(seg[:, 1] <= offsets[j - 1][par + 1])
            assert np.all(np.diff(seg[:, 5]) >= 0) and seg[:, 5].max() < n_ctas
            # runs: consecutive ids, constant (cta, region) inside a run, every region owns >= 1 run
            assert seg[0, 4] == 0 and np.all(np.isin(np.diff(seg[:, 4]), (0, 1))) and seg[-1, 4] == n_runs - 1
            for col in (2, 5):
                same_run = np.diff(seg[:, 4]) == 0
                assert np.all(np.diff(seg[:, col])[same_run] == 0)
            assert len(np.unique(seg[:, 2])) == len(off) - 1
            # balanced CTA ranges (multiple of 32 samples, last one shorter)
            per_cta = np.bincount(seg[:, 5], weights=seg[:, 1] - seg[:, 0])
            assert per_cta.max() % 32 == 0 or len(per_cta) == 1
            assert len(per_cta) == 1 or per_cta.max() - per_cta[:-1].min() == 0
    finally:
        lib.mrgp_destroy(h)


@pytest.mark.parametrize('case', ['uniform', 'ragged'])
def test_pieces_of_the_closed_form_statistics_tile_every_region(case):
    """Bookkeeping of the closed-form layer statistics (DESIGN.md §4): for every layer j > 0 and every coarser layer
    jp, the pieces (region of j) x (region of jp) must tile each region of j exactly once, in order, with the right
    coarser region; the reference's uniform index sets are NOT nested (1e6 / 64 = 15625 is odd), ragged ones less so."""
    if case == 'uniform':
        n = 1000000
        offsets = O.uniform_offsets(n, 9, 2)
    else:
        rng = np.random.RandomState(5)
        n = 5000
        offsets = [np.array([0, n], dtype=np.int64)]
        for r in (3, 7, 20, 41):
            cuts = np.sort(rng.choice(np.arange(1, n), size=r - 1, replace=False))
            offsets.append(np.concatenate([[0], cuts, [n]]).astype(np.int64))
    lib, rc, h = _create(n, offsets, n_ctas=16)
    assert rc == 0, lib.mrgp_last_error(None)
    try:
        nested = True
        for j in range(1, len(offsets)):
            cnt = C.c_int32()
            assert lib.mrgp_plan_pieces(h, j, C.byref(cnt), None) == 0
            pcs = np.zeros((cnt.value, 5), dtype=np.int64)
            assert lib.mrgp_plan_pieces(h, j, C.byref(cnt), pcs.ctypes.data_as(C.POINTER(C.c_int64))) == 0
            R = len(offsets[j]) - 1
            for jp in range(j):
                sel = pcs[pcs[:, 0] == jp]
                assert np.all(sel[:, 4] > sel[:, 3])
                # the pieces of (jp, .) tile [0, n) in order and respect both partitions
                assert sel[0, 3] == 0 and sel[-1, 4] == n and np.array_equal(sel[1:, 3], sel[:-1, 4])
                for c in range(R):
                    mine = sel[sel[:, 1] == c]
                    assert mine[0, 3] == offsets[j][c] and mine[-1, 4] == offsets[j][c + 1]
                    nested = nested and len(mine) == 1
                anc = np.searchsorted(offsets[jp], sel[:, 3], side='right') - 1
                assert np.array_equal(anc, sel[:, 2])
                assert np.all(sel[:, 4] <= offsets[jp][sel[:, 2] + 1])
        assert not nested      # both cases exercise regions that straddle coarser regions
    finally:
        lib.mrgp_destroy(h)


def test_create_rejects_what_the_reference_rejects():
    off = O.uniform_offsets(64, 2, 2)
    lib, rc, h = _create(64, off, dy=1)
    assert rc == _lib.EINVAL and b'greater than 1' in lib.mrgp_last_error(None)   # MRGP.py:65-66
    bad = [o.copy() for o in off]
    bad[1][1] = 0
    lib, rc, h = _create(64, bad)
    assert rc == _lib.EINVAL
    for kw in (dict(dy=3), dict(dx=2), dict(m=49), dict(m=0)):
        lib, rc, h = _create(64, off, **kw)
        assert rc == _lib.EINVAL, kw
    for kw in (dict(noise=0), dict(bias=0), dict(noise=0, bias=0)):      # shared noise / bias variants are accepted
        lib, rc, h = _create(64, off, **kw)
        assert rc == 0, kw
        lib.mrgp_destroy(h)


def test_create_checks_the_cluster_size_switch(monkeypatch):
    """MRGP_CHAIN_CLUSTER (DESIGN.md §5c) is refused at creation unless the fused sweep can launch it."""
    off = O.uniform_offsets(4096, 5, 2)
    for value in ('0', '1', '2', '4', '8', '16'):
        monkeypatch.setenv('MRGP_CHAIN_CLUSTER', value)
        lib, rc, h = _create(4096, off)
        assert rc == 0, (value, lib.mrgp_last_error(None))
        lib.mrgp_destroy(h)
    for value in ('3', '6', '12', '17', '32', '-1', '-16', '', 'x', '4x', '2.0', '99999999999'):
        monkeypatch.setenv('MRGP_CHAIN_CLUSTER', value)
        lib, rc, h = _create(4096, off)
        assert rc == _lib.EINVAL and not h.value, value
        assert b'MRGP_CHAIN_CLUSTER' in lib.mrgp_last_error(None), value


def test_no_gpu_means_no_compute():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    off = O.uniform_offsets(64, 2, 2)
    lib, rc, h = _create(64, off)
    assert rc == 0
    try:
        buf = np.zeros(1 << 20, dtype=np.uint8)
        assert lib.mrgp_workspace_bytes(h) > 0
        rc = lib.mrgp_bind_workspace(h, C.c_void_p((buf.ctypes.data + 255) & ~255), lib.mrgp_workspace_bytes(h))
        assert rc in (_lib.ENODEVICE, _lib.ENOMEM)
        assert lib.mrgp_sweep(h, 1) == _lib.ESTATE
        assert lib.mrgp_phase_a(h, 0) == _lib.ESTATE
    finally:
        lib.mrgp_destroy(h)
    from cimrgp_b200.engine import Engine
    with pytest.raises(_lib.MrgpError):
        Engine(np.zeros((64, 1)), np.zeros((64, 2)), off, 30)


def test_host_digamma_matches_scipy():
    from scipy.special import psi
    lib = _lib.load()
    xs = np.concatenate([[1e-45, 1e-30, 1e-10, 1e-3, 0.5, 1.0, 1.4616321449683623, 2.0, 9.999, 10.0, 33.5],
                         10 ** np.linspace(-3, 6.5, 200)])
    got = np.array([lib.mrgp_host_digamma(float(x)) for x in xs])
    ref = psi(xs)
    assert np.all(np.abs(got - ref) <= 4e-15 * np.maximum(1.0, np.abs(ref)))


def test_host_spectral_and_basis_match_reference_kats():
    lib = _lib.load()
    k = np.load(os.path.join(GOLD, 'kats.npz'))
    lam = k['basis.lam']
    got = np.array([lib.mrgp_host_matern_spectral(float(v), 1., 1., 1.) for v in lam])
    assert mismatch(got, k['basis.S'], 1e-13) is None
    got = np.array([lib.mrgp_host_matern_spectral(float(v), 2.5, .7, 1.3) for v in lam])
    assert mismatch(got, k['basis.S_nu2.5_l0.7_sf1.3'], 1e-13) is None
    phi = np.zeros((k['basis.x'].shape[0], 40))
    for n, x in enumerate(k['basis.x'][:, 0]):
        lib.mrgp_host_basis(float(x), 2.0, 40, phi[n].ctypes.data_as(C.POINTER(C.c_double)))
    # three-term recurrence vs. direct sin (SURVEY.md §8c: 2e-14 abs at M = 30)
    assert np.max(np.abs(phi - k['basis.phi'])) < 2e-13


def test_host_bingham_matches_reference_kats():
    lib = _lib.load()
    k = np.load(os.path.join(GOLD, 'kats.npz'))
    P = C.POINTER(C.c_double)
    for q, b_in in enumerate(k['bingham.B_in']):
        b_in = np.ascontiguousarray(b_in)
        b_out, kap, rho, cov = np.zeros((2, 2)), np.zeros(2), np.zeros(2), np.zeros((2, 2))
        logc, nch = C.c_double(), C.c_int32()
        lib.mrgp_host_bingham2(b_in.ctypes.data_as(P), b_out.ctypes.data_as(P), kap.ctypes.data_as(P),
                               rho.ctypes.data_as(P), C.byref(logc), cov.ctypes.data_as(P), C.byref(nch))
        scale = np.abs(k['bingham.B'][q]).max()
        assert np.max(np.abs(b_out - k['bingham.B'][q])) <= 1e-14 * scale, q
        assert np.max(np.abs(kap - k['bingham.kappa'][q])) <= 1e-13 * scale, q
        # brentq stops at xtol 2e-12 (computeRealBinghamConstant.py:92); the Newton root is exact
        assert mismatch(rho, k['bingham.rho'][q], 1e-9, atol_scale=1e-11) is None, q
        assert abs(logc.value - k['bingham.logC'][q]) <= 1e-10 * max(1.0, abs(k['bingham.logC'][q])), q
        assert mismatch(cov, k['bingham.axis_cov'][q], 1e-9, atol_scale=1e-11) is None, q
        assert nch.value >= 1
    # SURVEY.md §8c: Bingham([[2, .5], [.5, 1]])
    b_in = np.array([[2., .5], [.5, 1.]])
    b_out, kap, rho, cov = np.zeros((2, 2)), np.zeros(2), np.zeros(2), np.zeros((2, 2))
    logc, nch = C.c_double(), C.c_int32()
    lib.mrgp_host_bingham2(b_in.ctypes.data_as(P), b_out.ctypes.data_as(P), kap.ctypes.data_as(P),
                           rho.ctypes.data_as(P), C.byref(logc), cov.ctypes.data_as(P), C.byref(nch))
    assert np.allclose(kap, [2.2071067811865475, 0.7928932188134524], rtol=1e-15)
    assert np.allclose(rho, [0.6725460300683469, 0.3274539699316528], rtol=1e-10)
    assert abs(logc.value - 3.5103108648220838) < 1e-11


def test_host_omega_matches_reference_within_its_solver_tolerance():
    lib = _lib.load()
    k = np.load(os.path.join(GOLD, 'kats.npz'))
    P = C.POINTER(C.c_double)
    for lw, eta in zip(k['omega.log_omega_hat'], k['omega.ln_eta']):
        m = lw.shape[0]
        ref = np.exp(eta[:m, None] + eta[None, m:] + lw)
        lw = np.ascontiguousarray(lw)
        om = np.zeros((m, m))
        it = C.c_int32()
        assert lib.mrgp_host_omega(lw.ctypes.data_as(P), m, om.ctypes.data_as(P), C.byref(it)) == 0
        assert it.value < 1000
        assert np.max(np.abs(om.sum(0) - 1)) < 1e-10 and np.max(np.abs(om.sum(1) - 1)) < 1e-12   # kOmegaTol
        assert mismatch(om, ref, 1e-6) is None            # fsolve's own error is ~1e-8 (SURVEY.md App. D)
        assert mismatch(om, O.omega_sinkhorn(lw), 1e-8) is None


def test_host_omega_on_peaked_tables_from_the_device_run():
    """log omega_hat tables captured on the device at config 4 (layers 1 and 2, sweeps 2-7; scratch/dump_table.py):
    overall range 2e5, every row's maximum ~49 above its second entry.  A Newton step from a far start loses
    definiteness on them and plain Sinkhorn crawls on the flat ones; the step policy (omega_take_newton) must reach the
    tolerance in a few dozen steps, cold and warm-started alike."""
    lib = _lib.load()
    P = C.POINTER(C.c_double)
    g = np.load(os.path.join(GOLD, 'omega_hard.npz'))
    for key in g.files:
        lw = np.ascontiguousarray(g[key])
        m = lw.shape[0]
        om, it = np.zeros((m, m)), C.c_int32()
        assert lib.mrgp_host_omega(lw.ctypes.data_as(P), m, om.ctypes.data_as(P), C.byref(it)) == 0
        assert it.value <= 40, (key, it.value)
        assert np.max(np.abs(om.sum(0) - 1)) < 1e-10 and np.max(np.abs(om.sum(1) - 1)) < 1e-12
        assert mismatch(om, O.omega_sinkhorn(lw), 1e-8) is None, key


def test_index_sets_bit_exact():
    from cimrgp_b200.IndexSetGenerator import IndexSetUniform, offsets_of
    k = np.load(os.path.join(GOLD, 'kats.npz'))
    for (n, res, div) in k['index.cases']:
        idx = IndexSetUniform(n, res, div)
        assert idx.get_n_resolutions() == res
        for j, o in enumerate(idx.offsets):
            ref = k['index.%d_%d_%d.L%d' % (n, res, div, j)]
            assert o.dtype == np.int64 and np.array_equal(o, ref)
    idx = IndexSetUniform(37, 2, 3)
    assert idx.index_set[2][-1] == list(range(32, 37)) and idx.divider == 3
    assert [np.array_equal(a, b) for a, b in zip(offsets_of(idx), idx.offsets)]
    with pytest.raises(ValueError):
        IndexSetUniform(10, 5, 2)
    # random-boundary variant consumes the global RNG exactly as IndexSetGenerator.py:67-92
    np.random.seed(3)
    a = IndexSetUniform(1000, 2, 2, n_regions=[1, 3, 5])
    assert [len(o) - 1 for o in a.offsets] == [1, 3, 5] and all(o[0] == 0 and o[-1] == 1000 for o in a.offsets)
