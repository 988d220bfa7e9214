"""The oracle's index-set second moment and test likelihood (oracle/mrgp_oracle.py, predict_var_indexed and
test_likelihood) pinned to the unmodified reference's own output (tests/golden/predvar_*.npz), and their meaning on
test index sets with empty regions, which the reference cannot evaluate.  CPU only."""
import os

import numpy as np
import pytest

from oracle import mrgp_oracle as O
from parity import mismatch
from mrgp_helpers import prediction_ld, ragged, with_empty_regions

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
RTOL = 1e-9


def fitted(name):
    g = np.load(os.path.join(GOLD, name + '.npz'))
    res = int(g['meta.resolution'])
    m = O.OracleMRGP(g['x'], g['y'], int(g['meta.M']), O.uniform_offsets(g['x'].shape[0], res, 2),
                     mode='fi' if int(g['meta.fi']) else 'ci')
    for _ in range(int(g['meta.sweeps'])):
        m.sweep()
    return g, m, res


@pytest.mark.parametrize('name', ['predvar_ci', 'predvar_fi'])
def test_indexed_second_moment_and_test_likelihood_match_reference(name):
    g, m, res = fitted(name)
    xt, yt = g['pred.x'], g['pred.y']
    toff = O.uniform_offsets(xt.shape[0], res, 2)
    assert mismatch(m.predict_var_indexed(xt, toff), g['pred.var_indexed'], RTOL) is None
    assert mismatch(m.predict_var(xt), g['pred.var_global'], RTOL) is None
    assert mismatch(m.predict_mean(xt, toff), g['pred.mean_indexed'], RTOL) is None
    ref = float(g['pred.test_likelihood_indexed'])
    assert abs(m.test_likelihood([xt, yt], toff) - ref) <= RTOL * abs(ref)
    # the global form of the likelihood is the same formula over the layer-0 moments
    mf, vf = m.predict_mean(xt), m.predict_var(xt)
    want = np.mean(-0.5 * np.log(2 * np.pi * vf) - 0.5 * np.sum((yt - mf) ** 2, axis=1) / vf)
    assert abs(m.test_likelihood([xt, yt]) - want) <= 1e-13 * abs(want)


def _loop_moments(m, xt, toff):
    """Point by point and region by region as the reference walks them (MRGP.py:782-803, 863-932), skipping regions
    without test points: the mean and the index-set second moment.  A restatement of the same definition, not an
    independent oracle: it checks that the vectorised twin computes that definition; the skip itself is a choice (the
    reference cannot index the first point of an empty region), anchored to the reference only where no region is
    empty (the predvar pins above and the last check of the test below)."""
    xn = m._norm_test(xt)
    n = xn.shape[0]
    mean = np.zeros((n, m.dy))
    var = np.zeros(n)
    fvar = np.zeros(n)
    for j, off in enumerate(toff):
        ly = m.layers[j]
        contrib = np.zeros(n)
        for r in range(ly.R):
            a, b = int(off[r]), int(off[r + 1])
            for p in range(a, b):
                phi = O.eigenfunctions(xn[p:p + 1], np.array([[ly.L[r, 0]]]), m.M)[0]
                mean[p] += ly.A[r] @ phi + ly.bias_mean[r]
                contrib[p] = np.sum(phi * phi * ly.cm2[r]) + ly.bias_var[r]
            for p in range(a, b):
                var[p] += contrib[p] + (b - a) / ly.noise_mean[r] + fvar[a]
        fvar += contrib
    return mean, var


@pytest.mark.parametrize('mode', ['ci', 'fi'])
def test_prediction_with_empty_test_regions(mode):
    """A test index set with fewer points than regions: the mean is the sum over layers at each point's own region,
    and the second moment takes only the regions that hold test points (an empty region has no first point)."""
    g = np.load(os.path.join(GOLD, 'c1_ci.npz'))
    res = int(g['meta.resolution'])
    m = O.OracleMRGP(g['x'], g['y'], 30, O.uniform_offsets(g['x'].shape[0], res, 2), mode=mode)
    for _ in range(3):
        m.sweep()
    counts = [2 ** j for j in range(res + 1)]
    rng = np.random.RandomState(3)
    for n_test in (1, 7, 40):
        xt = rng.uniform(0.5, 3.5, size=(n_test, 1))
        toff = with_empty_regions(n_test, counts, seed=n_test)
        assert any(np.any(np.diff(o) == 0) for o in toff)
        mean, var = _loop_moments(m, xt, toff)
        assert mismatch(m.predict_mean(xt, toff), mean, 1e-12) is None
        got = m.predict_var_indexed(xt, toff)
        assert mismatch(got, var, 1e-12) is None and np.all(got > 0)
    # with every region non-empty the loop is the reference's own walk
    xt = np.atleast_2d(np.linspace(0.8, 3.2, 100)).T
    toff = O.uniform_offsets(100, res, 2)
    mean, var = _loop_moments(m, xt, toff)
    assert mismatch(m.predict_var_indexed(xt, toff), var, 1e-12) is None
    assert mismatch(m.predict_mean(xt, toff), mean, 1e-12) is None


def test_indexed_second_moment_needs_every_layer():
    _, m, res = fitted('predvar_ci')
    with pytest.raises(ValueError):
        m.predict_var_indexed(np.ones((10, 1)), O.uniform_offsets(10, res - 1, 2))


def edge_test_sets(st, counts, x_lo, x_hi, seed):
    """Normalised test points and test offsets at the edges of prediction: 1 to 129 points (across the 128-thread
    block of the kernels) with empty first, last and middle regions and with ragged regions that may be empty, points in
    random order with exact duplicates, and points exactly at -L, +L of every region of the last layer (each in that
    region) and at x = 0.  Yields (name, x (n,), offsets)."""
    rng = np.random.RandomState(seed)
    for n_test in (1, 7, 40, 127, 128, 129):
        x = rng.uniform(x_lo, x_hi, n_test)
        yield 'empty%d' % n_test, x, with_empty_regions(n_test, counts, seed=n_test)
        yield 'ragged%d' % n_test, x, ragged(n_test, counts, seed=n_test, min_len=0)
    pool = rng.uniform(x_lo, x_hi, 37)
    x = pool[rng.randint(0, 37, 500)]
    assert len(np.unique(x)) < 500 and np.any(np.diff(x) < 0)
    yield 'shuffled_duplicates', x, ragged(500, counts, seed=seed, min_len=0)
    j = len(counts) - 1
    L = st['L%d.L' % j][:, 0]
    x = np.r_[np.stack([-L, L], axis=1).ravel(), 0.0]
    offs = ragged(x.shape[0], counts[:-1], seed=seed + 1, min_len=0)
    last = np.r_[np.arange(counts[-1]) * 2, x.shape[0]].astype(np.int64)   # -L_r, +L_r in region r; 0 in the last
    yield 'interval_edges', x, offs + [last]


@pytest.mark.parametrize('mode', ['ci', 'fi'])
def test_long_double_prediction_matches_oracle(mode):
    """The long-double restatement of prediction (mrgp_helpers.prediction_ld), which the device tests use as the
    reference of the evaluation kernels, against the oracle's predictions on the oracle's own fitted state, at 1e-12:
    global and index-set mean and second moment, on the edge sets of the device tests (empty regions included)."""
    g = np.load(os.path.join(GOLD, 'c1_ci.npz'))
    res = int(g['meta.resolution'])
    m = O.OracleMRGP(g['x'], g['y'], 30, O.uniform_offsets(g['x'].shape[0], res, 2), mode=mode)
    for _ in range(3):
        m.sweep()
    st = m.state()
    counts = [2 ** j for j in range(res + 1)]
    raw = lambda xn: xn[:, None] * m.std_x + m.mean_x
    seen_empty = False
    for name, xn, toff in edge_test_sets(st, counts, -1.5, 1.5, seed=5):
        xt = raw(xn)
        xn = m._norm_test(xt)[:, 0]          # the oracle normalises again: use its points
        seen_empty |= any(np.any(np.diff(o) == 0) for o in toff)
        mean, _, var, _ = prediction_ld(st, xn, m.M)
        assert mismatch(mean, m.predict_mean(xt), 1e-12) is None, name
        assert mismatch(var, m.predict_var(xt), 1e-12) is None, name
        mean, _, var, _ = prediction_ld(st, xn, m.M, toff)
        assert mismatch(mean, m.predict_mean(xt, toff), 1e-12) is None, name
        assert mismatch(var, m.predict_var_indexed(xt, toff), 1e-12) is None, name
        mean, _, var, _ = prediction_ld(st, xn, m.M, toff[:2])
        assert var is None and mismatch(mean, m.predict_mean(xt, toff[:2]), 1e-12) is None, name
    assert seen_empty
