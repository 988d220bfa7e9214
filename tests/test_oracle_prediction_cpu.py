"""The oracle's index-set second moment and test likelihood (oracle/mrgp_oracle.py, predict_var_indexed and
test_likelihood) pinned to the unmodified reference's own output (tests/golden/predvar_*.npz), and their meaning on
test index sets with empty regions, which the reference cannot evaluate.  CPU only."""
import os

import numpy as np
import pytest

from oracle import mrgp_oracle as O
from parity import mismatch

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


def with_empty_regions(n_test, counts, seed):
    """Test offsets per layer with the given region counts; the first and last region of every layer with more than
    two regions are empty, and so is a run of three in the middle when there are more than eight.  With fewer test
    points than the remaining regions, a random choice of them holds one point each."""
    rng = np.random.RandomState(seed)
    out = []
    for r in counts:
        sizes = np.zeros(r, dtype=np.int64)
        full = np.arange(r)
        if r > 2:
            full = full[1:-1]
        if r > 8:
            full = np.setdiff1d(full, np.arange(r // 2 - 2, r // 2 + 1))
        if n_test < len(full):
            full = np.sort(rng.choice(full, n_test, replace=False))
        sizes[full] = rng.multinomial(n_test - len(full), np.ones(len(full)) / len(full)) + 1
        out.append(np.r_[0, np.cumsum(sizes)].astype(np.int64))
    return out


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
