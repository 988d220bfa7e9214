"""bench.py --dump-outputs: which arrays are written, in which type, and the bound on their size."""
import os

import numpy as np
import pytest

import bench


class _Engine(object):
    """Engine.state() / Engine.elbo() of a two-layer model with N samples (the shapes of cimrgp_b200.engine)."""
    N = 300000

    def state(self, latent=True):
        rng = np.random.RandomState(1)
        st = {}
        for j in range(2):
            st['L%d.A' % j] = rng.standard_normal((2 ** j, 2, 30))
            st['L%d.fbar' % j] = rng.standard_normal((self.N, 2))
            st['L%d.fvar' % j] = rng.standard_normal(self.N)
        st['S.omega'] = rng.standard_normal((30, 30))
        return st

    def elbo(self):
        return np.arange(12.).reshape(2, 6)


def test_dump_keeps_a_fixed_sample_of_per_sample_arrays_in_float64(tmp_path):
    eng = _Engine()
    full = eng.state()
    bench.dump_outputs(str(tmp_path), bench.engine_outputs(eng))
    got = {f[:-len('.npy')]: np.load(str(tmp_path / f)) for f in os.listdir(str(tmp_path))}
    assert set(got) == set(full) | {'latent_rows', 'elbo'}
    assert all(v.dtype == np.float64 for v in got.values())
    rows = got['latent_rows'].astype(np.int64)
    assert len(rows) == bench.DUMP_ROWS and np.all(np.diff(rows) > 0)
    assert np.array_equal(got['L1.fbar'], full['L1.fbar'][rows]) and np.array_equal(got['L0.fvar'], full['L0.fvar'][rows])
    assert np.array_equal(got['L1.A'], full['L1.A']) and np.array_equal(got['elbo'], eng.elbo())
    assert np.array_equal(bench.engine_outputs(eng)['latent_rows'], rows)       # the same rows on every run


def test_dump_refuses_outputs_over_the_limit(tmp_path):
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / 'd'), {'x': np.zeros(bench.DUMP_BYTES // 8 + 1)})
    assert not os.path.exists(str(tmp_path / 'd'))
