"""Helpers shared by the tests that hold a device model to the NumPy oracle: data and offsets, the oracle beside a
device model (with its exact-scaling fallback for the omega chain), test index sets with empty regions, and a
long-double restatement of prediction from a fitted state with a forward-error bound for the device's evaluation."""
import numpy as np

from oracle import mrgp_oracle as O
from parity import compare, mismatch

RTOL = 1e-6
# fields downstream of the chain of permutation weights (see test_parity_gpu.py, OMEGA_CHAIN)
OMEGA_CHAIN = ('S.B', 'S.kappa', 'S.logC', 'S.rho', 'S.omega')


def normed(x):
    return (x - np.mean(x, 0)) / np.std(x, 0)     # the oracle's standard normalisation (MRGP.py:278-295)


def ragged(n, counts, seed, min_len=3):
    """Random region boundaries per layer (not nested across layers), every region at least min_len samples."""
    rng = np.random.RandomState(seed)
    out = []
    for r in counts:
        extra = rng.multinomial(n - min_len * r, rng.dirichlet(np.ones(r)))
        out.append(np.r_[0, np.cumsum(min_len + extra)].astype(np.int64))
    return out


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


def engine(x, y, offsets, m, mode='ci', **kw):
    from cimrgp_b200.engine import Engine
    return Engine(normed(x), y, offsets, m, mode=mode, **kw)


def dropin(x, y, m, resolution, fi, **kw):
    from cimrgp_b200 import IndexSetUniform, LaplacianEigenpairs, MaternKernel
    from cimrgp_b200.MRGP import MultiResolutionGaussianProcess
    return MultiResolutionGaussianProcess([x, y], m, IndexSetUniform(x.shape[0], resolution, 2), LaplacianEigenpairs(),
                                          MaternKernel(1, 1, 1), forced_independence=fi, **kw)


def omega_exact(lw, tol=1e-15):
    """The doubly-stochastic scaling diag(e^a) exp(lw) diag(e^b) to roundoff: Newton's method on (a, b) with
    backtracking, from 50 Sinkhorn sweeps.  On the nearly decomposable tables of models with many small regions over
    many layers (log omega_hat spanning 1000 and more) plain Sinkhorn (mrgp_oracle.omega_sinkhorn) stops after its 10000
    sweeps at column sums 1e-4 off; Newton converges quadratically there, to column sums within 1e-13 of one."""
    from scipy.special import logsumexp
    lw = np.asarray(lw, dtype=np.float64)
    m = lw.shape[0]
    la, lb = np.zeros(m), np.zeros(m)
    for _ in range(50):
        la = -logsumexp(lw + lb[None, :], axis=1)
        lb = -logsumexp(lw + la[:, None], axis=0)

    def resid(la, lb):
        p = np.exp(lw + la[:, None] + lb[None, :])
        return p, np.r_[p.sum(1) - 1, p.sum(0) - 1]

    p, f = resid(la, lb)
    for _ in range(100):
        nf = np.max(np.abs(f))
        if nf < tol:
            break
        jac = np.block([[np.diag(p.sum(1)), p], [p.T, np.diag(p.sum(0))]])
        step = np.linalg.lstsq(jac, -f, rcond=None)[0]
        t = 1.0
        while t > 1e-6:
            p2, f2 = resid(la + t * step[:m], lb + t * step[m:])
            if np.max(np.abs(f2)) < nf:
                break
            t *= 0.5
        else:
            break
        la, lb, p, f = la + t * step[:m], lb + t * step[m:], p2, f2
    return p


class Oracle(object):
    """The NumPy oracle beside a device model.  In ci mode the reference solves for omega with MINPACK hybrd at xtol
    1.5e-8 (Stats.py:413) while the device computes the exact doubly-stochastic scaling.  On some models hybrd stalls
    ("not making good progress") and its slack in the omega chain exceeds the 1e-6 of the rule; every field downstream of
    omega (ARD means, scale precisions, the coefficients of every layer after the next sweep) inherits it.  There, and
    only after checking that the slack is the oracle's own (its omega chain differs from the exact scaling by more than
    1e-6), the model is held to the same oracle with the exact scaling (omega_exact): every array at the rule, the shared
    state at 1e-9, as test_config4_full_size_against_oracle does."""

    def __init__(self, x, y, m, offsets, mode='ci', **kw):
        self.args, self.kw = (x, y, m, offsets), dict(kw, mode=mode)
        self.ora = O.OracleMRGP(x, y, m, offsets, **self.kw)
        self.best = self.ora
        self.exact = None
        self.done = 0

    def _sweep_exact(self, k):
        saved = O.omega_sinkhorn
        O.omega_sinkhorn = lambda lw: omega_exact(lw)
        try:
            for _ in range(k):
                self.exact.sweep()
        finally:
            O.omega_sinkhorn = saved

    def sweep(self, k):
        for _ in range(k):
            self.ora.sweep()
        if self.exact is not None:
            self._sweep_exact(k)
        self.done += k

    def check(self, eng):
        got, ref = eng.state(), self.ora.state()
        self.best = self.ora
        try:
            compare(got, ref)
            return
        except AssertionError:
            if self.ora.mode == 'fi':
                raise
        if self.exact is None:
            self.exact = O.OracleMRGP(*self.args, omega_solver='sinkhorn', **self.kw)
            self._sweep_exact(self.done)
        ex = self.exact.state()
        assert any(mismatch(ref[k], ex[k], RTOL) is not None for k in OMEGA_CHAIN), \
            'device off the oracle where the oracle agrees with its exact-scaling form'
        self.best = self.exact
        compare(got, ex)
        for k in [k for k in ex if k.startswith('S.')]:
            assert mismatch(got[k], ex[k], 1e-9, atol_scale=1e-9 if k == 'S.omega' else 1e-12) is None, k

    def check_elbo(self, eng):
        assert mismatch(eng.elbo(), self.best.elbo()[2], RTOL) is None

    def check_predictions(self, eng, n_test=2000, seed=11):
        """predict_mean without and with an index set (every layer), predict_var."""
        ora = self.best
        counts = [len(o) - 1 for o in self.args[3]]
        n_test = max(n_test, 4 * max(counts))
        xt = np.atleast_2d(np.linspace(1, 3, n_test)).T
        xtn = (xt - ora.mean_x) / ora.std_x
        toff = ragged(n_test, counts, seed, min_len=1)
        assert mismatch(eng.predict_mean(xtn), ora.predict_mean(xt), RTOL) is None
        assert mismatch(eng.predict_mean(xtn, toff), ora.predict_mean(xt, toff), RTOL) is None
        assert mismatch(eng.predict_var(xtn), ora.predict_var(xt), RTOL) is None


# ---------------------------------------------------------------------------------------------------------------------
# Long-double restatement of prediction (k_eval_layers, k_eval_var_indexed) from a fitted state
# ---------------------------------------------------------------------------------------------------------------------
PI_LD = 4 * np.arctan(np.longdouble(1))
EPS = 2.0 ** -52       # spacing of float64 at 1
UNIT = 2.0 ** -53      # unit roundoff of float64
# Per-point error of the device's phi_i (basis_seed + the three-term recurrence), in units of EPS / sqrt(L):
#   C1 = 4: the seed.  sincospi_fast is exact to 2 ulp (mrgp_math.cuh), rsqrtL = 1 / sqrt(L) and phi_1 = rsqrtL * cos
#        round twice more; that relative error carries into every phi_i.
#   C2 = 8, times i (1 + |u|): u = x * (0.5 / L) is rounded twice, |du| <= EPS |u|, which moves the angle of phi_i by
#        pi i |du| (pi i |u| EPS).  The recurrence phi_(i+1) = c2 phi_i - phi_(i-1) adds the error of c2 = -2 sin(pi u),
#        amplified by |sin(theta) dU_(i-1)/dx (cos theta)| near an interval edge (theta -> 0 mod pi), and its own
#        rounding; a host run of basis_seed and the recurrence against this restatement over 2.4e6 points (half of them
#        within 0.05 of a half-integer u, i.e. next to an edge) found at most 6.6 i EPS / sqrt(L) for |u| <= 1 at i <= 48
#        (at u = 0.515), and at most 2.1 i (1 + |u|) EPS / sqrt(L) for |u| up to 1e6.  C2 = 8 bounds both with a margin
#        of 1.8 or more (8 (1 + |u|) >= 12 where the recurrence term peaks, |u| ~ 1/2).
C1, C2 = 4.0, 8.0


def phi_ld(x, L, m):
    """phi_i(x) = L^-1/2 sin(pi i (x + L) / (2L)), i = 1..m, in long double.  u = x / (2L) and i (u + 1/2) are reduced
    mod 2 exactly (fmod) before the sine, so the argument of the sine stays below 2 pi for any x.  Returns phi (n, m)
    and u (n,)."""
    x = np.asarray(x, dtype=np.longdouble)
    L = np.asarray(L, dtype=np.longdouble)
    u = x / (2 * L)
    i = np.arange(1, m + 1, dtype=np.longdouble)
    t = np.fmod(u[:, None] * i[None, :] + 0.5 * i[None, :], 2)
    return np.sin(PI_LD * t) / np.sqrt(L)[:, None], u


def _layer_ld(st, j, x, reg, m, chunk=1 << 15):
    """Layer j at the points x, each in its region reg: the mean term Phi A^T + b (n, dy), the variance term
    sum_i phi_i^2 cm2_i + bias_var (n,), both in long double, and their bounds from the basis error and from the
    rounding of the device's sums (M + 2 roundings per term; the sums over layers are added by the caller)."""
    n = x.shape[0]
    A, cm2 = st['L%d.A' % j], st['L%d.cm2' % j]
    L, b, bv = st['L%d.L' % j][:, 0], st['L%d.bias_mean' % j], st['L%d.bias_var' % j]
    dy = A.shape[1]
    mean = np.zeros((n, dy), dtype=np.longdouble)
    mean_err = np.zeros((n, dy))
    var = np.zeros(n, dtype=np.longdouble)
    var_err = np.zeros(n)
    for s in range(0, n, chunk):
        e = slice(s, min(n, s + chunk))
        r = reg[e]
        phi, u = phi_ld(x[e], L[r], m)
        i = np.arange(1, m + 1)[None, :]
        dphi = EPS / np.sqrt(L[r])[:, None] * (C1 + C2 * i * (1 + np.abs(u.astype(np.float64)))[:, None])   # per phi_i
        ar = A[r].astype(np.longdouble)                             # (n, dy, m)
        terms = phi[:, None, :] * ar
        mean[e] = np.sum(terms, axis=2) + b[r]
        absum = np.sum(np.abs(terms.astype(np.float64)), axis=2) + np.abs(b[r])
        mean_err[e] = np.sum(np.abs(A[r]) * dphi[:, None, :], axis=2) + (m + 2) * UNIT * absum
        c = cm2[r].astype(np.longdouble)
        vt = phi * phi * c
        var[e] = np.sum(vt, axis=1) + bv[r]
        pf = np.abs(phi.astype(np.float64))
        var_err[e] = np.sum(np.abs(cm2[r]) * (2 * pf + dphi) * dphi, axis=1) + \
            (m + 2) * UNIT * (np.sum(np.abs(vt.astype(np.float64)), axis=1) + np.abs(bv[r]))
    return mean, mean_err, var, var_err


def prediction_ld(st, x, m, test_offsets=None):
    """Prediction from the fitted state st (Engine.state() or OracleMRGP.state() keys) at the normalised test points x,
    in long double, with forward-error bounds of the device's float64 evaluation.

    test_offsets None: the global mean and second moment (layer 0, region 0; MRGP.py:726-755, 833-861).  Otherwise the
    index-set mean (sum over the given layers at each point's region) and the index-set second moment (every layer:
    sum_i phi_i^2 cm2_i + bias_var + n_test(region) / noise_mean + the variance terms of the coarser layers at the
    region's first test point; a region without test points contributes nothing, DESIGN.md §2).
    Returns (mean, mean_bound, var, var_bound) as float64 arrays; var is None for an index set with fewer layers than
    the model."""
    x = np.asarray(x, dtype=np.float64).reshape(-1)
    n = x.shape[0]
    if test_offsets is None:
        mean, mean_err, var, var_err = _layer_ld(st, 0, x, np.zeros(n, dtype=np.int64), m)
        return mean.astype(np.float64), mean_err, var.astype(np.float64), var_err
    J = len(test_offsets)
    n_layers = len([k for k in st if k.endswith('.L') and k.startswith('L')])
    mean = np.zeros((n, st['L0.A'].shape[1]), dtype=np.longdouble)
    mean_err = np.zeros(mean.shape)
    absmean = np.zeros(mean.shape)
    var = np.zeros(n, dtype=np.longdouble)
    var_err = np.zeros(n)
    fvar = np.zeros(n, dtype=np.longdouble)       # variance terms of the layers below the current one, per point
    fvar_err = np.zeros(n)
    for j, off in enumerate(test_offsets):
        off = np.asarray(off, dtype=np.int64)
        cnt = np.diff(off)
        reg = np.repeat(np.arange(len(cnt)), cnt)
        mj, mj_err, vj, vj_err = _layer_ld(st, j, x, reg, m)
        mean += mj
        mean_err += mj_err
        absmean += np.abs(mj.astype(np.float64))
        first = off[:-1][reg]
        noise = cnt[reg].astype(np.longdouble) / st['L%d.noise_mean' % j][reg]
        var += vj + noise + fvar[first]
        var_err += vj_err + UNIT * noise.astype(np.float64) + fvar_err[first]
        fvar = fvar + vj
        fvar_err = fvar_err + vj_err
    mean_err += (J + 1) * UNIT * absmean          # the sum over layers
    if J != n_layers:
        return mean.astype(np.float64), mean_err, None, None
    # every term of the second moment is non-negative: the device's J (J + 1) / 2 + 2 J additions of layer terms round
    # by at most that many units of the total
    var_err += (J * (J + 1) // 2 + 2 * J + 1) * UNIT * np.abs(var.astype(np.float64))
    return mean.astype(np.float64), mean_err, var.astype(np.float64), var_err
