"""CPU oracle for the ciMRGP / fiMRGP variational-inference hot path.

TEST INFRASTRUCTURE ONLY.  This is a vectorised NumPy restatement of the reference algorithm
(jtaghia/ciMRGP, `/root/reference/src`); it is the checker for the CUDA path and the "port" CPU
baseline of `bench.py`.  Nothing in the product package `cimrgp_b200/` imports it: only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` legs may.

Parity pin: the reference has no golden vectors or tests of its own (SURVEY.md §4).  The pin is the
reference itself, imported unmodified in the build container by `tests/golden/make_golden.py`; the
state it produces is committed under `tests/golden/*.npz` and `tests/test_oracle_golden.py` holds this
oracle to it (rtol 1e-7: the reference's own `fsolve` for the permutation weights is only converged to
~1e-8).  Third-party arithmetic that the reference reaches through NumPy/SciPy is reached here through
the same calls (numpy.linalg.eig/cholesky/svd/eigvals, scipy.optimize.fsolve/brentq/fminbound,
scipy.special.psi/gammaln); versions in this image: NumPy 2.3.5, SciPy 1.18.1 (unpinned upstream).

Every function cites the reference file:line it follows.  Regions of a layer are contiguous index
ranges (IndexSetGenerator.py:51-92 only ever builds `list(range(a, b))`), so a layer is described by an
int64 offsets array of length R+1 and per-region sums are `np.add.reduceat`.
"""
import time

import numpy as np
from numpy import linalg as la
from scipy.optimize import brentq, fminbound, fsolve
from scipy.special import gammaln, logsumexp, psi

EPSILON = 1e-45  # Priors.py:5


# ----------------------------------------------------------------------------------------------
# index sets  (IndexSetGenerator.py:51-65)
# ----------------------------------------------------------------------------------------------
def uniform_offsets(sample_length, resolution, divider):
    """Region offsets per layer for IndexSetUniform(sample_length, resolution, divider).

    IndexSetGenerator.py:51-65: divider**m regions of floor(N / divider**m) samples, the remainder
    goes to the last region; ValueError when a region would be empty.  `divider` is forced to 0 when
    resolution == 0 (:17-18), and 0**0 == 1 region.
    """
    resolution = int(resolution)
    divider = 0 if resolution == 0 else int(divider)
    n = int(sample_length)
    layers = []
    for m in range(resolution + 1):
        n_regions = divider ** m
        per = n // n_regions
        if per < 1:
            raise ValueError('*** Chosen resolution is too large! ***')
        off = np.arange(n_regions + 1, dtype=np.int64) * per
        off[-1] = n
        layers.append(off)
    return layers


def offsets_from_index_set(index_set):
    """index_set[j][l] (lists of ints) -> offsets; checks that the lists are contiguous ranges."""
    layers = []
    for regions in index_set:
        off = [regions[0][0]]
        for r in regions:
            if len(r) == 0 or r[0] != off[-1] or r[-1] - r[0] + 1 != len(r):
                raise ValueError('index sets must be contiguous, ordered ranges')
            off.append(r[-1] + 1)
        layers.append(np.asarray(off, dtype=np.int64))
    return layers


def seg_sum(a, off):
    """Per-region sums over the leading axis."""
    return np.add.reduceat(a, off[:-1], axis=0)


def seg_expand(v, off):
    """Per-region values -> per-sample values."""
    return np.repeat(v, np.diff(off), axis=0)


# ----------------------------------------------------------------------------------------------
# basis, eigenvalues, spectral density   (KernelClass.py:9-37, 80-90; MRGP.py:297-357)
# ----------------------------------------------------------------------------------------------
def eigenfunctions(x, L_per_sample, n_basis):
    """Phi[n, i] = prod_k L_k^-1/2 sin(pi (i+1) (x_k + L_k) / (2 L_k)).  KernelClass.py:21-37 with
    MRGP.py:344-350 (same basis index in every input dimension, product over dimensions)."""
    ids = np.arange(1, n_basis + 1, dtype=np.float64)
    phi = np.ones((x.shape[0], n_basis))
    for k in range(x.shape[1]):
        Lk = L_per_sample[:, k:k + 1]
        up = np.pi * ids[None, :] * (x[:, k:k + 1] + Lk)
        phi *= (1. / np.sqrt(Lk)) * np.sin(up / (2 * Lk))
    return phi


def eigenvalues(L, n_basis):
    """lambda[r, i] = sum_k (pi (i+1) / (2 L_rk))^2.  KernelClass.py:36, MRGP.py:349."""
    ids = np.arange(1, n_basis + 1, dtype=np.float64)
    return np.sum(np.power((np.pi * ids[None, :, None]) / (2 * L[:, None, :]), 2), axis=2)


def matern_spectral(s, nu, l, sf):
    """KernelClass.py:80-90 (log form) exponentiated as :57-58."""
    log_arg = np.log(2 * nu) - 2 * np.log(l)
    arg = np.exp(log_arg)
    log_const = 0.5 * np.log(2 * np.pi) + nu * log_arg
    log_gamma_term = gammaln(nu + 0.5) - gammaln(nu)
    log_power_term = -(nu + .5) * np.log(arg + s ** 2)
    return np.exp(np.log(sf) + log_const + log_gamma_term + log_power_term)


# ----------------------------------------------------------------------------------------------
# Bingham normaliser (computeRealBinghamConstant.py:12-155) and PD guard (SanityCheck.py:16-65)
# ----------------------------------------------------------------------------------------------
def log_partition_saddle(kappa):
    """First-order Kume-Wood saddle-point log C(kappa) and gradient.  kappa (..., p).
    computeRealBinghamConstant.py:42-53 shift, :72-95 root (brentq on [0.1-p, 0.1-0.5]),
    :101-119 logC, :125-147 gradient."""
    kappa = np.asarray(kappa, dtype=np.float64)
    shape = kappa.shape
    p = shape[-1]
    lam = -kappa.reshape(-1, p)
    adjust = 0.1 - np.min(lam, axis=-1, keepdims=True)
    lam = lam + adjust
    t = np.array([brentq(lambda t_, lk: 0.5 * np.sum(1 / (lk - t_)) - 1., 0.1 - p, 0.1 - 0.5, args=(lk,))
                  for lk in lam])[:, None]
    k2 = 0.5 * np.sum((lam - t) ** -2, axis=-1, keepdims=True)
    k3 = np.sum((lam - t) ** -3, axis=-1, keepdims=True)
    logc = 0.5 * (np.log(2) + (p - 1) * np.log(np.pi) - np.log(k2)
                  - np.sum(np.log(lam - t), axis=-1, keepdims=True)) - t
    dk1dlam = -0.5 * (lam - t) ** -2
    dk1dt = -np.sum(dk1dlam, axis=-1, keepdims=True)
    dtdlam = -dk1dlam / dk1dt
    dk2dlam = -(lam - t) ** -3 + k3 * dtdlam
    dlogk2 = dk2dlam / k2
    dsumlog = 1. / (lam - t)
    dsumlogdt = -np.sum(dsumlog, axis=-1, keepdims=True)
    dsumlog = dsumlog + dsumlogdt * dtdlam
    grad = 0.5 * dlogk2 + 0.5 * dsumlog + dtdlam
    logc = logc + adjust
    return logc.reshape(shape[:-1]), grad.reshape(shape)


def is_pd(b):
    """SanityCheck.py:59-65."""
    try:
        la.cholesky(b)
        return True
    except la.LinAlgError:
        return False


def nearest_pd(a):
    """SanityCheck.py:16-57 (Higham via SVD, then eigen-shift loop with spacing(norm(A)))."""
    b = (a + a.T) / 2
    _, s, v = la.svd(b)
    h = np.dot(v.T, np.dot(np.diag(s), v))
    a2 = (b + h) / 2
    a3 = (a2 + a2.T) / 2
    if is_pd(a3):
        return a3
    spacing = np.spacing(la.norm(a))
    eye = np.eye(a.shape[0])
    k = 1
    while not is_pd(a3):
        mineig = np.min(np.real(la.eigvals(a3)))
        a3 += eye * (-mineig * k ** 2 + spacing)
        k += 1
    return a3


def bingham_batch(b):
    """For a stack of dy x dy matrices: PD guard (Posteriors.py:519-523), eig sorted descending
    (CommonDensities.py:73-76), saddle-point constant from the unclamped eigenvalues (:77), stored
    kappa clamped at 0 (Posteriors.py:525-526).  Returns guarded B, kappa, axes, rho, logC, n_chol
    (the number of Cholesky factorisations performed, for the batched-Cholesky counter)."""
    b = np.array(b, dtype=np.float64)
    flat = b.reshape(-1, b.shape[-2], b.shape[-1])
    n_chol = 0
    for q in range(flat.shape[0]):
        n_chol += 1
        if not is_pd(flat[q]):
            flat[q] = nearest_pd(flat[q])
    w, v = la.eig(flat)
    w = np.real(w)
    v = np.real(v)
    idx = np.argsort(w, axis=-1)[:, ::-1]
    kappa = np.take_along_axis(w, idx, axis=-1)
    axes = np.take_along_axis(v, idx[:, None, :], axis=-1)
    logc, rho = log_partition_saddle(kappa)
    kappa = np.where(kappa < 0, 0., kappa)
    lead = b.shape[:-2]
    dy = b.shape[-1]
    return (flat.reshape(b.shape), kappa.reshape(lead + (dy,)), axes.reshape(b.shape),
            np.real(rho).reshape(lead + (dy,)), np.real(logc).reshape(lead), n_chol)


def axis_cov_from(rho, axes):
    """Stats.py:375-382 / :240-248: C = sum_d rho_d v_d v_d^T."""
    return np.einsum('...d,...ad,...bd->...ab', rho, axes, axes)


# ----------------------------------------------------------------------------------------------
# permutation-alignment weights   (Stats.py:390-445)
# ----------------------------------------------------------------------------------------------
def log_omega_hat(b_prime, logc_prime, shape_prime, scale_prime, axis_cov, ard_log_mean, ard_mean):
    """Stats.py:405-412 (a true matrix product inside the trace)."""
    tr = np.einsum('iab,kba->ik', axis_cov, b_prime)
    return (tr - logc_prime[None, :] + (shape_prime * np.log(scale_prime))[None, :]
            - gammaln(shape_prime)[None, :] + (shape_prime[None, :] - 1) * ard_log_mean[:, None]
            - scale_prime[None, :] * ard_mean[:, None])


def _omega_residual(ln_eta, ln_omega):
    """Stats.py:423-445, same equation order (row l, column l interleaved)."""
    m = ln_omega.shape[0]
    ln_alpha = ln_eta[:m]
    ln_beta = ln_eta[m:]
    rows = ln_alpha + logsumexp(ln_beta[None, :] + ln_omega, axis=1)
    cols = ln_beta + logsumexp(ln_alpha[:, None] + ln_omega, axis=0)
    out = np.empty(2 * m)
    out[0::2] = rows
    out[1::2] = cols
    return out


def omega_fsolve(lw):
    """Stats.py:413-420: MINPACK hybrd from zeros(2M), default xtol."""
    m = lw.shape[0]
    eta = fsolve(_omega_residual, np.zeros(2 * m), lw)
    return np.exp(eta[:m, None] + eta[None, m:] + lw)


def omega_sinkhorn(lw, tol=1e-14, max_iter=10000):
    """The exact solution the fsolve call approximates: diag(alpha) exp(lw) diag(beta) doubly
    stochastic (used to quantify the reference's own solver error, not part of the restatement)."""
    m = lw.shape[0]
    la_ = np.zeros(m)
    lb = np.zeros(m)
    for _ in range(max_iter):
        la_ = -logsumexp(lw + lb[None, :], axis=1)
        lb = -logsumexp(lw + la_[:, None], axis=0)
        p = np.exp(lw + la_[:, None] + lb[None, :])
        if np.max(np.abs(p.sum(1) - 1)) < tol:
            break
    return p


# ----------------------------------------------------------------------------------------------
# the model
# ----------------------------------------------------------------------------------------------
class _Layer(object):
    pass


class OracleMRGP(object):
    """State and sweeps of MultiResolutionGaussianProcess (MRGP.py:15-276 ctor, :571-724 sweeps),
    non-informative initialisation only (Priors.py; informative priors raise in the reference).

    mode 'ci' = shared Bingham axis / ARD chain (default reference flags), 'fi' = forced_independence.
    spectral = list of (nu, l, sf) per layer or None per layer (MRGP.py:325-335 -> ones).
    adaptive = None or dict(use_prior=True, opt_interval_factor=(lo, hi)) (BasisInterval.py:8).
    """

    def __init__(self, x, y, n_basis, offsets, mode='ci', spectral=(1., 1., 1.), interval_factor=1.,
                 standard_normalized_inputs=True, noise_region_specific=True, bias_region_specific=True,
                 snr_ratio=None, full_x=None, adaptive=None, omega_solver='fsolve'):
        x = np.asarray(x, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        self.mode = mode
        self.M = int(n_basis)
        self.dy = y.shape[1]
        if self.dy < 2:
            raise ValueError('output dimension must be greater than 1')  # MRGP.py:65-66
        self.N = x.shape[0]
        self.J = len(offsets)
        self.offsets = [np.asarray(o, dtype=np.int64) for o in offsets]
        self.noise_region_specific = noise_region_specific
        self.bias_region_specific = bias_region_specific
        self.omega_solver = omega_solver
        self.adaptive = None if mode == 'fi' else adaptive  # MRGP.py:108-109
        self.n_chol = 0
        self.t_omega = 0.0   # seconds spent in the permutation-weight solver (bench.py reports it)
        # MRGP.py:278-295
        ref = x if full_x is None else np.asarray(full_x, dtype=np.float64)
        if standard_normalized_inputs:
            self.std_x = np.std(ref, 0)
            self.std_x[self.std_x == 0] = 1
            self.mean_x = np.mean(ref, 0)
            x = (x - self.mean_x) / self.std_x
        else:
            self.mean_x = None
            self.std_x = None
        self.x = x
        self.y = y
        self.dx = x.shape[1]
        if isinstance(spectral, tuple) or spectral is None:
            spectral = [spectral] * self.J
        self.spectral = list(spectral)
        if not isinstance(interval_factor, (list, tuple)):
            interval_factor = [interval_factor] * self.J
        sf = [1. if s is None else s[2] for s in self.spectral]  # MRGP.py:174-179
        M, dy = self.M, self.dy

        self.layers = []
        for j in range(self.J):
            ly = _Layer()
            off = self.offsets[j]
            R = len(off) - 1
            ly.off = off
            ly.R = R
            ly.n = np.diff(off).astype(np.float64)
            # BasisInterval.py:15-16 via MRGP.py:144-149
            ly.L = interval_factor[j] * np.maximum.reduceat(np.abs(x), off[:-1], axis=0)
            self._rebuild_basis(ly, j)
            # Priors.py:74-78, 103-109, 132-135; MRGP.py:195-203 (snr only at layer 0)
            noise_var = 1.
            if j == 0 and snr_ratio is not None:
                y_var = (la.norm(y) ** 2) / self.N - np.dot(np.mean(y, axis=0), np.mean(y, axis=0))  # :966-971
                noise_var = y_var / snr_ratio
            ly.noise_shape0 = np.full(R, EPSILON)
            ly.noise_scale0 = np.full(R, (EPSILON + 1) * noise_var)
            ly.bias_mean0 = np.zeros((R, dy))
            ly.bias_prec0 = np.full(R, EPSILON)
            # Posteriors.py:17-25
            ly.scale_precision = 1. / ly.S
            ly.zeta = np.zeros((R, M))
            ly.ytil = np.zeros((R, dy, M))
            ly.noise_shape = ly.noise_shape0.copy()
            ly.noise_scale = ly.noise_scale0.copy()
            ly.bias_mean_q = ly.bias_mean0.copy()
            ly.bias_prec = ly.bias_prec0.copy()
            # Stats.py:22-49, 57-62
            ly.A = np.zeros((R, dy, M))
            ly.m2 = np.zeros((R, M))
            ly.cm2 = np.zeros((R, M))
            ly.noise_mean = ly.noise_shape / ly.noise_scale
            ly.noise_log_mean = psi(ly.noise_shape) - np.log(ly.noise_scale)
            ly.bias_mean = ly.bias_mean_q.copy()
            ly.bias_var = 1. / ly.bias_prec
            ly.fbar = np.zeros((self.N, dy))
            ly.fvar = np.zeros(self.N)
            ly.y_target = None
            ly.y_var = np.zeros(R)
            if mode == 'fi':
                # Priors.py:168-189, 205-210; Posteriors.py:220-227; Stats.py:170-185
                logc0, rho0 = log_partition_saddle(np.zeros(dy))
                ly.B0 = np.zeros((R, M, dy, dy))
                ly.logC0 = np.full((R, M), float(logc0))
                ly.ard_shape0 = np.full((R, M), EPSILON)
                ly.ard_scale0 = ly.ard_shape0 / np.mean(sf)
                ly.B = ly.B0.copy()
                ly.kappa = np.zeros((R, M, dy))
                ly.rho = np.tile(rho0, (R, M, 1))
                ly.axes = np.tile(np.eye(dy), (R, M, 1, 1))
                ly.logC = ly.logC0.copy()
                ly.ard_shape = ly.ard_shape0.copy()
                ly.ard_scale = ly.ard_scale0.copy()
                ly.axis_cov = np.zeros((R, M, dy, dy))
                ly.ard_mean = ly.ard_shape / ly.ard_scale
                ly.ard_log_mean = psi(ly.ard_shape) - np.log(ly.ard_scale)
            self.layers.append(ly)

        if mode == 'ci':
            # Priors.py:29-36, 51-53; Posteriors.py:483-491; Stats.py:361-369
            sh = _Layer()
            logc0, rho0 = log_partition_saddle(np.zeros(dy))
            sh.B0 = np.zeros((M, dy, dy))
            sh.logC0 = np.full(M, float(logc0))
            sh.ard_shape0 = np.full(M, EPSILON)
            sh.ard_scale0 = sh.ard_shape0 / np.mean(sf)
            sh.B = sh.B0.copy()
            sh.kappa = np.zeros((M, dy))
            sh.rho = np.tile(rho0, (M, 1))
            sh.axes = np.tile(np.eye(dy), (M, 1, 1))
            sh.logC = sh.logC0.copy()
            sh.ard_shape = sh.ard_shape0.copy()
            sh.ard_scale = sh.ard_scale0.copy()
            sh.axis_cov = np.zeros((M, dy, dy))
            sh.ard_mean = sh.ard_shape / sh.ard_scale
            sh.ard_log_mean = psi(sh.ard_shape) - np.log(sh.ard_scale)
            sh.omega = np.ones((M, M)) / M
            self.shared = sh
        self.lower_bound = []
        self.lower_bound_layer = [[] for _ in range(self.J)]
        self.lower_bound_terms = []

    # ------------------------------------------------------------------------------------------
    def _rebuild_basis(self, ly, j):
        """MRGP.py:305-357 (_update_basis_functions, _update_spectral_density)."""
        ly.Lx = seg_expand(ly.L, ly.off)
        ly.Phi = eigenfunctions(self.x, ly.Lx, self.M)
        ly.lam = eigenvalues(ly.L, self.M)
        if self.spectral[j] is None:
            ly.S = np.ones((ly.R, self.M))
        else:
            nu, l, sf = self.spectral[j]
            ly.S = matern_spectral(np.sqrt(ly.lam), nu, l, sf)
        ly.d = seg_sum(ly.Phi * ly.Phi, ly.off)  # sum_n Phi^2, Posteriors.py:41

    def _region_vals(self, ly, v):
        return seg_expand(v, ly.off)

    def _mean_function(self, ly, A=None):
        """sum_i Phi[:, i] a_i per sample with the sample's own region coefficients."""
        A = ly.A if A is None else A
        return np.einsum('ni,ndi->nd', ly.Phi, seg_expand(A, ly.off))

    # ------------------------------------------------------------------------------------------
    def sweep(self):
        if self.mode == 'ci':
            self._sweep_ci()
        else:
            self._sweep_fi()

    def _targets(self, ly, j):
        if j == 0 or self.mode == 'fi':
            # LatentOutputs.py:6-18
            return self.y, np.zeros(ly.R)
        # LatentOutputs.py:25-49 with the OLD A, b, noise
        e = self._mean_function(ly)
        y = e + (self._region_vals(ly, ly.bias_mean) + ly.fbar)
        return y, 1. / ly.noise_mean

    def _scale_given_axis(self, ly, y, ard_mean):
        """Posteriors.py:35-78 / :298-342.  ard_mean (M,) shared or (R, M) per region."""
        ly.scale_precision = ard_mean / ly.S + ly.noise_mean[:, None] * ly.d
        ly.zeta = ly.noise_mean[:, None] / ly.scale_precision
        e = self._mean_function(ly)
        base = y - (ly.fbar + self._region_vals(ly, ly.bias_mean))
        a_s = seg_expand(ly.A, ly.off)  # (N, dy, M)
        ytil = np.empty((ly.R, self.dy, self.M))
        for i in range(self.M):
            pen = e - ly.Phi[:, i:i + 1] * a_s[:, :, i]  # sum_{k != i}
            ytil[:, :, i] = seg_sum(ly.Phi[:, i:i + 1] * (base - pen), ly.off)
        ly.ytil = ytil

    def _scale_stats(self, ly, axis_cov):
        """Stats.py:67-100 / :257-290.  axis_cov (M, dy, dy) or (R, M, dy, dy)."""
        C = np.broadcast_to(axis_cov, (ly.R, self.M, self.dy, self.dy))
        yt = np.swapaxes(ly.ytil, 1, 2)  # (R, M, dy)
        Cy = np.einsum('rmab,rmb->rma', C, yt)
        ly.A = np.swapaxes(ly.zeta[:, :, None] * Cy, 1, 2)
        z2 = ly.zeta ** 2
        ly.m2 = 1. / ly.scale_precision + z2 * np.einsum('rma,rma->rm', yt, Cy)
        CC = C - np.einsum('rmab,rmbc->rmac', C, C)
        ly.cm2 = 1. / ly.scale_precision + z2 * np.einsum('rma,rmab,rmb->rm', yt, CC, yt)

    def _bias_noise(self, ly, y, y_var):
        """Posteriors.py:81-211 (bias, then the four noise variants), Stats.py:102-124."""
        e = self._mean_function(ly)
        r = y - e - ly.fbar
        sum_r = seg_sum(r, ly.off)
        mean_term = seg_sum(np.sum(r * r, axis=1), ly.off)
        var_f = seg_sum(ly.fvar, ly.off)
        var_au = seg_sum(np.sum((ly.Phi ** 2) * seg_expand(ly.cm2, ly.off), axis=1), ly.off)
        ly.sum_r, ly.mean_term, ly.var_f, ly.var_au = sum_r, mean_term, var_f, var_au
        dy = self.dy
        if self.bias_region_specific:
            ly.bias_prec = ly.bias_prec0 + ly.n
            ly.bias_mean_q = (ly.bias_mean0 * ly.bias_prec0[:, None] + sum_r) / ly.bias_prec[:, None]
            term3 = ly.bias_prec0 * np.sum(ly.bias_mean0 ** 2, axis=1)
            term4 = ly.bias_prec * np.sum(ly.bias_mean_q ** 2, axis=1)
        else:
            prec = ly.bias_prec0[0] + np.sum(ly.n)
            mean = (ly.bias_mean0[0] * ly.bias_prec0[0] + np.sum(sum_r, axis=0)) / prec
            ly.bias_prec = np.full(ly.R, prec)
            ly.bias_mean_q = np.tile(mean, (ly.R, 1))
            term3 = np.full(ly.R, ly.bias_prec0[0] * np.sum(ly.bias_mean0[0] ** 2))
            term4 = np.full(ly.R, prec * np.sum(mean ** 2))
        ci = self.mode == 'ci'
        if self.noise_region_specific:
            # y_var is NOT multiplied by n at Posteriors.py:138 (ci, regional bias) and :422 (fi, shared
            # bias); it is at :158 (ci, shared bias) and :402 (fi, regional bias).
            times_n = (ci and not self.bias_region_specific) or ((not ci) and self.bias_region_specific)
            yv = y_var * ly.n if times_n else y_var
            ly.noise_shape = ly.noise_shape0 + 0.5 * dy * ly.n
            ly.noise_scale = ly.noise_scale0 + 0.5 * (term3 - term4 + mean_term + var_f + var_au + yv)
        else:
            yv = y_var * ly.n
            if self.bias_region_specific:
                upd = np.sum(0.5 * (term3 - term4 + mean_term + var_f + var_au + yv))  # :168-187
            else:
                upd = 0.5 * (term3[0] - term4[0] + np.sum(mean_term) + np.sum(var_f) + np.sum(var_au)
                             + np.sum(yv))  # :189-211
            ly.noise_shape = np.full(ly.R, ly.noise_shape0[0] + np.sum(0.5 * dy * ly.n))
            ly.noise_scale = np.full(ly.R, ly.noise_scale0[0] + upd)
        ly.bias_mean = ly.bias_mean_q.copy()
        ly.bias_var = 1. / ly.bias_prec
        ly.noise_mean = ly.noise_shape / ly.noise_scale
        ly.noise_log_mean = psi(ly.noise_shape) - np.log(ly.noise_scale)

    def _propagate(self, j):
        """Stats.py:126-157 as a running prefix: contributions of layers < j do not change between
        their own step and step j of a sweep, so fbar^{j+1} = fbar^j + b_j + Phi_j A_j^T reproduces the
        reference's jp = 0, 1, ... summation order (SURVEY.md App. A)."""
        ly = self.layers[j]
        nxt = self.layers[j + 1]
        contrib_mean = self._region_vals(ly, ly.bias_mean) + self._mean_function(ly)
        contrib_var = self._region_vals(ly, ly.bias_var) + \
            np.sum((ly.Phi ** 2) * seg_expand(ly.cm2, ly.off), axis=1)
        nxt.fbar = ly.fbar + contrib_mean
        nxt.fvar = ly.fvar + contrib_var

    def _sweep_ci(self):
        """MRGP.py:571-652."""
        sh = self.shared
        M, dy = self.M, self.dy
        for j in range(self.J):
            ly = self.layers[j]
            if j == 0:
                pB, pLogC, pShape, pScale = sh.B0, sh.logC0, sh.ard_shape0, sh.ard_scale0  # :575
            else:
                pB, pLogC, pShape, pScale = sh.B.copy(), sh.logC.copy(), sh.ard_shape.copy(), \
                    sh.ard_scale.copy()  # :581
            y, y_var = self._targets(ly, j)
            self._scale_given_axis(ly, y, sh.ard_mean)
            # Posteriors.py:497-530
            w = 0.5 * ly.noise_mean[:, None] * ly.zeta  # (R, M)
            data = np.einsum('rm,ram,rbm->mab', w, ly.ytil, ly.ytil)
            b = np.einsum('ik,kab->iab', sh.omega, pB) + data
            sh.B, sh.kappa, sh.axes, sh.rho, sh.logC, nch = bingham_batch(b)
            self.n_chol += nch
            sh.axis_cov = axis_cov_from(sh.rho, sh.axes)
            self._scale_stats(ly, sh.axis_cov)
            # Posteriors.py:533-541, Stats.py:385-388
            sh.ard_shape = sh.omega @ pShape + 0.5 * ly.R
            sh.ard_scale = sh.omega @ pScale + 0.5 * np.sum(ly.m2 / ly.S, axis=0)
            sh.ard_mean = sh.ard_shape / sh.ard_scale
            sh.ard_log_mean = psi(sh.ard_shape) - np.log(sh.ard_scale)
            # Stats.py:390-420
            lw = log_omega_hat(pB, pLogC, pShape, pScale, sh.axis_cov, sh.ard_log_mean, sh.ard_mean)
            sh.log_omega_hat = lw
            _t0 = time.perf_counter()
            sh.omega = omega_fsolve(lw) if self.omega_solver == 'fsolve' else omega_sinkhorn(lw)
            self.t_omega += time.perf_counter() - _t0
            self._bias_noise(ly, y, y_var)
            if self.adaptive is not None:
                self._learn_intervals(ly, j, y, sh.ard_mean)  # MRGP.py:632-641
            if j + 1 < self.J:
                self._propagate(j)
            ly.y_target = y  # :650-652
            ly.y_var = y_var

    def _sweep_fi(self):
        """MRGP.py:654-724."""
        M = self.M
        for j in range(self.J):
            ly = self.layers[j]
            y, y_var = self._targets(ly, j)
            self._scale_given_axis(ly, y, ly.ard_mean)
            # Posteriors.py:253-285: prior B is the untouched zero prior, omega == 1/M
            w = 0.5 * ly.noise_mean[:, None] * ly.zeta
            data = np.einsum('rm,ram,rbm->rmab', w, ly.ytil, ly.ytil)
            b = np.sum((1. / M) * ly.B0, axis=1, keepdims=True) + data
            ly.B, ly.kappa, ly.axes, ly.rho, ly.logC, nch = bingham_batch(b)
            self.n_chol += nch
            ly.axis_cov = axis_cov_from(ly.rho, ly.axes)
            self._scale_stats(ly, ly.axis_cov)
            # Posteriors.py:288-295 (0.5 * n_regions of the layer, per region), Stats.py:251-255
            ly.ard_shape = np.sum((1. / M) * ly.ard_shape0, axis=1, keepdims=True) + 0.5 * ly.R + 0 * ly.m2
            ly.ard_scale = np.sum((1. / M) * ly.ard_scale0, axis=1, keepdims=True) + 0.5 * ly.m2 / ly.S
            ly.ard_mean = ly.ard_shape / ly.ard_scale
            ly.ard_log_mean = psi(ly.ard_shape) - np.log(ly.ard_scale)
            self._bias_noise(ly, y, y_var)
            if j + 1 < self.J:
                self._propagate(j)
            ly.y_target = y
            ly.y_var = y_var

    # ------------------------------------------------------------------------------------------
    def _interval_objective(self, L, xr, yr, noise_mean, ard_mean, m2, A, cm2, bias_mean, fbar, j):
        """BasisInterval.py:94-134 for dx == 1 (phi_penalty == 1, lambda_penalty == 0)."""
        Lx = np.full((xr.shape[0], 1), L)
        phi = eigenfunctions(xr, Lx, self.M)
        lam = eigenvalues(np.array([[L]]), self.M)[0]
        use_prior = self.adaptive.get('use_prior', True)
        if use_prior:
            nu, l, sf = self.spectral[j]
            S = matern_spectral(np.sqrt(lam + 0.), nu, l, sf)
        p2 = np.sum(phi ** 2, axis=0)  # (M,)
        term1 = np.sum(A ** 2, axis=0) * p2
        term2 = np.einsum('ni,nd,di->i', phi, bias_mean + fbar, A)
        term3 = np.einsum('ni,nd,di->i', phi, yr, A)
        term4 = cm2 * p2
        ll = -0.5 * noise_mean * np.sum(2 * term1 + 4 * term2 - 2 * term3 + term4)
        if not use_prior:
            return -ll
        prior = -0.5 * np.sum(np.log(S) - 0.5 * (ard_mean * m2) / S)
        return -(ll + prior)

    def _learn_intervals(self, ly, j, y, ard_mean):
        """BasisInterval.py:18-90 then MRGP.py:640-641.  dx == 1 only."""
        if self.dx != 1:
            raise NotImplementedError('oracle adaptive intervals: dx == 1 only')
        lo_f, hi_f = self.adaptive.get('opt_interval_factor', (1., 1.2))
        for r in range(ly.R):
            s, e = ly.off[r], ly.off[r + 1]
            xr = self.x[s:e]
            low = np.max(np.abs(xr)) * lo_f
            high = min(self.M, low * hi_f)
            if high < low:
                high = low * hi_f
            ly.L[r, 0] = fminbound(self._interval_objective, low, high,
                                   args=(xr, y[s:e], ly.noise_mean[r], ard_mean, ly.m2[r], ly.A[r],
                                         ly.cm2[r], ly.bias_mean[r], ly.fbar[s:e], j), full_output=0)
        self._rebuild_basis(ly, j)

    # ------------------------------------------------------------------------------------------
    def elbo(self):
        """MRGP.py:414-569 with prime == the current shared posterior for j > 0 (alias at :379) and
        the shared prior for j == 0.  ci only.  Returns total, per-layer list, (J, 6) terms in the
        order data, scale|axis, axis, ard, bias, noise."""
        sh = self.shared
        M, dy = self.M, self.dy
        terms = np.zeros((self.J, 6))
        for j, ly in enumerate(self.layers):
            if j == 0:
                pB, pLogC, pShape, pScale = sh.B0, sh.logC0, sh.ard_shape0, sh.ard_scale0
            else:
                pB, pLogC, pShape, pScale = sh.B, sh.logC, sh.ard_shape, sh.ard_scale
            # :535-569
            e = self._mean_function(ly)
            r = ly.y_target - e - ly.fbar - self._region_vals(ly, ly.bias_mean)
            mean_term = seg_sum(np.sum(r * r, axis=1), ly.off)
            var_f = seg_sum(ly.fvar, ly.off)
            var_au = seg_sum(np.sum((ly.Phi ** 2) * seg_expand(ly.cm2, ly.off), axis=1), ly.off)
            terms[j, 0] = np.sum(mean_term + var_f + var_au + ly.bias_var + ly.y_var * ly.n) + \
                np.sum(0.5 * dy * (ly.noise_log_mean - np.log(2 * np.pi)) * ly.n)
            # :520-533
            terms[j, 1] = np.sum(0.5 * sh.ard_log_mean / ly.S - 0.5 * sh.ard_mean * ly.m2 / ly.S) - \
                np.sum(0.5 * np.log(ly.scale_precision) - .5)
            # :499-518 (element-wise product inside the trace)
            diagC = np.einsum('iaa->ia', sh.axis_cov)
            log_term = -pLogC[None, :] + np.einsum('ia,ka->ik', diagC, np.einsum('kaa->ka', pB))
            log_q = np.sum(-sh.logC + np.einsum('ia,ia->i', diagC, np.einsum('iaa->ia', sh.B)))
            terms[j, 2] = np.sum(sh.omega * log_term) - log_q
            # :477-497
            lt = (pShape * np.log(pScale) - gammaln(pShape))[None, :] + \
                (pShape[None, :] - 1) * sh.ard_log_mean[:, None] - pScale[None, :] * sh.ard_mean[:, None]
            lq = np.sum(sh.ard_shape * np.log(sh.ard_scale) - gammaln(sh.ard_shape) +
                        (sh.ard_shape - 1) * sh.ard_log_mean - sh.ard_scale * sh.ard_mean)
            terms[j, 3] = np.sum(sh.omega * lt) - lq
            # :449-475
            w, tau = ly.bias_mean_q, ly.bias_prec
            w0, tau0 = ly.bias_mean0, ly.bias_prec0
            const = 0.5 * dy * (np.log(tau0) + ly.noise_log_mean - np.log(2 * np.pi))
            term1 = 1. / (tau * ly.noise_mean) + np.sum(w * w, 1) - 2 * np.sum(w * w0, 1) + np.sum(w0 * w0, 1)
            log_p = np.sum(const + 0.5 * tau0 * ly.noise_mean * term1)
            log_q = np.sum(0.5 * dy * (np.log(tau) + ly.noise_log_mean - np.log(2 * np.pi)) - 0.5)
            terms[j, 4] = log_p - log_q
            # :426-447
            c0, d0, c, d = ly.noise_shape0, ly.noise_scale0, ly.noise_shape, ly.noise_scale
            log_p = np.sum(c0 * np.log(d0) - gammaln(c0) + (c0 - 1) * ly.noise_log_mean - d0 * ly.noise_mean)
            log_q = np.sum(c * np.log(d) - gammaln(c) + (c - 1) * ly.noise_log_mean - d * ly.noise_mean)
            terms[j, 5] = log_p - log_q
        per_layer = list(np.sum(terms, axis=1))
        return float(np.sum(per_layer)), per_layer, terms

    def fit(self, n_iter=1, tol=1e-3, min_iter=10):
        """MRGP.py:367-412."""
        if tol is None or self.mode == 'fi':
            for _ in range(n_iter):
                self.sweep()
            return
        if n_iter < min_iter:
            min_iter = n_iter
        for it in range(1, n_iter + 1):
            self.sweep()
            total, per_layer, terms = self.elbo()
            self.lower_bound.append(total)
            self.lower_bound_terms.append(terms)
            for j in range(self.J):
                self.lower_bound_layer[j].append(per_layer[j])
            if it > min_iter:
                if abs(self.lower_bound_layer[0][-1] - self.lower_bound_layer[0][-2]) < abs(tol):
                    break

    # ------------------------------------------------------------------------------------------
    def _norm_test(self, test_x):
        test_x = np.asarray(test_x, dtype=np.float64)
        if self.mean_x is not None:
            test_x = (test_x - self.mean_x) / self.std_x  # MRGP.py:806-808
        return test_x

    def predict_mean(self, test_x, test_offsets=None):
        """MRGP.py:726-814.  Without an index set: layer 0, region 0 only.  With test offsets (same
        region counts per layer; points assigned to regions by array position): sum over layers."""
        xt = self._norm_test(test_x)
        if test_offsets is None:
            ly = self.layers[0]
            phi = eigenfunctions(xt, np.tile(ly.L[0], (xt.shape[0], 1)), self.M)
            return phi @ ly.A[0].T + ly.bias_mean[0]
        out = np.zeros((xt.shape[0], self.dy))
        for j, off in enumerate(test_offsets):
            ly = self.layers[j]
            phi = eigenfunctions(xt, seg_expand(ly.L, off), self.M)
            out += np.einsum('ni,ndi->nd', phi, seg_expand(ly.A, off)) + seg_expand(ly.bias_mean, off)
        return out

    def predict_var(self, test_x):
        """MRGP.py:833-861 (no index set): sum_i cm2_i phi_i^2 + bias_var at layer 0, region 0."""
        xt = self._norm_test(test_x)
        ly = self.layers[0]
        phi = eigenfunctions(xt, np.tile(ly.L[0], (xt.shape[0], 1)), self.M)
        return (phi ** 2) @ ly.cm2[0] + ly.bias_var[0]

    def predict_var_indexed(self, test_x, test_offsets):
        """MRGP.py:863-932 (index-set form of the second moment): per test point the sum over ALL layers j of
        sum_i phi_i^2 cm2_i + bias_var + n_test(region) / noise_mean + f_var_j(first test point of the region), where
        f_var_j is the latent variance of the layers < j (Stats.py:126-157) and the reference adds its value at the
        region's FIRST test point, `latent_f_var[l][0]`, to every point of the region (:929).  Test points are assigned
        to regions by position.  A region without test points contributes nothing (the reference cannot index its
        first point); every point lies in a non-empty region, so the result is defined for every point."""
        xt = self._norm_test(test_x)
        if len(test_offsets) != self.J:
            raise ValueError('the test index set must have the resolutions of the training index set')
        n = xt.shape[0]
        out = np.zeros(n)
        fvar = np.zeros(n)   # latent variance of the layers below the current one, per test point
        for j, off in enumerate(test_offsets):
            ly = self.layers[j]
            off = np.asarray(off, dtype=np.int64)
            cnt = np.diff(off)
            phi = eigenfunctions(xt, seg_expand(ly.L, off), self.M)
            contrib = np.sum((phi ** 2) * seg_expand(ly.cm2, off), axis=1) + seg_expand(ly.bias_var, off)
            first = np.zeros(ly.R)
            full = cnt > 0
            first[full] = fvar[off[:-1][full]]
            out += contrib + seg_expand(cnt / ly.noise_mean + first, off)
            fvar = fvar + contrib
        return out

    def test_likelihood(self, test, test_offsets=None):
        """MRGP.py:825-831: mean over the test points of the Gaussian log density of ||y - mean|| with variance var
        (index-set forms of both when test_offsets is given)."""
        test_x, test_y = test[0], np.asarray(test[1], dtype=np.float64)
        mf = self.predict_mean(test_x, test_offsets)
        vf = self.predict_var(test_x) if test_offsets is None else self.predict_var_indexed(test_x, test_offsets)
        ll = -0.5 * np.log(2 * np.pi * vf) - 0.5 * (la.norm(test_y - mf, axis=1) ** 2) / vf
        return float(np.mean(ll))

    # ------------------------------------------------------------------------------------------
    def state(self):
        """Flat dict of every state array, the comparison surface for parity tests."""
        out = {}
        for j, ly in enumerate(self.layers):
            p = 'L%d.' % j
            for name in ('L', 'lam', 'S', 'd', 'scale_precision', 'zeta', 'ytil', 'A', 'm2', 'cm2',
                         'noise_shape', 'noise_scale', 'noise_mean', 'noise_log_mean', 'bias_prec',
                         'bias_mean', 'bias_var', 'fbar', 'fvar'):
                out[p + name] = np.array(getattr(ly, name))
            if self.mode == 'fi':
                for name in ('B', 'kappa', 'rho', 'logC', 'axis_cov', 'ard_shape', 'ard_scale',
                             'ard_mean', 'ard_log_mean'):
                    out[p + name] = np.array(getattr(ly, name))
        if self.mode == 'ci':
            for name in ('B', 'kappa', 'rho', 'logC', 'axis_cov', 'ard_shape', 'ard_scale', 'ard_mean',
                         'ard_log_mean', 'omega'):
                out['S.' + name] = np.array(getattr(self.shared, name))
        return out
