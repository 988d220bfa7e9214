"""MultiResolutionGaussianProcess: drop-in for the reference's src/MRGP.py API (constructor, fit, predict,
public state) with the variational-inference sweep running on one B200 through libcimrgp.so.

Same constructor arguments, same exceptions for the same misuse (MRGP.py:37-126), same meaning of every
method.  `adaptive_inputs=True` without an `input_model` fits the input-warp GP of cimrgp_b200/RegressionInput.py (a
restatement of the reference's GPy call, Inputs.py:20-47; parity unpinned: GPy is absent).  What is NOT carried over
(raises NotImplementedError with the reason): dx > 1 and dy > 2 on the device.
"""
import numpy as np

from . import _lib
from .BasisInterval import BasisInterval
from .IndexSetGenerator import offsets_of
from .KernelClass import LaplacianEigenpairs, MaternKernel
from .engine import Engine


class _View(object):
    """Read-only, lazily materialised mirror of a reference state object."""

    def __init__(self, model, getters, consts):
        self.__dict__['_model'] = model
        self.__dict__['_getters'] = getters
        self.__dict__.update(consts)

    def __getattr__(self, name):
        g = self.__dict__['_getters'].get(name)
        if g is None:
            raise AttributeError(name)
        return g()


class MultiResolutionGaussianProcess(object):
    def __init__(self, train_xy,
                 n_basis,
                 index_set_obj,
                 basis_function_obj,
                 spectral_density_obj=None,
                 basis_interval_obj=None,
                 interval_factor=1,
                 adaptive_inputs=False,
                 standard_normalized_inputs=True,
                 axis_resolution_specific=False,
                 ard_resolution_specific=False,
                 noise_region_specific=True,
                 bias_region_specific=True,
                 noninformative_initialization=True,
                 snr_ratio=None,
                 full_x=None,
                 input_model=None,
                 forced_independence=False,
                 verbose=False,
                 device=0,
                 n_ctas=0,
                 distributed=False,
                 _engine_opts=None):
        self.verbose = verbose
        self.forced_independence = forced_independence
        # MRGP.py:38-50
        if forced_independence is True:
            self.axis_resolution_specific = True
            self.ard_resolution_specific = True
            if self.verbose is True:
                print("*** All GPs are forced to be independent *** ")
        else:
            if (axis_resolution_specific is False) and (ard_resolution_specific is False):
                self.axis_resolution_specific = False
                self.ard_resolution_specific = False
                if self.verbose is True:
                    print(" \n *** GPs are conditionally independent given the basis axes *** \n ")
            else:
                raise TypeError("not yet supported")
        self.adaptive_inputs = adaptive_inputs
        self.standard_normalized_inputs = standard_normalized_inputs
        self.noise_region_specific = noise_region_specific
        self.bias_region_specific = bias_region_specific
        self.n_layers = index_set_obj.get_n_resolutions() + 1
        self.index_set_obj = index_set_obj
        self.n_basis = n_basis
        x_train = np.asarray(train_xy[0], dtype=np.float64)
        y_train = np.asarray(train_xy[1], dtype=np.float64)
        self.observations = y_train
        self.dy = y_train.shape[1]
        if self.dy < 2:
            raise ValueError('output dimension must be greater than 1')   # MRGP.py:65-66
        if noninformative_initialization is not True:
            raise ValueError('not yet implemented...')                       # Priors.py:27, 49, 80
        x_train, self.full_x, self.mean_x_train, self.std_x_train = self._normalize_inputs(x_train, full_x)

        def per_layer(value, what):
            # MRGP.py:71-106
            if isinstance(value, list) is False:
                return [value] * self.n_layers
            if len(value) != self.n_layers:
                raise ValueError(what + ' must be a list of the same length as the number of resolutions + 1')
            return value
        self.spectral_density_obj = per_layer(spectral_density_obj, 'spectral_density_obj')
        self.basis_function_obj = per_layer(basis_function_obj, 'basis_function_obj')
        self.use_prior = [s is not None for s in self.spectral_density_obj]
        self.interval_factor = per_layer(interval_factor, 'interval_factor')
        if forced_independence is True:
            basis_interval_obj = None                                        # MRGP.py:108-109
        if basis_interval_obj is None:
            self.adaptive_basis_intervals = False
            self.basis_interval_obj = [BasisInterval() for _ in range(self.n_layers)]
        else:
            self.adaptive_basis_intervals = True                             # MRGP.py:110-124
            self.basis_interval_obj = per_layer(basis_interval_obj, 'basis_interval_obj')
            if distributed:
                raise NotImplementedError('adaptive basis intervals are not available on the sample-sharded path')
        for b in self.basis_function_obj:
            if getattr(b, 'name', None) != 'Laplacian':
                raise TypeError('the device path implements the Laplacian eigenfunction basis only')
        # Inputs.py:8-55
        if self.adaptive_inputs is True:
            z = np.atleast_2d(np.linspace(start=np.min(x_train), stop=np.max(x_train), num=x_train.shape[0])).T
            self.input_z = z if self.full_x is None else np.atleast_2d(
                np.linspace(start=np.min(self.full_x), stop=np.max(self.full_x), num=self.full_x.shape[0])).T
            if input_model is None:      # Inputs.py:20-47: the warp x -> z as an exact RBF GP on at most 3000 points
                input_model = self._learn_input_model(x_train if self.full_x is None else self.full_x, self.input_z, device)
            self.input_model = input_model
            x_used = z
        else:
            self.input_model = None
            x_used = x_train
        self._x_used = x_used
        self.dx = x_used.shape[1]
        self._offsets = offsets_of(index_set_obj)
        if int(self._offsets[0][-1]) != x_used.shape[0]:
            raise ValueError('index set does not cover the training samples')
        self.n_regions = [len(o) - 1 for o in self._offsets]
        self.n_samps = [list(np.diff(o).astype(int)) for o in self._offsets]
        sf = [1. if s is None else s.sf for s in self.spectral_density_obj]          # MRGP.py:174-179
        noise_var0 = 1.0
        if snr_ratio is not None:
            noise_var0 = self._compute_initial_noise_var_from_snr(y=y_train, snr_ratio=snr_ratio)
        spectral, host_spectral = [], []
        for s in self.spectral_density_obj:
            if s is None:
                spectral.append(None)
                host_spectral.append(None)
            elif isinstance(s, MaternKernel) or all(hasattr(s, a) for a in ('nu', 'l', 'sf')) and \
                    getattr(s, 'name', '') == 'Matern':
                spectral.append((s.nu, s.l, s.sf))
                host_spectral.append(None)
            else:
                spectral.append((1., 1., 1.))
                host_spectral.append(s)       # any object with .spectral(s): evaluated on the host, uploaded
        engine_kw = dict(mode='fi' if forced_independence else 'ci',
                         spectral=spectral, interval_factor=[float(f) for f in self.interval_factor],
                         noise_var0=noise_var0, ard_prior_influence=float(np.mean(sf)),
                         noise_region_specific=noise_region_specific, bias_region_specific=bias_region_specific,
                         device=device, n_ctas=n_ctas)
        if _engine_opts:
            engine_kw.update(_engine_opts)      # shared stream / workspace slice / pinned staging (cimrgp_b200/batch.py)
        if distributed:
            # one process per GPU (torch.distributed initialised by the caller): this rank keeps its chunk of
            # the samples, the region statistics are summed over the ranks by the peer exchange, the model state is
            # replicated on every rank
            import torch.distributed as dist
            from .distributed import ShardedEngine
            self._engine = ShardedEngine(x_used, y_train, self._offsets, n_basis, dist.get_rank(),
                                         dist.get_world_size(), **engine_kw)
        else:
            self._engine = Engine(x_used, y_train, self._offsets, n_basis, **engine_kw)
        if any(s is not None for s in host_spectral):
            eng = self._engine
            for j, s in enumerate(host_spectral):
                if s is not None:
                    lam = eng.get(j, _lib.F_LAMBDA, (self.n_regions[j], n_basis))
                    eng.put(j, _lib.F_SPECTRAL, np.vectorize(lambda v: s.spectral(np.sqrt(v)))(lam))
            eng._ck(eng.lib.mrgp_init_state(eng.handle, float(noise_var0), float(np.mean(sf))))
        if self.adaptive_basis_intervals:
            if self.dx != 1:
                raise NotImplementedError('adaptive basis intervals: one input dimension on the device path')
            for j, (b, s) in enumerate(zip(self.basis_interval_obj, host_spectral)):
                if s is not None and b.use_prior:
                    raise NotImplementedError('adaptive basis intervals with use_prior need the Matern spectral '
                                              'density on the device (custom spectral objects are host-evaluated)')
                self._engine.set_adaptive_intervals(j, bool(b.use_prior), tuple(b.opt_interval_factor))
        self.lower_bound_layer = [[] for _ in range(self.n_layers)]
        self.lower_bound = []
        self.lower_bound_terms = []
        self._noise_var0 = noise_var0
        self._ard_prior_influence = float(np.mean(sf))
        self._sweeps = 0

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _learn_input_model(x, z, device):
        """Inputs.py:20-47 with the reference's calls on the global RNGs in the reference's order (random.uniform, then one
        numpy permutation per region, then one for the rest): one GP_RBF on all points up to 3000 of them, otherwise on a
        subsample of 3000 that holds one random point of every region of a uniform split."""
        import random
        from .IndexSetGenerator import IndexSetUniform
        from .RegressionInput import GP_RBF
        train_data = [np.asarray(x, dtype=np.float64), np.asarray(z, dtype=np.float64)]
        n_samps = train_data[0].shape[0]
        if n_samps < 3001:
            model = GP_RBF(device=device)
            model.fit(train_data)
            return model
        n_repeats, min_length = 1, 3000
        rate = random.uniform(.1, .2)
        factor = (1.0 if n_samps < 10000 else 1e-1 if n_samps < 100000 else 1e-2 if n_samps < 1000000 else 1e-3) * rate
        n_divide = int(np.floor(factor * n_samps))                     # Inputs.py:62-72
        index_set = IndexSetUniform(sample_length=n_samps, resolution=1, divider=n_divide).index_set[-1]
        ids_all = list(range(n_samps))
        models = []
        for _ in range(n_repeats):
            ids_l = [np.random.permutation(index_set[l])[0] for l in range(len(index_set))]
            rem_ids = np.delete(ids_all, ids_l)
            if min_length > len(ids_l):
                ids_rep = list(np.random.permutation(rem_ids)[0:min_length - len(ids_l)]) + ids_l
            else:
                ids_rep = ids_l
            ids = list(np.sort(np.unique(ids_rep)))
            model = GP_RBF(device=device)
            model.fit([train_data[0][ids, :], train_data[1][ids, :]])
            models.append(model)
        return models

    def _normalize_inputs(self, x_train, full_x):
        # MRGP.py:278-295
        x = x_train if full_x is None else np.asarray(full_x, dtype=np.float64)
        if self.standard_normalized_inputs is True:
            std_x_train = np.std(x, 0)
            std_x_train[std_x_train == 0] = 1
            mean_x_train = np.mean(x, 0)
            x_train = (x_train - np.full(x_train.shape, mean_x_train)) / np.full(x_train.shape, std_x_train)
            if full_x is not None:
                full_x = (x - np.full(x.shape, mean_x_train)) / np.full(x.shape, std_x_train)
        else:
            mean_x_train = None
            std_x_train = None
        return x_train, full_x, mean_x_train, std_x_train

    @staticmethod
    def _compute_initial_noise_var_from_snr(y, snr_ratio):
        # MRGP.py:966-971
        n_samps = y.shape[0]
        y_var = (np.linalg.norm(y) ** 2) / n_samps - np.dot(np.mean(y, axis=0), np.mean(y, axis=0))
        return y_var / snr_ratio

    # ------------------------------------------------------------------------------------------
    def omega_solve_report(self):
        """Evaluations of the permutation-weight solve (Stats.py:413-420) per layer in the last sweep (ci mode).  Warns when a
        layer used up its budget (the accelerated iteration and the 2000 plain Sinkhorn sweeps behind it) without reaching
        the tolerance 1e-10 on the column sums: the weights of that layer are then the last iterate, rows exact.  Tables of
        the model converge in 2-15 evaluations.  Such a model is switched to the multi-kernel sweep (Sinkhorn / Newton solver,
        Engine.set_fused(False)) for the sweeps that follow."""
        if self.forced_independence or self._sweeps == 0:
            return None
        try:
            iters = np.asarray(self._engine.get(-1, 51, (self.n_layers,)), dtype=np.float64)
        except (AttributeError, _lib.MrgpError):      # (an engine without the per-layer counters)
            return None
        bad = [j for j in range(self.n_layers) if iters[j] >= 2040]
        if bad:
            import warnings
            warnings.warn('the omega solve of layer(s) %s did not reach its tolerance in the last sweep (%s evaluations); '
                          'this model takes the multi-kernel sweep with the Sinkhorn / Newton solver from now on'
                          % (bad, [int(iters[j]) for j in bad]), RuntimeWarning)
            if hasattr(self._engine, 'set_fused'):
                self._engine.set_fused(False)
        return iters

    def fit(self, n_iter=1, tol=1e-3, min_iter=10):
        # MRGP.py:367-412
        try:
            return self._fit_loop(n_iter, tol, min_iter)
        finally:
            if n_iter > 0:
                self.omega_solve_report()

    def _fit_loop(self, n_iter, tol, min_iter):
        if tol is None:
            self._engine.sweep(n_iter)
            self._engine.synchronize()
            self._sweeps += n_iter
            return
        if self.forced_independence:
            self._engine.sweep(n_iter)      # MRGP.py:400-401: no bound, no early stop in fi mode
            self._engine.synchronize()
            self._sweeps += n_iter
            return
        if n_iter < min_iter:
            min_iter = n_iter
        for iter_ in range(1, n_iter + 1):
            self._engine.sweep(1)
            self._sweeps += 1
            lower_bound, lower_bound_layer = self._compute_lower_bound()
            self.lower_bound.append(lower_bound)
            for j in range(self.n_layers):
                self.lower_bound_layer[j].append(lower_bound_layer[j])
            if iter_ > min_iter:
                delta_elbo_layer = [self.lower_bound_layer[j][-1] - self.lower_bound_layer[j][-2]
                                    for j in range(self.n_layers)]
                if self.verbose is True:
                    print("\nTotal ELBO: %.4f ... dELBO %.4f" % (self.lower_bound[-1],
                                                                 self.lower_bound[-1] - self.lower_bound[-2]))
                if abs(delta_elbo_layer[0]) < abs(tol):
                    if self.verbose is True:
                        print("converged: dELBO is smaller than %s" % str(tol))
                    break

    def _fit(self):
        self._engine.sweep(1)
        self._sweeps += 1

    def _independent_fit(self):
        self._engine.sweep(1)
        self._sweeps += 1

    def _compute_lower_bound(self, prime_shared_posterior=None):
        # MRGP.py:414-424; the six terms per layer are kept in lower_bound_terms
        terms = self._engine.elbo()
        self.lower_bound_terms.append(terms)
        ll = [float(v) for v in np.sum(terms, axis=1)]
        return float(np.sum(ll)), ll

    # ------------------------------------------------------------------------------------------
    def _warp(self, test_x):
        # MRGP.py:731-741
        if self.adaptive_inputs is True:
            if self.full_x is None:
                if isinstance(self.input_model, list) is True:
                    test_x = np.mean([m.predict(test_x) for m in self.input_model], axis=0)
                else:
                    test_x = self.input_model.predict(test_x)
            else:
                test_x = self.input_z
        return test_x

    def _norm(self, test_x):
        test_x = np.asarray(test_x, dtype=np.float64)
        if self.standard_normalized_inputs is True:
            test_x = (test_x - np.full(test_x.shape, self.mean_x_train)) / np.full(test_x.shape, self.std_x_train)
        return test_x

    def get_predicted_mean(self, test_x, index_set_obj=None, number_of_regions=None):
        # MRGP.py:805-814
        test_x = self._norm(test_x)
        if index_set_obj is None:
            return self._engine.predict_mean(self._warp(test_x))
        # MRGP.py:757-767
        if index_set_obj.get_n_resolutions() > self.index_set_obj.get_n_resolutions():
            raise ValueError('resolution in the test index set must be smaller or equal to that in the '
                             'train set.')
        if number_of_regions is None:
            if self.index_set_obj.divider != index_set_obj.divider:
                raise ValueError('divider on the training index_set must be'
                                 ' the same as in the test index_set.')
        if number_of_regions is not None:
            if (self.n_regions == number_of_regions) is False:
                raise ValueError('number of regions in the training must be the same as test.')
        test_offsets = offsets_of(index_set_obj)
        for j, off in enumerate(test_offsets):
            if len(off) - 1 != self.n_regions[j]:
                raise ValueError('number of regions in the training must be the same as test.')
        return self._engine.predict_mean(self._warp(test_x), test_offsets)

    def get_central_moment2(self, test_x, index_set_obj=None, number_of_regions=None):
        # MRGP.py:816-823
        test_x = self._norm(test_x)
        if index_set_obj is None:
            return self._engine.predict_var(self._warp(test_x))
        # MRGP.py:863-932.  The reference walks every layer of the MODEL with the test index set and overwrites the
        # model's latent functions on the way; here the state is left untouched.  A test region may be empty (fewer test
        # points than regions): it holds no point whose moment it could change, so only the regions that hold test
        # points are summed.  (The reference adds the latent variance at a region's first test point, :929, and cannot
        # index the first point of an empty region.)
        test_offsets = offsets_of(index_set_obj)
        if len(test_offsets) != self.n_layers:
            raise ValueError('the test index set must have the resolutions of the training index set')
        for j, off in enumerate(test_offsets):
            if len(off) - 1 != self.n_regions[j]:
                raise ValueError('number of regions in the training must be the same as test.')
        return self._engine.predict_var_indexed(self._warp(test_x), test_offsets)

    def get_test_likelihood(self, test, index_set_obj=None, number_of_regions=None):
        # MRGP.py:825-831
        test_x, test_y = test[0], test[1]
        mf = self.get_predicted_mean(test_x, index_set_obj, number_of_regions)
        vf = self.get_central_moment2(test_x, index_set_obj=index_set_obj)
        ll = -0.5 * np.log(2 * np.pi * vf) - 0.5 * (np.linalg.norm((test_y - mf), axis=1) ** 2) / vf
        return np.mean(ll)

    def get_basis_contributions(self):
        # MRGP.py:973-982
        out = []
        for j in range(self.n_layers):
            m2 = self._engine.get(j, _lib.F_M2, (self.n_regions[j], self.n_basis))
            out.append([m2[l] / sum(m2[l]) for l in range(self.n_regions[j])])
        return out

    # ------------------------------------------------------------------------------------------
    # public state (SURVEY.md §8b), materialised from the device on access
    # ------------------------------------------------------------------------------------------
    def _split(self, j, arr):
        off = self._offsets[j]
        return [arr[off[l]:off[l + 1]] for l in range(self.n_regions[j])]

    @property
    def x(self):
        return [self._split(j, self._x_used) for j in range(self.n_layers)]

    @property
    def train_basis_intervals(self):
        return [list(self._engine.get(j, _lib.F_L, (self.n_regions[j], 1))) for j in range(self.n_layers)]

    @property
    def lambda_(self):
        return [list(self._engine.get(j, _lib.F_LAMBDA, (self.n_regions[j], self.n_basis))) for j in range(self.n_layers)]

    @property
    def spectral_density_prior(self):
        return [list(self._engine.get(j, _lib.F_SPECTRAL, (self.n_regions[j], self.n_basis))) for j in range(self.n_layers)]

    @property
    def phi_x(self):
        """Feature matrices (n_jl, M) per region, rebuilt on the host on demand (KernelClass.py:21-37)."""
        out = []
        ids = np.arange(1, self.n_basis + 1, dtype=np.float64)[None, :]
        for j in range(self.n_layers):
            L = self._engine.get(j, _lib.F_L, (self.n_regions[j],))
            row = []
            for l, xs in enumerate(self._split(j, self._x_used)):
                row.append((1. / np.sqrt(L[l])) * np.sin((np.pi * ids * (xs + L[l])) / (2 * L[l])))
            out.append(row)
        return out

    def _posterior_view(self, j):
        e, R, M, dy = self._engine, self.n_regions[j], self.n_basis, self.dy
        F = _lib
        g = {
            'scale_precision': lambda: e.get(j, F.F_SCALE_PRECISION, (R, M)),
            'scale_mean_zeta': lambda: list(e.get(j, F.F_ZETA, (R, M))),
            'scale_mean_y_tilde': lambda: list(np.swapaxes(e.get(j, F.F_YTILDE, (R, M, dy)), 1, 2)),
            'noise_gamma_shape': lambda: self._shared(e.get(j, F.F_NOISE_SHAPE, (R,)), self.noise_region_specific),
            'noise_gamma_scale': lambda: self._shared(e.get(j, F.F_NOISE_SCALE, (R,)), self.noise_region_specific),
            'bias_normal_precision': lambda: self._shared(e.get(j, F.F_BIAS_PRECISION, (R,)), self.bias_region_specific),
            'bias_normal_mean': lambda: self._shared(e.get(j, F.F_BIAS_MEAN, (R, dy)), self.bias_region_specific),
        }
        if self.forced_independence:
            g.update({
                'axis_bingham_b': lambda: list(e.get(j, F.F_AXIS_B, (R, M, dy, dy))),
                'axis_bingham_kappa': lambda: list(e.get(j, F.F_AXIS_KAPPA, (R, M, dy))),
                'axis_bingham_rho': lambda: list(e.get(j, F.F_AXIS_RHO, (R, M, dy))),
                'axis_bingham_log_const': lambda: list(e.get(j, F.F_AXIS_LOGC, (R, M))),
                'ard_gamma_shape': lambda: list(e.get(j, F.F_ARD_SHAPE, (R, M))),
                'ard_gamma_scale': lambda: list(e.get(j, F.F_ARD_SCALE, (R, M))),
            })
        return _View(self, g, dict(dy=dy, n_basis=M, n_regions=R, noise_region_specific=self.noise_region_specific,
                                   bias_region_specific=self.bias_region_specific))

    def _stats_view(self, j):
        e, R, M, dy = self._engine, self.n_regions[j], self.n_basis, self.dy
        F = _lib
        g = {
            'scale_axis_mean': lambda: list(np.swapaxes(e.get(j, F.F_A, (R, M, dy)), 1, 2)),
            'scale_moment2': lambda: list(e.get(j, F.F_M2, (R, M))),
            'scale_axis_central_moment2': lambda: list(e.get(j, F.F_CM2, (R, M))),
            'noise_mean': lambda: self._shared(e.get(j, F.F_NOISE_MEAN, (R,)), self.noise_region_specific, True),
            'noise_log_mean': lambda: self._shared(e.get(j, F.F_NOISE_LOG_MEAN, (R,)), self.noise_region_specific, True),
            'bias_mean': lambda: self._shared(e.get(j, F.F_BIAS_MEAN, (R, dy)), self.bias_region_specific, True),
            'bias_var': lambda: self._shared(e.get(j, F.F_BIAS_VAR, (R,)), self.bias_region_specific, True),
            'latent_f_mean': lambda: self._split(j, e.latent(j)[0]),
            'latent_f_var': lambda: self._split(j, e.latent(j)[1][:, None]),
        }
        if self.forced_independence:
            g.update({
                'axis_cov': lambda: list(e.get(j, F.F_AXIS_COV, (R, M, dy, dy))),
                'ard_mean': lambda: list(e.get(j, F.F_ARD_MEAN, (R, M))),
                'ard_log_mean': lambda: list(e.get(j, F.F_ARD_LOG_MEAN, (R, M))),
                'omega': lambda: [np.ones((M, M)) / M for _ in range(R)],
            })
        return _View(self, g, dict(dy=dy, n_basis=M, n_regions=R, noise_region_specific=self.noise_region_specific,
                                   bias_region_specific=self.bias_region_specific))

    @staticmethod
    def _shared(per_region, region_specific, as_list=False):
        """A posterior shared by the regions of a layer is stored once per region on the device (all entries equal)
        and exposed with the reference's shape: a scalar / one (dy,) vector (Posteriors.py:17-25, Stats.py:29-49)."""
        if region_specific:
            return list(per_region) if as_list else per_region
        return per_region[0]

    @property
    def posterior_obj(self):
        return [self._posterior_view(j) for j in range(self.n_layers)]

    @property
    def stats_obj(self):
        return [self._stats_view(j) for j in range(self.n_layers)]

    @property
    def get_posterior(self):
        return self.posterior_obj

    @property
    def get_stats(self):
        return self.stats_obj

    # ---- priors (Priors.py; non-informative initialisation only, as in the reference) -----------------------------
    def _bingham_prior(self):
        """Bingham(0) of Priors.py:29-36 / :168-189: kappa = 0, rho = 1 / dy, axes = I, log C = log of the sphere's
        area (the saddle-point value the reference stores, computeRealBinghamConstant.py)."""
        import ctypes as C
        dy = self.dy
        if dy != 2:
            raise NotImplementedError('dy == 2 on the device path')
        b = np.zeros(4)
        out = np.zeros(4)
        kappa, rho, logc, cov = np.zeros(2), np.zeros(2), C.c_double(), np.zeros(4)
        D = C.POINTER(C.c_double)
        _lib.load().mrgp_host_bingham2(b.ctypes.data_as(D), out.ctypes.data_as(D), kappa.ctypes.data_as(D), rho.ctypes.data_as(D),
                                       C.byref(logc), cov.ctypes.data_as(D), None)
        return kappa, rho, float(logc.value)

    @property
    def shared_prior(self):
        """SharedPrior (Priors.py:8-53), MRGP.py:183-186."""
        self._require_ci()
        M, dy = self.n_basis, self.dy
        kappa, rho, logc = self._bingham_prior()
        shape = 1e-45 * np.ones(M)
        return _View(self, {}, dict(
            n_basis=M, dy=dy, axis_bingham_b=np.zeros((M, dy, dy)), axis_bingham_kappa=np.tile(kappa, (M, 1)),
            axis_bingham_rho=np.tile(rho, (M, 1)), axis_bingham_axes=np.tile(np.eye(dy), (M, 1, 1)),
            axis_bingham_log_const=np.full(M, logc), ard_gamma_shape=shape, ard_gamma_scale=shape / self._ard_prior_influence))

    @property
    def prior_obj(self):
        """Prior / IndependentPrior per layer (Priors.py:56-278), MRGP.py:187-226."""
        M, dy = self.n_basis, self.dy
        out = []
        for j in range(self.n_layers):
            R = self.n_regions[j]
            S = self._engine.get(j, _lib.F_SPECTRAL, (R, M))
            noise_var = self._noise_var0 if j == 0 else 1.0
            noise_scale, noise_shape = (1e-45 + 1) * noise_var, 1e-45                       # Priors.py:103-109
            consts = dict(
                n_basis=M, dy=dy, n_regions=R, scale_precision=[1 / S[l] for l in range(R)],                      # :74-78
                noise_region_specific=self.noise_region_specific, bias_region_specific=self.bias_region_specific,
                noise_gamma_scale=[noise_scale] * R if self.noise_region_specific else noise_scale,
                noise_gamma_shape=[noise_shape] * R if self.noise_region_specific else noise_shape,
                bias_normal_mean=[np.zeros(dy) for _ in range(R)] if self.bias_region_specific else np.zeros(dy),   # :132-135
                bias_normal_precision=[1e-45] * R if self.bias_region_specific else 1e-45)
            if self.forced_independence:
                kappa, rho, logc = self._bingham_prior()
                shape = 1e-45 * np.ones(M)
                consts.update(
                    axis_bingham_b=[np.zeros((M, dy, dy)) for _ in range(R)], axis_bingham_kappa=[np.tile(kappa, (M, 1)) for _ in range(R)],
                    axis_bingham_rho=[np.tile(rho, (M, 1)) for _ in range(R)], axis_bingham_axes=[np.tile(np.eye(dy), (M, 1, 1)) for _ in range(R)],
                    axis_bingham_log_const=[np.full(M, logc) for _ in range(R)], ard_gamma_shape=[shape.copy() for _ in range(R)],
                    ard_gamma_scale=[shape / self._ard_prior_influence for _ in range(R)])
            out.append(_View(self, {}, consts))
        return out

    # ---- targets of the last sweep (MRGP.py:650-652, kept there for the lower bound) --------------------------------
    @property
    def y_mean(self):
        """y_mean[j][l]: empty lists before the first sweep (MRGP.py:262-271); afterwards the observations at layer 0
        (LatentOutputs.py:6-9: ONE entry holding all of Y), in fi mode the observations of the region
        (LatentOutputs.py:11-18), in ci mode the targets inferred from the layer's own posterior BEFORE its update,
        Phi A_old^T + (b_old + latent_f_mean) (LatentOutputs.py:25-40), rebuilt on the host on demand."""
        if self._sweeps == 0:
            return [[[] for _ in range(R)] for R in self.n_regions]
        out = []
        phi = None
        for j in range(self.n_layers):
            R, M, dy = self.n_regions[j], self.n_basis, self.dy
            if self.forced_independence:
                out.append(self._split(j, self.observations))
            elif j == 0:
                out.append([self.observations] + [[] for _ in range(R - 1)])
            else:
                phi = self.phi_x if phi is None else phi
                a_old = self._engine.get(j, _lib.F_A_PREV, (R, M, dy))
                b_old = self._engine.get(j, _lib.F_BIAS_PREV, (R, dy))
                fbar = self._split(j, self._engine.latent(j)[0])
                out.append([phi[j][l] @ a_old[l] + (b_old[l] + fbar[l]) for l in range(R)])
        return out

    @property
    def y_var(self):
        if self._sweeps == 0:
            return [[[] for _ in range(R)] for R in self.n_regions]
        return [list(self._engine.get(j, _lib.F_YVAR, (self.n_regions[j],))) for j in range(self.n_layers)]

    def _require_ci(self):
        if self.forced_independence:
            raise AttributeError('shared posterior / stats exist in ci mode only (MRGP.py:229-246)')

    @property
    def shared_posterior(self):
        self._require_ci()
        e, M, dy = self._engine, self.n_basis, self.dy
        F = _lib
        return _View(self, {
            'axis_bingham_b': lambda: e.get(-1, F.F_AXIS_B, (M, dy, dy)),
            'axis_bingham_kappa': lambda: e.get(-1, F.F_AXIS_KAPPA, (M, dy)),
            'axis_bingham_rho': lambda: e.get(-1, F.F_AXIS_RHO, (M, dy)),
            'axis_bingham_log_const': lambda: e.get(-1, F.F_AXIS_LOGC, (M,)),
            'ard_gamma_shape': lambda: e.get(-1, F.F_ARD_SHAPE, (M,)),
            'ard_gamma_scale': lambda: e.get(-1, F.F_ARD_SCALE, (M,)),
        }, dict(dy=dy, n_basis=M))

    @property
    def shared_stats(self):
        self._require_ci()
        e, M, dy = self._engine, self.n_basis, self.dy
        F = _lib
        return _View(self, {
            'axis_cov': lambda: e.get(-1, F.F_AXIS_COV, (M, dy, dy)),
            'ard_mean': lambda: e.get(-1, F.F_ARD_MEAN, (M,)),
            'ard_log_mean': lambda: e.get(-1, F.F_ARD_LOG_MEAN, (M,)),
            'omega': lambda: e.get(-1, F.F_OMEGA, (M, M)),
        }, dict(dy=dy, n_basis=M))
