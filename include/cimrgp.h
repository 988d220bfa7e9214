/*
 * cimrgp.h - C ABI of the B200 (sm_100a) implementation of the ciMRGP / fiMRGP variational-
 * inference hot path.
 *
 * The reference (jtaghia/ciMRGP) is pure Python and has no FFI: its boundary is the object API of
 * src/MRGP.py.  The entry points below are the seams a binding for that path has to cross; each one
 * names the reference code it replaces (file:line under the reference's src/).  The Python package
 * `cimrgp_b200` binds them with ctypes; INTEGRATION.md shows the stub a maintainer of the reference
 * would add.
 *
 * Conventions
 *   - one handle per model, one process per GPU, one CUDA stream per handle; nothing is thread-safe
 *     per handle;
 *   - every function returns 0 on success or a negative MRGP_E* code; mrgp_last_error() gives text;
 *   - all arithmetic is IEEE float64; index sets are int64 region offsets (regions of a layer are the
 *     contiguous, ordered ranges [off[l], off[l+1]) that IndexSetGenerator.py:51-92 produces);
 *   - "dev" pointers are device pointers owned by the caller (torch tensors in the Python host),
 *     "host" pointers are ordinary host memory; the library allocates no device memory of its own:
 *     the caller binds one workspace of mrgp_workspace_bytes() bytes;
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     MRGP_ENODEVICE.
 *
 * Layouts (row-major, float64): x (N, dx); y (N, dy); per layer j with R regions and M basis
 * functions: region fields (R,), (R, M), (R, dy); coefficient fields A and ytil are (R, M, dy)
 * (the reference keeps (dy, M) per region; the Python host transposes on export).
 */
#ifndef CIMRGP_H
#define CIMRGP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRGP_ABI_VERSION 5

enum {
    MRGP_OK = 0,
    MRGP_EINVAL = -1,      /* bad argument / unsupported configuration                          */
    MRGP_ENODEVICE = -2,   /* no CUDA device, or the device is not sm_100                        */
    MRGP_ECUDA = -3,       /* a CUDA runtime call or kernel failed                               */
    MRGP_ESTATE = -4,      /* call made in the wrong order (no workspace, no data, no basis...)  */
    MRGP_ENOMEM = -5       /* workspace too small                                                */
};

enum { MRGP_MODE_CI = 0, MRGP_MODE_FI = 1 };   /* MRGP.py:37-50 (forced_independence)             */

/* Field ids for mrgp_get_state / mrgp_set_state.  Per-layer fields take layer >= 0; shared (ci) fields
 * take layer == -1.  Shapes in float64 elements.                                                    */
enum {
    /* static region data (MRGP.py:137-172) */
    MRGP_F_L = 1,               /* (R,)      basis half-interval L_jl, BasisInterval.py:15-16        */
    MRGP_F_LAMBDA = 2,          /* (R, M)    eigenvalues, KernelClass.py:36                          */
    MRGP_F_SPECTRAL = 3,        /* (R, M)    S(sqrt(lambda)), KernelClass.py:80-90                   */
    MRGP_F_PHI2SUM = 4,         /* (R, M)    sum_n phi^2, Posteriors.py:41                           */
    /* posterior_obj[j] (Posteriors.py:9-30) */
    MRGP_F_SCALE_PRECISION = 10,/* (R, M)                                                            */
    MRGP_F_ZETA = 11,           /* (R, M)    scale_mean_zeta                                         */
    MRGP_F_YTILDE = 12,         /* (R, M, dy) scale_mean_y_tilde (transposed)                        */
    MRGP_F_NOISE_SHAPE = 13,    /* (R,)                                                              */
    MRGP_F_NOISE_SCALE = 14,    /* (R,)                                                              */
    MRGP_F_BIAS_PRECISION = 15, /* (R,)                                                              */
    /* stats_obj[j] (Stats.py:7-62) */
    MRGP_F_A = 20,              /* (R, M, dy) scale_axis_mean (transposed)                           */
    MRGP_F_M2 = 21,             /* (R, M)    scale_moment2                                           */
    MRGP_F_CM2 = 22,            /* (R, M)    scale_axis_central_moment2                              */
    MRGP_F_NOISE_MEAN = 23,     /* (R,)                                                              */
    MRGP_F_NOISE_LOG_MEAN = 24, /* (R,)                                                              */
    MRGP_F_BIAS_MEAN = 25,      /* (R, dy)                                                           */
    MRGP_F_BIAS_VAR = 26,       /* (R,)                                                              */
    MRGP_F_FBAR = 27,           /* (N, dy)   latent_f_mean of the layer, as it was during the sweep   */
    MRGP_F_FVAR = 28,           /* (N,)      latent_f_var of the layer                                */
    MRGP_F_YVAR = 29,           /* (R,)      y_var used at the layer's step (MRGP.py:650-652)         */
    MRGP_F_PHASE_B_SUMS = 30,   /* (R, dy+3) sum r, sum |r|^2, sum f_var, sum phi^2 cm2 of the step   */
    MRGP_F_A_PREV = 31,         /* (R, M, dy) scale_axis_mean BEFORE the layer's last update: with MRGP_F_BIAS_PREV the
                                 * coefficients the inferred targets y_mean[j] of the last sweep were made of (MRGP.py:577, 650) */
    MRGP_F_BIAS_PREV = 32,      /* (R, dy)   bias_mean before the layer's last update                    */
    /* Bingham axis / ARD: shared_posterior + shared_stats in ci (layer == -1), posterior_obj[j] +
     * stats_obj[j] in fi (layer >= 0, leading R).  (Posteriors.py:482-541, Stats.py:354-388)        */
    MRGP_F_AXIS_B = 40,         /* ([R,] M, dy, dy)                                                  */
    MRGP_F_AXIS_KAPPA = 41,     /* ([R,] M, dy) clamped at 0 as stored by Posteriors.py:525-526      */
    MRGP_F_AXIS_RHO = 42,       /* ([R,] M, dy)                                                      */
    MRGP_F_AXIS_LOGC = 43,      /* ([R,] M)                                                          */
    MRGP_F_AXIS_COV = 44,       /* ([R,] M, dy, dy)                                                  */
    MRGP_F_ARD_SHAPE = 45,      /* ([R,] M)                                                          */
    MRGP_F_ARD_SCALE = 46,      /* ([R,] M)                                                          */
    MRGP_F_ARD_MEAN = 47,       /* ([R,] M)                                                          */
    MRGP_F_ARD_LOG_MEAN = 48,   /* ([R,] M)                                                          */
    MRGP_F_OMEGA = 49,          /* (M, M)    ci only, Stats.py:369, 390-420                          */
    MRGP_F_LOG_OMEGA_HAT = 50,  /* (M, M)    ci only, Stats.py:405-412 (last evaluation)             */
    MRGP_F_OMEGA_ITERS = 51,    /* (J,)      ci only: scaling iterations of the last omega solve per layer */
    MRGP_F_FUSED_GUARD = 55     /* (2,)      ci, fused sweep: [sum |r|^2 / sum |y|^2 of layer 0 in the last sweep, 1.0 once the
                                 * ratio fell below 1e-5 and the streamed fallback took over the statistics of layer 0] */
};

typedef struct mrgp_handle mrgp_handle;

typedef struct mrgp_config {
    int32_t abi_version;            /* MRGP_ABI_VERSION                                              */
    int32_t mode;                   /* MRGP_MODE_CI / MRGP_MODE_FI                                   */
    int64_t n_samples;              /* N                                                             */
    int32_t dx;                     /* input dimension (1 supported)                                 */
    int32_t dy;                     /* output dimension (>= 2, MRGP.py:65-66; 2 supported)           */
    int32_t n_basis;                /* M (<= 48)                                                     */
    int32_t n_layers;               /* J = resolution + 1                                            */
    int32_t noise_region_specific;  /* MRGP.py:27; 0 = one noise posterior per layer (stored once per region) */
    int32_t bias_region_specific;   /* MRGP.py:28; 0 = one bias posterior per layer (stored once per region)  */
    int32_t device;                 /* CUDA device ordinal                                           */
    int32_t n_ctas;                 /* streaming grid size; 0 = one persistent CTA per SM            */
    int64_t sample_begin;           /* sample sharding (multi-GPU): this handle owns samples           */
    int64_t sample_end;             /* [sample_begin, sample_end) of the N; 0, 0 = all of them         */
} mrgp_config;

/* ---- lifetime -------------------------------------------------------------------------------- */

/* Build the host-side plan (segment / run tables) for the index sets of a model.
 * region_offsets[j] points to n_regions[j]+1 int64 offsets of layer j (host memory).
 * Replaces the list-of-lists index sets read at MRGP.py:132-154 and Stats.py:155-157.              */
int mrgp_create(const mrgp_config *cfg, const int64_t *const *region_offsets, const int32_t *n_regions,
                mrgp_handle **out);
void mrgp_destroy(mrgp_handle *h);
const char *mrgp_last_error(const mrgp_handle *h);   /* h may be NULL: last create error          */
int mrgp_abi_version(void);

/* Device memory the caller has to provide, and binding it (256-byte aligned device pointer). */
size_t mrgp_workspace_bytes(const mrgp_handle *h);
int mrgp_bind_workspace(mrgp_handle *h, void *dev_ptr, size_t bytes);
int mrgp_set_stream(mrgp_handle *h, void *cuda_stream);

/* ---- data ------------------------------------------------------------------------------------ */

/* Normalised inputs x (N, dx) and observations y (N, dy), already on the device (MRGP.py:61-69).
 * The pointers are borrowed: they must stay valid while the handle is used.
 * NEW INPUTS INVALIDATE EVERYTHING DERIVED FROM x: after the first call, every further mrgp_set_data /
 * mrgp_set_data_host marks the basis of all layers (intervals, lambda, S, sum phi^2), the invariants of the
 * closed-form statistics and the captured sweep as stale; phases and sweeps then fail with MRGP_ESTATE until
 * mrgp_build_basis has run for every layer again (the reference needs a new model object for new inputs,
 * MRGP.py:128-172).  New observations at the SAME inputs go through mrgp_set_observations*, which keep all of
 * that (only the layer-0 sufficient statistics Phi^T y, sum y, sum |y|^2 are refreshed by the next sweep).     */
int mrgp_set_data(mrgp_handle *h, const double *x_dev, const double *y_dev);
/* Same from host buffers (pinned for full speed): asynchronous H2D copies on the handle's stream into the
 * workspace.                                                                                                   */
int mrgp_set_data_host(mrgp_handle *h, const double *x_host, const double *y_host);
/* New observations y (N, dy) at unchanged inputs: borrowed device pointer / asynchronous copy from host memory.
 * mrgp_set_observations_host is the entry the end-to-end benchmark times (16 B per sample and step).           */
int mrgp_set_observations(mrgp_handle *h, const double *y_dev);
int mrgp_set_observations_host(mrgp_handle *h, const double *y_host);
/* Double-buffered form of mrgp_set_observations_host for a stream of data sets at unchanged inputs: starts the copy of
 * the NEXT observations (pinned host memory) into the handle's spare buffer on a copy stream of its own and returns. The
 * copy runs beside whatever the handle's stream is doing - the fused ci sweep reads no sample. The observations take
 * effect at the next mrgp_refresh_statistics() (and only there: sweeps in between keep working on the current set): the
 * buffers are swapped and the statistics pass waits for the copy. One set can be pending (MRGP_ESTATE otherwise). Loop
 * of a pipelined consumer:
 *     mrgp_refresh_statistics(h);  mrgp_prefetch_observations_host(h, y_next);  mrgp_sweep(h, 1);  ... read results ...
 * (reference counterpart: a new MultiResolutionGaussianProcess([x, y_next], ...) per data set, MRGP.py:16-66).          */
int mrgp_prefetch_observations_host(mrgp_handle *h, const double *y_host);
/* Blocks until the last mrgp_prefetch_observations_host() has read its host buffer (the buffer may then be rewritten).
 * (No counterpart in the reference, which is synchronous NumPy.)                                                     */
int mrgp_prefetch_sync(mrgp_handle *h);

/* ---- K1-K3: basis intervals, eigenvalues, spectral density, sum phi^2 ---------------------------- */

/* Spectral density of a layer: use_prior = 0 -> S == 1 (MRGP.py:328-330), else Matern(nu, l, sf)
 * (KernelClass.py:43-90).                                                                         */
int mrgp_set_spectral(mrgp_handle *h, int32_t layer, int32_t use_prior, double nu, double l, double sf);
/* L_jl = factor * max|x_jl| (BasisInterval.py:15-16) unless L_host != NULL gives (R,) values;
 * then lambda, S and sum_n phi^2 for the layer (MRGP.py:305-357, KernelClass.py:9-37).              */
int mrgp_build_basis(mrgp_handle *h, int32_t layer, double interval_factor, const double *L_host);

/* ---- state ----------------------------------------------------------------------------------- */

/* Non-informative initialisation of priors, posteriors and stats (Priors.py, Posteriors.py:10-30,
 * Stats.py:8-62, 355-369; SURVEY.md App. E).  noise_var0 is the layer-0 prior noise variance
 * (1.0, or var(y)/snr from MRGP.py:966-971); ard_prior_influence = mean(sf) (MRGP.py:185).          */
int mrgp_init_state(mrgp_handle *h, double noise_var0, double ard_prior_influence);
int mrgp_get_state(mrgp_handle *h, int32_t layer, int32_t field, double *dst_host, size_t n_elems);
int mrgp_set_state(mrgp_handle *h, int32_t layer, int32_t field, const double *src_host, size_t n_elems);
int64_t mrgp_state_elems(const mrgp_handle *h, int32_t layer, int32_t field);

/* ---- the sweep, phase by phase (MRGP.py:571-724; SURVEY.md App. A/B) -------------------------- */

/* T1 + P1 statistics: stream x, y, latent mean of the layer and reduce Phi^T r per region
 * (LatentOutputs.py:6-49, Posteriors.py:35-78 / 298-342).                                           */
int mrgp_phase_a(mrgp_handle *h, int32_t layer);
/* P1 finish, P2, P2a-c, S1, S2, P3, S3 and (ci) S4: precision/zeta/y_tilde, Bingham axis update with
 * the PD guard, scale moments, ARD and permutation weights (Posteriors.py:35-59, 253-295, 497-541;
 * Stats.py:67-100, 240-290, 375-445; CommonDensities.py:71-77; SanityCheck.py:16-65).               */
int mrgp_axis_update(mrgp_handle *h, int32_t layer);
/* P4/P5 statistics with the new coefficients, fused with L1 propagation to the next layer
 * (Posteriors.py:81-211 / 345-475, Stats.py:126-157 / 316-348).                                     */
int mrgp_phase_b(mrgp_handle *h, int32_t layer);
/* P4, P5, S5 finish: bias and noise posteriors and their moments (Stats.py:102-124 / 292-314).     */
int mrgp_bias_noise(mrgp_handle *h, int32_t layer);
/* B1: BasisInterval.learn (BasisInterval.py:18-134) + rebuild of the layer's basis (MRGP.py:632-641), ci mode,
 * dx == 1.  mrgp_set_adaptive_intervals(layer | -1 = all, enabled, use_prior, opt_interval_factor[0], [1])
 * mirrors BasisInterval(use_prior, opt_interval_factor) of that layer; once enabled every sweep learns the
 * intervals of the layer after its bias / noise update (bounded search, scipy fminbound semantics: xatol
 * 1e-5, run in lock-step over all regions).  mrgp_learn_intervals runs the search for one layer (per-phase
 * use).  mrgp_interval_failures: regions whose search had not converged when the fixed iteration budget
 * ran out, summed since mrgp_init_state.                                                             */
int mrgp_set_adaptive_intervals(mrgp_handle *h, int32_t layer, int32_t enabled, int32_t use_prior, double factor_lo, double factor_hi);
int mrgp_learn_intervals(mrgp_handle *h, int32_t layer);
int mrgp_interval_failures(mrgp_handle *h, uint64_t *out);
/* n_iter full sweeps (all layers, Gauss-Seidel order), replayed from one captured CUDA graph.  Same results as
 * the per-phase calls above up to summation order (1e-11): in ci mode with static intervals the sweep does not
 * stream the layers whose targets are inferred from their own posterior (LatentOutputs.py:20-49) - their P1
 * residual vanishes identically and their P4 / P5 sums are evaluated in closed form from basis invariants built
 * on the first call (DESIGN.md §4); MRGP_STREAM_ALL=1 in the environment streams every layer.        */
int mrgp_sweep(mrgp_handle *h, int32_t n_iter);
/* The fused ci sweep (ci mode, static intervals, region-specific noise and bias, n_basis <= 32: one kernel per sweep,
 * DESIGN.md §4) reads layer 0 through the sufficient statistics of its observations, Phi^T y, sum y, sum |y|^2: one
 * pass over x and y (24 B per sample) whenever the observations, the inputs or the intervals of layer 0 changed.
 * mrgp_sweep refreshes them on demand; this entry does it now (asynchronously on the handle's stream), e.g. right after
 * mrgp_set_observations_host.  A no-op for models that take the multi-kernel sweep.                             */
int mrgp_refresh_statistics(mrgp_handle *h);
/* on = 0: this handle takes the multi-kernel sweep (Sinkhorn / Newton omega solve) from now on; on = 1: the fused sweep
 * again where it applies.  Same state either way (results agree to summation order).  The host mirror switches a model
 * over when the accelerated omega solve of the fused sweep used up its budget on a layer (MRGP.omega_solve_report).
 * Both are the sweep of MRGP.py:571-652; the permutation weights are Stats.py:390-445 either way.                    */
int mrgp_set_fused(mrgp_handle *h, int32_t on);
int mrgp_synchronize(mrgp_handle *h);

/* E1-E6: the six ELBO terms per layer, out_host (J, 6) in the order data, scale|axis, axis, ard, bias,
 * noise (MRGP.py:414-569; ci only).  Under adaptive intervals the data term uses the re-learnt basis of every
 * layer against the targets inferred with the previous one, as the reference does (MRGP.py:535-569 after :640). */
int mrgp_elbo(mrgp_handle *h, double *out_host);
/* The same (MRGP.py:414-569) without blocking: the terms are copied into PINNED host memory behind the kernel on the handle's stream and
 * mrgp_elbo_wait(h, slot) blocks until the copy of that slot (0 or 1) has arrived.  A consumer that reads the bound of step k
 * after queueing step k + 1 keeps the host round trip off the chain of a step (bench.py, e2e).                          */
int mrgp_elbo_async(mrgp_handle *h, double *out_pinned_host, int32_t slot);
int mrgp_elbo_wait(mrgp_handle *h, int32_t slot);

/* ---- O1: prediction (MRGP.py:726-861) --------------------------------------------------------- */

/* x_test_dev (n_test, dx) normalised.  test_offsets == NULL: layer 0 / region 0 only (MRGP.py:726-755);
 * else test_offsets[j] (host, n_regions[j]+1 int64) assigns test points to regions by position for
 * the first n_test_layers layers (MRGP.py:757-803).  out_dev (n_test, dy).
 * Test offsets of every layer run from 0 to n_test and must be non-decreasing; a region may be empty (equal
 * neighbouring offsets).  Otherwise, as for n_test < 1 or n_test_layers outside [1, n_layers], MRGP_EINVAL with a
 * message naming the layer.  The same holds for mrgp_predict_var_indexed, which takes exactly n_layers layers.
 * Prediction is valid for test points with |x| / (2 L) < 2^30 in every layer (the range of the basis evaluation).  */
int mrgp_predict_mean(mrgp_handle *h, const double *x_test_dev, int64_t n_test,
                      const int64_t *const *test_offsets, int32_t n_test_layers, double *out_dev);
/* Layer-0 central second moment sum_i cm2_i phi_i^2 + bias_var (MRGP.py:833-861). out_dev (n_test,). */
int mrgp_predict_var(mrgp_handle *h, const double *x_test_dev, int64_t n_test, double *out_dev);
/* Index-set form of the second moment (MRGP.py:863-932): sum over ALL layers of sum_i cm2_i phi_i^2 + bias_var +
 * n_test(region) / noise_mean + the latent variance of the region's first test point (MRGP.py:929).  The reference
 * overwrites the model's latent functions with their values at the test points while doing so (MRGP.py:893-901);
 * here they are derived quantities and the model state is left untouched.  Test regions may be empty: a point takes
 * the terms of the non-empty region that holds it in every layer.  out_dev (n_test,).                        */
int mrgp_predict_var_indexed(mrgp_handle *h, const double *x_test_dev, int64_t n_test,
                             const int64_t *const *test_offsets, int32_t n_test_layers, double *out_dev);

/* ---- sample sharding over several GPUs (SURVEY.md §8e) ------------------------------------------ */

/* A handle created with [sample_begin, sample_end) streams only its chunk of x, y (mrgp_set_data* take the
 * LOCAL rows) but knows every region.  The per-region sufficient statistics of a phase (<= R x 60 doubles) are
 * summed over the ranks and consumed by the replicated small-matrix step; no per-sample data ever leaves a GPU.
 *
 * The sums go through a peer-memory exchange: every rank keeps a small arena that the peers map over
 * NVLink / NVSwitch (CUDA IPC between processes, plain pointers inside one process).
 *     mrgp_comm_export(h, blob)                     -> 128-byte description of this rank's arena
 *     (all-gather the blobs of all ranks with any transport: torch.distributed, MPI, a file)
 *     mrgp_comm_bind(h, rank, world, blobs, bounds) -> maps the peers; bounds[q], bounds[q+1] = samples of rank q
 * Afterwards mrgp_build_basis, mrgp_sweep (one CUDA graph, exchanges included) and mrgp_exchange work on the
 * sharded handle; before it they are refused.  One exchange = dense local sums -> arena, a release-store of the next
 * sequence number into every peer's flag array, and a reduce kernel that waits for all peers and sums, per region,
 * the arenas of exactly the ranks that own samples of the region, in rank order: every rank computes bit-identical
 * sums.  A peer that never publishes makes the wait time out (15 s) and mrgp_synchronize return MRGP_ECUDA.
 *     mrgp_phase_a -> mrgp_exchange(layer, MRGP_X_PHASE_A) -> mrgp_axis_update
 *     mrgp_phase_b -> mrgp_exchange(layer, MRGP_X_PHASE_B) -> mrgp_bias_noise                                */
enum { MRGP_X_PHASE_A = 0, MRGP_X_PHASE_B = 1 };
#define MRGP_COMM_BLOB_BYTES 128
#define MRGP_COMM_MAX_RANKS 16
int mrgp_comm_export(mrgp_handle *h, void *blob_out);
int mrgp_comm_bind(mrgp_handle *h, int32_t rank, int32_t world, const void *blobs, const int64_t *bounds);
int mrgp_exchange(mrgp_handle *h, int32_t layer, int32_t which);
/* Optional on a sharded ci handle: the normalised inputs of ALL ranks (n_samples x dx doubles, host memory; 8 MB at
 * N = 1e6).  With them every rank builds the basis invariants of the closed-form statistics (DESIGN.md §4) and
 * the layers above the first need neither their samples nor an exchange in mrgp_sweep.  y never leaves its rank. */
int mrgp_set_all_inputs_host(mrgp_handle *h, const double *x_all_host);

/* ---- groups of independent models (BASELINE config 5: a batch of series) --------------------------------- */

/* The reference fits its models one after the other; they are independent.  A group sweeps all of its models with one
 * launch per iteration:
 *   - batched form (every member is a ci model with static intervals, region-specific noise and bias, n_basis <= 32,
 *     layer-0 regions of at most 32768 samples): one launch of the fused sweep kernel with one thread-block cluster per
 *     model, and one launch for the layer-0 statistics of all members when observations changed;
 *   - otherwise: the members' sweeps captured as parallel branches of ONE CUDA graph.
 * The models must be initialised, unsharded and on one device; their state is what mrgp_sweep would leave.  Work queued
 * on a member's own stream (uploads, state writes) is ordered before the group's next launch; a member whose captured
 * sweep went stale (new pointers, intervals, re-initialisation) makes the group prepare itself again.  The batched
 * form keeps a small table of descriptor pointers in device memory of its own (n x 8 bytes, cudaMalloc).
 * cuda_stream: the stream the group launches on (NULL: the group creates one).
 * mrgp_group_observations_changed: the caller overwrote the members' (borrowed) observation buffers in place.          */
typedef struct mrgp_group mrgp_group;
int mrgp_group_create(mrgp_handle *const *handles, int32_t n, void *cuda_stream, mrgp_group **out);
int mrgp_group_sweep(mrgp_group *g, int32_t n_iter);
int mrgp_group_observations_changed(mrgp_group *g);
int64_t mrgp_group_launch_count(const mrgp_group *g);
int mrgp_group_synchronize(mrgp_group *g);
void mrgp_group_destroy(mrgp_group *g);

/* ---- counters and micro-benchmarks ------------------------------------------------------------ */

/* Number of kernels launched on the handle so far (for bench.py's gpu_launches). */
int64_t mrgp_launch_count(const mrgp_handle *h);
/* Number of dy x dy Cholesky factorisations performed by the PD guard so far (SanityCheck.py:59-65). */
int64_t mrgp_cholesky_count(mrgp_handle *h);
/* Batched Cholesky of `batch` symmetric n x n matrices (n <= 32), one warp per matrix, in place
 * (lower triangle); info_dev[b] = 0 or the failing pivot (1-based), as LAPACK potrf.               */
int mrgp_batched_cholesky(void *cuda_stream, double *a_dev, int32_t n, int64_t batch, int32_t *info_dev);
/* FP64 FMA throughput probe: runs `iters` dependent-chain-free DFMAs per thread on a full grid and
 * writes the elapsed milliseconds; used to measure the FP64 pipe roofline.                          */
int mrgp_fp64_probe(void *cuda_stream, int64_t iters, double *sink_dev, float *ms_out);

/* Debug aid: global-timer stamps written by the kernels of the captured sweep graph.  Enable before the first
 * mrgp_sweep(); mrgp_timeline_read() runs ONE sweep and returns n = 4 * n_layers entries: tags[k] = layer * 4 + kind
 * (0 phase A, 1 mid-step, 2 phase B, 3 omega), ms[2k] / ms[2k+1] = begin / end of that kernel in ms since the first
 * begin (-1 when the kernel did not run).  cap = capacity of tags[]; ms[] must hold 2 * cap floats.              */
int mrgp_timeline_enable(mrgp_handle *h, int32_t on);
int mrgp_timeline_read(mrgp_handle *h, int32_t *tags, float *ms, int32_t cap);

/* ---- host-only hooks (no GPU needed; used by the CPU tests) ------------------------------------ */

/* Plan introspection: number of streaming CTAs, segments and runs of a layer. */
int mrgp_plan_info(const mrgp_handle *h, int32_t layer, int32_t *n_ctas, int32_t *n_segments, int32_t *n_runs);
/* Copy the plan of a layer: seg (n_segments, 6) int64 = start, end, region, parent, run, cta. */
int mrgp_plan_segments(const mrgp_handle *h, int32_t layer, int64_t *seg_out);
/* Pieces of the closed-form statistics (ci mode, layers > 0): every intersection of a region of `layer` with a
 * region of a coarser layer.  piece_out == NULL: only the count; else (n_pieces, 5) int64 = coarser layer, region
 * of `layer`, region of the coarser layer, first sample, one past the last sample.                   */
int mrgp_plan_pieces(const mrgp_handle *h, int32_t layer, int32_t *n_pieces, int64_t *piece_out);
/* The device math routines compiled for the host (same source): digamma, Matern spectral density,
 * the 2x2 Bingham update (guard, eigen-solve, saddle point), basis recurrence, omega scaling.       */
double mrgp_host_digamma(double x);
double mrgp_host_matern_spectral(double lambda, double nu, double l, double sf);
void mrgp_host_bingham2(const double *b_in, double *b_out, double *kappa, double *rho, double *logc,
                        double *axis_cov, int32_t *n_chol);
void mrgp_host_basis(double x, double L, int32_t n_basis, double *phi_out);
int mrgp_host_omega(const double *log_omega_hat, int32_t m, double *omega_out, int32_t *iters_out);

#ifdef __cplusplus
}
#endif
#endif /* CIMRGP_H */
