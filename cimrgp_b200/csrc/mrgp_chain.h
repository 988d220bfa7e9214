// Descriptors of the fused ci sweep (csrc/chain.cu): one ChainModel per model, in device memory.
//
// The fused sweep runs ONE kernel per variational sweep of a ci model with static basis intervals
// (MRGP.py:571-652): one thread-block cluster per model walks the layers on the device, so the serial chain
//   omega(j-1) -> B_j, C_j (Bingham) -> ARD_j -> log omega_hat_j -> omega(j)
// (Posteriors.py:497-541, Stats.py:375-445) costs no kernel launch and no graph edge, and a batch of independent
// models (BASELINE config 5) is one launch with one cluster per model.  No sample is touched: layer 0 reads the
// sufficient statistics of its observations (Phi^T y, sum y, sum |y|^2; rebuilt when y changes) and every layer
// the basis invariants s = Phi^T 1, G = Phi^T Phi, D (DESIGN.md §4).
#pragma once
#include <stdint.h>

namespace mrgp {

constexpr int kChainMaxLayers = 24;
constexpr int kChainThreads = 256;
constexpr int kChainMaxCluster = 16;   // above 8: non-portable cluster size (allowed on sm_100a)

// One piece of a region with a region of a coarser layer, for sum f_var of the closed-form statistics: offsets in
// doubles from the base of the small-matrix state (ChainModel::sbase) of the coarser region's cm2 row and bias variance
// and of the piece's D row; its number of samples (len < 0: unused slot of the fixed-stride table).
struct AncEntry {
    uint32_t cm2_off, bv_off, d_off;
    int32_t len;
};

struct ChainLayer {
    int32_t R, P;                  // regions; pieces region x coarser region (layers > 0)
    int32_t E, pad;                // slots per region of anc_tab (largest number of pieces of a region)
    const AncEntry *anc_tab;       // (R, E)
    const double *rconst;          // (R, 8): n, bias_prec0, bias_mean0 (2), noise_shape0, noise_scale0, psi(noise shape), -
    const int64_t *offsets;        // (R + 1)
    // static
    const double *inv2L, *rsqrtL;  // (R) 1 / (2 L), L^-1/2 of the basis interval
    const double *S, *d;           // (R, M) spectral density, sum phi^2
    const double *sumPhi, *gram;   // (R, M) Phi^T 1, (R, M, M) Phi^T Phi
    const double *ancD;            // (P, M) sum over the piece of the squared basis functions of its coarser layer
    const int32_t *pc_ptr, *pc_anc;   // piece table: (layer, R + 1) CSR, coarser region per piece
    const int64_t *pc_lo, *pc_hi;
    double *yc, *ysum;             // layer 0: (R, M, 2) Phi^T y and (R, 4) sum y_0, sum y_1, sum |y|^2, -
    // posterior / stats
    double *prec, *zeta, *ytil, *A, *A_prev, *m2, *cm2;
    double *noise_shape, *noise_scale, *noise_mean, *noise_log_mean;
    const double *noise_shape0, *noise_scale0, *bias_prec0, *bias_mean0;
    double *bias_prec, *bias_mean, *bias_prev, *bias_var, *yvar, *sumsB;
};

struct ChainModel {
    int32_t J, M, DY;
    double *sbase;                 // base of the small-matrix state in the workspace (AncEntry offsets are relative to it)
    const char *pf_base;           // range pulled into L2 at the start of a sweep (the small-matrix state), 128-byte lines
    unsigned long long pf_lines;
    const double *x, *y;           // (N), (N, DY) normalised inputs and observations, indexed by the global sample number
    // shared posterior / stats (Posteriors.py:482-541, Stats.py:354-420)
    double *axB, *axKappa, *axRho, *axLogC, *axCov, *ardShape, *ardScale, *ardMean, *ardLogMean;
    double *omega, *logOmegaHat, *omegaIters, *omegaEta, *omegaWarm;
    const double *priorB, *priorLogC, *priorShape, *priorScale, *priorSk;
    unsigned long long *chol_count;
    unsigned int *status;          // [0]: layer-0 closed-form guard tripped (sum |r|^2 / sum |y|^2 below kChainGuard)
    double guard_threshold;        // kChainGuard unless overridden (MRGP_CHAIN_GUARD, tests of the fallback)
    double *guard;                 // [0]: last ratio sum |r|^2 / sum |y|^2 of layer 0; [1]: 1.0 once the guard tripped
    unsigned long long *ts;        // timeline stamps or null
    double *prof;                  // (J, 16) SM-clock stamps inside CTA 0 (MRGP_CHAIN_PROF=1) or null
    double *tables;                // (J, M, M) log omega_hat of every layer of the sweep (MRGP_CHAIN_PROF=1) or null
    ChainLayer layer[kChainMaxLayers];
};

// sum |r|^2 of layer 0 is formed as sum |y|^2 - 2 tr(A^T Phi^T y) + tr(A^T G A): below this ratio to sum |y|^2 the
// cancellation would cost more than 1e-16 / kChainGuard relative accuracy and the streamed pass takes over.
constexpr double kChainGuard = 1e-5;

// Smallest compiled solver size that holds M basis functions (0: none, M > 32).
inline int chain_solver_size(int M) {
    if (M == 30) return 30;
    if (M <= 8) return 8;
    if (M <= 16) return 16;
    if (M <= 24) return 24;
    if (M <= 32) return 32;
    return 0;
}

// Launch n_models clusters of `cluster` CTAs on `stream`.  models_dev: device array of pointers to ChainModel.
// Returns a cudaError_t as int.
int launch_ci_sweep(int solver_size, const ChainModel *const *models_dev, int n_models, int cluster, void *stream);
// Sufficient statistics of the observations for layer 0 (Phi^T y, sum y, sum |y|^2), one CTA per (model, region of
// layer 0): the form for models whose layer-0 regions are small (a batch of short series: one launch for all of them).
// r0_max: largest number of layer-0 regions among the models.
int launch_ystats_small(int solver_size, const ChainModel *const *models_dev, int n_models, int r0_max, void *stream);
// Streamed fallback of layer 0 for the models whose guard tripped (status != 0), same geometry as launch_ystats_small:
// exact P4 / P5 statistics by a pass over the samples and the bias / noise update of layer 0 again.
int launch_l0_fix_small(int solver_size, const ChainModel *const *models_dev, int n_models, int r0_max, void *stream);
constexpr int64_t kYstatsSmallMaxRegion = 32768;   // longest layer-0 region this form is used for
size_t ci_sweep_smem_bytes(int solver_size);

}  // namespace mrgp
