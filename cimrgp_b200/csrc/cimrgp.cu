// C ABI (include/cimrgp.h) over the sm_100a kernels of mrgp_kernels.cuh: host-side plan, workspace
// carving, kernel dispatch, the per-layer composition of a sweep and its CUDA-graph replay.
#include "../../include/cimrgp.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include <unistd.h>

#include "mrgp_kernels.cuh"
#include "mrgp_chain.h"

using namespace mrgp;

namespace {

std::string g_create_error;

struct LayerPlan {
    std::vector<int64_t> offsets;     // R + 1
    // pieces region x coarser region (closed-form statistics): CSR over (coarser layer, region)
    std::vector<int32_t> pc_ptr, pc_jp, pc_anc;
    std::vector<int64_t> pc_lo, pc_hi;
    std::vector<Segment> segs;
    std::vector<int32_t> cta_seg;     // n_ctas + 1
    std::vector<int32_t> seg_cta;     // per segment (host only)
    std::vector<int32_t> region_run;  // R + 1
    std::vector<int32_t> ident_run;   // 0 .. R (dense exchange buffer: one "run" per region)
    int32_t R = 0, n_runs = 0;
    int32_t E = 0;                    // largest number of pieces (over all coarser layers) of a region
};

struct LayerDev {
    // plan
    Segment *segs = nullptr;
    int32_t *cta_seg = nullptr, *region_run = nullptr, *ident_run = nullptr;
    int64_t *offsets = nullptr;
    // static
    double *L = nullptr, *inv2L = nullptr, *rsqrtL = nullptr, *lam = nullptr, *S = nullptr, *d = nullptr, *absx = nullptr;
    double *bias_prev = nullptr, *brent = nullptr, *trial_inv2L = nullptr, *trial_rsqrtL = nullptr, *wq = nullptr;
    double *inv2L_old = nullptr, *rsqrtL_old = nullptr, *sumsE = nullptr;   // adaptive intervals: basis of the step's targets, ELBO sums
    bool adaptive = false;
    int32_t ad_use_prior = 1;
    double ad_lo = 1.0, ad_hi = 1.2;
    // posterior / stats
    double *prec = nullptr, *zeta = nullptr, *ytil = nullptr, *A = nullptr, *A_prev = nullptr, *m2 = nullptr, *cm2 = nullptr;
    double *noise_shape = nullptr, *noise_scale = nullptr, *noise_shape0 = nullptr, *noise_scale0 = nullptr;
    double *noise_mean = nullptr, *noise_log_mean = nullptr;
    double *bias_prec = nullptr, *bias_prec0 = nullptr, *bias_mean = nullptr, *bias_mean0 = nullptr, *bias_var = nullptr;
    double *yvar = nullptr, *sumsB = nullptr, *bcontrib = nullptr, *wcontrib = nullptr;
    // fi: per-region axis / ARD
    double *axB = nullptr, *axKappa = nullptr, *axRho = nullptr, *axLogC = nullptr, *axCov = nullptr;
    double *ardShape = nullptr, *ardScale = nullptr, *ardMean = nullptr, *ardLogMean = nullptr;
    // spectral settings
    int32_t use_prior = 1;
    double nu = 1.0, ell = 1.0, sf = 1.0;
    bool basis_built = false;
    // invariants of the closed-form statistics (ci layers above the first): s (R, M), G (R, M, M), D (layer, R, M)
    double *sumPhi = nullptr, *gram = nullptr, *ancD = nullptr;
    int32_t *pc_ptr = nullptr, *pc_jp = nullptr, *pc_anc = nullptr;
    int64_t *pc_lo = nullptr, *pc_hi = nullptr;
    bool inv_built = false;
    double *rconst = nullptr;                // (R, 8) constants of the regions for the fused sweep (k_init_layer)
    AncEntry *anc_tab = nullptr;             // (R, E) pieces of every region, flattened (fused sweep)
    double *yc = nullptr, *ysum = nullptr;   // layer 0 (ci): Phi^T y (R, M, dy) and sum y, sum |y|^2 (R, 4) of the fused sweep
};

struct SharedDev {
    double *axB = nullptr, *axKappa = nullptr, *axRho = nullptr, *axLogC = nullptr, *axCov = nullptr;
    double *ardShape = nullptr, *ardScale = nullptr, *ardMean = nullptr, *ardLogMean = nullptr;
    double *omega = nullptr, *logOmegaHat = nullptr, *omegaIters = nullptr, *ardPartial = nullptr, *omegaEta = nullptr, *omegaWarm = nullptr, *omegaK = nullptr;
    double *primeB = nullptr, *primeLogC = nullptr, *primeShape = nullptr, *primeScale = nullptr, *primeSk = nullptr, *skTag = nullptr;
    double *priorB = nullptr, *priorLogC = nullptr, *priorShape = nullptr, *priorScale = nullptr;
};

}  // namespace

struct mrgp_handle {
    mrgp_config cfg{};
    int32_t n_ctas = 0;
    int64_t cta_quantum = 0;
    int32_t sm_count = 0;
    std::vector<LayerPlan> plan;
    std::vector<LayerDev> dev;
    SharedDev sh;
    size_t ws_bytes = 0;
    char *ws = nullptr;
    bool bound = false, have_data = false, state_init = false;
    bool ystats_valid = false;   // layer-0 sufficient statistics Phi^T y, sum y, sum |y|^2 match the current x, y, intervals
    bool sharded = false;
    int64_t lo = 0, hi = 0;   // owned samples [lo, hi)
    double *xchg = nullptr;   // dense exchange buffer (max R) x part_stride
    const double *x = nullptr, *y = nullptr;
    double *x_ws = nullptr, *y_ws = nullptr, *y_ws2 = nullptr, *g = nullptr, *hvar = nullptr, *tmp_mean = nullptr, *tmp_var = nullptr;
    double *part = nullptr, *elbo_out = nullptr, *elbo_part = nullptr;
    unsigned int *elbo_counter = nullptr;
    int elbo_chunks = 1;             // region chunks of the finest layer (grid.y of k_elbo)
    RegionArgs *elbo_args = nullptr;
    int64_t *off_staging = nullptr;
    size_t off_total = 0;
    int32_t part_stride = 0, max_runs = 0;
    unsigned long long *chol_count = nullptr;
    unsigned int *done_counter = nullptr, *mid_sync = nullptr;
    cudaStream_t stream = nullptr, side = nullptr;
    bool own_stream = false;
    std::vector<cudaEvent_t> ev_fork, ev_join, ev_ard, ev_mid2;
    cudaEvent_t ev_prefetch = nullptr, ev_b0_fork = nullptr, ev_b0_done = nullptr;
    cudaStream_t copy_stream = nullptr;   // mrgp_prefetch_observations_host: uploads beside the handle's stream
    cudaEvent_t ev_copy_done = nullptr, ev_y_free = nullptr, ev_elbo[2] = {nullptr, nullptr};
    bool elbo_no_sync = false;
    bool prefetch_pending = false, y_free_recorded = false;
    cudaStream_t side2 = nullptr;    // layer 0's phase B beside the chain of layer 1 (closed-form ci sweeps)
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graph_exec = nullptr;
    int64_t launches = 0, launches_per_sweep = 0, sweeps_done = 0;
    bool timeline = false;
    double *x_all = nullptr;         // sharded handles: inputs of ALL ranks (mrgp_set_all_inputs_host), else unused
    bool have_x_all = false;
    size_t state_begin = 0, state_end = 0;
    double *build_part = nullptr;    // split partials of the invariant builds
    size_t build_part_doubles = 0;
    // fused ci sweep (csrc/chain.cu): descriptor of this model in device memory, its host copy, guard status
    ChainModel *chain_dev = nullptr;
    const ChainModel **chain_ptr_dev = nullptr;
    ChainModel chain_host{};
    unsigned int *chain_status = nullptr;
    double *chain_guard = nullptr, *chain_prof = nullptr, *chain_tables = nullptr;
    double chain_guard_threshold = kChainGuard;   // MRGP_CHAIN_GUARD overrides (tests of the streamed fallback)
    bool chain_prof_on = false;      // MRGP_CHAIN_PROF=1: SM-clock stamps of the fused sweep (field 54)
    bool elbo_args_valid = false;    // the per-layer argument blocks of k_elbo on the device match generation / sweeps_done
    uint64_t elbo_args_key = 0;
    bool chain_uploaded = false;     // the device descriptor matches the current pointers (reset by drop_graph)
    uint64_t generation = 0;         // bumped whenever a captured sweep / descriptor becomes stale (groups re-capture)
    uint64_t stream_ops = 0;         // asynchronous work queued on the handle's stream from outside a sweep (groups order after it)
    bool fused = true;               // MRGP_FUSED=0: the multi-kernel sweep of round 1
    bool direct_launch = false;      // the fused sweep is launched on the stream, not through a graph (set once prefetched
                                     // observations are taken over: the buffers alternate, a graph would hold one pointer)
    int chain_cluster = 0;           // CTAs per model of the fused sweep (0: by the number of regions)
    bool inferred_shortcut = true;   // skip phase A where Phi^T r == 0 identically (MRGP_STREAM_ALL=1: stream everything)
    // peer-memory exchange (multi-GPU): arena + flags in one cudaMalloc'ed block that the peers map through CUDA IPC
    struct Comm {
        bool exported = false, ready = false;
        void *mem = nullptr;
        size_t bytes = 0, slot_doubles = 0;
        double *arena = nullptr;
        unsigned long long *flags = nullptr, *seq = nullptr;
        unsigned int *err = nullptr, *counter = nullptr;
        void *peer_base[kMaxRanks] = {};
        bool opened[kMaxRanks] = {};
        CommArgs args{};
    } comm;
    // adaptive basis intervals (BasisInterval.learn): the per-layer switches live in LayerDev
    int32_t ad_iters = 40;
    unsigned long long *brent_fail = nullptr;
    unsigned long long *ts = nullptr;   // (kMaxLayers * 4) x {begin, end} global-timer stamps
    double fi_shape0_mix = 0.0, fi_scale0_mix = 0.0;
    std::string err;
};

namespace {

int fail(mrgp_handle *h, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h)
        h->err = buf;
    else
        g_create_error = buf;
    return code;
}

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) cudaGetLastError();                                                       \
        if (e_ != cudaSuccess) return fail(h, MRGP_ECUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// Any number of basis functions up to 48: the streaming kernels are instantiated for 8, 20, 30, 40 and 48 functions and a
// model runs on the smallest instantiation that holds its basis, the extra functions carrying zero weight.
bool basis_supported(int m) { return m >= 1 && m <= 48; }
int padded_basis(int m) { return m <= 8 ? 8 : m <= 20 ? 20 : m <= 30 ? 30 : m <= 40 ? 40 : 48; }

// ---- plan -------------------------------------------------------------------------------------
void build_plan(mrgp_handle *h) {
    const int64_t lo = h->lo, N = h->hi;   // the owned chunk [lo, N)
    const int J = h->cfg.n_layers;
    const int64_t Q = h->cta_quantum;
    const int G = h->n_ctas;
    for (int j = 0; j < J; ++j) {
        LayerPlan &lp = h->plan[j];
        std::vector<int64_t> cuts;
        for (int64_t o : lp.offsets)
            if (o > lo && o < N) cuts.push_back(o);
        if (j > 0)
            for (int64_t o : h->plan[j - 1].offsets)
                if (o > lo && o < N) cuts.push_back(o);
        for (int c = 0; c < G; ++c) cuts.push_back(std::min<int64_t>(N, lo + (int64_t)c * Q));
        cuts.push_back(lo);
        cuts.push_back(N);
        std::sort(cuts.begin(), cuts.end());
        cuts.erase(std::unique(cuts.begin(), cuts.end()), cuts.end());
        lp.segs.clear();
        lp.seg_cta.clear();
        lp.cta_seg.assign(G + 1, 0);
        lp.region_run.assign(lp.R + 1, 0);
        int region = 0, parent = 0, run = -1, prev_cta = -1, prev_region = -1;
        const std::vector<int64_t> *poff = (j > 0) ? &h->plan[j - 1].offsets : nullptr;
        for (size_t k = 0; k + 1 < cuts.size(); ++k) {
            const int64_t s = cuts[k], e = cuts[k + 1];
            while (lp.offsets[region + 1] <= s) ++region;
            if (poff)
                while ((*poff)[parent + 1] <= s) ++parent;
            const int cta = (int)((s - lo) / Q);
            if (cta != prev_cta || region != prev_region) {
                ++run;
                if (region != prev_region)
                    for (int r = prev_region + 1; r <= region; ++r) lp.region_run[r] = run;
            }
            Segment sg;
            sg.start = s;
            sg.len = (int32_t)(e - s);
            sg.region = region;
            sg.parent = parent;
            sg.run = run;
            sg.flush = 0;
            sg.pad = 0;
            lp.segs.push_back(sg);
            lp.seg_cta.push_back(cta);
            prev_cta = cta;
            prev_region = region;
        }
        lp.n_runs = run + 1;
        for (int r = prev_region + 1; r <= lp.R; ++r) lp.region_run[r] = lp.n_runs;   // regions past the chunk: empty
        lp.ident_run.resize(lp.R + 1);
        for (int r = 0; r <= lp.R; ++r) lp.ident_run[r] = r;
        for (size_t k = 0; k < lp.segs.size(); ++k)
            lp.segs[k].flush = (k + 1 == lp.segs.size() || lp.segs[k + 1].run != lp.segs[k].run) ? 1 : 0;
        // first segment of each CTA (CTAs past the data get an empty range)
        size_t k = 0;
        for (int c = 0; c <= G; ++c) {
            while (k < lp.segs.size() && lp.seg_cta[k] < c) ++k;
            lp.cta_seg[c] = (int32_t)k;
        }
    }
}

// ---- workspace --------------------------------------------------------------------------------
struct Carver {
    char *base;
    size_t off = 0;
    explicit Carver(char *b) : base(b) {}
    template <typename T>
    T *take(size_t n) {
        off = (off + 255) & ~(size_t)255;
        T *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
        off += n * sizeof(T);
        return p;
    }
};

// Blocks per region of the invariant builds: about two waves of the SMs per layer.
int build_splits(int R) { return std::max(1, (296 + R - 1) / R); }

size_t carve(mrgp_handle *h, char *base) {
    Carver c(base);
    const int64_t N = h->hi - h->lo;   // local samples
    const int DY = h->cfg.dy, M = h->cfg.n_basis, J = h->cfg.n_layers;
    const bool fi = h->cfg.mode == MRGP_MODE_FI;
    h->x_ws = c.take<double>(N * h->cfg.dx);
    h->y_ws = c.take<double>(N * DY);
    h->y_ws2 = c.take<double>(N * DY);   // spare buffer of mrgp_prefetch_observations_host
    h->g = c.take<double>(N * DY);
    h->hvar = c.take<double>(N);
    h->tmp_mean = c.take<double>(N * DY);
    h->tmp_var = c.take<double>(N);
    h->max_runs = 0;
    for (int j = 0; j < J; ++j) h->max_runs = std::max(h->max_runs, h->plan[j].n_runs);
    h->part_stride = std::max(padded_basis(M) * DY + DY + 2, kPartBStride);   // phase A: MP*DY sums; y statistics: MP*DY + DY + 1
    h->part = c.take<double>((size_t)h->max_runs * h->part_stride);
    {
        int rmax = 1;
        for (int j = 0; j < J; ++j) rmax = std::max(rmax, h->plan[j].R);
        h->xchg = c.take<double>((size_t)rmax * h->part_stride);
    }
    if (!fi) {   // closed-form statistics (layers above the first) and sufficient statistics (layer 0)
        if (h->sharded) h->x_all = c.take<double>((size_t)h->cfg.n_samples * h->cfg.dx);   // replicated inputs: the invariants need every sample
        const size_t MPb = (size_t)padded_basis(M), np = MPb * (MPb + 1) / 2 + MPb;
        size_t need = 0;
        for (int j = 0; j < J; ++j) {
            const size_t blocks = (size_t)h->plan[j].R * build_splits(h->plan[j].R);
            const size_t P = h->plan[j].pc_jp.size();
            need = std::max(need, std::max(blocks * np, P * build_splits((int)std::max<size_t>(P, 1)) * MPb));
        }
        h->build_part_doubles = need;
        h->build_part = c.take<double>(need);
    }
    h->elbo_out = c.take<double>((size_t)J * 6);
    {
        int r_max = 1;
        for (int j = 0; j < J; ++j) r_max = std::max(r_max, h->plan[j].R);
        h->elbo_chunks = (r_max + kElboRegions - 1) / kElboRegions;
        h->elbo_part = c.take<double>((size_t)J * h->elbo_chunks * 6);
        h->elbo_counter = c.take<unsigned int>(J);
    }
    h->elbo_args = c.take<RegionArgs>(J);
    h->off_total = 0;
    for (int j = 0; j < J; ++j) h->off_total += h->plan[j].R + 1;
    h->off_staging = c.take<int64_t>(h->off_total);
    h->chol_count = c.take<unsigned long long>(1);
    h->done_counter = c.take<unsigned int>(1);
    h->brent_fail = c.take<unsigned long long>(1);
    h->mid_sync = c.take<unsigned int>(2 * kMaxLayers);
    h->ts = c.take<unsigned long long>(kMaxLayers * 8);
    h->state_begin = c.off;   // everything from here to state_end is the small-matrix state (L2 prefetch range)
    for (int j = 0; j < J; ++j) {
        const LayerPlan &lp = h->plan[j];
        LayerDev &d = h->dev[j];
        const size_t R = lp.R, RM = R * M;
        d.segs = c.take<Segment>(lp.segs.size());
        d.cta_seg = c.take<int32_t>(lp.cta_seg.size());
        d.region_run = c.take<int32_t>(lp.region_run.size());
        d.ident_run = c.take<int32_t>(lp.ident_run.size());
        d.offsets = c.take<int64_t>(lp.offsets.size());
        d.L = c.take<double>(R);
        d.inv2L = c.take<double>(R);
        d.rsqrtL = c.take<double>(R);
        d.lam = c.take<double>(RM);
        d.S = c.take<double>(RM);
        d.d = c.take<double>(RM);
        d.absx = c.take<double>(R);
        if (!fi) {
            d.sumPhi = c.take<double>(RM);
            d.rconst = c.take<double>(R * 8);
            if (j > 0) d.anc_tab = c.take<AncEntry>(R * (size_t)std::max(lp.E, 1));
        }
        if (!fi && j == 0) {
            d.yc = c.take<double>(RM * DY);
            d.ysum = c.take<double>(R * 4);
        }
        if (!fi && j > 0) {
            const size_t P = lp.pc_jp.size();
            d.ancD = c.take<double>(P * M);
            d.pc_ptr = c.take<int32_t>(lp.pc_ptr.size());
            d.pc_jp = c.take<int32_t>(P);
            d.pc_anc = c.take<int32_t>(P);
            d.pc_lo = c.take<int64_t>(P);
            d.pc_hi = c.take<int64_t>(P);
        }
        d.bias_prev = c.take<double>(R * DY);
        d.brent = c.take<double>(R * BrentState::NFIELDS);
        d.trial_inv2L = c.take<double>(R);
        d.trial_rsqrtL = c.take<double>(R);
        d.wq = c.take<double>(RM);
        d.inv2L_old = c.take<double>(R);
        d.rsqrtL_old = c.take<double>(R);
        d.sumsE = c.take<double>(R * (DY + 3));
        d.prec = c.take<double>(RM);
        d.zeta = c.take<double>(RM);
        d.ytil = c.take<double>(RM * DY);
        d.A = c.take<double>(RM * DY);
        d.A_prev = c.take<double>(RM * DY);
        d.m2 = c.take<double>(RM);
        d.cm2 = c.take<double>(RM);
        d.noise_shape = c.take<double>(R);
        d.noise_scale = c.take<double>(R);
        d.noise_shape0 = c.take<double>(R);
        d.noise_scale0 = c.take<double>(R);
        d.noise_mean = c.take<double>(R);
        d.noise_log_mean = c.take<double>(R);
        d.bias_prec = c.take<double>(R);
        d.bias_prec0 = c.take<double>(R);
        d.bias_mean = c.take<double>(R * DY);
        d.bias_mean0 = c.take<double>(R * DY);
        d.bias_var = c.take<double>(R);
        d.yvar = c.take<double>(R);
        d.sumsB = c.take<double>(R * (DY + 3));
        d.bcontrib = c.take<double>(std::max<size_t>(RM * 3, 48 * 160));
        d.wcontrib = c.take<double>((size_t)48 * 192);
        if (fi) {
            d.axB = c.take<double>(RM * DY * DY);
            d.axKappa = c.take<double>(RM * DY);
            d.axRho = c.take<double>(RM * DY);
            d.axLogC = c.take<double>(RM);
            d.axCov = c.take<double>(RM * DY * DY);
            d.ardShape = c.take<double>(RM);
            d.ardScale = c.take<double>(RM);
            d.ardMean = c.take<double>(RM);
            d.ardLogMean = c.take<double>(RM);
        }
    }
    SharedDev &s = h->sh;
    s.axB = c.take<double>((size_t)M * DY * DY);
    s.axKappa = c.take<double>((size_t)M * DY);
    s.axRho = c.take<double>((size_t)M * DY);
    s.axLogC = c.take<double>(M);
    s.axCov = c.take<double>((size_t)M * DY * DY);
    s.ardShape = c.take<double>(M);
    s.ardScale = c.take<double>(M);
    s.ardMean = c.take<double>(M);
    s.ardLogMean = c.take<double>(M);
    s.omega = c.take<double>((size_t)M * M);
    s.logOmegaHat = c.take<double>((size_t)M * M);
    s.omegaIters = c.take<double>(kMaxLayers);
    s.ardPartial = c.take<double>((size_t)256 * M);
    s.omegaEta = c.take<double>((size_t)kMaxLayers * 64);
    s.omegaWarm = c.take<double>(kMaxLayers);
    s.omegaK = c.take<double>((size_t)64 * 64 + 64);   // shifted, exponentiated table (column-major) + column shifts
    s.primeB = c.take<double>((size_t)M * DY * DY);
    s.primeLogC = c.take<double>(M);
    s.primeShape = c.take<double>(M);
    s.primeScale = c.take<double>(M);
    s.primeSk = c.take<double>(3 * 64);   // k-only terms of log omega_hat: slots for odd / even layers and layer 0
    s.skTag = c.take<double>(4);
    s.priorB = c.take<double>((size_t)M * DY * DY);
    s.priorLogC = c.take<double>(M);
    s.priorShape = c.take<double>(M);
    s.priorScale = c.take<double>(M);
    h->state_end = c.off;
    if (!fi) {
        for (int j = 0; j < J; ++j) h->dev[j].gram = c.take<double>((size_t)h->plan[j].R * M * M);   // layers > 0: read only when dA != 0
        h->chain_dev = c.take<ChainModel>(1);
        h->chain_ptr_dev = c.take<const ChainModel *>(1);
        h->chain_status = c.take<unsigned int>(4);
        h->chain_guard = c.take<double>(2);
        h->chain_prof = c.take<double>((size_t)kMaxLayers * 16);
        h->chain_tables = c.take<double>((size_t)kMaxLayers * 32 * 32);   // MRGP_CHAIN_PROF=1: log omega_hat of every layer (field 56)
    }
    return (c.off + 255) & ~(size_t)255;
}

// ---- argument packs -----------------------------------------------------------------------------
StreamArgs stream_args(mrgp_handle *h, int j) {
    const LayerDev &d = h->dev[j];
    StreamArgs a{};
    a.segs = d.segs;
    a.cta_seg = d.cta_seg;
    // kernels index samples by their global number: shift the (local) arrays by the chunk start
    a.x = h->x - h->lo;
    a.y = h->y - h->lo * h->cfg.dy;
    a.g = h->g - h->lo * h->cfg.dy;
    a.h = h->hvar - h->lo;
    a.inv2L = d.inv2L;
    a.rsqrtL = d.rsqrtL;
    a.A = d.A;
    a.A_prev = d.A_prev;
    a.cm2 = d.cm2;
    a.bias = d.bias_mean;
    a.pbias = j > 0 ? h->dev[j - 1].bias_mean : nullptr;
    a.pbias_var = j > 0 ? h->dev[j - 1].bias_var : nullptr;
    a.part = h->part;
    a.part_stride = h->part_stride;
    a.sample_begin = h->lo;
    a.n_samples = h->hi;
    a.cta_quantum = h->cta_quantum;
    a.done_counter = h->done_counter;
    a.region_run = d.region_run;
    a.offsets = d.offsets;
    a.R = h->plan[j].R;
    a.n_basis = h->cfg.n_basis;
    a.infer = (h->cfg.mode == MRGP_MODE_CI && j > 0) ? 1 : 0;
    a.fuse_tail = 0;
    a.layer = j;
    a.ts = h->timeline ? h->ts : nullptr;
    a.bias_prec0 = d.bias_prec0;
    a.bias_mean0 = d.bias_mean0;
    a.noise_shape0 = d.noise_shape0;
    a.noise_scale0 = d.noise_scale0;
    a.noise_rs = h->cfg.noise_region_specific ? 1 : 0;
    a.bias_rs = h->cfg.bias_region_specific ? 1 : 0;
    a.ci = h->cfg.mode == MRGP_MODE_CI ? 1 : 0;
    a.bias_mean_out = d.bias_mean;
    a.bias_prev_out = d.bias_prev;
    a.bias_prec = d.bias_prec;
    a.bias_var = d.bias_var;
    a.noise_shape = d.noise_shape;
    a.noise_scale = d.noise_scale;
    a.noise_mean = d.noise_mean;
    a.noise_log_mean = d.noise_log_mean;
    a.yvar = d.yvar;
    a.sumsB = d.sumsB;
    return a;
}

RegionArgs region_args(mrgp_handle *h, int j) {
    const LayerDev &d = h->dev[j];
    const SharedDev &s = h->sh;
    const bool fi = h->cfg.mode == MRGP_MODE_FI;
    RegionArgs a{};
    a.R = h->plan[j].R;
    a.M = h->cfg.n_basis;
    a.DY = h->cfg.dy;
    a.layer = j;
    a.mode = h->cfg.mode;
    a.infer = (!fi && j > 0) ? 1 : 0;
    a.region_run = d.region_run;
    a.offsets = d.offsets;
    a.part = h->part;
    a.part_stride = h->part_stride;
    a.L = d.L;
    a.inv2L = d.inv2L;
    a.rsqrtL = d.rsqrtL;
    a.lam = d.lam;
    a.S = d.S;
    a.d = d.d;
    a.absx = d.absx;
    a.prec = d.prec;
    a.zeta = d.zeta;
    a.ytil = d.ytil;
    a.A = d.A;
    a.A_prev = d.A_prev;
    a.m2 = d.m2;
    a.cm2 = d.cm2;
    a.noise_shape = d.noise_shape;
    a.noise_scale = d.noise_scale;
    a.noise_shape0 = d.noise_shape0;
    a.noise_scale0 = d.noise_scale0;
    a.noise_mean = d.noise_mean;
    a.noise_log_mean = d.noise_log_mean;
    a.bias_prec = d.bias_prec;
    a.bias_prec0 = d.bias_prec0;
    a.bias_mean = d.bias_mean;
    a.bias_mean0 = d.bias_mean0;
    a.bias_var = d.bias_var;
    a.yvar = d.yvar;
    a.sumsB = d.sumsB;
    a.bcontrib = d.bcontrib;
    a.wcontrib = d.wcontrib;
    if (fi) {
        a.axB = d.axB;
        a.axKappa = d.axKappa;
        a.axRho = d.axRho;
        a.axLogC = d.axLogC;
        a.axCov = d.axCov;
        a.ardShape = d.ardShape;
        a.ardScale = d.ardScale;
        a.ardMean = d.ardMean;
        a.ardLogMean = d.ardLogMean;
    } else {
        a.axB = s.axB;
        a.axKappa = s.axKappa;
        a.axRho = s.axRho;
        a.axLogC = s.axLogC;
        a.axCov = s.axCov;
        a.ardShape = s.ardShape;
        a.ardScale = s.ardScale;
        a.ardMean = s.ardMean;
        a.ardLogMean = s.ardLogMean;
    }
    a.omega = s.omega;
    a.logOmegaHat = s.logOmegaHat;
    a.omegaIters = s.omegaIters;
    a.ardPartial = s.ardPartial;
    a.omegaEta = s.omegaEta;
    a.omegaWarm = s.omegaWarm;
    a.omegaK = s.omegaK;
    a.primeB = s.primeB;
    a.primeLogC = s.primeLogC;
    a.primeShape = s.primeShape;
    a.primeScale = s.primeScale;
    a.primeSk = s.primeSk;
    a.skTag = s.skTag;
    a.priorB = s.priorB;
    a.priorLogC = s.priorLogC;
    a.priorShape = s.priorShape;
    a.priorScale = s.priorScale;
    a.chol_count = h->chol_count;
    a.ts = h->timeline ? h->ts : nullptr;
    a.fi_shape0_mix = h->fi_shape0_mix;
    a.fi_scale0_mix = h->fi_scale0_mix;
    if (h->sharded) {   // the small-matrix steps read the all-reduced dense statistics: one "run" per region
        a.region_run = d.ident_run;
        a.part = h->xchg;
    }
    a.rconst = d.rconst;
    a.use_prior = d.use_prior;
    a.nu = d.nu;
    a.ell = d.ell;
    a.sf = d.sf;
    a.interval_factor = 1.0;
    a.L_given = 0;
    a.zero_T = 0;
    return a;
}

// ---- kernel dispatch ----------------------------------------------------------------------------
constexpr size_t kRedSmemBytes = kRedSmemDoubles * sizeof(double);

// Every kernel of the sweep asks for the same (maximum) shared-memory carveout: switching the L1 / shared split
// between consecutive kernels drains and reconfigures the SMs, which costs more than the small kernels run.
// The dynamic shared-memory limit of a kernel is process-wide state that captured graphs of other models rely on:
// it is only ever RAISED (a high-water mark per kernel function, guarded by a mutex), never rewritten to a smaller
// launch's size.
std::mutex g_smem_mu;
std::map<const void *, size_t> g_smem_high_water;

template <typename K>
cudaError_t set_smem(K kernel, size_t bytes) {
    std::lock_guard<std::mutex> lock(g_smem_mu);
    const void *key = reinterpret_cast<const void *>(kernel);
    auto it = g_smem_high_water.find(key);
    if (it == g_smem_high_water.end()) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        it = g_smem_high_water.emplace(key, 0).first;
    }
    bytes = std::max<size_t>(bytes, 1);
    if (bytes <= it->second) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) it->second = bytes;
    return e;
}

template <int M>
cudaError_t launch_phase_a(mrgp_handle *h, cudaStream_t stream, const StreamArgs &a, bool infer, bool latent) {
    constexpr int DY = 2;
    dim3 grid(h->n_ctas), block(kThreads);
#define LA(I, L)                                                                                               \
    {                                                                                                          \
        const size_t smem = (size_t)(kStages * TileLayout<DY, !(I), (L), false>::kDoubles + kRedSmemDoubles) * sizeof(double); \
        cudaError_t e = set_smem(k_phase_a<DY, M, I, L>, smem);                                                \
        if (e != cudaSuccess) return e;                                                                        \
        k_phase_a<DY, M, I, L><<<grid, block, smem, stream>>>(a);                                              \
    }
    if (infer)
        LA(true, true)
    else if (latent)
        LA(false, true)
    else
        LA(false, false)
#undef LA
    return cudaGetLastError();
}

template <int M>
cudaError_t launch_phase_b(mrgp_handle *h, cudaStream_t stream, const StreamArgs &a, bool infer, bool latent, bool prop) {
    constexpr int DY = 2;
    dim3 grid(h->n_ctas), block(kThreadsB);
#define LB(I, L, P)                                                                                         \
    {                                                                                                       \
        const size_t smem = (size_t)(kStages * TileLayout<DY, !(I), (L), (L)>::kDoubles) * sizeof(double);  \
        cudaError_t e = set_smem(k_phase_b<DY, M, I, L, P>, smem);                                          \
        if (e != cudaSuccess) return e;                                                                     \
        k_phase_b<DY, M, I, L, P><<<grid, block, smem, stream>>>(a);                                        \
    }
    if (infer) {
        if (prop)
            LB(true, true, true)
        else
            LB(true, true, false)
    } else if (latent) {
        if (prop)
            LB(false, true, true)
        else
            LB(false, true, false)
    } else {
        if (prop)
            LB(false, false, true)
        else
            LB(false, false, false)
    }
#undef LB
    return cudaGetLastError();
}

template <int M>
cudaError_t launch_phi2sum(mrgp_handle *h, cudaStream_t stream, const StreamArgs &a) {
    cudaError_t e = set_smem(k_phi2sum<M>, kRedSmemBytes);
    if (e != cudaSuccess) return e;
    k_phi2sum<M><<<h->n_ctas, kThreads, kRedSmemBytes, stream>>>(a);
    return cudaGetLastError();
}

#define DISPATCH_M(m, expr)                     \
    switch (padded_basis(m)) {                  \
        case 8: { constexpr int MM = 8; expr; } break;   \
        case 20: { constexpr int MM = 20; expr; } break; \
        case 30: { constexpr int MM = 30; expr; } break; \
        case 40: { constexpr int MM = 40; expr; } break; \
        case 48: { constexpr int MM = 48; expr; } break; \
        default: break;                         \
    }

int check_ready(mrgp_handle *h, int layer, bool need_state) {
    if (!h) return MRGP_EINVAL;
    if (!h->bound) return fail(h, MRGP_ESTATE, "no workspace bound");
    if (!h->have_data) return fail(h, MRGP_ESTATE, "no data set");
    if (layer < 0 || layer >= h->cfg.n_layers) return fail(h, MRGP_EINVAL, "layer %d out of range", layer);
    if (need_state && !h->state_init) return fail(h, MRGP_ESTATE, "state not initialised");
    if (need_state)
        for (int j = 0; j < h->cfg.n_layers; ++j)
            if (!h->dev[j].basis_built)
                return fail(h, MRGP_ESTATE, "the inputs changed: rebuild the basis of layer %d (mrgp_build_basis) before the next phase or sweep", j);
    return MRGP_OK;
}

// Where a helper enqueues its work and which counter its kernel launches add to: the handle's stream and
// mrgp_handle::launches outside a sweep; a captured sweep counts into its own per-sweep count, and a branch of a sweep
// onto another stream keeps the counter of the sweep.
struct Launch {
    cudaStream_t stream;
    int64_t *count;
};

// ---- the phases ---------------------------------------------------------------------------------
int do_phase_a(mrgp_handle *h, const Launch &L, int j) {
    const bool fi = h->cfg.mode == MRGP_MODE_FI;
    const bool infer = !fi && j > 0, latent = j > 0;
    StreamArgs a = stream_args(h, j);
    cudaError_t e = cudaErrorInvalidValue;
    DISPATCH_M(h->cfg.n_basis, e = launch_phase_a<MM>(h, L.stream, a, infer, latent));
    CK(e);
    *L.count += 1;
    return MRGP_OK;
}

int reduce_threads(int nv, int max_runs_per_region, int cap) {
    const int nval = (nv + 31) & ~31;
    int slices = std::max(1, std::min(cap / nval, max_runs_per_region));
    return nval * slices;
}

int max_region_runs(const LayerPlan &lp) {
    int m = 1;
    for (int r = 0; r < lp.R; ++r) m = std::max(m, lp.region_run[r + 1] - lp.region_run[r]);
    return m;
}

int do_mid_ci(mrgp_handle *h, const Launch &L, int j, bool fork_omega, bool zero_T = false);

int do_axis_update(mrgp_handle *h, const Launch &L, int j, bool fork_omega, bool zero_T = false) {
    const bool fi = h->cfg.mode == MRGP_MODE_FI;
    const int M = h->cfg.n_basis, DY = h->cfg.dy;
    if (!fi) return do_mid_ci(h, L, j, fork_omega, zero_T);
    RegionArgs a = region_args(h, j);
    const LayerPlan &lp = h->plan[j];
    {
        const int nv = M * DY, nval = (nv + 31) & ~31;
        const int threads = std::max(reduce_threads(nv, h->sharded ? 1 : max_region_runs(lp), 512), ((M + 31) & ~31));
        const int slices = threads / nval;
        const size_t smem = (size_t)(slices * nval + nv) * sizeof(double);
        CK(set_smem(k_reduce_scale<2>, smem));
        k_reduce_scale<2><<<lp.R, threads, smem, L.stream>>>(a);
        CK(cudaGetLastError());
        *L.count += 1;
    }
    return MRGP_OK;
}

int do_mid_ci(mrgp_handle *h, const Launch &L, int j, bool fork_omega, bool zero_T) {
    const int M = h->cfg.n_basis;
    RegionArgs a = region_args(h, j);
    a.zero_T = zero_T ? 1 : 0;
    const LayerPlan &lp = h->plan[j];
    if (fork_omega && j > 0) CK(cudaStreamWaitEvent(L.stream, h->ev_ard[j - 1], 0));   // k_mid1 reads ard_mean
    int n_partials = 1;
    {
        const int mr = h->sharded ? 1 : max_region_runs(lp);
        int nb = std::min(32, lp.R);
        const int rpc = (lp.R + nb - 1) / nb;
        nb = (lp.R + rpc - 1) / rpc;
        const int items_cta = std::min(rpc, 32) * M;
        int lpi = 1;
        while (lpi < 32 && lpi * 2 <= mr && lpi * 2 * items_cta <= kMidThreads) lpi *= 2;
        const int nvp = (M * 3 + 31) & ~31, nvwp = (M * 4 + 31) & ~31;
        const size_t smem1 = (size_t)(2 * 32 * M * 4 + nvp + nvwp) * sizeof(double);
        CK(set_smem(k_mid1<2>, smem1));
        k_mid1<2><<<nb, kMidThreads, smem1, L.stream>>>(a, lpi, rpc);
        CK(cudaGetLastError());
        *L.count += 1;
        n_partials = nb;
        // The critical chain of the sweep is omega(j-1) -> axis / ARD update and table (k_ard) -> omega(j): k_ard only
        // needs the region sums of k_mid1, so it is forked here and runs beside k_mid2 (S2 of the regions).
        cudaStream_t st = L.stream;
        if (fork_omega) {
            CK(cudaEventRecord(h->ev_fork[j], L.stream));
            CK(cudaStreamWaitEvent(h->side, h->ev_fork[j], 0));
            st = h->side;
        }
        const size_t smem = omega_smem_doubles(M) * sizeof(double);
        if (fork_omega) {
            CK(set_smem(k_ard, smem));
            k_ard<<<1, kOmegaThreads, smem, st>>>(a, n_partials);
            CK(cudaGetLastError());
            CK(cudaEventRecord(h->ev_ard[j], h->side));
        }
        int nb2 = std::min(48, lp.R);
        const int rpc2 = (lp.R + nb2 - 1) / nb2;
        nb2 = (lp.R + rpc2 - 1) / rpc2;
        const size_t smem2 = (size_t)(std::max(33 * M, M * M + 4 * M + 3 * nvp) + 4 * M) * sizeof(double);
        if (fork_omega && j > 0) CK(cudaStreamWaitEvent(L.stream, h->ev_join[j - 1], 0));   // k_mid2 reads omega
        CK(set_smem(k_mid2<2>, smem2));
        k_mid2<2><<<nb2, kMidThreads, smem2, L.stream>>>(a, rpc2, nb);
        CK(cudaGetLastError());
        *L.count += 1;
        if (fork_omega) {
            // k_scale_warp overwrites omega, which k_mid2 reads
            CK(cudaEventRecord(h->ev_mid2[j], L.stream));
            CK(cudaStreamWaitEvent(h->side, h->ev_mid2[j], 0));
        } else {
            CK(set_smem(k_ard, smem));
            k_ard<<<1, kOmegaThreads, smem, st>>>(a, n_partials);
            CK(cudaGetLastError());
        }
        if (M == 30) {
            CK(cudaFuncSetAttribute(k_scale_warp<30>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
            k_scale_warp<30><<<1, 64, 0, st>>>(a);
        } else if (M == 20) {
            CK(cudaFuncSetAttribute(k_scale_warp<20>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
            k_scale_warp<20><<<1, 64, 0, st>>>(a);
        } else if (M == 8) {
            CK(cudaFuncSetAttribute(k_scale_warp<8>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
            k_scale_warp<8><<<1, 64, 0, st>>>(a);
        } else {
            CK(set_smem(k_scale, smem));
            k_scale<<<1, kOmegaThreads, smem, st>>>(a);
        }
        CK(cudaGetLastError());
        *L.count += 2;
        if (fork_omega) CK(cudaEventRecord(h->ev_join[j], h->side));
    }
    return MRGP_OK;
}

int do_bias_noise_shared(mrgp_handle *h, const Launch &L, int j);

// `gate`: when not null the kernel runs only if *gate != 0 (the streamed fallback of the fused sweep).
int do_phase_b(mrgp_handle *h, const Launch &L, int j, bool fuse_tail, int prop_override = -1, const unsigned int *gate = nullptr) {
    const bool fi = h->cfg.mode == MRGP_MODE_FI;
    const bool infer = !fi && j > 0, latent = j > 0;
    const bool prop = prop_override < 0 ? (j + 1 < h->cfg.n_layers) : (prop_override != 0);
    StreamArgs a = stream_args(h, j);
    a.fuse_tail = fuse_tail ? 1 : 0;
    a.gate = gate;
    cudaError_t e = cudaErrorInvalidValue;
    DISPATCH_M(h->cfg.n_basis, e = launch_phase_b<MM>(h, L.stream, a, infer, latent, prop));
    CK(e);
    *L.count += 1;
    return fuse_tail ? do_bias_noise_shared(h, L, j) : MRGP_OK;
}

// Second stage of the bias / noise update when noise or bias is shared by the regions of a layer.
int do_bias_noise_shared(mrgp_handle *h, const Launch &L, int j) {
    if (h->cfg.noise_region_specific && h->cfg.bias_region_specific) return MRGP_OK;
    StreamArgs a = stream_args(h, j);
    k_bias_noise_shared<2><<<1, 256, 0, L.stream>>>(a);
    CK(cudaGetLastError());
    *L.count += 1;
    return MRGP_OK;
}

int do_bias_noise(mrgp_handle *h, const Launch &L, int j) {
    StreamArgs a = stream_args(h, j);
    if (h->sharded) {
        a.region_run = h->dev[j].ident_run;
        a.part = h->xchg;
    }
    k_bias_noise<2><<<std::max(1, std::min(32, (h->plan[j].R + 7) / 8)), kThreadsB, 0, L.stream>>>(a);
    CK(cudaGetLastError());
    *L.count += 1;
    return do_bias_noise_shared(h, L, j);
}

// One exchange over peer memory: local dense sums -> arena slot (picked on the device from the exchange number),
// publish, reduce over the owning ranks -> h->xchg.
int do_exchange(mrgp_handle *h, const Launch &L, int j, int nv, bool is_max) {
    if (!h->comm.ready) return fail(h, MRGP_ESTATE, "no peer exchange bound: mrgp_comm_export / mrgp_comm_bind first");
    const LayerPlan &lp = h->plan[j];
    LayerDev &d = h->dev[j];
    const int total = lp.R * h->part_stride;
    if (h->part_stride > 256) return fail(h, MRGP_EINVAL, "exchange rows of more than 256 values are not supported");
    if (is_max)
        k_comm_sums_signal<true><<<lp.R, 256, 0, L.stream>>>(h->comm.args, d.region_run, h->part, h->part_stride, nv, h->comm.arena, h->comm.counter);
    else
        k_comm_sums_signal<false><<<lp.R, 256, 0, L.stream>>>(h->comm.args, d.region_run, h->part, h->part_stride, nv, h->comm.arena, h->comm.counter);
    CK(cudaGetLastError());
    const int grid = std::max(1, std::min(96, (total + 255) / 256));
    if (is_max)
        k_comm_reduce<true><<<grid, 256, 0, L.stream>>>(h->comm.args, d.offsets, lp.R, h->part_stride, nv, h->xchg);
    else
        k_comm_reduce<false><<<grid, 256, 0, L.stream>>>(h->comm.args, d.offsets, lp.R, h->part_stride, nv, h->xchg);
    CK(cudaGetLastError());
    *L.count += 2;
    return MRGP_OK;
}

template <int M>
cudaError_t launch_objective(mrgp_handle *h, cudaStream_t stream, const IntervalArgs &q, bool infer, bool latent) {
    dim3 grid(h->n_ctas), block(kThreads);
    if (infer)
        k_interval_objective<2, M, true, true><<<grid, block, 0, stream>>>(q);
    else if (latent)
        k_interval_objective<2, M, false, true><<<grid, block, 0, stream>>>(q);
    else
        k_interval_objective<2, M, false, false><<<grid, block, 0, stream>>>(q);
    return cudaGetLastError();
}

template <int M>
cudaError_t launch_elbo_sums(mrgp_handle *h, cudaStream_t stream, const IntervalArgs &q, bool infer, bool latent) {
    dim3 grid(h->n_ctas), block(kThreads);
    if (infer)
        k_adaptive_elbo_sums<2, M, true, true><<<grid, block, 0, stream>>>(q);
    else if (latent)
        k_adaptive_elbo_sums<2, M, false, true><<<grid, block, 0, stream>>>(q);
    else
        k_adaptive_elbo_sums<2, M, false, false><<<grid, block, 0, stream>>>(q);
    return cudaGetLastError();
}

// B1: BasisInterval.learn for one layer (BasisInterval.py:18-134), then the rebuild of lambda, S and sum phi^2
// (MRGP.py:640-641).  ci mode only (MRGP.py:108-109 switches it off for fi).
int do_learn_intervals(mrgp_handle *h, const Launch &L, int j) {
    LayerDev &d = h->dev[j];
    const LayerPlan &lp = h->plan[j];
    const int M = h->cfg.n_basis;
    const bool infer = j > 0, latent = j > 0;
    BrentArgs b{};
    b.R = lp.R;
    b.M = M;
    b.first = 1;
    b.region_run = d.region_run;
    b.part = h->part;
    b.part_stride = h->part_stride;
    b.st = d.brent;
    b.trial_inv2L = d.trial_inv2L;
    b.trial_rsqrtL = d.trial_rsqrtL;
    b.noise_mean = d.noise_mean;
    b.ard_mean = h->sh.ardMean;
    b.m2 = d.m2;
    b.use_prior = d.ad_use_prior ? 1 : 0;
    b.nu = d.nu;
    b.ell = d.ell;
    b.sf = d.sf;
    b.xatol = 1e-5;
    b.maxfun = 500;
    const int total = lp.R * M;
    k_brent_start<<<(total + 127) / 128, 128, 0, L.stream>>>(b, d.absx, d.ad_lo, d.ad_hi, d.A, d.cm2, d.wq);
    CK(cudaGetLastError());
    *L.count += 1;
    IntervalArgs q{};
    q.s = stream_args(h, j);
    q.trial_inv2L = d.trial_inv2L;
    q.trial_rsqrtL = d.trial_rsqrtL;
    q.w = d.wq;
    q.bias_old = d.bias_prev;
    for (int it = 0; it < h->ad_iters; ++it) {
        cudaError_t e = cudaErrorInvalidValue;
        DISPATCH_M(M, e = launch_objective<MM>(h, L.stream, q, infer, latent));
        CK(e);
        b.first = (it == 0) ? 1 : 0;
        k_brent_step<<<(lp.R + 3) / 4, 128, 0, L.stream>>>(b);
        CK(cudaGetLastError());
        *L.count += 2;
    }
    k_brent_finish<<<(lp.R + 127) / 128, 128, 0, L.stream>>>(b, d.L, h->brent_fail);
    CK(cudaGetLastError());
    // the targets of this step were inferred with the current basis: keep it for the lower bound
    CK(cudaMemcpyAsync(d.inv2L_old, d.inv2L, lp.R * sizeof(double), cudaMemcpyDeviceToDevice, L.stream));
    CK(cudaMemcpyAsync(d.rsqrtL_old, d.rsqrtL, lp.R * sizeof(double), cudaMemcpyDeviceToDevice, L.stream));
    RegionArgs ra = region_args(h, j);
    ra.L_given = 1;
    k_region_setup<<<(lp.R + 7) / 8, 256, 0, L.stream>>>(ra);
    CK(cudaGetLastError());
    StreamArgs sa = stream_args(h, j);
    cudaError_t e = cudaErrorInvalidValue;
    DISPATCH_M(M, e = launch_phi2sum<MM>(h, L.stream, sa));
    CK(e);
    k_reduce_d<<<lp.R, 64, 0, L.stream>>>(ra);
    CK(cudaGetLastError());
    *L.count += 4;
    // data-term sums of the lower bound with the re-learnt basis (before the propagation overwrites g, h)
    {
        IntervalArgs qe{};
        qe.s = stream_args(h, j);
        qe.trial_inv2L = d.inv2L_old;
        qe.trial_rsqrtL = d.rsqrtL_old;
        qe.w = nullptr;
        qe.bias_old = d.bias_prev;
        cudaError_t ee = cudaErrorInvalidValue;
        DISPATCH_M(M, ee = launch_elbo_sums<MM>(h, L.stream, qe, infer, latent));
        CK(ee);
        StreamArgs se = stream_args(h, j);
        se.sums_only = 1;
        se.sumsB = d.sumsE;
        k_bias_noise<2><<<std::max(1, std::min(32, (lp.R + 7) / 8)), kThreadsB, 0, L.stream>>>(se);
        CK(cudaGetLastError());
        *L.count += 2;
    }
    return MRGP_OK;
}

int fill_eval_layers(mrgp_handle *h, EvalArgs &ea, int n_layers, const int64_t *const *dev_offsets);

// ci, static intervals, nested regions, one GPU: the layers above the first take their P4 / P5 statistics in closed
// form (k_stats_b) instead of streaming the samples.
bool use_closed_form(const mrgp_handle *h) {
    if (h->cfg.mode != MRGP_MODE_CI || !h->inferred_shortcut || !h->build_part) return false;
    if (h->sharded && !h->have_x_all) return false;
    for (const auto &d : h->dev)
        if (d.adaptive) return false;
    return h->cfg.n_layers > 1;
}

// The fused sweep (csrc/chain.cu): ci, static intervals, region-specific noise and bias, M <= 32.  Everything else
// (fi, adaptive intervals, shared noise / bias, M > 32, MRGP_STREAM_ALL=1, MRGP_FUSED=0) takes the multi-kernel sweep.
bool use_fused(const mrgp_handle *h) {
    if (!h->fused || h->cfg.mode != MRGP_MODE_CI || !h->inferred_shortcut || !h->build_part || !h->chain_dev) return false;
    if (h->sharded && !h->have_x_all) return false;
    if (!h->cfg.noise_region_specific || !h->cfg.bias_region_specific) return false;
    if (h->cfg.dy != 2 || chain_solver_size(h->cfg.n_basis) == 0) return false;
    if (h->timeline && h->cfg.n_layers > kMaxLayersTs) return false;
    for (const auto &d : h->dev)
        if (d.adaptive) return false;
    return true;
}

template <int M>
int launch_build_invariants(mrgp_handle *h, const Launch &L, int j) {
    LayerDev &d = h->dev[j];
    const LayerPlan &lp = h->plan[j];
    const int splits = build_splits(lp.R), blocks = lp.R * splits;
    constexpr int NP = M * (M + 1) / 2;
    CK(cudaFuncSetAttribute(k_build_gram<M>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    const double *xg = h->sharded ? h->x_all : h->x;   // indexed by the global sample number
    k_build_gram<M><<<blocks, 256, 0, L.stream>>>(xg, d.offsets, d.inv2L, d.rsqrtL, splits, h->build_part);
    CK(cudaGetLastError());
    k_reduce_gram<<<(lp.R * (NP + M) + 255) / 256, 256, 0, L.stream>>>(h->build_part, splits, lp.R, h->cfg.n_basis, M, d.gram, d.sumPhi);
    CK(cudaGetLastError());
    *L.count += 2;
    if (j > 0) {
        EvalArgs ea{};
        int rc = fill_eval_layers(h, ea, j, nullptr);
        if (rc) return rc;
        const int P = (int)lp.pc_jp.size(), psplits = build_splits(P);
        const PieceTable pt{d.pc_ptr, d.pc_jp, d.pc_anc, d.pc_lo, d.pc_hi, P};
        k_build_ancD<M><<<P * psplits, 256, 0, L.stream>>>(ea, xg, pt, psplits, h->build_part);
        CK(cudaGetLastError());
        k_reduce_ancD<<<(P * h->cfg.n_basis + 255) / 256, 256, 0, L.stream>>>(h->build_part, psplits, P, h->cfg.n_basis, M, d.ancD);
        CK(cudaGetLastError());
        *L.count += 2;
    }
    d.inv_built = true;
    return MRGP_OK;
}

int build_invariants(mrgp_handle *h, const Launch &L) {
    const bool fused = use_fused(h);
    if (!use_closed_form(h) && !fused) return MRGP_OK;
    for (int j = fused ? 0 : 1; j < h->cfg.n_layers; ++j) {
        if (h->dev[j].inv_built) continue;
        int rc = MRGP_EINVAL;
        DISPATCH_M(h->cfg.n_basis, rc = launch_build_invariants<MM>(h, L, j));
        if (rc) return rc;
    }
    return MRGP_OK;
}

int do_stats_b(mrgp_handle *h, const Launch &L, int j) {
    LayerDev &d = h->dev[j];
    StatsBArgs q{};
    q.p = stream_args(h, j);
    q.p.infer = 1;
    int rc = fill_eval_layers(h, q.anc, j, nullptr);
    if (rc) return rc;
    q.s = d.sumPhi;
    q.G = d.gram;
    q.D = d.ancD;
    q.pt = PieceTable{d.pc_ptr, d.pc_jp, d.pc_anc, d.pc_lo, d.pc_hi, (int32_t)h->plan[j].pc_jp.size()};
    q.A = d.A;
    q.A_prev = d.A_prev;
    q.d = d.d;
    q.cm2 = d.cm2;
    CK(cudaFuncSetAttribute(k_stats_b<2>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    k_stats_b<2><<<(h->plan[j].R + 7) / 8, 256, 0, L.stream>>>(q);
    CK(cudaGetLastError());
    *L.count += 1;
    return do_bias_noise_shared(h, L, j);
}

// Sufficient statistics of the observations for layer 0 of the fused sweep: Phi^T y, sum y, sum |y|^2 per region
// (one pass over x and y; again whenever y, x or the intervals of layer 0 change).
template <int M>
cudaError_t launch_ystats(mrgp_handle *h, cudaStream_t stream, const StreamArgs &a) {
    constexpr int DY = 2;
    const size_t smem = (size_t)(kStages * TileLayout<DY, true, false, false>::kDoubles + kRedSmemDoubles) * sizeof(double);
    cudaError_t e = set_smem(k_ystats<DY, M>, smem);
    if (e != cudaSuccess) return e;
    k_ystats<DY, M><<<h->n_ctas, kThreads, smem, stream>>>(a);
    return cudaGetLastError();
}

int upload_chain_model(mrgp_handle *h);

bool ystats_small(const mrgp_handle *h) {
    if (h->sharded) return false;
    const LayerPlan &lp = h->plan[0];
    for (int r = 0; r < lp.R; ++r)
        if (lp.offsets[r + 1] - lp.offsets[r] > kYstatsSmallMaxRegion) return false;
    return true;
}

int do_ystats(mrgp_handle *h, const Launch &L) {
    LayerDev &d = h->dev[0];
    const LayerPlan &lp = h->plan[0];
    const int M = h->cfg.n_basis, DY = h->cfg.dy;
    if (ystats_small(h)) {   // one CTA per region of layer 0, straight from the descriptor (the form a batch of series uses)
        int rc = h->chain_uploaded ? MRGP_OK : upload_chain_model(h);
        if (rc) return rc;
        const int e = launch_ystats_small(chain_solver_size(M), h->chain_ptr_dev, 1, lp.R, L.stream);
        if (e != 0) return fail(h, MRGP_ECUDA, "y statistics launch: %s", cudaGetErrorString((cudaError_t)e));
        *L.count += 1;
        h->ystats_valid = true;
        return MRGP_OK;
    }
    StreamArgs a = stream_args(h, 0);
    // one handle: the last CTA of the pass sums the run partials itself (no second launch); sharded: the partials of
    // the ranks' chunks are exchanged first
    const bool fuse = !h->sharded && lp.R <= 64;
    a.fuse_tail = fuse ? 1 : 0;
    a.yc_out = d.yc;
    a.ysum_out = d.ysum;
    cudaError_t e = cudaErrorInvalidValue;
    DISPATCH_M(M, e = launch_ystats<MM>(h, L.stream, a));
    CK(e);
    *L.count += 1;
    if (!fuse) {
        const int32_t *rr = d.region_run;
        const double *part = h->part;
        if (h->sharded) {   // sum the statistics of the ranks' chunks
            int rc = do_exchange(h, L, 0, padded_basis(M) * DY + DY + 1, false);
            if (rc) return rc;
            rr = d.ident_run;
            part = h->xchg;
        }
        k_reduce_ystats<<<lp.R, 1024, 0, L.stream>>>(rr, part, h->part_stride, lp.R, M, padded_basis(M), DY, d.yc, d.ysum);
        CK(cudaGetLastError());
        *L.count += 1;
    }
    h->ystats_valid = true;
    return MRGP_OK;
}

int chain_cluster_size(const mrgp_handle *h) {
    if (h->chain_cluster > 0) return h->chain_cluster;
    int rmax = 1;
    for (const auto &lp : h->plan) rmax = std::max(rmax, lp.R);
    return rmax <= 32 ? 1 : rmax <= 64 ? 2 : rmax <= 128 ? 4 : rmax <= 256 ? 8 : 16;
}

// Descriptor of the model for the fused sweep (device pointers only; uploaded before the sweep is captured).
int upload_chain_model(mrgp_handle *h) {
    ChainModel &m = h->chain_host;
    const SharedDev &s = h->sh;
    std::memset(&m, 0, sizeof m);
    m.J = h->cfg.n_layers;
    m.M = h->cfg.n_basis;
    m.DY = h->cfg.dy;
    m.sbase = reinterpret_cast<double *>(h->ws + h->state_begin);
    m.pf_base = h->ws + h->state_begin;
    m.pf_lines = (h->state_end - h->state_begin + 127) / 128;
    m.x = h->x - h->lo;
    m.y = h->y - h->lo * h->cfg.dy;
    m.axB = s.axB; m.axKappa = s.axKappa; m.axRho = s.axRho; m.axLogC = s.axLogC; m.axCov = s.axCov;
    m.ardShape = s.ardShape; m.ardScale = s.ardScale; m.ardMean = s.ardMean; m.ardLogMean = s.ardLogMean;
    m.omega = s.omega; m.logOmegaHat = s.logOmegaHat; m.omegaIters = s.omegaIters; m.omegaEta = s.omegaEta; m.omegaWarm = s.omegaWarm;
    m.priorB = s.priorB; m.priorLogC = s.priorLogC; m.priorShape = s.priorShape; m.priorScale = s.priorScale;
    m.priorSk = s.primeSk + 2 * 64;    // k-only terms of the table for layer 0 (k_init_shared)
    m.chol_count = h->chol_count;
    m.status = h->chain_status;
    m.guard = h->chain_guard;
    m.guard_threshold = h->chain_guard_threshold;
    m.ts = h->timeline ? h->ts : nullptr;
    m.prof = h->chain_prof_on ? h->chain_prof : nullptr;
    m.tables = (h->chain_prof_on && h->cfg.n_basis <= 32) ? h->chain_tables : nullptr;
    for (int j = 0; j < m.J; ++j) {
        const LayerDev &d = h->dev[j];
        ChainLayer &l = m.layer[j];
        l.R = h->plan[j].R;
        l.P = (int32_t)h->plan[j].pc_jp.size();
        l.offsets = d.offsets;
        l.E = std::max(h->plan[j].E, 1);
        l.anc_tab = d.anc_tab;
        l.rconst = d.rconst;
        l.inv2L = d.inv2L; l.rsqrtL = d.rsqrtL;
        l.S = d.S; l.d = d.d; l.sumPhi = d.sumPhi; l.gram = d.gram; l.ancD = d.ancD;
        l.pc_ptr = d.pc_ptr; l.pc_anc = d.pc_anc; l.pc_lo = d.pc_lo; l.pc_hi = d.pc_hi;
        l.yc = d.yc; l.ysum = d.ysum;
        l.prec = d.prec; l.zeta = d.zeta; l.ytil = d.ytil; l.A = d.A; l.A_prev = d.A_prev; l.m2 = d.m2; l.cm2 = d.cm2;
        l.noise_shape = d.noise_shape; l.noise_scale = d.noise_scale; l.noise_mean = d.noise_mean; l.noise_log_mean = d.noise_log_mean;
        l.noise_shape0 = d.noise_shape0; l.noise_scale0 = d.noise_scale0; l.bias_prec0 = d.bias_prec0; l.bias_mean0 = d.bias_mean0;
        l.bias_prec = d.bias_prec; l.bias_mean = d.bias_mean; l.bias_prev = d.bias_prev; l.bias_var = d.bias_var;
        l.yvar = d.yvar; l.sumsB = d.sumsB;
    }
    CK(cudaMemcpyAsync(h->chain_dev, &m, sizeof m, cudaMemcpyHostToDevice, h->stream));
    const ChainModel *ptr = h->chain_dev;
    CK(cudaMemcpyAsync(h->chain_ptr_dev, &ptr, sizeof ptr, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));   // `ptr` is a local; the descriptor must be in place before any capture
    h->chain_uploaded = true;
    return MRGP_OK;
}

int do_fused_sweep(mrgp_handle *h, const Launch &L) {
    const int rc = launch_ci_sweep(chain_solver_size(h->cfg.n_basis), h->chain_ptr_dev, 1, chain_cluster_size(h), L.stream);
    if (rc != 0) return fail(h, MRGP_ECUDA, "fused sweep launch: %s", cudaGetErrorString((cudaError_t)rc));
    *L.count += 1;
    // Guarded fallback for layer 0: its sum |r|^2 is formed from the sufficient statistics of y as a difference of large
    // terms; when the residual is tiny against sum |y|^2 (ratio below kChainGuard: high-SNR data) the sweep sets the
    // model's status word and the kernel below - a no-op otherwise - takes the statistics of layer 0 by a pass over the
    // samples and repeats its bias / noise update (nothing else of the sweep depends on them).
    if (h->sharded) return MRGP_OK;   // (the sharded handle reports the status; its fallback would need an exchange)
    if (ystats_small(h)) {
        const int e = launch_l0_fix_small(chain_solver_size(h->cfg.n_basis), h->chain_ptr_dev, 1, h->plan[0].R, L.stream);
        if (e != 0) return fail(h, MRGP_ECUDA, "layer-0 fallback launch: %s", cudaGetErrorString((cudaError_t)e));
        *L.count += 1;
        return MRGP_OK;
    }
    return do_phase_b(h, L, 0, true, 0, h->chain_status);
}

int sweep_once(mrgp_handle *h, const Launch &L) {
    const int J = h->cfg.n_layers;
    const bool ci = h->cfg.mode == MRGP_MODE_CI;
    const bool closed = use_closed_form(h);
    int rc;
    if (use_fused(h)) return do_fused_sweep(h, L);   // the whole sweep is one kernel (csrc/chain.cu)
    if (ci && h->state_end > h->state_begin) {
        // the small-matrix state (a few MB) is pulled into L2 by the side stream while layer 0 streams the samples:
        // the short kernels that follow are chains of dependent loads and would otherwise each pay HBM latency
        CK(cudaEventRecord(h->ev_prefetch, L.stream));
        CK(cudaStreamWaitEvent(h->side, h->ev_prefetch, 0));
        const size_t lines = (h->state_end - h->state_begin + 127) / 128;
        k_prefetch_l2<<<(unsigned)std::min<size_t>((lines + 255) / 256, 1024), 256, 0, h->side>>>(h->ws + h->state_begin, lines);
        CK(cudaGetLastError());
        *L.count += 1;
    }
    // the third stream: layer 0's phase B (b0_forked once it is there), then the closed-form statistics of the layers above
    const Launch b0{h->side2, L.count};
    bool b0_forked = false;
    for (int j = 0; j < J; ++j) {
        // ci layers above the first regress on targets inferred from their own posterior, y = Phi A + b + fbar
        // (LatentOutputs.py:20-49), so the residual of the P1 statistics, y - fbar - b - Phi A with the same A and b
        // (Posteriors.py:61-78), vanishes identically: Phi^T r == 0 and y_tilde == d a.  The streaming pass that
        // would add up those zeros (plus roundoff) is not launched; mrgp_phase_a still runs it on request and
        // MRGP_STREAM_ALL=1 puts it back into the sweep.
        const bool zero_T = ci && j > 0 && h->inferred_shortcut;
        if (!zero_T && (rc = do_phase_a(h, L, j))) return rc;
        if (h->sharded) {
            // sample-sharded: the region statistics of both streaming phases are summed over the ranks
            if (!zero_T && (rc = do_exchange(h, L, j, h->cfg.n_basis * h->cfg.dy, false))) return rc;
            if ((rc = do_axis_update(h, L, j, ci, zero_T))) return rc;
            if (closed && j > 0) {   // replicated closed form: no samples, no exchange
                if ((rc = do_stats_b(h, L, j))) return rc;
                continue;
            }
            if ((rc = do_phase_b(h, L, j, false, closed ? 0 : -1))) return rc;
            if ((rc = do_exchange(h, L, j, h->cfg.dy + 3, false))) return rc;
            if ((rc = do_bias_noise(h, L, j))) return rc;
            continue;
        }
        if ((rc = do_axis_update(h, L, j, ci, zero_T))) return rc;
        if (h->dev[j].adaptive && ci) {
            // the latent functions of the next layer use the re-learnt basis (MRGP.py:632-649): statistics first,
            // then the interval search, then a second pass that only propagates
            if ((rc = do_phase_b(h, L, j, true, 0))) return rc;
            if ((rc = do_learn_intervals(h, L, j))) return rc;
            if (j + 1 < J && (rc = do_phase_b(h, L, j, false, 1))) return rc;
        } else if (closed && j > 0) {
            // inferred targets: statistics from the basis invariants.  In the captured sweep they follow layer 0's pass
            // on the third stream (they read the bias variances of the coarser layers, nothing of the chain waits for
            // them): k_mid1 of the next layer starts as soon as the ARD moments are there.
            if (b0_forked) CK(cudaStreamWaitEvent(h->side2, h->ev_mid2[j], 0));   // A, cm2 of this layer (k_mid2)
            if ((rc = do_stats_b(h, b0_forked ? b0 : L, j))) return rc;
        } else if (closed && j == 0 && J > 1) {
            // Layer 0's statistics pass (26 us on 147 SMs) runs on a third stream: the small-matrix chain of layer 1
            // (k_mid1 -> k_ard -> k_scale_warp on the SM left free) does not depend on it, only k_stats_b does.
            CK(cudaEventRecord(h->ev_b0_fork, L.stream));
            CK(cudaStreamWaitEvent(h->side2, h->ev_b0_fork, 0));
            if ((rc = do_phase_b(h, b0, j, true, 0))) return rc;
            b0_forked = true;
        } else {
            // bias / noise update fused into the kernel tail; nothing reads the latent buffers when the layers below
            // take the closed form
            if ((rc = do_phase_b(h, L, j, true, closed ? 0 : -1))) return rc;
        }
    }
    if (ci) {
        CK(cudaStreamWaitEvent(L.stream, h->ev_ard[J - 1], 0));
        CK(cudaStreamWaitEvent(L.stream, h->ev_join[J - 1], 0));
    }
    if (b0_forked) {   // join the third stream (layer 0's pass and the closed-form statistics of the other layers)
        CK(cudaEventRecord(h->ev_b0_done, h->side2));
        CK(cudaStreamWaitEvent(L.stream, h->ev_b0_done, 0));
    }
    return MRGP_OK;
}

struct FieldRef {
    void *ptr = nullptr;
    int64_t n = 0;
};

FieldRef field_ref(mrgp_handle *h, int layer, int field) {
    FieldRef f;
    const int M = h->cfg.n_basis, DY = h->cfg.dy;
    const bool fi = h->cfg.mode == MRGP_MODE_FI;
    if (field >= MRGP_F_AXIS_B && !fi) {
        if (layer != -1) return f;
        SharedDev &s = h->sh;
        switch (field) {
            case 54: f = {h->chain_prof, (int64_t)h->cfg.n_layers * 16}; break;   // MRGP_CHAIN_PROF=1: clock stamps of the fused sweep
            case 56: f = {h->chain_tables, (int64_t)h->cfg.n_layers * h->cfg.n_basis * h->cfg.n_basis}; break;   // (J, M, M) tables of the last sweep
            case MRGP_F_FUSED_GUARD: f = {h->chain_guard, 2}; break;
            case MRGP_F_AXIS_B: f = {s.axB, (int64_t)M * DY * DY}; break;
            case MRGP_F_AXIS_KAPPA: f = {s.axKappa, (int64_t)M * DY}; break;
            case MRGP_F_AXIS_RHO: f = {s.axRho, (int64_t)M * DY}; break;
            case MRGP_F_AXIS_LOGC: f = {s.axLogC, M}; break;
            case MRGP_F_AXIS_COV: f = {s.axCov, (int64_t)M * DY * DY}; break;
            case MRGP_F_ARD_SHAPE: f = {s.ardShape, M}; break;
            case MRGP_F_ARD_SCALE: f = {s.ardScale, M}; break;
            case MRGP_F_ARD_MEAN: f = {s.ardMean, M}; break;
            case MRGP_F_ARD_LOG_MEAN: f = {s.ardLogMean, M}; break;
            case MRGP_F_OMEGA: f = {s.omega, (int64_t)M * M}; break;
            case MRGP_F_LOG_OMEGA_HAT: f = {s.logOmegaHat, (int64_t)M * M}; break;
            case MRGP_F_OMEGA_ITERS: f = {s.omegaIters, h->cfg.n_layers}; break;
            default: break;
        }
        return f;
    }
    if (layer < 0 || layer >= h->cfg.n_layers) return f;
    LayerDev &d = h->dev[layer];
    const int64_t R = h->plan[layer].R, RM = R * M;
    switch (field) {
        case MRGP_F_L: f = {d.L, R}; break;
        case MRGP_F_LAMBDA: f = {d.lam, RM}; break;
        case MRGP_F_SPECTRAL: f = {d.S, RM}; break;
        case MRGP_F_PHI2SUM: f = {d.d, RM}; break;
        case MRGP_F_SCALE_PRECISION: f = {d.prec, RM}; break;
        case MRGP_F_ZETA: f = {d.zeta, RM}; break;
        case MRGP_F_YTILDE: f = {d.ytil, RM * DY}; break;
        case MRGP_F_NOISE_SHAPE: f = {d.noise_shape, R}; break;
        case MRGP_F_NOISE_SCALE: f = {d.noise_scale, R}; break;
        case MRGP_F_BIAS_PRECISION: f = {d.bias_prec, R}; break;
        case MRGP_F_A: f = {d.A, RM * DY}; break;
        case MRGP_F_M2: f = {d.m2, RM}; break;
        case MRGP_F_CM2: f = {d.cm2, RM}; break;
        case MRGP_F_NOISE_MEAN: f = {d.noise_mean, R}; break;
        case MRGP_F_NOISE_LOG_MEAN: f = {d.noise_log_mean, R}; break;
        case MRGP_F_BIAS_MEAN: f = {d.bias_mean, R * DY}; break;
        case MRGP_F_BIAS_VAR: f = {d.bias_var, R}; break;
        case MRGP_F_FBAR: f = {h->tmp_mean, h->cfg.n_samples * DY}; break;
        case MRGP_F_FVAR: f = {h->tmp_var, h->cfg.n_samples}; break;
        case MRGP_F_YVAR: f = {d.yvar, R}; break;
        case MRGP_F_PHASE_B_SUMS: f = {d.sumsB, R * (DY + 3)}; break;
        case MRGP_F_A_PREV: f = {d.A_prev, RM * DY}; break;
        case MRGP_F_BIAS_PREV: f = {d.bias_prev, R * DY}; break;
        default: break;
    }
    if (fi) {
        switch (field) {
            case MRGP_F_AXIS_B: f = {d.axB, RM * DY * DY}; break;
            case MRGP_F_AXIS_KAPPA: f = {d.axKappa, RM * DY}; break;
            case MRGP_F_AXIS_RHO: f = {d.axRho, RM * DY}; break;
            case MRGP_F_AXIS_LOGC: f = {d.axLogC, RM}; break;
            case MRGP_F_AXIS_COV: f = {d.axCov, RM * DY * DY}; break;
            case MRGP_F_ARD_SHAPE: f = {d.ardShape, RM}; break;
            case MRGP_F_ARD_SCALE: f = {d.ardScale, RM}; break;
            case MRGP_F_ARD_MEAN: f = {d.ardMean, RM}; break;
            case MRGP_F_ARD_LOG_MEAN: f = {d.ardLogMean, RM}; break;
            default: break;
        }
    }
    return f;
}

int fill_eval_layers(mrgp_handle *h, EvalArgs &ea, int n_layers, const int64_t *const *dev_offsets) {
    if (n_layers > kMaxLayers) return fail(h, MRGP_EINVAL, "too many layers");
    ea.n_layers = n_layers;
    ea.M = h->cfg.n_basis;
    for (int j = 0; j < n_layers; ++j) {
        const LayerDev &d = h->dev[j];
        EvalLayer &l = ea.layer[j];
        l.offsets = dev_offsets ? dev_offsets[j] : d.offsets;
        l.inv2L = d.inv2L;
        l.rsqrtL = d.rsqrtL;
        l.A = d.A;
        l.cm2 = d.cm2;
        l.bias = d.bias_mean;
        l.bias_var = d.bias_var;
        l.noise_mean = d.noise_mean;
        l.R = h->plan[j].R;
    }
    return MRGP_OK;
}

void drop_graph(mrgp_handle *h) {
    if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
    if (h->graph) cudaGraphDestroy(h->graph);
    h->graph_exec = nullptr;
    h->graph = nullptr;
    h->launches_per_sweep = 0;
    h->chain_uploaded = false;
    h->generation += 1;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int mrgp_abi_version(void) { return MRGP_ABI_VERSION; }

const char *mrgp_last_error(const mrgp_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int mrgp_create(const mrgp_config *cfg, const int64_t *const *region_offsets, const int32_t *n_regions, mrgp_handle **out) {
    mrgp_handle *h = nullptr;
    if (!cfg || !region_offsets || !n_regions || !out) return fail(h, MRGP_EINVAL, "null argument");
    *out = nullptr;
    if (cfg->abi_version != MRGP_ABI_VERSION) return fail(h, MRGP_EINVAL, "abi version %d != %d", cfg->abi_version, MRGP_ABI_VERSION);
    if (cfg->mode != MRGP_MODE_CI && cfg->mode != MRGP_MODE_FI) return fail(h, MRGP_EINVAL, "unknown mode");
    if (cfg->dy < 2) return fail(h, MRGP_EINVAL, "output dimension must be greater than 1");
    if (cfg->dy != 2) return fail(h, MRGP_EINVAL, "dy = %d: only dy == 2 is implemented on the device", cfg->dy);
    if (cfg->dx != 1) return fail(h, MRGP_EINVAL, "dx = %d: only dx == 1 is implemented on the device", cfg->dx);
    if (!basis_supported(cfg->n_basis)) return fail(h, MRGP_EINVAL, "n_basis = %d: 1 .. 48 basis functions are supported", cfg->n_basis);
    if (cfg->n_layers < 1 || cfg->n_layers > kMaxLayers) return fail(h, MRGP_EINVAL, "n_layers out of range");
    if (cfg->n_samples < 1) return fail(h, MRGP_EINVAL, "n_samples < 1");
    if (cfg->sample_begin < 0 || cfg->sample_end < cfg->sample_begin || cfg->sample_end > cfg->n_samples)
        return fail(h, MRGP_EINVAL, "bad sample range");
    // the cluster size of the fused sweep must be a power of two the launch supports (0: chosen by the regions);
    // anything else would only fail at the first sweep, far from its cause
    int chain_cluster = 0;
    if (const char *e = getenv("MRGP_CHAIN_CLUSTER")) {
        char *end = nullptr;
        const long c = strtol(e, &end, 10);
        if (end == e || *end != '\0' || c < 0 || c > kChainMaxCluster || (c & (c - 1)))
            return fail(h, MRGP_EINVAL, "MRGP_CHAIN_CLUSTER=\"%s\": must be 0 (by the regions), 1, 2, 4, 8 or %d", e, kChainMaxCluster);
        chain_cluster = (int)c;
    }
    h = new mrgp_handle();
    h->cfg = *cfg;
    if (const char *e = getenv("MRGP_STREAM_ALL")) h->inferred_shortcut = !(e[0] == '1');
    if (const char *e = getenv("MRGP_FUSED")) h->fused = !(e[0] == '0');
    if (const char *e = getenv("MRGP_CHAIN_PROF")) h->chain_prof_on = e[0] == '1';
    if (const char *e = getenv("MRGP_CHAIN_GUARD")) h->chain_guard_threshold = atof(e);
    h->chain_cluster = chain_cluster;
    h->sharded = cfg->sample_end > cfg->sample_begin;   // an explicit range selects the exchange-buffer path
    h->lo = h->sharded ? cfg->sample_begin : 0;
    h->hi = h->sharded ? cfg->sample_end : cfg->n_samples;
    h->plan.resize(cfg->n_layers);
    h->dev.resize(cfg->n_layers);
    for (int j = 0; j < cfg->n_layers; ++j) {
        LayerPlan &lp = h->plan[j];
        lp.R = n_regions[j];
        if (lp.R < 1) {
            delete h;
            return fail(nullptr, MRGP_EINVAL, "layer %d has no regions", j);
        }
        lp.offsets.assign(region_offsets[j], region_offsets[j] + lp.R + 1);
        bool ok = lp.offsets.front() == 0 && lp.offsets.back() == cfg->n_samples;
        for (int r = 0; r < lp.R && ok; ++r) ok = lp.offsets[r + 1] > lp.offsets[r];
        if (!ok) {
            delete h;
            return fail(nullptr, MRGP_EINVAL, "layer %d: offsets must be strictly increasing from 0 to n_samples", j);
        }
    }
    // streaming geometry: one persistent CTA per SM unless told otherwise; small problems use fewer CTAs
    int sms = 148;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0) {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, cfg->device) == cudaSuccess) sms = prop.multiProcessorCount;
    } else {
        cudaGetLastError();
    }
    h->sm_count = sms;
    // ci: one SM is left to the omega solver, which runs beside phase B / phase A on a side stream (a phase-A CTA
    // takes the whole register file of its SM, and sharing an SM with phase B halves the solver's FP64 rate)
    int want = cfg->n_ctas > 0 ? cfg->n_ctas : (cfg->mode == MRGP_MODE_CI && sms > 8 ? sms - 1 : sms);
    const int64_t min_per_cta = 4 * kThreads;
    const int64_t n_local = h->hi - h->lo;
    const int64_t cap = std::max<int64_t>(1, (n_local + min_per_cta - 1) / min_per_cta);
    want = (int)std::min<int64_t>(want, cap);
    int64_t q = (n_local + want - 1) / want;
    q = ((q + 31) / 32) * 32;
    h->cta_quantum = q;
    h->n_ctas = (int)((n_local + q - 1) / q);
    build_plan(h);
    if (cfg->mode == MRGP_MODE_CI)
        for (int j = 1; j < cfg->n_layers; ++j) {
            LayerPlan &lp = h->plan[j];
            lp.pc_ptr.assign((size_t)j * (lp.R + 1), 0);
            for (int jp = 0; jp < j; ++jp) {
                const auto &po = h->plan[jp].offsets;
                size_t a = 0;
                for (int c = 0; c < lp.R; ++c) {
                    lp.pc_ptr[(size_t)jp * (lp.R + 1) + c] = (int32_t)lp.pc_jp.size();
                    const int64_t lo = lp.offsets[c], hi = lp.offsets[c + 1];
                    while (po[a + 1] <= lo) ++a;
                    for (size_t q = a; q + 1 < po.size() && po[q] < hi; ++q) {
                        lp.pc_jp.push_back(jp);
                        lp.pc_anc.push_back((int32_t)q);
                        lp.pc_lo.push_back(std::max(lo, po[q]));
                        lp.pc_hi.push_back(std::min(hi, po[q + 1]));
                    }
                }
                lp.pc_ptr[(size_t)jp * (lp.R + 1) + lp.R] = (int32_t)lp.pc_jp.size();
            }
            lp.E = 0;
            for (int c = 0; c < lp.R; ++c) {
                int cnt = 0;
                for (int jp = 0; jp < j; ++jp) cnt += lp.pc_ptr[(size_t)jp * (lp.R + 1) + c + 1] - lp.pc_ptr[(size_t)jp * (lp.R + 1) + c];
                lp.E = std::max(lp.E, cnt);
            }
        }
    h->ws_bytes = carve(h, nullptr);
    *out = h;
    return MRGP_OK;
}

void mrgp_destroy(mrgp_handle *h) {
    if (!h) return;
    drop_graph(h);
    for (auto e : h->ev_fork) cudaEventDestroy(e);
    for (auto e : h->ev_join) cudaEventDestroy(e);
    for (auto e : h->ev_ard) cudaEventDestroy(e);
    for (auto e : h->ev_mid2) cudaEventDestroy(e);
    if (h->ev_prefetch) cudaEventDestroy(h->ev_prefetch);
    if (h->ev_b0_fork) cudaEventDestroy(h->ev_b0_fork);
    if (h->ev_b0_done) cudaEventDestroy(h->ev_b0_done);
    if (h->side2) cudaStreamDestroy(h->side2);
    if (h->ev_copy_done) cudaEventDestroy(h->ev_copy_done);
    for (int q = 0; q < 2; ++q)
        if (h->ev_elbo[q]) cudaEventDestroy(h->ev_elbo[q]);
    if (h->ev_y_free) cudaEventDestroy(h->ev_y_free);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for (int q = 0; q < kMaxRanks; ++q)
        if (h->comm.opened[q]) cudaIpcCloseMemHandle(h->comm.peer_base[q]);
    if (h->comm.mem) cudaFree(h->comm.mem);
    if (h->side) cudaStreamDestroy(h->side);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

size_t mrgp_workspace_bytes(const mrgp_handle *h) { return h ? h->ws_bytes : 0; }

int mrgp_bind_workspace(mrgp_handle *h, void *dev_ptr, size_t bytes) {
    if (!h || !dev_ptr) return fail(h, MRGP_EINVAL, "null argument");
    if (bytes < h->ws_bytes) return fail(h, MRGP_ENOMEM, "workspace %zu < %zu bytes", bytes, h->ws_bytes);
    if (((uintptr_t)dev_ptr & 255) != 0) return fail(h, MRGP_EINVAL, "workspace must be 256-byte aligned");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(h, MRGP_ENODEVICE, "no CUDA device");
    }
    CK(cudaSetDevice(h->cfg.device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->cfg.device));
    if (prop.major != 10) return fail(h, MRGP_ENODEVICE, "device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor);
    if (!h->stream) {
        CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        h->own_stream = true;
    }
    if (!h->side) CK(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
    if (!h->ev_prefetch) {
        CK(cudaEventCreateWithFlags(&h->ev_prefetch, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_b0_fork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_b0_done, cudaEventDisableTiming));
        CK(cudaStreamCreateWithFlags(&h->side2, cudaStreamNonBlocking));
    }
    if (h->ev_fork.empty()) {
        h->ev_fork.resize(h->cfg.n_layers);
        h->ev_join.resize(h->cfg.n_layers);
        h->ev_ard.resize(h->cfg.n_layers);
        h->ev_mid2.resize(h->cfg.n_layers);
        for (int j = 0; j < h->cfg.n_layers; ++j) {
            CK(cudaEventCreateWithFlags(&h->ev_fork[j], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->ev_join[j], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->ev_ard[j], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->ev_mid2[j], cudaEventDisableTiming));
        }
    }
    h->ws = static_cast<char *>(dev_ptr);
    carve(h, h->ws);
    drop_graph(h);
    // upload the plan
    for (int j = 0; j < h->cfg.n_layers; ++j) {
        const LayerPlan &lp = h->plan[j];
        LayerDev &d = h->dev[j];
        CK(cudaMemcpyAsync(d.segs, lp.segs.data(), lp.segs.size() * sizeof(Segment), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(d.cta_seg, lp.cta_seg.data(), lp.cta_seg.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(d.region_run, lp.region_run.data(), lp.region_run.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(d.ident_run, lp.ident_run.data(), lp.ident_run.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(d.offsets, lp.offsets.data(), lp.offsets.size() * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
        if (d.pc_ptr) {
            const size_t P = lp.pc_jp.size();
            CK(cudaMemcpyAsync(d.pc_ptr, lp.pc_ptr.data(), lp.pc_ptr.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(d.pc_jp, lp.pc_jp.data(), P * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(d.pc_anc, lp.pc_anc.data(), P * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(d.pc_lo, lp.pc_lo.data(), P * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(d.pc_hi, lp.pc_hi.data(), P * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
        }
    }
    // flattened piece table of the fused sweep: for every region its pieces over all coarser layers, coarse to fine
    for (int j = 1; j < h->cfg.n_layers && h->cfg.mode == MRGP_MODE_CI; ++j) {
        const LayerPlan &lp = h->plan[j];
        LayerDev &d = h->dev[j];
        const int E = std::max(lp.E, 1), M = h->cfg.n_basis;
        std::vector<AncEntry> tab((size_t)lp.R * E);
        const double *base = reinterpret_cast<const double *>(h->ws + h->state_begin);
        if ((h->state_end - h->state_begin) / sizeof(double) >= 0xffffffffull)
            return fail(h, MRGP_EINVAL, "small-matrix state of more than 32 GB: not supported by the fused sweep tables");
        for (int c = 0; c < lp.R; ++c) {
            int e = 0;
            for (int jp = 0; jp < j; ++jp)
                for (int pc = lp.pc_ptr[(size_t)jp * (lp.R + 1) + c]; pc < lp.pc_ptr[(size_t)jp * (lp.R + 1) + c + 1]; ++pc, ++e) {
                    AncEntry &a = tab[(size_t)c * E + e];
                    a.cm2_off = (uint32_t)((h->dev[jp].cm2 - base) + (long long)lp.pc_anc[pc] * M);
                    a.bv_off = (uint32_t)((h->dev[jp].bias_var - base) + lp.pc_anc[pc]);
                    a.d_off = (uint32_t)((d.ancD - base) + (long long)pc * M);
                    a.len = (int32_t)(lp.pc_hi[pc] - lp.pc_lo[pc]);
                }
            for (; e < E; ++e) tab[(size_t)c * E + e] = AncEntry{0, 0, 0, -1};
        }
        CK(cudaMemcpyAsync(d.anc_tab, tab.data(), tab.size() * sizeof(AncEntry), cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));   // `tab` is a local
    }
    CK(cudaMemsetAsync(h->chol_count, 0, sizeof(unsigned long long), h->stream));
    CK(cudaMemsetAsync(h->done_counter, 0, sizeof(unsigned int), h->stream));
    CK(cudaMemsetAsync(h->elbo_counter, 0, (size_t)h->cfg.n_layers * sizeof(unsigned int), h->stream));
    CK(cudaMemsetAsync(h->brent_fail, 0, sizeof(unsigned long long), h->stream));
    CK(cudaMemsetAsync(h->mid_sync, 0, 2 * kMaxLayers * sizeof(unsigned int), h->stream));
    if (h->chain_status) {
        CK(cudaMemsetAsync(h->chain_status, 0, 4 * sizeof(unsigned int), h->stream));
        CK(cudaMemsetAsync(h->chain_guard, 0, 2 * sizeof(double), h->stream));
    }
    CK(cudaMemsetAsync(h->g, 0, (size_t)(h->hi - h->lo) * h->cfg.dy * sizeof(double), h->stream));
    CK(cudaMemsetAsync(h->hvar, 0, (size_t)(h->hi - h->lo) * sizeof(double), h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->bound = true;
    return MRGP_OK;
}

int mrgp_set_stream(mrgp_handle *h, void *cuda_stream) {
    if (!h) return MRGP_EINVAL;
    if (!cuda_stream) return fail(h, MRGP_EINVAL, "a non-default stream is required (graph capture)");
    drop_graph(h);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    h->own_stream = false;
    h->stream = static_cast<cudaStream_t>(cuda_stream);
    return MRGP_OK;
}

// New inputs x: everything derived from them (intervals, lambda, S, sum phi^2, the invariants of the closed-form
// statistics, the captured graph) is stale.  The basis of every layer has to be rebuilt before the next phase / sweep.
static void invalidate_inputs(mrgp_handle *h) {
    for (auto &d : h->dev) {
        d.basis_built = false;
        d.inv_built = false;
    }
    h->ystats_valid = false;
    drop_graph(h);
}

int mrgp_set_data(mrgp_handle *h, const double *x_dev, const double *y_dev) {
    if (!h || !x_dev || !y_dev) return fail(h, MRGP_EINVAL, "null argument");
    if (!h->bound) return fail(h, MRGP_ESTATE, "no workspace bound");
    if (((uintptr_t)y_dev & 15) != 0 || ((uintptr_t)x_dev & 15) != 0) return fail(h, MRGP_EINVAL, "x and y must be 16-byte aligned (bulk copies)");
    if (h->have_data) invalidate_inputs(h);
    h->x = x_dev;
    h->y = y_dev;
    h->have_data = true;
    return MRGP_OK;
}

int mrgp_set_data_host(mrgp_handle *h, const double *x_host, const double *y_host) {
    if (h) h->stream_ops += 1;
    if (!h || !x_host || !y_host) return fail(h, MRGP_EINVAL, "null argument");
    if (!h->bound) return fail(h, MRGP_ESTATE, "no workspace bound");
    const size_t N = (size_t)(h->hi - h->lo);
    CK(cudaMemcpyAsync(h->x_ws, x_host, N * h->cfg.dx * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->y_ws, y_host, N * h->cfg.dy * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if (h->have_data) invalidate_inputs(h);
    h->x = h->x_ws;
    h->y = h->y_ws;
    h->have_data = true;
    return MRGP_OK;
}

int mrgp_set_observations(mrgp_handle *h, const double *y_dev) {
    if (!h || !y_dev) return fail(h, MRGP_EINVAL, "null argument");
    if (!h->have_data) return fail(h, MRGP_ESTATE, "no inputs yet: mrgp_set_data / mrgp_set_data_host first");
    if (((uintptr_t)y_dev & 15) != 0) return fail(h, MRGP_EINVAL, "y must be 16-byte aligned (bulk copies)");
    if (h->prefetch_pending) return fail(h, MRGP_ESTATE, "prefetched observations are waiting to be taken over");
    if (h->y != y_dev) drop_graph(h);   // the captured kernels hold the pointer
    h->y = y_dev;
    h->ystats_valid = false;
    return MRGP_OK;
}

// Host-to-device copy in pieces of kH2DChunk bytes.  In isolation 16 MB from pinned memory took 0.47 ms as one
// cudaMemcpyAsync and 0.31 ms as 4 MB pieces on the boxes of this project (scratch/h2d_bw.py, noisy); inside bench.py the
// piece size made no difference (the copy is hidden behind the sweep).
constexpr size_t kH2DChunk = (size_t)4 << 20;

static cudaError_t copy_h2d_chunked(void *dst, const void *src, size_t bytes, cudaStream_t st) {
    if (bytes <= kH2DChunk) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
    for (size_t off = 0; off < bytes; off += kH2DChunk) {
        const size_t n = bytes - off < kH2DChunk ? bytes - off : kH2DChunk;
        cudaError_t e = cudaMemcpyAsync(static_cast<char *>(dst) + off, static_cast<const char *>(src) + off, n, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

int mrgp_set_observations_host(mrgp_handle *h, const double *y_host) {
    if (h) h->stream_ops += 1;
    if (!h || !y_host) return fail(h, MRGP_EINVAL, "null argument");
    if (!h->have_data) return fail(h, MRGP_ESTATE, "no inputs yet: mrgp_set_data / mrgp_set_data_host first");
    if (h->prefetch_pending) return fail(h, MRGP_ESTATE, "prefetched observations are waiting to be taken over");
    const size_t N = (size_t)(h->hi - h->lo);
    CK(copy_h2d_chunked(h->y_ws, y_host, N * h->cfg.dy * sizeof(double), h->stream));
    if (h->y != h->y_ws) drop_graph(h);
    h->y = h->y_ws;
    h->ystats_valid = false;
    return MRGP_OK;
}

// Double-buffered upload: the copy of the NEXT observations runs on the handle's own copy stream into the spare buffer
// while the handle's stream works on the current ones (a fused ci sweep reads no sample at all).
int mrgp_prefetch_observations_host(mrgp_handle *h, const double *y_host) {
    if (h) h->stream_ops += 1;
    if (!h || !y_host) return fail(h, MRGP_EINVAL, "null argument");
    if (!h->have_data) return fail(h, MRGP_ESTATE, "no inputs yet: mrgp_set_data / mrgp_set_data_host first");
    if (h->prefetch_pending)
        return fail(h, MRGP_ESTATE, "prefetched observations are waiting to be taken over (mrgp_refresh_statistics)");
    if (!h->copy_stream) {
        CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&h->ev_copy_done, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_y_free, cudaEventDisableTiming));
    }
    // the spare buffer held the observations before the current ones: its last readers were enqueued before the marker
    if (h->y_free_recorded) CK(cudaStreamWaitEvent(h->copy_stream, h->ev_y_free, 0));
    const size_t N = (size_t)(h->hi - h->lo);
    CK(copy_h2d_chunked(h->y_ws2, y_host, N * h->cfg.dy * sizeof(double), h->copy_stream));
    CK(cudaEventRecord(h->ev_copy_done, h->copy_stream));
    h->prefetch_pending = true;
    return MRGP_OK;
}

// Switch between the fused ci sweep and the multi-kernel sweep (the environment variable MRGP_FUSED sets the start value).
// Both keep the same state arrays; the captured graph is dropped.
int mrgp_set_fused(mrgp_handle *h, int32_t on) {
    if (!h) return MRGP_EINVAL;
    if (h->fused != (on != 0)) {
        h->fused = on != 0;
        h->direct_launch = false;
        drop_graph(h);
    }
    return MRGP_OK;
}

// Blocks the caller until the last mrgp_prefetch_observations_host() has read its host buffer (which may then be reused).
int mrgp_prefetch_sync(mrgp_handle *h) {
    if (!h) return MRGP_EINVAL;
    if (h->ev_copy_done) CK(cudaEventSynchronize(h->ev_copy_done));
    return MRGP_OK;
}

namespace {
// Take over prefetched observations: swap the buffers, make the stream wait for the copy, invalidate what depends on y.
int adopt_prefetched(mrgp_handle *h) {
    if (!h->prefetch_pending) return MRGP_OK;
    CK(cudaEventRecord(h->ev_y_free, h->stream));   // everything enqueued so far may read the buffer that becomes the spare
    h->y_free_recorded = true;
    CK(cudaStreamWaitEvent(h->stream, h->ev_copy_done, 0));
    std::swap(h->y_ws, h->y_ws2);
    h->y = h->y_ws;
    h->ystats_valid = false;
    h->prefetch_pending = false;
    if (use_fused(h) && !ystats_small(h)) {
        // the sweep kernel reads no sample and the guarded fallback takes y from its launch arguments: launch on the
        // stream from now on (a captured graph would hold the old pointer; two launches per sweep either way)
        h->direct_launch = true;
        if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
        if (h->graph) cudaGraphDestroy(h->graph);
        h->graph_exec = nullptr;
        h->graph = nullptr;
    } else {
        drop_graph(h);
    }
    return MRGP_OK;
}
}  // namespace

int mrgp_set_all_inputs_host(mrgp_handle *h, const double *x_all_host) {
    if (!h || !x_all_host) return fail(h, MRGP_EINVAL, "null argument");
    if (!h->bound) return fail(h, MRGP_ESTATE, "no workspace bound");
    if (!h->sharded) return fail(h, MRGP_ESTATE, "not a sharded handle: mrgp_set_data* already holds every sample");
    if (!h->x_all) return fail(h, MRGP_ESTATE, "this handle has no use for the replicated inputs (fi mode or one layer)");
    CK(cudaMemcpyAsync(h->x_all, x_all_host, (size_t)h->cfg.n_samples * h->cfg.dx * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    h->have_x_all = true;
    for (auto &d : h->dev) d.inv_built = false;
    drop_graph(h);
    return MRGP_OK;
}

int mrgp_set_spectral(mrgp_handle *h, int32_t layer, int32_t use_prior, double nu, double l, double sf) {
    if (!h || layer < 0 || layer >= h->cfg.n_layers) return fail(h, MRGP_EINVAL, "bad layer");
    LayerDev &d = h->dev[layer];
    d.use_prior = use_prior;
    d.nu = nu;
    d.ell = l;
    d.sf = sf;
    return MRGP_OK;
}

int mrgp_build_basis(mrgp_handle *h, int32_t layer, double interval_factor, const double *L_host) {
    if (h) h->stream_ops += 1;
    int rc = check_ready(h, layer, false);
    if (rc) return rc;
    if (h->sharded && !h->comm.ready) return fail(h, MRGP_ESTATE, "sharded handle: bind the peer exchange first (mrgp_comm_export / mrgp_comm_bind)");
    if (h->sharded && L_host) return fail(h, MRGP_EINVAL, "given intervals are not supported on a sharded handle");
    LayerDev &d = h->dev[layer];
    const LayerPlan &lp = h->plan[layer];
    const Launch L{h->stream, &h->launches};
    StreamArgs sa = stream_args(h, layer);
    RegionArgs ra = region_args(h, layer);
    ra.interval_factor = interval_factor;
    if (L_host) {
        CK(cudaMemcpyAsync(d.L, L_host, lp.R * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        ra.L_given = 1;
    } else {
        k_absmax<<<h->n_ctas, kThreads, 0, h->stream>>>(sa);
        CK(cudaGetLastError());
        h->launches += 1;
    }
    // sharded: L, lambda, S from the max|x| of the region over all ranks, d from the sum of phi^2 over all ranks
    if (h->sharded && (rc = do_exchange(h, L, layer, 1, true))) return rc;
    k_region_setup<<<(lp.R + 7) / 8, 256, 0, h->stream>>>(ra);
    CK(cudaGetLastError());
    h->launches += 1;
    cudaError_t e = cudaErrorInvalidValue;
    DISPATCH_M(h->cfg.n_basis, e = launch_phi2sum<MM>(h, h->stream, sa));
    CK(e);
    h->launches += 1;
    if (h->sharded && (rc = do_exchange(h, L, layer, h->cfg.n_basis, false))) return rc;
    k_reduce_d<<<lp.R, 64, 0, h->stream>>>(ra);
    CK(cudaGetLastError());
    h->launches += 1;
    d.basis_built = true;
    for (int jj = layer; jj < h->cfg.n_layers; ++jj) h->dev[jj].inv_built = false;   // s, G of the layer; D of the finer ones
    h->ystats_valid = false;
    drop_graph(h);
    return MRGP_OK;
}

int mrgp_init_state(mrgp_handle *h, double noise_var0, double ard_prior_influence) {
    if (h) h->stream_ops += 1;
    int rc = check_ready(h, 0, false);
    if (rc) return rc;
    for (int j = 0; j < h->cfg.n_layers; ++j)
        if (!h->dev[j].basis_built) return fail(h, MRGP_ESTATE, "basis of layer %d not built", j);
    const int M = h->cfg.n_basis;
    const double zero2[2] = {0.0, 0.0};
    double logc0, rho0[2];
    saddle_point<2>(zero2, logc0, rho0);
    // fi ARD mixing of the (never updated) prior: sum_k (1/M) shape0_k in index order (Posteriors.py:293-295)
    double sh = 0.0, sc = 0.0;
    const double w = 1.0 / (double)M;
    for (int k = 0; k < M; ++k) {
        sh += w * kEps;
        sc += w * (kEps / ard_prior_influence);
    }
    h->fi_shape0_mix = sh;
    h->fi_scale0_mix = sc;
    for (int j = 0; j < h->cfg.n_layers; ++j) {
        RegionArgs a = region_args(h, j);
        const int total = h->plan[j].R * M;
        k_init_layer<2><<<(total + 127) / 128, 128, 0, h->stream>>>(a, j == 0 ? noise_var0 : 1.0, ard_prior_influence, logc0, rho0[0]);
        CK(cudaGetLastError());
        h->launches += 1;
    }
    {
        RegionArgs a = region_args(h, 0);
        SharedDev &s = h->sh;
        // region_args points the axis/ARD fields at per-layer arrays in fi mode; the shared block is
        // initialised in both modes so that every buffer is defined
        a.axB = s.axB; a.axKappa = s.axKappa; a.axRho = s.axRho; a.axLogC = s.axLogC; a.axCov = s.axCov;
        a.ardShape = s.ardShape; a.ardScale = s.ardScale; a.ardMean = s.ardMean; a.ardLogMean = s.ardLogMean;
        k_init_shared<2><<<1, 256, 0, h->stream>>>(a, s.priorB, s.priorLogC, s.priorShape, s.priorScale, ard_prior_influence, logc0, rho0[0]);
        CK(cudaGetLastError());
        h->launches += 1;
    }
    CK(cudaMemsetAsync(h->g, 0, (size_t)(h->hi - h->lo) * h->cfg.dy * sizeof(double), h->stream));
    CK(cudaMemsetAsync(h->hvar, 0, (size_t)(h->hi - h->lo) * sizeof(double), h->stream));
    CK(cudaMemsetAsync(h->sh.omegaWarm, 0, kMaxLayers * sizeof(double), h->stream));
    if (h->chain_status) {
        CK(cudaMemsetAsync(h->chain_status, 0, 4 * sizeof(unsigned int), h->stream));
        CK(cudaMemsetAsync(h->chain_guard, 0, 2 * sizeof(double), h->stream));
    }
    drop_graph(h);
    h->sweeps_done = 0;
    h->state_init = true;
    return MRGP_OK;
}

int64_t mrgp_state_elems(const mrgp_handle *h, int32_t layer, int32_t field) {
    if (!h) return -1;
    FieldRef f = field_ref(const_cast<mrgp_handle *>(h), layer, field);
    return f.n > 0 ? f.n : -1;
}

int mrgp_get_state(mrgp_handle *h, int32_t layer, int32_t field, double *dst_host, size_t n_elems) {
    if (!h || !dst_host) return fail(h, MRGP_EINVAL, "null argument");
    if (!h->bound) return fail(h, MRGP_ESTATE, "no workspace bound");
    FieldRef f = field_ref(h, layer, field);
    if (!f.ptr || f.n <= 0) return fail(h, MRGP_EINVAL, "unknown field %d for layer %d", field, layer);
    if ((int64_t)n_elems != f.n) return fail(h, MRGP_EINVAL, "field %d has %lld elements, caller passed %zu", field, (long long)f.n, n_elems);
    if ((field == MRGP_F_FBAR || field == MRGP_F_FVAR) && h->sharded) return fail(h, MRGP_EINVAL, "latent export is not available on a sharded handle");
    if (field == MRGP_F_FBAR || field == MRGP_F_FVAR) {
        // latent functions of `layer`: sum over coarser layers (Stats.py:126-157), recomputed on demand
        int rc = check_ready(h, layer, true);
        if (rc) return rc;
        const int64_t N = h->cfg.n_samples;
        if (layer == 0 || h->sweeps_done == 0) {   // Stats.py:57-62: zeros until the first sweep
            CK(cudaMemsetAsync(h->tmp_mean, 0, (size_t)N * h->cfg.dy * sizeof(double), h->stream));
            CK(cudaMemsetAsync(h->tmp_var, 0, (size_t)N * sizeof(double), h->stream));
        } else {
            EvalArgs ea{};
            if ((rc = fill_eval_layers(h, ea, layer, nullptr))) return rc;
            ea.n = N;
            ea.x = h->x;
            ea.out_mean = h->tmp_mean;
            ea.out_var = h->tmp_var;
            ea.single_region = 0;
            k_eval_layers<2><<<(unsigned)((N + 127) / 128), 128, 0, h->stream>>>(ea);
            CK(cudaGetLastError());
            h->launches += 1;
        }
    }
    CK(cudaMemcpyAsync(dst_host, f.ptr, (size_t)f.n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MRGP_OK;
}

int mrgp_set_state(mrgp_handle *h, int32_t layer, int32_t field, const double *src_host, size_t n_elems) {
    if (h) h->stream_ops += 1;
    if (!h || !src_host) return fail(h, MRGP_EINVAL, "null argument");
    if (!h->bound) return fail(h, MRGP_ESTATE, "no workspace bound");
    if (field == MRGP_F_FBAR || field == MRGP_F_FVAR) return fail(h, MRGP_EINVAL, "latent functions are derived, not settable");
    FieldRef f = field_ref(h, layer, field);
    if (!f.ptr || f.n <= 0) return fail(h, MRGP_EINVAL, "unknown field %d for layer %d", field, layer);
    if ((int64_t)n_elems != f.n) return fail(h, MRGP_EINVAL, "field %d has %lld elements, caller passed %zu", field, (long long)f.n, n_elems);
    CK(cudaMemcpyAsync(f.ptr, src_host, (size_t)f.n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if (h->sh.skTag) {   // terms prepared from the shared posterior by the previous layer's k_ard may be stale now
        const double invalid[2] = {-1.0, -1.0};
        CK(cudaMemcpyAsync(h->sh.skTag, invalid, sizeof(invalid), cudaMemcpyHostToDevice, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return MRGP_OK;
}

int mrgp_phase_a(mrgp_handle *h, int32_t layer) {
    if (h) h->stream_ops += 1;
    int rc = check_ready(h, layer, true);
    return rc ? rc : do_phase_a(h, Launch{h->stream, &h->launches}, layer);
}

int mrgp_axis_update(mrgp_handle *h, int32_t layer) {
    if (h) h->stream_ops += 1;
    int rc = check_ready(h, layer, true);
    return rc ? rc : do_axis_update(h, Launch{h->stream, &h->launches}, layer, false);
}

int mrgp_phase_b(mrgp_handle *h, int32_t layer) {
    if (h) h->stream_ops += 1;
    int rc = check_ready(h, layer, true);
    return rc ? rc : do_phase_b(h, Launch{h->stream, &h->launches}, layer, false);
}

int mrgp_bias_noise(mrgp_handle *h, int32_t layer) {
    if (h) h->stream_ops += 1;
    int rc = check_ready(h, layer, true);
    if (!rc && layer == h->cfg.n_layers - 1) h->sweeps_done += 1;
    return rc ? rc : do_bias_noise(h, Launch{h->stream, &h->launches}, layer);
}

int mrgp_set_adaptive_intervals(mrgp_handle *h, int32_t layer, int32_t enabled, int32_t use_prior, double factor_lo, double factor_hi) {
    if (!h) return MRGP_EINVAL;
    if (layer < -1 || layer >= h->cfg.n_layers) return fail(h, MRGP_EINVAL, "layer out of range");
    if (enabled && h->cfg.mode != MRGP_MODE_CI) return fail(h, MRGP_EINVAL, "adaptive intervals exist in ci mode only (MRGP.py:108-109)");
    if (enabled && h->sharded) return fail(h, MRGP_EINVAL, "adaptive intervals are not available on a sharded handle");
    if (enabled && !(factor_lo > 0.0 && factor_hi > 0.0)) return fail(h, MRGP_EINVAL, "opt_interval_factor must be positive");
    for (int j = 0; j < h->cfg.n_layers; ++j) {
        if (layer >= 0 && j != layer) continue;
        LayerDev &d = h->dev[j];
        if (enabled && use_prior && !d.use_prior)
            return fail(h, MRGP_EINVAL, "use_prior needs a spectral density on the layer (BasisInterval.py:121)");
        d.adaptive = enabled != 0;
        for (auto &dd : h->dev) dd.inv_built = false;
        d.ad_use_prior = use_prior;
        d.ad_lo = factor_lo;
        d.ad_hi = factor_hi;
    }
    drop_graph(h);
    return MRGP_OK;
}

int mrgp_learn_intervals(mrgp_handle *h, int32_t layer) {
    int rc = check_ready(h, layer, true);
    if (rc) return rc;
    if (!h->dev[layer].adaptive) return fail(h, MRGP_ESTATE, "adaptive intervals are not enabled on this layer");
    return do_learn_intervals(h, Launch{h->stream, &h->launches}, layer);
}

int mrgp_interval_failures(mrgp_handle *h, uint64_t *out) {
    if (!h || !out) return MRGP_EINVAL;
    if (!h->brent_fail) return fail(h, MRGP_ESTATE, "workspace not bound");
    unsigned long long v = 0;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(&v, h->brent_fail, sizeof(v), cudaMemcpyDeviceToHost));
    *out = v;
    return MRGP_OK;
}

int mrgp_refresh_statistics(mrgp_handle *h) {
    int rc = check_ready(h, 0, true);
    if (rc) return rc;
    h->stream_ops += 1;
    if ((rc = adopt_prefetched(h))) return rc;
    if (!use_fused(h)) return MRGP_OK;   // the multi-kernel sweep streams layer 0: nothing to prepare
    const Launch L{h->stream, &h->launches};
    if ((rc = build_invariants(h, L))) return rc;
    if (!h->chain_uploaded && (rc = upload_chain_model(h))) return rc;
    return do_ystats(h, L);
}

int mrgp_sweep(mrgp_handle *h, int32_t n_iter) {
    if (h) h->stream_ops += 1;
    int rc = check_ready(h, 0, true);
    if (rc) return rc;
    if (n_iter < 0) return fail(h, MRGP_EINVAL, "n_iter < 0");
    if (h->sharded && !h->comm.ready)
        return fail(h, MRGP_ESTATE, "mrgp_sweep on a sharded handle needs the peer exchange (mrgp_comm_export / mrgp_comm_bind)");
    const bool fused = use_fused(h);
    const Launch L{h->stream, &h->launches};
    if (fused) {
        if ((rc = build_invariants(h, L))) return rc;
        if (!h->chain_uploaded && (rc = upload_chain_model(h))) return rc;
        if (!h->ystats_valid && (rc = do_ystats(h, L))) return rc;
    }
    if (fused && h->direct_launch) {
        for (int it = 0; it < n_iter; ++it)
            if ((rc = sweep_once(h, L))) return rc;
        h->sweeps_done += n_iter;
        return MRGP_OK;
    }
    if (!h->graph_exec) {
        if ((rc = build_invariants(h, L))) return rc;
        h->launches_per_sweep = 0;
        cudaError_t e = cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) return fail(h, MRGP_ECUDA, "cudaStreamBeginCapture: %s", cudaGetErrorString(e));
        rc = sweep_once(h, Launch{h->stream, &h->launches_per_sweep});
        cudaGraph_t graph = nullptr;
        e = cudaStreamEndCapture(h->stream, &graph);
        if (rc) {
            if (graph) cudaGraphDestroy(graph);
            return rc;
        }
        if (e != cudaSuccess) return fail(h, MRGP_ECUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
        h->graph = graph;
        CK(cudaGraphInstantiate(&h->graph_exec, h->graph, 0));
    }
    for (int it = 0; it < n_iter; ++it) CK(cudaGraphLaunch(h->graph_exec, h->stream));
    h->launches += h->launches_per_sweep * n_iter;
    h->sweeps_done += n_iter;
    return MRGP_OK;
}

// ---- groups of independent models ---------------------------------------------------------------------------
// Batched form (every member takes the fused ci sweep with the same solver and cluster size): ONE launch of
// k_ci_sweep with one cluster per model (plus one launch of k_ystats_small when observations changed).
// Otherwise: one captured graph with the members' sweeps as parallel branches.
struct mrgp_group {
    std::vector<mrgp_handle *> handles;
    std::vector<uint64_t> generation, stream_ops;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    bool batched = false;
    int solver = 0, cluster = 1, r0_max = 1;
    const ChainModel **ptrs_dev = nullptr;     // batched: device array of the members' descriptors
    cudaEvent_t ev = nullptr;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    std::vector<int64_t> launches_per_sweep;
    int64_t launches = 0;
    std::string error;
};

static int gfail(mrgp_group *g, int code, const char *what, cudaError_t e) {
    if (g) g->error = std::string(what) + ": " + cudaGetErrorString(e);
    cudaGetLastError();
    return code;
}

// Everything a member queued on its own stream (uploads, state writes, basis builds) precedes the group's next launch.
static int group_order_after_members(mrgp_group *g) {
    for (size_t i = 0; i < g->handles.size(); ++i) {
        mrgp_handle *h = g->handles[i];
        if (h->stream_ops == g->stream_ops[i] || h->stream == g->stream) continue;
        cudaError_t e = cudaEventRecord(g->ev, h->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(g->stream, g->ev, 0);
        if (e != cudaSuccess) return gfail(g, MRGP_ECUDA, "ordering after a member stream", e);
        g->stream_ops[i] = h->stream_ops;
    }
    return MRGP_OK;
}

static void group_drop(mrgp_group *g) {
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    g->exec = nullptr;
    g->graph = nullptr;
}

// (Re)build what the group replays: descriptors of the members (batched) or the branch graph.
static int group_prepare(mrgp_group *g) {
    const int n = (int)g->handles.size();
    group_drop(g);
    bool batched = true;
    int r0 = 1;
    for (int i = 0; i < n; ++i) {
        mrgp_handle *h = g->handles[i];
        int rc = check_ready(h, 0, true);
        if (rc) {
            g->error = h->err;
            return rc;
        }
        if ((rc = build_invariants(h, Launch{h->stream, &h->launches}))) return rc;
        const bool f = use_fused(h) && ystats_small(h);
        batched = batched && f && chain_solver_size(h->cfg.n_basis) == chain_solver_size(g->handles[0]->cfg.n_basis) &&
                  chain_cluster_size(h) == chain_cluster_size(g->handles[0]);
        if (use_fused(h) && !h->chain_uploaded && (rc = upload_chain_model(h))) return rc;
        r0 = std::max(r0, h->plan[0].R);
        if (cudaStreamSynchronize(h->stream) != cudaSuccess) return fail(h, MRGP_ECUDA, "stream synchronisation failed");
    }
    g->batched = batched;
    g->r0_max = r0;
    cudaError_t e;
    if (batched) {
        g->solver = chain_solver_size(g->handles[0]->cfg.n_basis);
        g->cluster = chain_cluster_size(g->handles[0]);
        if (!g->ptrs_dev && (e = cudaMalloc(&g->ptrs_dev, (size_t)n * sizeof(ChainModel *))) != cudaSuccess)
            return gfail(g, MRGP_ECUDA, "cudaMalloc of the descriptor table", e);
        std::vector<const ChainModel *> ptrs(n);
        for (int i = 0; i < n; ++i) ptrs[i] = g->handles[i]->chain_dev;
        if ((e = cudaMemcpy(g->ptrs_dev, ptrs.data(), (size_t)n * sizeof(ChainModel *), cudaMemcpyHostToDevice)) != cudaSuccess)
            return gfail(g, MRGP_ECUDA, "upload of the descriptor table", e);
        for (int i = 0; i < n; ++i) {
            g->generation[i] = g->handles[i]->generation;
            g->launches_per_sweep[i] = 0;
        }
        return MRGP_OK;
    }
    // the streams only shape the captured DAG (one branch per model); the replay does not use them
    std::vector<cudaStream_t> tmp(n, nullptr);
    std::vector<cudaEvent_t> done(n, nullptr);
    cudaEvent_t start = nullptr;
    int rc = MRGP_OK;
    auto cleanup = [&]() {
        for (auto st : tmp)
            if (st) cudaStreamDestroy(st);
        for (auto ev : done)
            if (ev) cudaEventDestroy(ev);
        if (start) cudaEventDestroy(start);
    };
    for (int i = 0; i < n && rc == MRGP_OK; ++i) {
        mrgp_handle *h = g->handles[i];
        if (use_fused(h) && !h->ystats_valid && (rc = do_ystats(h, Launch{h->stream, &h->launches}))) break;
        if (cudaStreamSynchronize(h->stream) != cudaSuccess) rc = MRGP_ECUDA;
        if (cudaStreamCreateWithFlags(&tmp[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) != cudaSuccess)
            rc = MRGP_ECUDA;
    }
    if (rc == MRGP_OK && cudaEventCreateWithFlags(&start, cudaEventDisableTiming) != cudaSuccess) rc = MRGP_ECUDA;
    if (rc == MRGP_OK && (e = cudaStreamBeginCapture(g->stream, cudaStreamCaptureModeThreadLocal)) != cudaSuccess)
        rc = gfail(g, MRGP_ECUDA, "cudaStreamBeginCapture", e);
    if (rc == MRGP_OK) {
        cudaEventRecord(start, g->stream);
        for (int i = 0; i < n; ++i) {
            mrgp_handle *h = g->handles[i];
            cudaStreamWaitEvent(tmp[i], start, 0);
            g->launches_per_sweep[i] = 0;
            const int r = sweep_once(h, Launch{tmp[i], &g->launches_per_sweep[i]});
            if (r && rc == MRGP_OK) rc = r;
            cudaEventRecord(done[i], tmp[i]);
            cudaStreamWaitEvent(g->stream, done[i], 0);
        }
        e = cudaStreamEndCapture(g->stream, &g->graph);
        if (rc == MRGP_OK && e != cudaSuccess) rc = gfail(g, MRGP_ECUDA, "cudaStreamEndCapture", e);
        if (rc == MRGP_OK && (e = cudaGraphInstantiate(&g->exec, g->graph, 0)) != cudaSuccess)
            rc = gfail(g, MRGP_ECUDA, "cudaGraphInstantiate", e);
    }
    cleanup();
    if (rc != MRGP_OK) {
        group_drop(g);
        return rc;
    }
    for (int i = 0; i < n; ++i) g->generation[i] = g->handles[i]->generation;
    return MRGP_OK;
}

int mrgp_group_create(mrgp_handle *const *handles, int32_t n, void *cuda_stream, mrgp_group **out) {
    if (!handles || !out || n < 1) return MRGP_EINVAL;
    *out = nullptr;
    for (int i = 0; i < n; ++i) {
        mrgp_handle *h = handles[i];
        int rc = check_ready(h, 0, true);
        if (rc) return rc;
        if (h->sharded) return fail(h, MRGP_EINVAL, "sharded handles cannot join a group");
        if (h->cfg.device != handles[0]->cfg.device) return fail(h, MRGP_EINVAL, "all models of a group live on one device");
    }
    mrgp_group *g = new mrgp_group();
    g->handles.assign(handles, handles + n);
    g->launches_per_sweep.assign(n, 0);
    g->generation.assign(n, ~0ull);
    g->stream_ops.assign(n, ~0ull);
    if (cuda_stream) {
        g->stream = static_cast<cudaStream_t>(cuda_stream);
    } else {
        if (cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete g;
            return MRGP_ECUDA;
        }
        g->own_stream = true;
    }
    int rc = cudaEventCreateWithFlags(&g->ev, cudaEventDisableTiming) == cudaSuccess ? MRGP_OK : MRGP_ECUDA;
    if (rc == MRGP_OK) rc = group_prepare(g);
    if (rc != MRGP_OK) {
        g_create_error = g->error;
        mrgp_group_destroy(g);
        return rc;
    }
    *out = g;
    return MRGP_OK;
}

int mrgp_group_sweep(mrgp_group *g, int32_t n_iter) {
    if (!g || n_iter < 0) return MRGP_EINVAL;
    const int n = (int)g->handles.size();
    // a member whose captured sweep / descriptor went stale (new pointers, new intervals, re-initialised state ...)
    // since the group was prepared: prepare again
    bool stale = false;
    for (int i = 0; i < n; ++i) stale = stale || g->handles[i]->generation != g->generation[i];
    int rc;
    if (stale && (rc = group_prepare(g))) return rc;
    if ((rc = group_order_after_members(g))) return rc;
    if (g->batched) {
        bool need_y = false;
        for (int i = 0; i < n; ++i) need_y = need_y || !g->handles[i]->ystats_valid;
        if (need_y) {   // new observations somewhere: the statistics of all members in one launch
            const int e = launch_ystats_small(g->solver, g->ptrs_dev, n, g->r0_max, g->stream);
            if (e != 0) return gfail(g, MRGP_ECUDA, "y statistics launch", (cudaError_t)e);
            for (int i = 0; i < n; ++i) g->handles[i]->ystats_valid = true;
            g->launches += 1;
        }
        for (int it = 0; it < n_iter; ++it) {
            int e = launch_ci_sweep(g->solver, g->ptrs_dev, n, g->cluster, g->stream);
            if (e != 0) return gfail(g, MRGP_ECUDA, "fused sweep launch", (cudaError_t)e);
            e = launch_l0_fix_small(g->solver, g->ptrs_dev, n, g->r0_max, g->stream);   // no-op for models whose guard did not trip
            if (e != 0) return gfail(g, MRGP_ECUDA, "layer-0 fallback launch", (cudaError_t)e);
        }
        g->launches += 2 * n_iter;
        for (int i = 0; i < n; ++i) g->handles[i]->sweeps_done += n_iter;
        return MRGP_OK;
    }
    for (int it = 0; it < n_iter; ++it) {
        cudaError_t e = cudaGraphLaunch(g->exec, g->stream);
        if (e != cudaSuccess) return gfail(g, MRGP_ECUDA, "cudaGraphLaunch", e);
    }
    for (int i = 0; i < n; ++i) {
        g->handles[i]->launches += g->launches_per_sweep[i] * n_iter;
        g->launches += g->launches_per_sweep[i] * n_iter;
        g->handles[i]->sweeps_done += n_iter;
    }
    return MRGP_OK;
}

int mrgp_group_observations_changed(mrgp_group *g) {
    if (!g) return MRGP_EINVAL;
    for (auto h : g->handles) h->ystats_valid = false;
    return MRGP_OK;
}

int64_t mrgp_group_launch_count(const mrgp_group *g) { return g ? g->launches : -1; }

int mrgp_group_synchronize(mrgp_group *g) {
    if (!g) return MRGP_EINVAL;
    cudaError_t e = cudaStreamSynchronize(g->stream);
    return e == cudaSuccess ? MRGP_OK : gfail(g, MRGP_ECUDA, "cudaStreamSynchronize", e);
}

void mrgp_group_destroy(mrgp_group *g) {
    if (!g) return;
    group_drop(g);
    if (g->ptrs_dev) cudaFree(g->ptrs_dev);
    if (g->ev) cudaEventDestroy(g->ev);
    if (g->own_stream && g->stream) cudaStreamDestroy(g->stream);
    delete g;
}

int mrgp_synchronize(mrgp_handle *h) {
    if (!h || !h->stream) return fail(h, MRGP_ESTATE, "no stream");
    CK(cudaStreamSynchronize(h->stream));
    if (h->comm.ready) {
        unsigned int err = 0;
        CK(cudaMemcpy(&err, h->comm.err, sizeof(err), cudaMemcpyDeviceToHost));
        if (err) return fail(h, MRGP_ECUDA, "peer exchange timed out: a rank did not publish its region sums");
    }
    return MRGP_OK;
}

int mrgp_elbo(mrgp_handle *h, double *out_host) {
    int rc = check_ready(h, 0, true);
    if (rc) return rc;
    if (!out_host) return fail(h, MRGP_EINVAL, "null argument");
    if (h->cfg.mode != MRGP_MODE_CI) return fail(h, MRGP_EINVAL, "the lower bound is defined for ci mode only (MRGP.py:378-401)");
    // the argument blocks of the layers live on the device; they change only with what drop_graph() tracks (pointers,
    // intervals, adaptive switches) and with the first sweep of an adaptive model
    const uint64_t key = h->generation * 2 + (h->sweeps_done > 0 ? 1 : 0);
    if (!h->elbo_args_valid || h->elbo_args_key != key) {
        std::vector<RegionArgs> args(h->cfg.n_layers);
        for (int j = 0; j < h->cfg.n_layers; ++j) {
            args[j] = region_args(h, j);
            args[j].ts = nullptr;
            // adaptive intervals: the data sums with the re-learnt basis (MRGP.py:535-569 reads phi_x after MRGP.py:640)
            if (h->dev[j].adaptive && h->sweeps_done > 0) args[j].sumsB = h->dev[j].sumsE;
        }
        CK(cudaMemcpyAsync(h->elbo_args, args.data(), args.size() * sizeof(RegionArgs), cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));   // args is a local
        h->elbo_args_valid = true;
        h->elbo_args_key = key;
    }
    k_elbo<2><<<dim3((unsigned)h->cfg.n_layers, (unsigned)h->elbo_chunks), 256, 0, h->stream>>>(h->elbo_args, h->elbo_out, h->elbo_part, h->elbo_counter);
    CK(cudaGetLastError());
    h->launches += 1;
    CK(cudaMemcpyAsync(out_host, h->elbo_out, (size_t)h->cfg.n_layers * 6 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (h->elbo_no_sync) return MRGP_OK;
    CK(cudaStreamSynchronize(h->stream));
    return MRGP_OK;
}

// The lower bound without the host round trip on the chain of a step: the terms are copied into pinned host memory behind the
// kernel and an event marks the copy; mrgp_elbo_wait(h, slot) blocks until the terms of that slot have arrived.  Two slots:
// a consumer that reads the result of step k while step k + 1 is already queued never idles the GPU.
int mrgp_elbo_async(mrgp_handle *h, double *out_pinned_host, int32_t slot) {
    if (!h || slot < 0 || slot > 1) return fail(h, MRGP_EINVAL, "slot must be 0 or 1");
    if (!h->ev_elbo[slot]) CK(cudaEventCreateWithFlags(&h->ev_elbo[slot], cudaEventDisableTiming));
    h->elbo_no_sync = true;
    const int rc = mrgp_elbo(h, out_pinned_host);
    h->elbo_no_sync = false;
    if (rc) return rc;
    CK(cudaEventRecord(h->ev_elbo[slot], h->stream));
    return MRGP_OK;
}

int mrgp_elbo_wait(mrgp_handle *h, int32_t slot) {
    if (!h || slot < 0 || slot > 1) return fail(h, MRGP_EINVAL, "slot must be 0 or 1");
    if (!h->ev_elbo[slot]) return fail(h, MRGP_ESTATE, "no mrgp_elbo_async on this slot yet");
    CK(cudaEventSynchronize(h->ev_elbo[slot]));
    return MRGP_OK;
}

// Test offsets of one layer: cnt entries from 0 to n_test, non-decreasing (a test region may be empty).  The region
// search of the prediction kernels assumes this order; decreasing offsets would put points in the wrong regions and
// give k_eval_var_indexed a negative region count.
static int check_test_offsets(mrgp_handle *h, const int64_t *off, size_t cnt, int64_t n_test, int j) {
    if (off[0] != 0 || off[cnt - 1] != n_test) return fail(h, MRGP_EINVAL, "test offsets of layer %d do not cover the test points", j);
    for (size_t r = 0; r + 1 < cnt; ++r)
        if (off[r + 1] < off[r])
            return fail(h, MRGP_EINVAL, "test offsets of layer %d must be non-decreasing (offset %zu: %lld < %lld)", j, r + 1,
                        (long long)off[r + 1], (long long)off[r]);
    return MRGP_OK;
}

int mrgp_predict_mean(mrgp_handle *h, const double *x_test_dev, int64_t n_test, const int64_t *const *test_offsets,
                      int32_t n_test_layers, double *out_dev) {
    int rc = check_ready(h, 0, true);
    if (rc) return rc;
    if (!x_test_dev || !out_dev || n_test < 1) return fail(h, MRGP_EINVAL, "bad argument");
    EvalArgs ea{};
    std::vector<const int64_t *> dev_off;
    int64_t *staging = nullptr;
    if (test_offsets) {
        if (n_test_layers < 1 || n_test_layers > h->cfg.n_layers)
            return fail(h, MRGP_EINVAL, "resolution in the test index set must be smaller or equal to that in the train set");
        staging = h->off_staging;
        size_t o = 0;
        for (int j = 0; j < n_test_layers; ++j) {
            const size_t cnt = h->plan[j].R + 1;
            if ((rc = check_test_offsets(h, test_offsets[j], cnt, n_test, j))) return rc;
            CK(cudaMemcpyAsync(staging + o, test_offsets[j], cnt * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
            dev_off.push_back(staging + o);
            o += cnt;
        }
        if ((rc = fill_eval_layers(h, ea, n_test_layers, dev_off.data()))) return rc;
        ea.single_region = 0;
    } else {
        if ((rc = fill_eval_layers(h, ea, 1, nullptr))) return rc;
        ea.single_region = 1;
    }
    ea.n = n_test;
    ea.x = x_test_dev;
    ea.out_mean = out_dev;
    ea.out_var = nullptr;
    k_eval_layers<2><<<(unsigned)((n_test + 127) / 128), 128, 0, h->stream>>>(ea);
    CK(cudaGetLastError());
    h->launches += 1;
    CK(cudaStreamSynchronize(h->stream));
    return MRGP_OK;
}

int mrgp_predict_var_indexed(mrgp_handle *h, const double *x_test_dev, int64_t n_test, const int64_t *const *test_offsets,
                             int32_t n_test_layers, double *out_dev) {
    int rc = check_ready(h, 0, true);
    if (rc) return rc;
    if (!x_test_dev || !out_dev || !test_offsets || n_test < 1) return fail(h, MRGP_EINVAL, "bad argument");
    if (n_test_layers != h->cfg.n_layers)
        return fail(h, MRGP_EINVAL, "the test index set must have the resolutions of the train set (MRGP.py:877-879 walks every layer)");
    EvalArgs ea{};
    std::vector<const int64_t *> dev_off;
    size_t o = 0;
    for (int j = 0; j < n_test_layers; ++j) {
        const size_t cnt = h->plan[j].R + 1;
        if ((rc = check_test_offsets(h, test_offsets[j], cnt, n_test, j))) return rc;
        CK(cudaMemcpyAsync(h->off_staging + o, test_offsets[j], cnt * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
        dev_off.push_back(h->off_staging + o);
        o += cnt;
    }
    if ((rc = fill_eval_layers(h, ea, n_test_layers, dev_off.data()))) return rc;
    ea.single_region = 0;
    ea.n = n_test;
    ea.x = x_test_dev;
    ea.out_mean = nullptr;
    ea.out_var = out_dev;
    k_eval_var_indexed<2><<<(unsigned)((n_test + 127) / 128), 128, 0, h->stream>>>(ea);
    CK(cudaGetLastError());
    h->launches += 1;
    CK(cudaStreamSynchronize(h->stream));
    return MRGP_OK;
}

int mrgp_predict_var(mrgp_handle *h, const double *x_test_dev, int64_t n_test, double *out_dev) {
    int rc = check_ready(h, 0, true);
    if (rc) return rc;
    if (!x_test_dev || !out_dev || n_test < 1) return fail(h, MRGP_EINVAL, "bad argument");
    EvalArgs ea{};
    if ((rc = fill_eval_layers(h, ea, 1, nullptr))) return rc;
    ea.single_region = 1;
    ea.n = n_test;
    ea.x = x_test_dev;
    ea.out_mean = nullptr;
    ea.out_var = out_dev;
    k_eval_layers<2><<<(unsigned)((n_test + 127) / 128), 128, 0, h->stream>>>(ea);
    CK(cudaGetLastError());
    h->launches += 1;
    CK(cudaStreamSynchronize(h->stream));
    return MRGP_OK;
}

namespace {
struct CommBlob {          // what the ranks all-gather; MRGP_COMM_BLOB_BYTES in the header
    uint64_t magic;
    int64_t pid;
    uint64_t ptr;
    int32_t device, pad;
    uint64_t bytes;
    cudaIpcMemHandle_t handle;
};
static_assert(sizeof(CommBlob) <= 128, "blob must fit MRGP_COMM_BLOB_BYTES");
constexpr uint64_t kBlobMagic = 0x6d726770636f6d31ull;
}   // namespace

int mrgp_comm_export(mrgp_handle *h, void *blob_out) {
    if (!h || !blob_out) return fail(h, MRGP_EINVAL, "null argument");
    if (!h->bound) return fail(h, MRGP_ESTATE, "no workspace bound");
    if (!h->sharded) return fail(h, MRGP_ESTATE, "not a sharded handle");
    auto &c = h->comm;
    if (!c.exported) {
        int rmax = 0;
        for (auto &lp : h->plan) rmax = std::max(rmax, lp.R);
        c.slot_doubles = ((size_t)rmax * h->part_stride + 31) & ~(size_t)31;
        c.bytes = 512 + kCommSlots * c.slot_doubles * sizeof(double);
        CK(cudaSetDevice(h->cfg.device));
        CK(cudaMalloc(&c.mem, c.bytes));
        CK(cudaMemset(c.mem, 0, c.bytes));
        c.flags = reinterpret_cast<unsigned long long *>(c.mem);
        c.seq = reinterpret_cast<unsigned long long *>(static_cast<char *>(c.mem) + 256);
        c.err = reinterpret_cast<unsigned int *>(static_cast<char *>(c.mem) + 320);
        c.counter = reinterpret_cast<unsigned int *>(static_cast<char *>(c.mem) + 384);
        c.arena = reinterpret_cast<double *>(static_cast<char *>(c.mem) + 512);
        c.exported = true;
    }
    CommBlob b{};
    b.magic = kBlobMagic;
    b.pid = (int64_t)getpid();
    b.ptr = (uint64_t)(uintptr_t)c.mem;
    b.device = h->cfg.device;
    b.bytes = c.bytes;
    CK(cudaIpcGetMemHandle(&b.handle, c.mem));
    std::memset(blob_out, 0, 128);
    std::memcpy(blob_out, &b, sizeof b);
    return MRGP_OK;
}

int mrgp_comm_bind(mrgp_handle *h, int32_t rank, int32_t world, const void *blobs, const int64_t *bounds) {
    if (!h || !blobs || !bounds) return fail(h, MRGP_EINVAL, "null argument");
    auto &c = h->comm;
    if (!c.exported) return fail(h, MRGP_ESTATE, "mrgp_comm_export first");
    if (c.ready) return fail(h, MRGP_ESTATE, "peer exchange already bound");
    if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world) return fail(h, MRGP_EINVAL, "rank / world out of range (at most %d ranks)", kMaxRanks);
    if (bounds[0] != 0 || bounds[world] != h->cfg.n_samples || bounds[rank] != h->lo || bounds[rank + 1] != h->hi)
        return fail(h, MRGP_EINVAL, "bounds do not match the sample range of this handle");
    for (int q = 0; q < world; ++q)
        if (bounds[q + 1] < bounds[q]) return fail(h, MRGP_EINVAL, "bounds must be non-decreasing");
    CK(cudaSetDevice(h->cfg.device));
    CommArgs a{};
    a.rank = rank;
    a.world = world;
    a.seq = c.seq;
    a.err = c.err;
    a.slot_doubles = c.slot_doubles;
    for (int q = 0; q <= world; ++q) a.bounds[q] = bounds[q];
    for (int q = 0; q < world; ++q) {
        CommBlob b;
        std::memcpy(&b, static_cast<const char *>(blobs) + (size_t)q * 128, sizeof b);
        if (b.magic != kBlobMagic || b.bytes != c.bytes) return fail(h, MRGP_EINVAL, "blob of rank %d is not from a matching handle", q);
        void *base = nullptr;
        if (q == rank) {
            base = c.mem;
        } else if (b.pid == (int64_t)getpid()) {
            base = reinterpret_cast<void *>((uintptr_t)b.ptr);      // same process (several handles, threads): plain pointer
            if (b.device != h->cfg.device) {
                int can = 0;
                CK(cudaDeviceCanAccessPeer(&can, h->cfg.device, b.device));
                if (!can) return fail(h, MRGP_ENODEVICE, "device %d cannot map the memory of device %d", h->cfg.device, b.device);
                cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
                cudaGetLastError();
            }
        } else {
            CK(cudaIpcOpenMemHandle(&base, b.handle, cudaIpcMemLazyEnablePeerAccess));
            c.peer_base[q] = base;
            c.opened[q] = true;
        }
        a.flags[q] = reinterpret_cast<unsigned long long *>(base);
        a.arena[q] = reinterpret_cast<const double *>(static_cast<char *>(base) + 512);
    }
    // same shared-memory carveout as the rest of the sweep: no SM reconfiguration around the exchanges
    CK(cudaFuncSetAttribute(k_comm_sums_signal<false>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    CK(cudaFuncSetAttribute(k_comm_sums_signal<true>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    CK(cudaFuncSetAttribute(k_comm_reduce<false>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    CK(cudaFuncSetAttribute(k_comm_reduce<true>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    CK(cudaFuncSetAttribute(k_bias_noise<2>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    c.args = a;
    c.ready = true;
    drop_graph(h);
    return MRGP_OK;
}

int mrgp_exchange(mrgp_handle *h, int32_t layer, int32_t which) {
    int rc = check_ready(h, layer, false);
    if (rc) return rc;
    if (!h->sharded) return fail(h, MRGP_ESTATE, "not a sharded handle");
    if (which != MRGP_X_PHASE_A && which != MRGP_X_PHASE_B) return fail(h, MRGP_EINVAL, "which must be MRGP_X_PHASE_A or MRGP_X_PHASE_B");
    return do_exchange(h, Launch{h->stream, &h->launches}, layer, which == MRGP_X_PHASE_A ? h->cfg.n_basis * h->cfg.dy : h->cfg.dy + 3, false);
}

int64_t mrgp_launch_count(const mrgp_handle *h) { return h ? h->launches : -1; }

int64_t mrgp_cholesky_count(mrgp_handle *h) {
    if (!h || !h->bound) return -1;
    unsigned long long v = 0;
    if (cudaMemcpyAsync(&v, h->chol_count, sizeof v, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) return -1;
    return (int64_t)v;
}

int mrgp_batched_cholesky(void *cuda_stream, double *a_dev, int32_t n, int64_t batch, int32_t *info_dev) {
    mrgp_handle *h = nullptr;
    if (!a_dev || !info_dev || n < 1 || n > 32 || batch < 1) return fail(h, MRGP_EINVAL, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    const unsigned small_grid = (unsigned)((batch + 255) / 256);
    switch (n) {   // n <= 8: one thread per matrix; larger: one warp per matrix
        case 1: k_batched_cholesky_small<1><<<small_grid, 256, 0, st>>>(a_dev, batch, info_dev); break;
        case 2: k_batched_cholesky_small<2><<<small_grid, 256, 0, st>>>(a_dev, batch, info_dev); break;
        case 3: k_batched_cholesky_small<3><<<small_grid, 256, 0, st>>>(a_dev, batch, info_dev); break;
        case 4: k_batched_cholesky_small<4><<<small_grid, 256, 0, st>>>(a_dev, batch, info_dev); break;
        case 5: k_batched_cholesky_small<5><<<small_grid, 256, 0, st>>>(a_dev, batch, info_dev); break;
        case 6: k_batched_cholesky_small<6><<<small_grid, 256, 0, st>>>(a_dev, batch, info_dev); break;
        case 7: k_batched_cholesky_small<7><<<small_grid, 256, 0, st>>>(a_dev, batch, info_dev); break;
        case 8: k_batched_cholesky_small<8><<<small_grid, 256, 0, st>>>(a_dev, batch, info_dev); break;
        default: {
            const int64_t threads = batch * 32;
            k_batched_cholesky<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(a_dev, n, batch, info_dev);
        }
    }
    CK(cudaGetLastError());
    return MRGP_OK;
}

int mrgp_fp64_probe(void *cuda_stream, int64_t iters, double *sink_dev, float *ms_out) {
    mrgp_handle *h = nullptr;
    if (!sink_dev || !ms_out || iters < 1) return fail(h, MRGP_EINVAL, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    int dev = 0, sms = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    k_fp64_probe<<<sms * 4, 256, 0, st>>>(iters / 8 + 1, sink_dev);   // warm-up
    CK(cudaEventRecord(e0, st));
    k_fp64_probe<<<sms * 4, 256, 0, st>>>(iters, sink_dev);
    CK(cudaEventRecord(e1, st));
    CK(cudaEventSynchronize(e1));
    CK(cudaEventElapsedTime(ms_out, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return MRGP_OK;
}

// Debug aid (not part of the reference-facing surface): per-kernel completion times of one sweep.
// mrgp_timeline_enable(h, 1) before the first mrgp_sweep() makes the captured graph carry timing events;
// mrgp_timeline_read() returns (tag, ms since sweep start) pairs: tag 1 phase A, 2 mid-step, 3 phase B, 4 omega.
int mrgp_timeline_enable(mrgp_handle *h, int32_t on) {
    if (!h) return MRGP_EINVAL;
    h->timeline = on != 0;
    drop_graph(h);
    return MRGP_OK;
}

int mrgp_timeline_read(mrgp_handle *h, int32_t *tags, float *ms, int32_t cap) {
    // Runs one sweep with fresh stamps and returns, per kernel in issue order, its begin and end in ms relative to
    // the earliest begin: tags[k] = layer * 4 + kind (0 phase A, 1 mid-step, 2 phase B, 3 omega), ms[2k], ms[2k+1].
    if (!h || !tags || !ms || !h->timeline) return MRGP_EINVAL;
    if (h->cfg.n_layers > kMaxLayersTs) return MRGP_EINVAL;
    const int n = kMaxLayersTs * 4 + h->cfg.n_layers * 4;   // kernel slots, then the debug slots of the omega solve
    if (cap < n) return MRGP_EINVAL;
    std::vector<unsigned long long> init((size_t)kMaxLayers * 8), got((size_t)kMaxLayers * 8);
    for (size_t k = 0; k < init.size(); k += 2) {
        init[k] = ~0ull;
        init[k + 1] = 0ull;
    }
    CK(cudaMemcpyAsync(h->ts, init.data(), init.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, h->stream));
    int rc = mrgp_sweep(h, 1);
    if (rc) return rc;
    CK(cudaMemcpyAsync(got.data(), h->ts, got.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    unsigned long long t0 = ~0ull;
    for (int k = 0; k < n; ++k)
        if (got[2 * k + 1] != 0ull) t0 = std::min(t0, got[2 * k]);
    for (int k = 0; k < n; ++k) {
        tags[k] = k;
        const bool ran = got[2 * k + 1] != 0ull;
        ms[2 * k] = ran ? (float)((got[2 * k] - t0) * 1e-6) : -1.f;
        ms[2 * k + 1] = ran ? (float)((got[2 * k + 1] - t0) * 1e-6) : -1.f;
    }
    return n;
}

// ---- host-only hooks ----------------------------------------------------------------------------
int mrgp_plan_info(const mrgp_handle *h, int32_t layer, int32_t *n_ctas, int32_t *n_segments, int32_t *n_runs) {
    if (!h || layer < 0 || layer >= h->cfg.n_layers) return MRGP_EINVAL;
    if (n_ctas) *n_ctas = h->n_ctas;
    if (n_segments) *n_segments = (int32_t)h->plan[layer].segs.size();
    if (n_runs) *n_runs = h->plan[layer].n_runs;
    return MRGP_OK;
}

int mrgp_plan_segments(const mrgp_handle *h, int32_t layer, int64_t *seg_out) {
    if (!h || !seg_out || layer < 0 || layer >= h->cfg.n_layers) return MRGP_EINVAL;
    const LayerPlan &lp = h->plan[layer];
    for (size_t k = 0; k < lp.segs.size(); ++k) {
        seg_out[k * 6 + 0] = lp.segs[k].start;
        seg_out[k * 6 + 1] = lp.segs[k].start + lp.segs[k].len;
        seg_out[k * 6 + 2] = lp.segs[k].region;
        seg_out[k * 6 + 3] = lp.segs[k].parent;
        seg_out[k * 6 + 4] = lp.segs[k].run;
        seg_out[k * 6 + 5] = lp.seg_cta[k];
    }
    return MRGP_OK;
}

int mrgp_plan_pieces(const mrgp_handle *h, int32_t layer, int32_t *n_pieces, int64_t *piece_out) {
    if (!h || !n_pieces || layer < 0 || layer >= h->cfg.n_layers) return MRGP_EINVAL;
    const LayerPlan &lp = h->plan[layer];
    *n_pieces = (int32_t)lp.pc_jp.size();
    if (!piece_out) return MRGP_OK;
    const int R = lp.R;
    for (size_t k = 0; k < lp.pc_jp.size(); ++k) {
        const int jp = lp.pc_jp[k];
        int c = 0;   // region of the layer that owns the piece: the CSR row of (jp, c) containing k
        while (!(lp.pc_ptr[(size_t)jp * (R + 1) + c] <= (int32_t)k && (int32_t)k < lp.pc_ptr[(size_t)jp * (R + 1) + c + 1])) ++c;
        piece_out[k * 5 + 0] = jp;
        piece_out[k * 5 + 1] = c;
        piece_out[k * 5 + 2] = lp.pc_anc[k];
        piece_out[k * 5 + 3] = lp.pc_lo[k];
        piece_out[k * 5 + 4] = lp.pc_hi[k];
    }
    return MRGP_OK;
}

double mrgp_host_digamma(double x) { return digamma(x); }

double mrgp_host_matern_spectral(double lambda, double nu, double l, double sf) { return matern_spectral(lambda, nu, l, sf); }

void mrgp_host_bingham2(const double *b_in, double *b_out, double *kappa, double *rho, double *logc, double *axis_cov, int32_t *n_chol) {
    Bingham2 bg;
    bingham2(b_in[0], 0.5 * (b_in[1] + b_in[2]), b_in[3], bg);
    b_out[0] = bg.b[0];
    b_out[1] = b_out[2] = bg.b[1];
    b_out[3] = bg.b[2];
    kappa[0] = bg.kappa[0];
    kappa[1] = bg.kappa[1];
    rho[0] = bg.rho[0];
    rho[1] = bg.rho[1];
    *logc = bg.logc;
    axis_cov[0] = bg.cov[0];
    axis_cov[1] = axis_cov[2] = bg.cov[1];
    axis_cov[3] = bg.cov[2];
    if (n_chol) *n_chol = bg.n_chol;
}

void mrgp_host_basis(double x, double L, int32_t n_basis, double *phi_out) {
    double f1, c2;
    basis_seed(x, 0.5 / L, 1.0 / std::sqrt(L), f1, c2);
    double fm = 0.0, f = f1;
    for (int i = 0; i < n_basis; ++i) {
        phi_out[i] = f;
        const double fn = std::fma(c2, f, -fm);
        fm = f;
        f = fn;
    }
}

int mrgp_host_omega(const double *lw, int32_t m, double *omega_out, int32_t *iters_out) {
    std::vector<double> w((size_t)3 * m * m + 4 * m);
    double *K = w.data(), *P = K + m * m, *S = P + m * m, *v = S + m * m, *c = v + m, *rhs = c + m, *dinv = rhs + m;
    const int it = omega_solve_serial(lw, m, omega_out, K, P, S, v, c, rhs, dinv);
    if (iters_out) *iters_out = it;
    return MRGP_OK;
}

}  // extern "C"

