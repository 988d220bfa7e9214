// Fused ci sweep for sm_100a: one thread-block cluster per model runs ALL layers of one variational sweep
// (MRGP.py:571-652, static basis intervals) in a single kernel.  See mrgp_chain.h for the why.
//
// Roles inside a cluster of C CTAs x 256 threads:
//   * warp 0 of CTA 0 is the SOLVER: the doubly-stochastic scaling omega (Stats.py:413-420) with the table in its
//     registers (one lane per row), exactly the scheme of omega_solve_serial (mrgp_math.cuh);
//   * every other warp is a WORKER: a region of a layer belongs to one worker warp (lane = basis function) for all
//     of its per-region steps: P1-finish (y_tilde, precision, zeta: Posteriors.py:35-78), S2 (a, m2, cm2:
//     Stats.py:67-100), P4 / P5 / S5 (bias and noise posteriors from closed-form statistics: Posteriors.py:81-148,
//     Stats.py:102-124);
//   * CTA 0 as a whole does the shared step of a layer (P2, P2a-c, S1, P3, S3 and the log omega_hat table:
//     Posteriors.py:497-541, Stats.py:375-412) from the region sums that the CTAs leave in their shared memory
//     (read over DSMEM).
// Per layer: the region sums reach CTA 0, shared step on CTA 0, its results reach the workers, then the solver works
// on omega(j) WHILE the workers finish layer j (S2, P4/P5) and prepare the region sums of layer j + 1 (which need the
// ARD moments of layer j but not omega(j)).  Sums are formed in a fixed order: results are bit-reproducible for a
// cluster size.
//
// Hand-offs inside a cluster of C >= 2 CTAs are PUSHES over DSMEM, signalled through mbarriers (a hardware cluster
// barrier costs ~1.2k cycles with 16 CTAs and waits for every thread; a remote store + remote mbarrier arrive costs one
// DSMEM hop and only the consumer waits):
//   A(j): every worker CTA stores its region sums into its slot of CTA 0 with st.async, counted on CTA 0's barA;
//   B(j): CTA 0 stores the axis covariances / ARD means of layer j into loc[j & 1] of every worker CTA with st.async,
//         counted on its barB - and goes on to the solve without waiting for anybody;
//         (st.async: data and completion travel together - a release.cluster arrive costs a MEMBAR.GPU instead)
//   F(j): S2 / P4 / P5 of layer j + 1 read moments that OTHER worker CTAs wrote for layer j (global memory): every worker
//         CTA arrives on every worker's barF when its share of layer j is done and waits for phase j before layer j + 1.
// A cluster of one CTA (batch of small models) keeps the two barriers per layer (its "cluster" barrier is a CTA barrier).
#include "mrgp_chain.h"

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdlib>

#include "mrgp_math.cuh"

namespace cg = cooperative_groups;

namespace mrgp {
namespace {

constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ double wsum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ double wmax(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define PROF(k)                                                              \
    do {                                                                     \
        if (m.prof) m.prof[j * 16 + (k)] = (double)clock64();                \
    } while (0)
// 1 / x for normal positive x to the last bit or two: the hardware's reciprocal estimate (20 bits) and two Newton steps.  The
// IEEE division of the compiler is a subroutine of ~30 instructions with its special-case paths; the chain has five of them
// in a row per layer (Bingham constants, digamma, ARD mean), the solver two per evaluation and the workers three per region.
__device__ __forceinline__ double rcp_fast(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
}
// Maximum over the warp for a stabilising shift: rounded UP to single precision (the shift only has to bound the largest
// entry; any common shift of a row or column leaves omega unchanged) and reduced with one REDUX on an order-preserving
// integer image instead of a five-step butterfly of 64-bit shuffles and compares.
__device__ __forceinline__ double wmax_shift(double v) {
    unsigned b = __float_as_uint(__double2float_ru(v));
    b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
    b = __reduce_max_sync(kFull, b);
    b = (b & 0x80000000u) ? (b & 0x7fffffffu) : ~b;
    return (double)__uint_as_float(b);
}
// N sums over the warp in lock-step: the butterflies of the N values overlap instead of running one after the other
template <int N>
__device__ __forceinline__ void wsum_n(double (&v)[N]) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < N; ++k) v[k] += __shfl_xor_sync(kFull, v[k], o);
    }
}
// ---- DSMEM pushes and mbarriers at cluster scope ----------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// address of the same shared-memory variable in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t remote_addr(uint32_t local, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
    return r;
}
// asynchronous store of one double into the shared memory of another CTA of the cluster; its completion is counted (8
// bytes) on the mbarrier `bar` of that CTA: data and signal travel together, no fence on either side
__device__ __forceinline__ void st_async_remote(uint32_t addr, double v, uint32_t bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f64 [%0], %1, [%2];" ::"r"(addr), "d"(v), "r"(bar) : "memory");
}
// arm the current phase of a barrier of this CTA: one arrival (the barriers of the pushes are initialised with count 1)
// and `bytes` of asynchronous stores to come
__device__ __forceinline__ void bar_expect(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
// one arrival on the mbarrier at cluster address `addr`; publishes the writes that happen before it (cumulative over
// __syncwarp / CTA barriers) to the CTA that owns the barrier
__device__ __forceinline__ void bar_arrive_remote(uint32_t addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(addr) : "memory");
}
// wait for the phase of parity `parity` of a barrier that counts asynchronous stores (their data is visible with it)
__device__ __forceinline__ void bar_wait_tx(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_addr(bar)),
        "r"(parity)
        : "memory");
}
// wait for the phase of parity `parity` of a barrier of this CTA; acquires what the arriving CTAs published (global memory)
__device__ __forceinline__ void bar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_addr(bar)),
        "r"(parity)
        : "memory");
}
// split cluster barrier: arrive publishes this thread's writes, wait makes the others' visible
__device__ __forceinline__ void cl_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cl_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void worker_bar(int count) { asm volatile("bar.sync 1, %0;" ::"r"(count) : "memory"); }

constexpr int kChainAndersonIters = 48;   // accelerated evaluations before the plain Sinkhorn sweeps take over
constexpr unsigned kSumBytes = 7 * 32 * 8, kPubBytes = 4 * 32 * 8;   // region sums of a CTA, covariances + ARD means of a layer
constexpr int LD = 34;    // row stride of the transposed tables: conflict-free columns, 16-byte aligned rows
constexpr int LW = 33;    // row stride of the log omega_hat table

struct ChainSmem {
    double omT[32 * LD];      // omega transposed: omT[k * LD + i] = omega_ik
    double Kt[32 * LD];       // shifted, exponentiated table, column-major: Kt[k * LD + i] = K_ik
    double lw[32 * LW];       // log omega_hat, row-major
    double primeB[32 * 4], primeLogC[32], primeShape[32], primeScale[32], sk[32], skNext[32];
    double B[32 * 4], kappa[32 * 2], rho[32 * 2], logC[32], cov[32 * 4], shape[32], scale[32], mean[32], lmean[32];
    double part[8][7][32];    // per-warp region sums of the P1-finish step
    double ctaPart[7 * 32];   // per-CTA sums (cluster of one CTA; a cluster of several pushes them into `slots` of CTA 0)
    double slots[kChainMaxCluster][7 * 32];   // CTA 0: the per-CTA sums of the worker CTAs, written by them over DSMEM
    uint64_t barA, barB, barF;                // mbarriers of the hand-offs (see the head of the file)
    double data[7 * 32];      // cluster sums (CTA 0)
    double pub[4 * 32];       // CTA 0: axis covariance (c00, c01, c11) and ARD mean of the layer, read by every CTA
    double loc[2][4 * 32];    // local copies of pub, by layer parity (the background step of layer j reads its copy while
                              // the copy of layer j + 1 is being written)
    double rowmax[32], colmax[32];
    double dg[32], sh[32], sc[32];              // shared step: digamma(shape), mixed prior shape / scale
    alignas(16) double sv[32], su[32];          // solver: column and row scalings of the current iterate (broadcast reads)
    double eta[kChainMaxLayers][32];            // warm start of the solver: log column scalings of the previous sweep
    double vout[kChainMaxLayers][32], cshift[kChainMaxLayers][32];   // column scalings and shifts of this sweep's solves
    double warm[kChainMaxLayers];
    int nchol;
    // the model's descriptor: every pointer of the sweep comes from here (a descriptor left in global memory costs an L2
    // round trip before each data access: the cluster barriers invalidate L1)
    alignas(16) unsigned char model[sizeof(ChainModel)];
};

// ---- worker steps (one warp per region, lane = basis function) --------------------------------------------------

// P1-finish of a region (Posteriors.py:35-78) and its contribution to the sums over regions that the shared step
// needs: 0.5 noise zeta y y^T (B_i, Posteriors.py:507-517) and the two terms that make sum_l m2/S linear in the axis
// covariance (ARD, Posteriors.py:533-541; see k_mid1).
__device__ __forceinline__ void p1_finish(const ChainLayer &ly, size_t ri, double y0, double y1, double dsum, double S, double noise,
                                          double ard, double (&acc)[7]) {
    const double is = rcp_fast(S);
    const double prec = fma(ard, is, noise * dsum);      // Posteriors.py:40-42: ard / S + noise sum phi^2
    const double ip = rcp_fast(prec);
    const double zeta = noise * ip;
    *reinterpret_cast<double2 *>(ly.ytil + ri * 2) = make_double2(y0, y1);
    ly.prec[ri] = prec;
    ly.zeta[ri] = zeta;
    const double w = 0.5 * noise * zeta;
    acc[0] += w * (y0 * y0);
    acc[1] += w * (y0 * y1);
    acc[2] += w * (y1 * y1);
    const double z2s = zeta * zeta * is;
    acc[3] += is * ip;
    acc[4] += z2s * (y0 * y0);
    acc[5] += z2s * (y0 * y1);
    acc[6] += z2s * (y1 * y1);
}

// Layer 0 (observed targets, no latent function), from the sufficient statistics of y:
//     y_tilde_i = (Phi^T y)_i - s_i b - sum_{k != i} G_ik a_k
__device__ __forceinline__ void mid1_layer0(const ChainModel &m, const ChainLayer &ly, int l, int lane, const double *ardMean, double (&acc)[7]) {
    const int M = m.M;
    const bool on = lane < M;
    const size_t ri = (size_t)l * M + (on ? lane : 0);
    const double2 a = on ? __ldcg(reinterpret_cast<const double2 *>(ly.A) + ri) : make_double2(0.0, 0.0);
    const double dsum = on ? __ldg(ly.d + ri) : 0.0, S = on ? __ldg(ly.S + ri) : 1.0;
    const double noise = __ldcg(ly.noise_mean + l);
    const double b0 = __ldcg(ly.bias_mean + (size_t)l * 2), b1 = __ldcg(ly.bias_mean + (size_t)l * 2 + 1);
    const double s = on ? __ldg(ly.sumPhi + ri) : 0.0;
    double t0 = on ? fma(-s, b0, ly.yc[ri * 2]) : 0.0, t1 = on ? fma(-s, b1, ly.yc[ri * 2 + 1]) : 0.0;
    const double *G = ly.gram + (size_t)l * M * M;
    double g[32];      // column `lane` of G without its diagonal entry, all loads in flight at once
#pragma unroll
    for (int k = 0; k < 32; ++k) g[k] = (on && k < M && k != lane) ? __ldg(G + (size_t)k * M + lane) : 0.0;
#pragma unroll
    for (int k = 0; k < 32; ++k) {
        t0 = fma(-g[k], __shfl_sync(kFull, a.x, k), t0);
        t1 = fma(-g[k], __shfl_sync(kFull, a.y, k), t1);
    }
    if (on) p1_finish(ly, ri, t0, t1, dsum, S, noise, ardMean[lane], acc);
}

// Regions a worker warp takes at once in P1-finish / in S2 + P4 / P5 of the layers above the first: ONE form per step,
// whatever the number of regions (unused slots are masked), so that its code is fetched once, at the first layer, and
// not for the first time on the fine layers after an L2 flush.  Layer 9 at config 4 (512 regions on 120 worker warps)
// is one batch of each.
constexpr int kMid1Batch = 8, kFinishBatch = 5;

// Layers above the first (targets inferred from the layer's own posterior, LatentOutputs.py:20-49): y_tilde_i = d_i a_i.
// NB regions l0, l0 + stride, ... at once: their loads are issued together (the step is a chain of L2 round trips).
template <int NB>
__device__ __forceinline__ void mid1_upper(const ChainModel &m, const ChainLayer &ly, int l0, int stride, int lane, const double *ardMean,
                                           double (&acc)[7]) {
    const int M = m.M;
    const bool on = lane < M;
    double2 a[NB];
    double dsum[NB], S[NB], noise[NB];
    size_t ri[NB];
    bool act[NB];
#pragma unroll
    for (int q = 0; q < NB; ++q) {
        const int l = l0 + q * stride;
        act[q] = on && l < ly.R;
        ri[q] = (size_t)(act[q] ? l : 0) * M + (on ? lane : 0);
        a[q] = act[q] ? __ldcg(reinterpret_cast<const double2 *>(ly.A) + ri[q]) : make_double2(0.0, 0.0);
        dsum[q] = act[q] ? __ldg(ly.d + ri[q]) : 0.0;
        S[q] = act[q] ? __ldg(ly.S + ri[q]) : 1.0;
        noise[q] = act[q] ? __ldcg(ly.noise_mean + l) : 0.0;
    }
    const double ard = ardMean[lane];
#pragma unroll
    for (int q = 0; q < NB; ++q)
        if (act[q]) p1_finish(ly, ri[q], dsum[q] * a[q].x, dsum[q] * a[q].y, dsum[q], S[q], noise[q], ard, acc);
}

// P4 / P5 / S5 of one region from its statistics sums = [sum r_0, sum r_1, sum |r|^2, sum f_var, sum phi^2 cm2]
// (region-specific noise and bias: Posteriors.py:81-93, 132-148 - y_var NOT times n, :138; Stats.py:102-124).
// rc: the region's constants [n, bias_prec0, bias_mean0 (2), noise_shape0, noise_scale0, digamma(noise shape), -].
__device__ __forceinline__ void bias_noise_update(const ChainLayer &ly, int l, bool infer, const double (&sums)[5], const double (&rc)[7],
                                                  double noise_old, double b0, double b1) {
    const double n = rc[0], bp0 = rc[1], bp = bp0 + n, ibp = rcp_fast(bp);
    const double mn0 = ibp * (rc[2] * bp0 + sums[0]), mn1 = ibp * (rc[3] * bp0 + sums[1]);
    const double t3 = bp0 * (rc[2] * rc[2] + rc[3] * rc[3]), t4 = bp * (mn0 * mn0 + mn1 * mn1);
    const double yvar = infer ? rcp_fast(noise_old) : 0.0;
    const double shape = rc[4] + 0.5 * 2.0 * n;
    const double scale = rc[5] + 0.5 * (t3 - t4 + sums[2] + sums[3] + sums[4] + yvar);
    *reinterpret_cast<double2 *>(ly.bias_prev + (size_t)l * 2) = make_double2(b0, b1);
    *reinterpret_cast<double2 *>(ly.bias_mean + (size_t)l * 2) = make_double2(mn0, mn1);
    ly.yvar[l] = yvar;
    ly.bias_prec[l] = bp;
    ly.bias_var[l] = ibp;
    ly.noise_shape[l] = shape;
    ly.noise_scale[l] = scale;
    ly.noise_mean[l] = shape * rcp_fast(scale);
    ly.noise_log_mean[l] = rc[6] - log(scale);
#pragma unroll
    for (int d = 0; d < 5; ++d) ly.sumsB[(size_t)l * 5 + d] = sums[d];
}

// S2 of a region (Stats.py:67-100) with the layer's new axis covariance; returns the new coefficients and cm2.
__device__ __forceinline__ void s2_region(const ChainLayer &ly, size_t ri, bool on, double c00, double c01, double c11, double2 yt,
                                          double zeta, double prec, double2 ao, double2 &an, double &cm2) {
    const double cy0 = c00 * yt.x + c01 * yt.y, cy1 = c01 * yt.x + c11 * yt.y;
    an = make_double2(zeta * cy0, zeta * cy1);
    const double z2 = zeta * zeta;
    const double ccy0 = c00 * cy0 + c01 * cy1, ccy1 = c01 * cy0 + c11 * cy1;
    const double ip = rcp_fast(prec);
    const double m2 = ip + z2 * (yt.x * cy0 + yt.y * cy1);
    cm2 = ip + z2 * (yt.x * (cy0 - ccy0) + yt.y * (cy1 - ccy1));
    if (on) {
        *reinterpret_cast<double2 *>(ly.A_prev + ri * 2) = ao;
        *reinterpret_cast<double2 *>(ly.A + ri * 2) = an;
        ly.m2[ri] = m2;
        ly.cm2[ri] = cm2;
    }
}

// Layer 0: S2, then the P4 / P5 statistics from the sufficient statistics of y and the bias / noise update:
//   r = y - Phi A_new:   sum r = sum y - A^T s,   sum |r|^2 = sum |y|^2 - 2 tr(A^T Phi^T y) + tr(A^T G A)
__device__ __forceinline__ void mid2_stats_layer0(const ChainModel &m, const ChainLayer &ly, int l, int lane, const double *cov) {
    const int M = m.M;
    const bool on = lane < M;
    const size_t ri = (size_t)l * M + (on ? lane : 0);
    const double2 yt = on ? __ldcg(reinterpret_cast<const double2 *>(ly.ytil) + ri) : make_double2(0.0, 0.0);
    const double zeta = on ? __ldcg(ly.zeta + ri) : 0.0, prec = on ? __ldcg(ly.prec + ri) : 1.0;
    const double2 ao = on ? __ldcg(reinterpret_cast<const double2 *>(ly.A) + ri) : make_double2(0.0, 0.0);
    const double dsum = on ? __ldg(ly.d + ri) : 0.0, si = on ? __ldg(ly.sumPhi + ri) : 0.0;
    const double2 yc = on ? *reinterpret_cast<const double2 *>(ly.yc + ri * 2) : make_double2(0.0, 0.0);
    const double rcl = lane < 7 ? __ldg(ly.rconst + (size_t)l * 8 + lane) : 0.0;
    const double b0 = __ldcg(ly.bias_mean + (size_t)l * 2), b1 = __ldcg(ly.bias_mean + (size_t)l * 2 + 1);
    const double ys0 = ly.ysum[(size_t)l * 4 + 0], ys1 = ly.ysum[(size_t)l * 4 + 1], y2 = ly.ysum[(size_t)l * 4 + 2];
    double2 an;
    double cm2;
    s2_region(ly, ri, on, cov[lane], cov[32 + lane], cov[64 + lane], yt, zeta, prec, ao, an, cm2);
    const double *G = ly.gram + (size_t)l * M * M;
    double g[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) g[k] = (on && k < M) ? __ldg(G + (size_t)k * M + lane) : 0.0;
    double t0 = 0.0, t1 = 0.0;
#pragma unroll
    for (int k = 0; k < 32; ++k) {
        t0 = fma(g[k], __shfl_sync(kFull, an.x, k), t0);
        t1 = fma(g[k], __shfl_sync(kFull, an.y, k), t1);
    }
    const double sa0 = wsum(si * an.x), sa1 = wsum(si * an.y);
    const double cross = wsum(an.x * yc.x + an.y * yc.y);
    const double quad = wsum(an.x * t0 + an.y * t1);
    double sums[5];
    sums[0] = ys0 - sa0;
    sums[1] = ys1 - sa1;
    sums[2] = (y2 - 2.0 * cross) + quad;
    sums[3] = 0.0;
    sums[4] = wsum(dsum * cm2);
    double rc[7];
#pragma unroll
    for (int t = 0; t < 7; ++t) rc[t] = __shfl_sync(kFull, rcl, t);
    if (lane == 0) {
        if (l == 0) {
            const double ratio = y2 > 0.0 ? sums[2] / y2 : 1.0;
            m.guard[0] = ratio;
            if (!(ratio >= m.guard_threshold)) {
                atomicOr(m.status, 1u);
                m.guard[1] = 1.0;
            }
        }
        bias_noise_update(ly, l, false, sums, rc, 1.0, b0, b1);
    }
}

// Layers above the first: S2, then the statistics of r = Phi (A_old - A_new) + b_old in closed form (see k_stats_b):
//   sum r = dA^T s + n b,  sum |r|^2 = sum_d dA_d^T G dA_d + 2 b . (dA^T s) + n |b|^2,  sum phi^2 cm2 = d . cm2,
//   sum f_var = sum over the region's pieces with coarser regions of (len bias_var_anc + cm2_anc . D_piece)
// and the bias / noise update.  NB regions at once: two L2 round trips per batch (own data + piece table, then the
// coarser regions' moments), all warp sums of the batch in one lock-step butterfly, the NB updates on NB lanes side
// by side (lane q loads the constants of region q itself).
template <int NB>
__device__ __forceinline__ void mid2_stats_upper(const ChainModel &m, const ChainLayer &ly, int l0, int stride, int lane, const double *cov) {
    const int M = m.M, E = ly.E;
    const bool on = lane < M;
    const double c00 = cov[lane], c01 = cov[32 + lane], c11 = cov[64 + lane];
    double2 yt[NB], ao[NB];
    double zeta[NB], prec[NB], dsum[NB], si[NB];
    size_t ri[NB];
    bool live[NB];
    AncEntry en[NB];
#pragma unroll
    for (int q = 0; q < NB; ++q) {
        const int l = l0 + q * stride;
        live[q] = l < ly.R;
        const bool act = on && live[q];
        ri[q] = (size_t)(live[q] ? l : 0) * M + (on ? lane : 0);
        yt[q] = act ? __ldcg(reinterpret_cast<const double2 *>(ly.ytil) + ri[q]) : make_double2(0.0, 0.0);
        zeta[q] = act ? __ldcg(ly.zeta + ri[q]) : 0.0;
        prec[q] = act ? __ldcg(ly.prec + ri[q]) : 1.0;
        ao[q] = act ? __ldcg(reinterpret_cast<const double2 *>(ly.A) + ri[q]) : make_double2(0.0, 0.0);
        dsum[q] = act ? __ldg(ly.d + ri[q]) : 0.0;
        si[q] = act ? __ldg(ly.sumPhi + ri[q]) : 0.0;
        en[q].len = -1;
        en[q].cm2_off = en[q].bv_off = en[q].d_off = 0;
        if (live[q] && lane < E) en[q] = ly.anc_tab[(size_t)l * E + lane];
    }
    // lane q < NB: constants and old noise / bias of region q for its update
    const int lq = l0 + lane * stride;
    const bool tail = lane < NB && lq < ly.R;
    double rc[7] = {1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0}, noise_old = 1.0, b0 = 0.0, b1 = 0.0;
    if (tail) {
#pragma unroll
        for (int k = 0; k < 7; ++k) rc[k] = __ldg(ly.rconst + (size_t)lq * 8 + k);
        noise_old = __ldcg(ly.noise_mean + lq);
        const double2 b = __ldcg(reinterpret_cast<const double2 *>(ly.bias_mean) + lq);
        b0 = b.x;
        b1 = b.y;
    }
    double2 an[NB];
    double cm2[NB];
#pragma unroll
    for (int q = 0; q < NB; ++q) s2_region(ly, ri[q], on && live[q], c00, c01, c11, yt[q], zeta[q], prec[q], ao[q], an[q], cm2[q]);
    // pieces: lane e holds piece e of the region (E <= 32 per pass); len * bias_var lane-parallel, cm2 . D by all lanes
    double t[NB];
#pragma unroll
    for (int q = 0; q < NB; ++q) t[q] = en[q].len >= 0 ? (double)en[q].len * __ldcg(m.sbase + en[q].bv_off) : 0.0;
    int e_pass = 0;      // the slots of a region are filled from the front: the longest list of the batch
#pragma unroll
    for (int q = 0; q < NB; ++q) e_pass = max(e_pass, __popc(__ballot_sync(kFull, en[q].len >= 0)));
    constexpr int UE = NB >= 4 ? 4 : (NB == 2 ? 8 : 16);   // 2 NB UE loads in flight per round trip
#pragma unroll UE
    for (int e = 0; e < e_pass; ++e) {
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            const unsigned oc = __shfl_sync(kFull, en[q].cm2_off, e), od = __shfl_sync(kFull, en[q].d_off, e);
            const int len = __shfl_sync(kFull, en[q].len, e);
            if (on && len >= 0) t[q] = fma(__ldcg(m.sbase + oc + lane), __ldg(m.sbase + od + lane), t[q]);
        }
    }
    for (int e0 = 32; e0 < E; e0 += 32) {     // more than 32 pieces per region (deep, non-nested index sets): further passes
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            AncEntry x;
            x.len = -1;
            x.cm2_off = x.bv_off = x.d_off = 0;
            if (live[q] && e0 + lane < E) x = ly.anc_tab[(size_t)(l0 + q * stride) * E + e0 + lane];
            t[q] += x.len >= 0 ? (double)x.len * __ldcg(m.sbase + x.bv_off) : 0.0;
            for (int e = 0; e < 32 && e0 + e < E; ++e) {
                const unsigned oc = __shfl_sync(kFull, x.cm2_off, e), od = __shfl_sync(kFull, x.d_off, e);
                const int len = __shfl_sync(kFull, x.len, e);
                if (on && len >= 0) t[q] = fma(__ldcg(m.sbase + oc + lane), __ldg(m.sbase + od + lane), t[q]);
            }
        }
    }
    // warp sums: [dA . s (2), d . cm2, f_var] per region, all in one lock-step butterfly
    double red[NB * 4];
    bool any = false;
#pragma unroll
    for (int q = 0; q < NB; ++q) {
        const double dA0 = ao[q].x - an[q].x, dA1 = ao[q].y - an[q].y;
        any = any || dA0 != 0.0 || dA1 != 0.0;
        red[q * 4 + 0] = si[q] * dA0;
        red[q * 4 + 1] = si[q] * dA1;
        red[q * 4 + 2] = dsum[q] * cm2[q];
        red[q * 4 + 3] = t[q];
    }
    wsum_n<NB * 4>(red);
    double quad[NB];
#pragma unroll
    for (int q = 0; q < NB; ++q) quad[q] = 0.0;
    if (__any_sync(kFull, any)) {      // dA^T G dA (zero in the inert regime of the published model: skipped)
        // column `lane` of G of each region, all 32 loads of a column in flight at once; those of region q + 1 are issued
        // before the FMA chain of region q, so the batch costs about one L2 round trip instead of one per region
        double g[2][32];
#pragma unroll
        for (int q = 0; q <= NB; ++q) {
            if (q < NB) {
                const double *G = ly.gram + (size_t)(live[q] ? l0 + q * stride : 0) * M * M;
#pragma unroll
                for (int k = 0; k < 32; ++k) g[q & 1][k] = (on && live[q] && k < M) ? __ldg(G + (size_t)k * M + lane) : 0.0;
            }
            if (q > 0) {
                const int p = q - 1;
                const double dA0 = ao[p].x - an[p].x, dA1 = ao[p].y - an[p].y;
                double t0 = 0.0, t1 = 0.0;
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    t0 = fma(g[p & 1][k], __shfl_sync(kFull, dA0, k), t0);
                    t1 = fma(g[p & 1][k], __shfl_sync(kFull, dA1, k), t1);
                }
                quad[p] = dA0 * t0 + dA1 * t1;
            }
        }
        wsum_n<NB>(quad);
    }
    double sums[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int q = 0; q < NB; ++q)
        if (lane == q) {
            const double n = rc[0], sd0 = red[q * 4 + 0], sd1 = red[q * 4 + 1];
            sums[0] = sd0 + n * b0;
            sums[1] = sd1 + n * b1;
            sums[2] = quad[q] + 2.0 * (b0 * sd0 + b1 * sd1) + n * (b0 * b0 + b1 * b1);
            sums[3] = red[q * 4 + 3];
            sums[4] = red[q * 4 + 2];
        }
    if (tail) bias_noise_update(ly, lq, true, sums, rc, noise_old, b0, b1);
}

// ---- the solver (one warp) ---------------------------------------------------------------------------------------
// The fixed point of omega_solve_serial (mrgp_math.cuh; tolerance kOmegaTol on the column sums, rows exact), reached by
// Anderson-accelerated Sinkhorn instead of Sinkhorn / Newton steps: on x = log v the Sinkhorn map is g(x) = -log(K^T u),
// u = 1 / (K e^x); with the residual f = g(x) - x (its mean removed: g(x + a) = g(x) + a) and the last three differences
// dX, dF of the iterates and residuals, the next iterate is x + f - sum_a gamma_a (dX_a + dF_a), gamma the least-squares
// solution of dF gamma = f (3 x 3 normal equations, columns scaled, ridge).  On the tables of the model this takes 2-15
// evaluations where Sinkhorn needs up to 160 and where a Newton step (Cholesky of the 30 x 30 dual Hessian by one warp)
// costs as much as 16 evaluations (profiles/r02_chain_cycles.md).  Warm start from the previous sweep's column
// scalings, history dropped when the residual grows, cold restart on a non-finite residual, plain Sinkhorn sweeps as the
// last resort.  MP rows / columns live in the registers of MP lanes; for M < MP the table is padded with an identity
// block (its scalings stay at 1 and do not couple to the model's block).
// One evaluation of the scaling iteration: u = 1 / (K v) (rows normalised exactly), s = K^T u, c = v s (column sums of
// P = diag(u) K diag(v)).  Lane i keeps BOTH row i (Kr) and column i (Kc) of the table in registers, v and u travel
// through two 32-entry arrays in shared memory (broadcast loads): no transposes and no shuffles inside the loop.
// Returns max |c - 1| (reduced in single precision: one REDUX instead of a five-step butterfly; it only steers the
// iteration) - NaN if any entry is NaN - and the column sums s (the Sinkhorn column step is v / c = 1 / s).
template <int MP>
__device__ __forceinline__ float omega_eval(const double (&Kr)[MP], const double (&Kc)[MP], double *sv, double *su, double v, double &u,
                                            double &c, double &v_sinkhorn, bool row, int lane) {
    sv[lane] = v;
    __syncwarp();
    double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;
    const double2 *pv = reinterpret_cast<const double2 *>(sv);
#pragma unroll
    for (int k = 0; k < MP; k += 2) {
        const double2 t = pv[k >> 1];
        if (k & 2) {
            r2 = fma(Kr[k], t.x, r2);
            r3 = fma(Kr[k + 1], t.y, r3);
        } else {
            r0 = fma(Kr[k], t.x, r0);
            r1 = fma(Kr[k + 1], t.y, r1);
        }
    }
    u = row ? rcp_fast((r0 + r1) + (r2 + r3)) : 0.0;
    su[lane] = u;
    __syncwarp();
    double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
    const double2 *pu = reinterpret_cast<const double2 *>(su);
#pragma unroll
    for (int i = 0; i < MP; i += 2) {
        const double2 t = pu[i >> 1];
        if (i & 2) {
            c2 = fma(Kc[i], t.x, c2);
            c3 = fma(Kc[i + 1], t.y, c3);
        } else {
            c0 = fma(Kc[i], t.x, c0);
            c1 = fma(Kc[i + 1], t.y, c1);
        }
    }
    const double s = (c0 + c1) + (c2 + c3);
    c = row ? v * s : 1.0;
    v_sinkhorn = row ? s : 1.0;                                 // (the column sum itself: the Sinkhorn step is v / c = 1 / s)
    const float e = row ? fabsf((float)(c - 1.0)) : 0.0f;      // NaN stays NaN; |.| >= 0: floats order like their bit patterns
    const unsigned bits = __reduce_max_sync(kFull, __float_as_uint(e));
    return __uint_as_float(bits);
}

template <int MP>
__device__ __noinline__ void omega_solve_warp(const ChainModel &m, ChainSmem &sm, int layer, int lane) {
    static_assert(MP <= 32 && (MP & 1) == 0, "one lane per row, columns in pairs");
    const int M = m.M, j = layer;
    if (lane == 0) PROF(6);
    const bool row = lane < MP, real = lane < M;
    double *sv = sm.sv, *su = sm.su;
    double Kr[MP], Kc[MP];
    // padding (M <= index < MP): an identity block, its scalings stay at 1 and do not couple to the model's block
    if (M == MP) {   // no padding (the headline M = 30): plain loads - the per-element selects of the general form cost 1.2 k cycles
#pragma unroll
        for (int k = 0; k < MP; ++k) Kr[k] = row ? sm.Kt[k * LD + lane] : 0.0;
        const double2 *col = reinterpret_cast<const double2 *>(sm.Kt + (row ? lane : 0) * LD);
#pragma unroll
        for (int i = 0; i < MP; i += 2) {
            const double2 t = col[i >> 1];
            Kc[i] = row ? t.x : 0.0;
            Kc[i + 1] = row ? t.y : 0.0;
        }
    } else {
#pragma unroll
        for (int k = 0; k < MP; ++k) Kr[k] = (real && k < M) ? sm.Kt[k * LD + lane] : ((row && !real && k == lane) ? 1.0 : 0.0);
        const double2 *col = reinterpret_cast<const double2 *>(sm.Kt + (real ? lane : 0) * LD);
#pragma unroll
        for (int i = 0; i < MP; i += 2) {
            const double2 t = col[i >> 1];
            Kc[i] = (real && i < M) ? t.x : ((row && !real && i == lane) ? 1.0 : 0.0);
            Kc[i + 1] = (real && i + 1 < M) ? t.y : ((row && !real && i + 1 == lane) ? 1.0 : 0.0);
        }
    }
    const double cshift = real ? sm.colmax[lane] : 0.0;
    const bool warm = sm.warm[layer] > 0.5;
    double x = 0.0;                                     // log v of this lane's column (0 on the padding)
    if (real) {
        const double eta = sm.eta[layer][lane] + cshift;
        x = (warm && isfinite(eta)) ? fmax(-600.0, fmin(600.0, eta)) : 0.0;
    }
    int iters = 0;
    double err_prev = INFINITY, c = 1.0, u = 0.0, vs = 1.0, v = 1.0;
    bool converged = false;
    const double dm = (double)M, inv_m = 1.0 / dm;
    // Anderson history, newest first: differences of the iterates / centred residuals (per lane) and their Gram matrix
    double xp = 0.0, fp = 0.0, dX0 = 0.0, dX1 = 0.0, dX2 = 0.0, dF0 = 0.0, dF1 = 0.0, dF2 = 0.0;
    double g00 = 0.0, g01 = 0.0, g02 = 0.0, g11 = 0.0, g12 = 0.0, g22 = 0.0, d1 = 0.0, d2 = 0.0;   // d: 1 / length of dF1, dF2
    int nh = 0;
    bool have_prev = false;
    if (lane == 0) PROF(7);
    for (int it = 0; it < kChainAndersonIters; ++it) {
        ++iters;
        v = real ? exp(x) : 1.0;
        const double err = (double)omega_eval<MP>(Kr, Kc, sv, su, v, u, c, vs, row, lane);
        if (err < kOmegaTol) {
            converged = true;
            break;
        }
        if (!isfinite(err)) {   // a bad (warm) start: start again from the shifts alone
            x = 0.0;
            nh = 0;
            have_prev = false;
            err_prev = INFINITY;
            continue;
        }
        const double fr = real ? -log(vs) - x : 0.0;      // g(x) - x = -log(K^T u) - x, not centred yet
        if (!(err <= err_prev)) {                         // the residual grew: drop the history, plain step from here
            nh = 0;
            have_prev = false;
        }
        double fc, b0 = 0.0, b1 = 0.0, b2 = 0.0;
        if (have_prev) {
            dX2 = dX1;
            dX1 = dX0;
            dF2 = dF1;
            dF1 = dF0;
            g22 = g11;
            g12 = g01;
            g11 = g00;
            const double w = real ? fr - fp : 0.0;        // newest residual difference before centring (sum fp = 0)
            dX0 = x - xp;
            double sums[7] = {w, w * w, w * dF1, w * dF2, fr * w, fr * dF1, fr * dF2};
            wsum_n<7>(sums);
            const double mu = sums[0] * inv_m, mm = dm * mu * mu;
            g00 = sums[1] - mm;
            g01 = sums[2];
            g02 = sums[3];
            b0 = sums[4] - mm;
            b1 = sums[5];
            b2 = sums[6];
            dF0 = real ? w - mu : 0.0;
            fc = real ? fr - mu : 0.0;
            nh = min(nh + 1, 3);
        } else {
            const double mu = wsum(fr) * inv_m;
            fc = real ? fr - mu : 0.0;
        }
        xp = x;
        fp = fc;
        have_prev = true;
        double xn = x + fc;                               // the Sinkhorn step (up to the scale of v)
        if (nh > 0 && g00 > 0.0) {
            // normal equations of the nh newest differences, columns scaled to unit length (the matrix holds the cosines
            // between the differences), ridge on the diagonal; 3 x 3 by Cramer's rule: one division, no chain of square
            // roots (gamma only steers the iteration - the fixed point is judged by the column sums)
            const bool h1 = nh > 1 && g11 > 0.0, h2 = nh > 2 && h1 && g22 > 0.0;
            const double d0 = rsqrt(g00);
            if (!h1) d1 = 0.0;
            if (!h2) d2 = 0.0;
            const double a01 = g01 * d0 * d1, a02 = g02 * d0 * d2, a12 = g12 * d1 * d2;
            const double r0 = b0 * d0, r1 = b1 * d1, r2 = b2 * d2;
            constexpr double kD = 1.0 + 1e-7;
            const double m00 = kD * kD - a12 * a12, m01 = a02 * a12 - kD * a01, m02 = a01 * a12 - kD * a02;
            const double m11 = kD * kD - a02 * a02, m12 = a01 * a02 - kD * a12, m22 = kD * kD - a01 * a01;
            const double det = kD * m00 + a01 * m01 + a02 * m02;
            if (det > 1e-12) {
                const double idet = rcp_fast(det);
                const double c0 = (m00 * r0 + m01 * r1 + m02 * r2) * idet * d0;     // gamma
                const double c1 = (m01 * r0 + m11 * r1 + m12 * r2) * idet * d1;
                const double c2 = (m02 * r0 + m12 * r1 + m22 * r2) * idet * d2;
                xn -= c0 * (dX0 + dF0) + c1 * (dX1 + dF1) + c2 * (dX2 + dF2);
            }
            d2 = d1;      // scalings of the differences, shifted with them
            d1 = d0;
        } else {
            d2 = d1;
            d1 = 0.0;
        }
        x = real ? fmax(-640.0, fmin(640.0, xn)) : 0.0;
        err_prev = err;
    }
    if (!converged) v = real ? exp(x) : 1.0;
    if (lane == 0) PROF(8);
    // last resort: plain Sinkhorn sweeps (see omega_solve_serial); on model tables the loop is not entered
    for (int it = 0; it < kOmegaFallbackSweeps && !converged; ++it) {
        const double err = (double)omega_eval<MP>(Kr, Kc, sv, su, v, u, c, vs, row, lane);
        if (err < kOmegaTol || !isfinite(err)) break;
        ++iters;
        if (real) v = fmax(1e-280, fmin(1e280, rcp_fast(vs)));
    }
    if (real) {   // omega = diag(u) K diag(v), kept transposed for the mixing step of the next layer
        const double2 *pv = reinterpret_cast<const double2 *>(sv);
        if (M == MP) {
            double2 tv[MP / 2];      // all column scalings first (the column registers are free now): the loads overlap
#pragma unroll
            for (int k = 0; k < MP / 2; ++k) tv[k] = pv[k];
#pragma unroll
            for (int k = 0; k < MP; k += 2) {
                sm.omT[k * LD + lane] = (Kr[k] * u) * tv[k >> 1].x;
                sm.omT[(k + 1) * LD + lane] = (Kr[k + 1] * u) * tv[k >> 1].y;
            }
        } else {
#pragma unroll
            for (int k = 0; k < MP; k += 2) {
                const double2 t = pv[k >> 1];
                if (k < M) sm.omT[k * LD + lane] = Kr[k] * u * t.x;
                if (k + 1 < M) sm.omT[(k + 1) * LD + lane] = Kr[k + 1] * u * t.y;
            }
        }
        sm.vout[layer][lane] = v;           // log(v) - column shift (next sweep's warm start): taken at the end of the kernel
        sm.cshift[layer][lane] = cshift;
    }
    if (lane == 0) {
        m.omegaIters[layer] = (double)iters;
        m.omegaWarm[layer] = 1.0;
        PROF(9);
    }
}

// One Bingham axis update for dy == 2 on the critical chain (same mathematics as bingham2 of mrgp_math.cuh, arranged
// for latency: division-free PD test, one rsqrt for the eigen-solve, the saddle point of
// computeRealBinghamConstant.py:42-147 in the closed form of its root for p = 2 with one logarithm:
//   Lam = (0.1, 0.1 + gap), gap = kappa_1 - kappa_2;  t = 0.1 - u,  u = (1 + 1 / (sqrt(1 + gap^2) + gap)) / 2;
//   log C = (log 2 pi - log(K2 u (u + gap))) / 2 + u + kappa_1,   K2 u (u + gap) = (q + 1 / q) / 2,  q = (u + gap) / u.
// The rare non-PD input takes the guard of bingham2 (SanityCheck.py:16-65).
__device__ __forceinline__ void bingham2_chain(double a, double b, double c, Bingham2 &out) {
    if (!(a > 0.0 && fma(a, c, -b * b) > 0.0)) {
        bingham2(a, b, c, out);
        return;
    }
    const double mid = 0.5 * (a + c), d = 0.5 * (a - c), qq = fma(d, d, b * b);
    double h = 0.0, p00 = 1.0, p01 = 0.0, p11 = 0.0;
    if (qq > 0.0) {
        const double rh = rsqrt(qq);
        h = qq * rh;
        const double ih = 0.5 * rh;
        p00 = fma(d, ih, 0.5);
        p11 = fma(-d, ih, 0.5);
        p01 = b * ih;
    }
    const double l1 = mid + h, l2 = mid - h, gap = l1 - l2;
    const double g1 = fma(gap, gap, 1.0);
    const double u = 0.5 * (1.0 + rcp_fast(g1 * rsqrt(g1) + gap));       // sqrt(1 + gap^2) as x rsqrt(x), x >= 1
    const double ug = u + gap;
    const double r0 = rcp_fast(u), r1 = rcp_fast(ug);
    const double k2 = 0.5 * (r0 * r0 + r1 * r1), k3 = r0 * r0 * r0 + r1 * r1 * r1;
    const double q = ug * r0;
    out.logc = 0.5 * (kLog2Pi - log(0.5 * (q + u * r1))) + u + l1;
    const double ik2 = rcp_fast(k2), dsumlogdt = -(r0 + r1);
    const double rr[2] = {r0, r1};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double dtdlam = 0.5 * rr[k] * rr[k] * ik2;
        const double dk2dlam = fma(k3, dtdlam, -(rr[k] * rr[k] * rr[k]));
        out.rho[k] = 0.5 * (dk2dlam * ik2) + 0.5 * fma(dsumlogdt, dtdlam, rr[k]) + dtdlam;
    }
    out.b[0] = a;
    out.b[1] = b;
    out.b[2] = c;
    out.kappa[0] = l1 < 0.0 ? 0.0 : l1;
    out.kappa[1] = l2 < 0.0 ? 0.0 : l2;
    out.cov[0] = out.rho[0] * p00 + out.rho[1] * (1.0 - p00);
    out.cov[1] = out.rho[0] * p01 - out.rho[1] * p01;
    out.cov[2] = out.rho[0] * p11 + out.rho[1] * (1.0 - p11);
    out.n_chol = 1;
}

// psi(x) as digamma() of mrgp_math.cuh with the recurrence below 10 summed as ONE fraction (a chain of multiplications
// and a single division instead of up to ten divisions in a row: the coarse layers have shapes of 0.5 .. 8).
__device__ __forceinline__ double digamma_chain(double x) {
    double num = 0.0, den = 1.0;
    while (x < 10.0) {
        num = fma(num, x, den);
        den *= x;
        x += 1.0;
    }
    const double inv = rcp_fast(x);
    const double i2 = inv * inv;
    const double series =
        i2 * (1.0 / 12.0 -
              i2 * (1.0 / 120.0 -
                    i2 * (1.0 / 252.0 - i2 * (1.0 / 240.0 - i2 * (1.0 / 132.0 - i2 * (691.0 / 32760.0 - i2 * (1.0 / 12.0)))))));
    return (log(x) - 0.5 * inv - series) - num * rcp_fast(den);
}

// ---- the shared step of a layer on CTA 0 (256 threads) ------------------------------------------------------------
__device__ __forceinline__ void shared_step(const ChainModel &m, ChainSmem &sm, int j, int tid, unsigned C) {
    const int M = m.M, lane = tid & 31, warp = __shfl_sync(kFull, tid >> 5, 0);   // (warp-uniform for the compiler)
    const ChainLayer &ly = m.layer[j];
    if (tid == 0) PROF(0);
    // region sums of the cluster, in rank order (all DSMEM loads of a thread in flight at once)
    if (tid < 7 * 32) {
        if (C >= 2) {    // the slots of the worker CTAs (local shared memory: they pushed), in rank order
            double s = 0.0;
            for (unsigned r = 1; r < C; ++r) s += sm.slots[r][tid];
            sm.data[tid] = s;
        } else {
            sm.data[tid] = sm.ctaPart[tid];
        }
    }
    // snapshot of the previous posterior: the pristine prior for layer 0, the posterior of layer j - 1 otherwise
    // (MRGP.py:575 / :581); its k-only terms of the table were prepared beside the previous solve BY THIS WARP (the
    // warps of CTA 0 other than the solver arrive here while the solve of layer j - 1 is still running: nothing that
    // the solver reads or writes may be touched before the barrier below)
    if (warp == 1 && lane < M) {
        const int t = lane;
        if (j == 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q) sm.primeB[t * 4 + q] = m.priorB[t * 4 + q];
            sm.primeLogC[t] = m.priorLogC[t];
            sm.primeShape[t] = m.priorShape[t];
            sm.primeScale[t] = m.priorScale[t];
            sm.sk[t] = m.priorSk[t];
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) sm.primeB[t * 4 + q] = sm.B[t * 4 + q];
            sm.primeLogC[t] = sm.logC[t];
            sm.primeShape[t] = sm.shape[t];
            sm.primeScale[t] = sm.scale[t];
            sm.sk[t] = sm.skNext[t];
        }
    }
    __syncthreads();
    if (tid == 0) PROF(1);
    if (warp == 0 && lane < M) {
        const int i = lane;
        // P2: B_i = sum_k omega_ik B'_k + sum_l 0.5 noise zeta y y^T (Posteriors.py:502-518); PD guard, eigen-solve,
        // saddle point (P2a-c), axis covariance (S1)
        double b00 = 0.0, b01 = 0.0, b11 = 0.0;
#pragma unroll 6
        for (int k = 0; k < M; ++k) {
            const double w = sm.omT[k * LD + i];
            b00 = fma(w, sm.primeB[k * 4 + 0], b00);
            b01 = fma(w, sm.primeB[k * 4 + 1], b01);
            b11 = fma(w, sm.primeB[k * 4 + 3], b11);
        }
        Bingham2 bg;
        bingham2_chain(b00 + sm.data[0 * 32 + i], b01 + sm.data[1 * 32 + i], b11 + sm.data[2 * 32 + i], bg);
        sm.cov[i * 4 + 0] = bg.cov[0];
        sm.cov[i * 4 + 1] = bg.cov[1];
        sm.cov[i * 4 + 2] = bg.cov[1];
        sm.cov[i * 4 + 3] = bg.cov[2];
        sm.pub[i] = bg.cov[0];
        sm.pub[32 + i] = bg.cov[1];
        sm.pub[64 + i] = bg.cov[2];
        sm.B[i * 4 + 0] = bg.b[0];
        sm.B[i * 4 + 1] = bg.b[1];
        sm.B[i * 4 + 2] = bg.b[1];
        sm.B[i * 4 + 3] = bg.b[2];
        sm.kappa[i * 2 + 0] = bg.kappa[0];
        sm.kappa[i * 2 + 1] = bg.kappa[1];
        sm.rho[i * 2 + 0] = bg.rho[0];
        sm.rho[i * 2 + 1] = bg.rho[1];
        sm.logC[i] = bg.logc;
        atomicAdd(&sm.nchol, bg.n_chol);
    } else if (warp == 1 && lane < M) {
        // P3 beside it (Posteriors.py:533-541): the mixed prior shape / scale and psi(shape) do not depend on the axis update
        const int i = lane;
        double sh = 0.0, sc = 0.0;
#pragma unroll 6
        for (int k = 0; k < M; ++k) {
            const double w = sm.omT[k * LD + i];
            sh = fma(w, sm.primeShape[k], sh);
            sc = fma(w, sm.primeScale[k], sc);
        }
        const double shape = sh + 0.5 * (double)ly.R;
        sm.sh[i] = shape;
        sm.sc[i] = sc;
        sm.dg[i] = digamma_chain(shape);
    }
    __syncthreads();
    if (tid == 0) PROF(2);
    if (tid < M) {
        // S3 (Stats.py:385-388): sum_l m2/S = sum_l 1/(prec S) + tr((sum_l zeta^2 y y^T / S) C_i)
        const int i = tid;
        const double beta2 = sm.data[3 * 32 + i] +
                             (sm.data[4 * 32 + i] * sm.cov[i * 4 + 0] + 2.0 * sm.data[5 * 32 + i] * sm.cov[i * 4 + 1] + sm.data[6 * 32 + i] * sm.cov[i * 4 + 3]);
        const double shape = sm.sh[i];
        const double scale = sm.sc[i] + 0.5 * beta2;
        const double mean = shape * rcp_fast(scale), lmean = sm.dg[i] - log(scale);
        sm.shape[i] = shape;
        sm.scale[i] = scale;
        sm.mean[i] = mean;
        sm.lmean[i] = lmean;
        sm.pub[96 + i] = mean;
    }
    __syncthreads();
    if (tid == 0) PROF(3);
    // S4, the table (Stats.py:405-412; a true matrix product inside the trace): a warp per row, the row maxima on the
    // way; the (at most 4) rows of a warp are independent instruction streams
    const bool last_layer = j == m.J - 1;
    {
        double lwv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = warp + u * 8;
            lwv[u] = -INFINITY;
            if (i < M && lane < M) {
                const int k = lane;
                const double *Cc = sm.cov + i * 4, *Bp = sm.primeB + k * 4;
                const double tr = Cc[0] * Bp[0] + Cc[1] * Bp[2] + Cc[2] * Bp[1] + Cc[3] * Bp[3];
                lwv[u] = tr + sm.sk[k] + (sm.primeShape[k] - 1.0) * sm.lmean[i] - sm.primeScale[k] * sm.mean[i];
                sm.lw[i * LW + k] = lwv[u];
                if (last_layer) m.logOmegaHat[i * M + k] = lwv[u];
                if (m.tables) m.tables[((size_t)j * M + i) * M + k] = lwv[u];
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) lwv[u] = wmax_shift(lwv[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (lane == 0 && warp + u * 8 < M) sm.rowmax[warp + u * 8] = lwv[u];
    }
    __syncthreads();
    if (tid == 0) PROF(4);
    // shifts and exponentials, a warp per column: every row and column of K holds a 1 (no overflow, no empty line)
    {
        double v[4], mx[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = warp + u * 8;
            v[u] = (k < M && lane < M) ? sm.lw[lane * LW + k] - sm.rowmax[lane] : -INFINITY;
            mx[u] = v[u];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) mx[u] = wmax_shift(mx[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = warp + u * 8;
            if (k < M && lane < M) sm.Kt[k * LD + lane] = exp(v[u] - mx[u]);
            if (k < M && lane == 0) sm.colmax[k] = mx[u];
        }
    }
    if (tid == 0) PROF(5);
}

// Worker steps of one warp for a whole layer: regions ww, ww + n_workers, ..., a batch at a time (the order in which
// a warp adds its regions into acc does not depend on the batch size).
// (Inlined at their three call sites: as separate functions they cost 4 % - the calls spill around the 255-register solver.)
__device__ __forceinline__ void layer_mid1(const ChainModel &m, int j, int ww, int n_workers, int lane, const double *ardMean, double (&acc)[7]) {
    const ChainLayer &ly = m.layer[j];
    if (j == 0) {
        for (int l = ww; l < ly.R; l += n_workers) mid1_layer0(m, ly, l, lane, ardMean, acc);
    } else {
        for (int l = ww; l < ly.R; l += kMid1Batch * n_workers) mid1_upper<kMid1Batch>(m, ly, l, n_workers, lane, ardMean, acc);
    }
}

__device__ __forceinline__ void layer_finish(const ChainModel &m, int j, int ww, int n_workers, int lane, const double *cov) {
    const ChainLayer &ly = m.layer[j];
    if (j == 0) {
        for (int l = ww; l < ly.R; l += n_workers) mid2_stats_layer0(m, ly, l, lane, cov);
    } else {
        for (int l = ww; l < ly.R; l += kFinishBatch * n_workers) mid2_stats_upper<kFinishBatch>(m, ly, l, n_workers, lane, cov);
    }
}

// Region sums of a worker CTA for the shared step: the warps' partial sums (registers) are added in warp order; a
// cluster of several CTAs pushes the result into this CTA's slot of CTA 0 (counted on its barA).
__device__ __forceinline__ void publish_sums(ChainSmem &sm, const double (&acc)[7], bool early, unsigned rank, int warp, int lane, int w0, int wt,
                                             int wthreads) {
#pragma unroll
    for (int q = 0; q < 7; ++q) sm.part[warp][q][lane] = acc[q];
    worker_bar(wthreads);
    const uint32_t slot = early ? remote_addr(smem_addr(&sm.slots[rank][0]), 0) : 0u;
    const uint32_t bar = early ? remote_addr(smem_addr(&sm.barA), 0) : 0u;
    for (int v = wt; v < 7 * 32; v += wthreads) {
        double s = 0.0;
        for (int w = w0; w < 8; ++w) s += sm.part[w][v >> 5][v & 31];
        if (early)
            st_async_remote(slot + (uint32_t)v * 8u, s, bar);
        else
            sm.ctaPart[v] = s;
    }
}

// Cluster of C CTAs per model.  C >= 2: CTA 0 runs the shared step and the solver, the warps of CTAs 1 .. C-1 are the
// workers and finish layer j (S2, P4 / P5) in the BACKGROUND: they arrive at the cluster barrier as soon as the region
// sums of layer j + 1 are published and do that work before they wait, so the chain on CTA 0 never waits for it.
// C == 1 (a batch of small models, one CTA each): warp 0 solves while warps 1-7 do the worker steps of the layer.
template <int MP>
__global__ void __launch_bounds__(kChainThreads, 1) k_ci_sweep(const ChainModel *const *models) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ChainSmem &sm = *reinterpret_cast<ChainSmem *>(smem_raw);
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned C = cluster.num_blocks(), rank = cluster.block_rank();
    // the warp index as a broadcast: the compiler then knows that every branch on it is warp-uniform and emits plain
    // shuffles inside the solver / worker roles (otherwise each one is bracketed by a WARPSYNC and serialised)
    const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(kFull, tid >> 5, 0);
    const long long t_begin = clock64();
    if (C >= 2) {    // the hand-off barriers; their initialisation is cluster-visible after the (one) cluster barrier of the prologue
        if (tid == 0) {
            bar_init(&sm.barA, 1u);              // armed by this CTA per layer; counts the bytes of the pushed region sums
            bar_init(&sm.barB, 1u);              // likewise, the bytes of the pushed covariances / ARD means
            bar_init(&sm.barF, C - 1u);          // every worker CTA, once its share of a layer is finished
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            if (rank == 0)
                bar_expect(&sm.barA, (C - 1u) * kSumBytes);
            else
                bar_expect(&sm.barB, kPubBytes);
        }
        cl_arrive();
    }
    {
        const ChainModel *gm = models[blockIdx.x / C];
        const int J0 = gm->J;
        const size_t bytes = offsetof(ChainModel, layer) + (size_t)J0 * sizeof(ChainLayer);   // multiples of 8
        const unsigned long long *src = reinterpret_cast<const unsigned long long *>(gm);
        unsigned long long *dst = reinterpret_cast<unsigned long long *>(sm.model);
        for (size_t t = tid; t < bytes / 8; t += kChainThreads) dst[t] = src[t];
    }
    __syncthreads();
    const ChainModel &m = *reinterpret_cast<const ChainModel *>(sm.model);
    const int M = m.M, J = m.J;
    const bool early = C >= 2;
    const bool solver = rank == 0 && warp == 0;
    const bool worker = early ? rank > 0 : warp > 0;
    const int n_workers = early ? ((int)C - 1) * 8 : 7;                   // worker warps of the cluster
    const int ww = early ? ((int)rank - 1) * 8 + warp : warp - 1;         // this warp's worker index
    const int w0 = early ? 0 : 1;                                         // first worker warp of a CTA
    const int wthreads = early ? kChainThreads : kChainThreads - 32;      // worker threads of a CTA
    const int wt = tid - w0 * 32;
    unsigned long long *ts = m.ts;
    if (ts && rank == 0 && tid == 0) atomicMin(&ts[(0 * 4 + 1) * 2], gtimer());

    // ---- prologue: the small-matrix state into L2 (the sweep is a chain of dependent loads), omega (transposed) and the
    //      warm starts on CTA 0, the ARD mean of the previous sweep everywhere ---------------------------------------
    if (C >= 4 && rank >= 2) {   // CTAs that are neither on the chain (0) nor own layer 0's region (1) pull the state into L2
        const unsigned long long lines = m.pf_lines, nthr = (unsigned long long)(C - 2) * kChainThreads;
        const unsigned long long first = (unsigned long long)(rank - 2) * kChainThreads + tid;
        for (unsigned long long l = first; l < lines; l += nthr) asm volatile("prefetch.global.L2 [%0];" ::"l"(m.pf_base + l * 128));
    }
    if (rank == 0) {
        for (int t = tid; t < M * M; t += kChainThreads) {
            const int i = t / M, k = t - i * M;
            sm.omT[k * LD + i] = m.omega[t];
        }
        if (tid == 0) sm.nchol = 0;
        for (int t = tid; t < J * 32; t += kChainThreads) sm.eta[t >> 5][t & 31] = m.omegaEta[(t >> 5) * 64 + (t & 31)];
        if (tid < J) sm.warm[tid] = m.omegaWarm[tid];
    }
    if (tid < 4 * 32) {   // lanes past M must hold finite values (they are multiplied by zeros)
        const double am = (tid >= 96 && tid - 96 < M) ? m.ardMean[tid - 96] : (tid >= 96 ? 1.0 : 0.0);
        sm.pub[tid] = 0.0;
        sm.loc[0][tid] = am;
        sm.loc[1][tid] = am;
    }
    if (tid < 7 * 32) sm.ctaPart[tid] = 0.0;
    __syncthreads();
    if (early) cl_wait();
    double acc[7];
#pragma unroll
    for (int q = 0; q < 7; ++q) acc[q] = 0.0;
    if (worker) {
        layer_mid1(m, 0, ww, n_workers, lane, sm.loc[0] + 96, acc);
        publish_sums(sm, acc, early, rank, warp, lane, w0, wt, wthreads);
    }

    if (m.prof && J >= 4 && rank == 0 && tid == 0) {   // whole-kernel stamps of CTA 0 in slot 15 of rows 0 .. 3 (needs J >= 4)
        m.prof[0 * 16 + 15] = (double)t_begin;
        m.prof[1 * 16 + 15] = (double)clock64();
    }
    // Iteration j = J only finishes the last layer (the one call site of layer_finish: the sweep's code is mostly the
    // unrolled worker steps and has to stay in the instruction caches).
    for (int j = 0; j <= J; ++j) {
        if (j == J && m.prof && J >= 4 && rank == 0 && tid == 0) m.prof[2 * 16 + 15] = (double)clock64();
        if (!early) cl_arrive();                           // A_j: this thread's share of the region sums of layer j is published
        if (worker && j > 0) {   // S2 and P4 / P5 of layer j - 1 in the background of the chain (C >= 2) / of the solve (C == 1)
            const long long tf = clock64();
            if (early && j > 1) bar_wait(&sm.barF, (unsigned)(j - 2) & 1u);   // F(j - 2): the moments of the coarser layers are complete
            if (ts && lane == 0) atomicMin(&ts[((j - 1) * 4 + 0) * 2], gtimer());
            layer_finish(m, j - 1, ww, n_workers, lane, sm.loc[(j - 1) & 1]);
            if (ts && lane == 0) atomicMax(&ts[((j - 1) * 4 + 0) * 2 + 1], gtimer());
            if (early && j < J) {                                             // F(j - 1) to every worker CTA
                worker_bar(wthreads);
                if (warp == 0 && lane + 1 < (int)C) bar_arrive_remote(remote_addr(smem_addr(&sm.barF), lane + 1));
            }
            if (m.prof && j > 4 && ww == 0 && lane == 0) m.prof[(j - 1) * 16 + 15] = (double)(clock64() - tf);   // rows >= 4: its cycles
        }
        if (!early) cl_wait();
        if (j == J) break;
        if (rank == 0) {
            if (early) {                                                     // A(j): the region sums of every worker CTA are in `slots`
                bar_wait_tx(&sm.barA, (unsigned)j & 1u);
                if (tid == 0 && j + 1 < J) bar_expect(&sm.barA, (C - 1u) * kSumBytes);   // (phase j + 1 cannot complete before B(j) is out)
            }
            if (ts && tid == 0) atomicMin(&ts[(j * 4 + 3) * 2], gtimer());
            shared_step(m, sm, j, tid, C);
        }
        if (!early) {
            cl_arrive();                                   // B_j: axis covariance, ARD moments and the table of layer j
            cl_wait();
        } else if (rank == 0) {
            __syncthreads();                               // the table of layer j is complete (the solver reads all of it)
            if (warp >= 4) {   // B(j): warps 4-7 push the 4 x 32 values to every worker CTA while warp 0 starts the solve
                const int t = tid - 128;
                const double v = sm.pub[t];
                const uint32_t dst = smem_addr(&sm.loc[j & 1][t]), bar = smem_addr(&sm.barB);
                for (unsigned r = 1; r < C; ++r) st_async_remote(remote_addr(dst, r), v, remote_addr(bar, r));
            }
        }
        if (solver) {
            omega_solve_warp<MP>(m, sm, j, lane);
            if (ts && lane == 0) atomicMax(&ts[(j * 4 + 3) * 2 + 1], gtimer());
        }
        // k-only terms of the NEXT layer's table from the posterior of this layer (one lgamma per basis function), beside the solve
        if (rank == 0 && warp == 1 && lane < M) sm.skNext[lane] = -sm.logC[lane] + sm.shape[lane] * log(sm.scale[lane]) - lgamma(sm.shape[lane]);
        if (worker) {
            const bool stamp = ww == 0 && lane == 0;
            if (stamp) PROF(10);
            double *loc = sm.loc[j & 1];
            if (early) {
                bar_wait_tx(&sm.barB, (unsigned)j & 1u);   // B(j): CTA 0 has pushed the layer's covariances / ARD means into loc
                if (tid == 0 && j + 1 < J) bar_expect(&sm.barB, kPubBytes);
            } else {
                for (int v = wt; v < 4 * 32; v += wthreads) loc[v] = sm.pub[v];
                worker_bar(wthreads);
            }
            if (stamp) PROF(11);
            if (ts && lane == 0) atomicMin(&ts[(j * 4 + 1) * 2], gtimer());
#pragma unroll
            for (int q = 0; q < 7; ++q) acc[q] = 0.0;
            if (j + 1 < J) {
                layer_mid1(m, j + 1, ww, n_workers, lane, loc + 96, acc);
                if (stamp) PROF(12);
                publish_sums(sm, acc, early, rank, warp, lane, w0, wt, wthreads);
            }
            if (stamp) PROF(13);
            if (ts && lane == 0) atomicMax(&ts[(j * 4 + 1) * 2 + 1], gtimer());
            if (stamp) PROF(14);
        }
    }
    if (m.prof && J >= 4 && rank == 0 && tid == 0) m.prof[3 * 16 + 15] = (double)clock64();
    // ---- the shared posterior / stats left by the last layer (Posteriors.py:482-541, Stats.py:354-420) ----------
    if (rank == 0) {
        __syncthreads();   // the last solve (warp 0) is complete
        for (int t = tid; t < M * M; t += kChainThreads) {
            const int i = t / M, k = t - i * M;
            m.omega[t] = sm.omT[k * LD + i];
        }
        for (int t = tid; t < M * 4; t += kChainThreads) {
            m.axB[t] = sm.B[t];
            m.axCov[t] = sm.cov[t];
        }
        for (int t = tid; t < M * 2; t += kChainThreads) {
            m.axKappa[t] = sm.kappa[t];
            m.axRho[t] = sm.rho[t];
        }
        for (int t = tid; t < M; t += kChainThreads) {
            m.axLogC[t] = sm.logC[t];
            m.ardShape[t] = sm.shape[t];
            m.ardScale[t] = sm.scale[t];
            m.ardMean[t] = sm.mean[t];
            m.ardLogMean[t] = sm.lmean[t];
        }
        for (int t = tid; t < J * 32; t += kChainThreads)
            if ((t & 31) < M) m.omegaEta[(t >> 5) * 64 + (t & 31)] = log(sm.vout[t >> 5][t & 31]) - sm.cshift[t >> 5][t & 31];
        if (tid == 0) atomicAdd(m.chol_count, (unsigned long long)sm.nchol);
        if (ts && tid == 0) atomicMax(&ts[((J - 1) * 4 + 1) * 2 + 1], gtimer());
    }
    // timeline, slots kind 2 of layers 0 and 1: the exits of the warps of CTA 0 and of every warp of the cluster (the
    // workers' finish of the last layers runs after the chain)
    if (ts && lane == 0) {
        const unsigned long long t = gtimer();
        if (rank == 0) {
            atomicMin(&ts[(0 * 4 + 2) * 2], t);
            atomicMax(&ts[(0 * 4 + 2) * 2 + 1], t);
        }
        atomicMin(&ts[(1 * 4 + 2) * 2], t);
        atomicMax(&ts[(1 * 4 + 2) * 2 + 1], t);
    }
}

// Sufficient statistics of y for layer 0, one CTA per (model, region): c[i][d] = sum_n phi_i y_d, sum y_d, sum |y|^2
// in a fixed order (thread-strided samples, shuffles inside the warps, warps in order).
template <int MP>
__global__ void __launch_bounds__(256) k_ystats_small(const ChainModel *const *models, int r0_max) {
    constexpr int NV = MP * 2 + 3;
    __shared__ double red[8][NV];
    const ChainModel &m = *models[blockIdx.x / r0_max];
    const int r = blockIdx.x % r0_max;
    const ChainLayer &ly = m.layer[0];
    if (r >= ly.R) return;
    const int M = m.M, tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(kFull, tid >> 5, 0);
    const int64_t lo = ly.offsets[r], hi = ly.offsets[r + 1];
    const double inv2L = ly.inv2L[r], rs = ly.rsqrtL[r];
    double T[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) T[i] = 0.0;
    for (int64_t n = lo + tid; n < hi; n += 256) {
        const double y0 = m.y[n * 2], y1 = m.y[n * 2 + 1];
        double f, c2;
        basis_seed(m.x[n], inv2L, rs, f, c2);
        double fm = 0.0;
        T[MP * 2] += y0;
        T[MP * 2 + 1] += y1;
        T[MP * 2 + 2] += fma(y1, y1, y0 * y0);
#pragma unroll
        for (int i = 0; i < MP; ++i) {
            T[i * 2] = fma(f, y0, T[i * 2]);
            T[i * 2 + 1] = fma(f, y1, T[i * 2 + 1]);
            const double fn = fma(c2, f, -fm);
            fm = f;
            f = fn;
        }
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const double t = wsum(T[i]);
        if (lane == 0) red[warp][i] = t;
    }
    __syncthreads();
    for (int v = tid; v < NV; v += 256) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w][v];
        if (v < M * 2)
            ly.yc[(size_t)r * M * 2 + v] = t;
        else if (v >= MP * 2)
            ly.ysum[(size_t)r * 4 + (v - MP * 2)] = t;
    }
}

// Streamed fallback for layer 0 of the fused sweep, one CTA per (model, region): runs only for models whose guard
// tripped (ChainModel::status, see kChainGuard): the P4 / P5 statistics of the region by a pass over its samples with
// the NEW coefficients (r = y - Phi A^T; Posteriors.py:81-148) and the bias / noise update again from those sums.
template <int MP>
__global__ void __launch_bounds__(256) k_l0_fix_small(const ChainModel *const *models, int r0_max) {
    __shared__ double red[8][4];
    __shared__ double sA[MP * 2], sC[MP];
    const ChainModel &m = *models[blockIdx.x / r0_max];
    if (m.status[0] == 0u) return;
    const int r = blockIdx.x % r0_max;
    const ChainLayer &ly = m.layer[0];
    if (r >= ly.R) return;
    const int M = m.M, tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(kFull, tid >> 5, 0);
    for (int t = tid; t < MP * 2; t += 256) sA[t] = t < M * 2 ? ly.A[(size_t)r * M * 2 + t] : 0.0;
    for (int t = tid; t < MP; t += 256) sC[t] = t < M ? ly.cm2[(size_t)r * M + t] : 0.0;
    __syncthreads();
    const int64_t lo = ly.offsets[r], hi = ly.offsets[r + 1];
    const double inv2L = ly.inv2L[r], rs = ly.rsqrtL[r];
    double acc[4] = {0.0, 0.0, 0.0, 0.0};      // sum r_0, sum r_1, sum |r|^2, sum phi^2 cm2
    for (int64_t n = lo + tid; n < hi; n += 256) {
        double f, c2, fm = 0.0, e0 = 0.0, e1 = 0.0, v = 0.0;
        basis_seed(m.x[n], inv2L, rs, f, c2);
#pragma unroll 6
        for (int i = 0; i < MP; ++i) {
            e0 = fma(f, sA[i * 2], e0);
            e1 = fma(f, sA[i * 2 + 1], e1);
            v = fma(f * sC[i], f, v);
            const double fn = fma(c2, f, -fm);
            fm = f;
            f = fn;
        }
        const double r0 = m.y[n * 2] - e0, r1 = m.y[n * 2 + 1] - e1;
        acc[0] += r0;
        acc[1] += r1;
        acc[2] += fma(r1, r1, r0 * r0);
        acc[3] += v;
    }
    wsum_n<4>(acc);
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < 4; ++k) red[warp][k] = acc[k];
    __syncthreads();
    if (tid == 0) {
        double sums[5] = {0.0, 0.0, 0.0, 0.0, 0.0}, rc[7];
        for (int w = 0; w < 8; ++w) {
            sums[0] += red[w][0];
            sums[1] += red[w][1];
            sums[2] += red[w][2];
            sums[4] += red[w][3];
        }
        for (int k = 0; k < 7; ++k) rc[k] = ly.rconst[(size_t)r * 8 + k];
        bias_noise_update(ly, r, false, sums, rc, 1.0, ly.bias_prev[(size_t)r * 2], ly.bias_prev[(size_t)r * 2 + 1]);
    }
}

template <int MP>
int launch_l0_fix_impl(const ChainModel *const *models_dev, int n_models, int r0_max, cudaStream_t stream) {
    k_l0_fix_small<MP><<<(unsigned)(n_models * r0_max), 256, 0, stream>>>(models_dev, r0_max);
    return (int)cudaGetLastError();
}

template <int MP>
int launch_ystats_impl(const ChainModel *const *models_dev, int n_models, int r0_max, cudaStream_t stream) {
    k_ystats_small<MP><<<(unsigned)(n_models * r0_max), 256, 0, stream>>>(models_dev, r0_max);
    return (int)cudaGetLastError();
}

template <int MP>
int launch_impl(const ChainModel *const *models_dev, int n_models, int cluster, cudaStream_t stream) {
    static bool configured = false;
    const size_t smem = sizeof(ChainSmem);
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(k_ci_sweep<MP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        e = cudaFuncSetAttribute(k_ci_sweep<MP>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return (int)e;
        e = cudaFuncSetAttribute(k_ci_sweep<MP>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return (int)e;
        configured = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(n_models * cluster));
    cfg.blockDim = dim3(kChainThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return (int)cudaLaunchKernelEx(&cfg, k_ci_sweep<MP>, models_dev);
}

}  // namespace

size_t ci_sweep_smem_bytes(int) { return sizeof(ChainSmem); }

int launch_ystats_small(int solver_size, const ChainModel *const *models_dev, int n_models, int r0_max, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n_models < 1 || r0_max < 1) return (int)cudaErrorInvalidValue;
    switch (solver_size) {
        case 8: return launch_ystats_impl<8>(models_dev, n_models, r0_max, st);
        case 16: return launch_ystats_impl<16>(models_dev, n_models, r0_max, st);
        case 24: return launch_ystats_impl<24>(models_dev, n_models, r0_max, st);
        case 30: return launch_ystats_impl<30>(models_dev, n_models, r0_max, st);
        case 32: return launch_ystats_impl<32>(models_dev, n_models, r0_max, st);
        default: return (int)cudaErrorInvalidValue;
    }
}

int launch_l0_fix_small(int solver_size, const ChainModel *const *models_dev, int n_models, int r0_max, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n_models < 1 || r0_max < 1) return (int)cudaErrorInvalidValue;
    switch (solver_size) {
        case 8: return launch_l0_fix_impl<8>(models_dev, n_models, r0_max, st);
        case 16: return launch_l0_fix_impl<16>(models_dev, n_models, r0_max, st);
        case 24: return launch_l0_fix_impl<24>(models_dev, n_models, r0_max, st);
        case 30: return launch_l0_fix_impl<30>(models_dev, n_models, r0_max, st);
        case 32: return launch_l0_fix_impl<32>(models_dev, n_models, r0_max, st);
        default: return (int)cudaErrorInvalidValue;
    }
}

int launch_ci_sweep(int solver_size, const ChainModel *const *models_dev, int n_models, int cluster, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (cluster < 1 || cluster > kChainMaxCluster || (cluster & (cluster - 1))) return (int)cudaErrorInvalidValue;
    switch (solver_size) {
        case 8: return launch_impl<8>(models_dev, n_models, cluster, st);
        case 16: return launch_impl<16>(models_dev, n_models, cluster, st);
        case 24: return launch_impl<24>(models_dev, n_models, cluster, st);
        case 30: return launch_impl<30>(models_dev, n_models, cluster, st);
        case 32: return launch_impl<32>(models_dev, n_models, cluster, st);
        default: return (int)cudaErrorInvalidValue;
    }
}

}  // namespace mrgp
