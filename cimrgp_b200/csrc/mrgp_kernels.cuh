// Device kernels of the ciMRGP / fiMRGP sweep for sm_100a.
//
// Layout of the streaming kernels (phase A, phase B, basis build): the sample axis [0, N) is cut into
// one contiguous range per persistent CTA; each range is cut further at the region boundaries of the
// layer and of its parent layer into SEGMENTS (host-built table).  Inside a segment all 256 threads
// stride over the samples (coalesced 8/16-byte loads per lane, one sample ahead prefetched), the basis
// functions of a sample are produced by the three-term sine recurrence from one sincospi, and per-thread
// FP64 register accumulators hold the region statistics.  At the end of a RUN (last segment of a region
// inside the CTA range) the block reduces the accumulators through shared memory in a fixed order and
// writes one partial per run: no atomics, results are reproducible for a given launch geometry.
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "mrgp_math.cuh"
#include "mrgp_tma.cuh"

namespace mrgp {

// Debug timeline: when `ts` is non-null every kernel of the sweep stamps the global timer at the entry of its
// first-scheduled CTA (min) and at the exit of every CTA (max) into slot (layer * 4 + kind).
__device__ __forceinline__ unsigned long long global_timer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void ts_begin(unsigned long long *ts, int slot) {
    if (ts && threadIdx.x == 0) atomicMin(&ts[slot * 2], global_timer());
}
__device__ __forceinline__ void ts_end(unsigned long long *ts, int slot) {
    if (ts && threadIdx.x == 0) atomicMax(&ts[slot * 2 + 1], global_timer());
}

constexpr int kMaxLayersTs = 12;    // timeline: 4 kernel slots per layer, then 4 debug slots per layer
__device__ __forceinline__ void ts_dbg(unsigned long long *ts, int layer, int k, bool end) {
    if (layer >= kMaxLayersTs) return;
    if (end)
        ts_end(ts, kMaxLayersTs * 4 + layer * 4 + k);
    else
        ts_begin(ts, kMaxLayersTs * 4 + layer * 4 + k);
}
constexpr int kThreads = 256;      // streaming CTA size (8 warps)
constexpr int kPartBStride = 8;    // doubles per phase-B partial (dy + 3 <= 8)
constexpr int kRedSmemDoubles = (kThreads / 32) * 128;   // block_reduce_store: one row of (padded) sums per warp

struct Segment {
    int64_t start;
    int32_t len;
    int32_t region;
    int32_t parent;
    int32_t run;
    int32_t flush;   // 1: last segment of its run
    int32_t pad;
};

// Arguments of the streaming kernels for one layer.
struct StreamArgs {
    const Segment *segs;
    const int32_t *cta_seg;      // (n_ctas + 1) first segment of each CTA
    const double *x;             // (N)
    const double *y;             // (N, DY)
    double *g;                   // (N, DY) latent mean of the layer minus the parent's bias (in place)
    double *h;                   // (N)     latent variance minus the parent's bias variance (in place)
    const double *inv2L;         // (R)
    const double *rsqrtL;        // (R)
    const double *A;             // (R, M, DY) current coefficients
    const double *A_prev;        // (R, M, DY) coefficients before this layer's update (phase B, inferred)
    const double *cm2;           // (R, M)
    const double *bias;          // (R, DY) current (old) bias of the layer
    const double *pbias;         // (Rp, DY) parent-layer bias (new)
    const double *pbias_var;     // (Rp)
    double *part;                // partial sums per run
    int32_t part_stride;
    int64_t sample_begin;        // first sample of this handle's chunk (0 unless sharded over GPUs)
    int64_t n_samples;           // end of the chunk (exclusive)
    int64_t cta_quantum;         // samples per CTA range (multiple of 32)
    // bias / noise update fused into the tail of phase B (run by the last CTA to finish)
    unsigned int *done_counter;
    const int32_t *region_run;   // (R + 1)
    const int64_t *offsets;      // (R + 1)
    int32_t R, infer, fuse_tail, layer;
    const unsigned int *gate;    // phase B only: when non-null the kernel runs only if *gate != 0 (streamed fallback of the fused sweep)
    int32_t n_basis;             // basis functions of the model; the kernels are instantiated for a padded M >= n_basis and
                                 // treat the extra functions as zero-weight (their sums are never read)
    unsigned long long *ts;
    const double *bias_prec0, *bias_mean0, *noise_shape0, *noise_scale0;
    int32_t sums_only;               // bias_noise_*: only store the per-region sums in sumsB
    int32_t noise_rs, bias_rs, ci;   // noise / bias region specific (MRGP.py:27-28); ci or fi (Posteriors.py:113-211 vs 377-475)
    double *bias_mean_out, *bias_prev_out, *bias_prec, *bias_var, *noise_shape, *noise_scale, *noise_mean, *noise_log_mean, *yvar, *sumsB;
    double *yc_out, *ysum_out;       // k_ystats with fuse_tail: the last CTA to finish sums the run partials into the region statistics
};

// ------------------------------------------------------------------------------------------------
// block reductions
// ------------------------------------------------------------------------------------------------

// Sum NV per-thread values over the 256 threads of the block, fixed order.  Inside a warp a halving butterfly: at every
// level a lane sends one half of its values to its partner and adds the partner's other half, so NP values cost NP - NP/32
// exchanges (not 5 NP) and lane l ends with the warp's sums of values l NP/32 .. ; the 8 warps then meet in shared memory
// (red: 8 x NP doubles) and are added in warp order.  (Round 1 staged all values through 66 KB of shared memory with three
// block barriers per 32 values: a quarter of the time of k_ystats and more on layers with several regions per CTA.)

template <int NV, bool NAMED = false>
__device__ __forceinline__ void block_reduce_store(double (&v)[NV], double *red, double *out) {
    static_assert(NV <= 128, "block_reduce_store: at most 128 values");
    constexpr int NP = NV <= 32 ? 32 : (NV <= 64 ? 64 : 128), PER = NP / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    auto sync = [] {
        if (NAMED)
            compute_sync<kThreads>();
        else
            __syncthreads();
    };
    double a[NP];
#pragma unroll
    for (int k = 0; k < NP; ++k) a[k] = k < NV ? v[k] : 0.0;
#pragma unroll
    for (int o = 16, half = NP / 2; o > 0; o >>= 1, half >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int k = 0; k < half; ++k) {
            const double send = up ? a[k] : a[k + half];
            const double keep = up ? a[k + half] : a[k];
            a[k] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
    sync();                                       // the previous call's readers are done with `red`
#pragma unroll
    for (int k = 0; k < PER; ++k) red[warp * NP + lane * PER + k] = a[k];
    sync();
    if (tid < NV) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) t += red[w * NP + tid];
        out[tid] = t;
    }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Few values (NV <= 8): shuffle inside the warp, then across the 8 warps through shared memory.
template <int NV, bool MAX, int NT = kThreads, bool NAMED = false>
__device__ __forceinline__ void block_reduce_small(double (&v)[NV], double *sm /* >= (NT/32)*8 */, double *out) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    auto sync = [] {
        if (NAMED)
            compute_sync<NT>();
        else
            __syncthreads();
    };
    sync();
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        const double s = MAX ? warp_max(v[k]) : warp_sum(v[k]);
        if (lane == 0) sm[warp * 8 + k] = s;
    }
    sync();
    if (tid < NV) {
        double t = sm[tid];
#pragma unroll
        for (int q = 1; q < NT / 32; ++q) t = MAX ? fmax(t, sm[q * 8 + tid]) : t + sm[q * 8 + tid];
        out[tid] = t;
    }
}

// ------------------------------------------------------------------------------------------------
// K3 / K1: max|x| per run, then sum phi^2 per run
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_absmax(StreamArgs p) {
    __shared__ double sm[64];
    const int tid = threadIdx.x;
    double acc[1] = {0.0};
    const int s0 = p.cta_seg[blockIdx.x], s1 = p.cta_seg[blockIdx.x + 1];
    for (int s = s0; s < s1; ++s) {
        const Segment sg = p.segs[s];
        const int64_t end = sg.start + sg.len;
        for (int64_t n = sg.start + tid; n < end; n += kThreads) acc[0] = fmax(acc[0], fabs(p.x[n]));
        if (sg.flush) {
            block_reduce_small<1, true>(acc, sm, p.part + (size_t)sg.run * p.part_stride);
            acc[0] = 0.0;
        }
    }
}

template <int M>
__global__ void __launch_bounds__(kThreads, 1) k_phi2sum(StreamArgs p) {
    extern __shared__ double red[];
    __shared__ double sScal[2];
    const int tid = threadIdx.x;
    double acc[M];
#pragma unroll
    for (int i = 0; i < M; ++i) acc[i] = 0.0;
    const int s0 = p.cta_seg[blockIdx.x], s1 = p.cta_seg[blockIdx.x + 1];
    for (int s = s0; s < s1; ++s) {
        const Segment sg = p.segs[s];
        __syncthreads();
        if (tid == 0) {
            sScal[0] = p.inv2L[sg.region];
            sScal[1] = p.rsqrtL[sg.region];
        }
        __syncthreads();
        const double inv2L = sScal[0], rs = sScal[1];
        const int64_t end = sg.start + sg.len;
        for (int64_t n = sg.start + tid; n < end; n += kThreads) {
            double f1, c2;
            basis_seed(p.x[n], inv2L, rs, f1, c2);
            double fm = 0.0, f = f1;
#pragma unroll
            for (int i = 0; i < M; ++i) {
                acc[i] = fma(f, f, acc[i]);
                const double fn = fma(c2, f, -fm);
                fm = f;
                f = fn;
            }
        }
        if (sg.flush) {
            block_reduce_store<M>(acc, red, p.part + (size_t)sg.run * p.part_stride);
#pragma unroll
            for (int i = 0; i < M; ++i) acc[i] = 0.0;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// P4, P5, S5 for one region from the summed phase-B statistics sm[0..DY+2] = [sum r_d, sum |r|^2, sum fvar,
// sum phi^2 cm2] (region-specific noise and bias: Posteriors.py:81-93, 132-148 (ci) / 396-412 (fi);
// Stats.py:102-124).  y_var is 1/noise_mean(old) for inferred targets and is NOT multiplied by n in the ci
// regional/regional variant (Posteriors.py:138); fi targets are observations with y_var == 0.
// ------------------------------------------------------------------------------------------------
template <int DY>
__device__ __forceinline__ void bias_noise_region(const StreamArgs &p, int r, const double *sums) {
    if (p.sums_only || !(p.noise_rs && p.bias_rs)) {   // shared noise and / or bias: the sums of all regions first (k_bias_noise_shared)
#pragma unroll
        for (int d = 0; d < DY + 3; ++d) p.sumsB[(size_t)r * (DY + 3) + d] = sums[d];
        return;
    }
    const double n = (double)(p.offsets[r + 1] - p.offsets[r]);
    const double bp0 = p.bias_prec0[r];
    const double bp = bp0 + n;
    double t3 = 0.0, t4 = 0.0;
#pragma unroll
    for (int d = 0; d < DY; ++d) {
        const double m0 = p.bias_mean0[(size_t)r * DY + d];
        const double m = (1.0 / bp) * (m0 * bp0 + sums[d]);
        p.bias_prev_out[(size_t)r * DY + d] = p.bias_mean_out[(size_t)r * DY + d];
        p.bias_mean_out[(size_t)r * DY + d] = m;
        t3 += m0 * m0;
        t4 += m * m;
    }
    t3 *= bp0;
    t4 *= bp;
    const double yvar = p.infer ? 1.0 / p.noise_mean[r] : 0.0;
    const double shape = p.noise_shape0[r] + 0.5 * (double)DY * n;
    const double scale = p.noise_scale0[r] + 0.5 * (t3 - t4 + sums[DY] + sums[DY + 1] + sums[DY + 2] + yvar);
    p.yvar[r] = yvar;
    p.bias_prec[r] = bp;
    p.bias_var[r] = 1.0 / bp;
    p.noise_shape[r] = shape;
    p.noise_scale[r] = scale;
    p.noise_mean[r] = shape / scale;
    p.noise_log_mean[r] = digamma(shape) - log(scale);
#pragma unroll
    for (int d = 0; d < DY + 3; ++d) p.sumsB[(size_t)r * (DY + 3) + d] = sums[d];
}

// All regions of the layer by one block: `lpr` lanes (power of two <= 32) share the run loop of a region,
// the lane sums are combined by shuffles in a fixed order.
template <int DY, int NT>
__device__ __forceinline__ void bias_noise_all(const StreamArgs &p, int lpr, int block = 0, int n_blocks = 1) {
    const int groups = NT / lpr;
    const int grp = threadIdx.x / lpr, sl = threadIdx.x % lpr;
    for (int base = block * groups; base < p.R; base += n_blocks * groups) {
        const int r = base + grp;
        double acc[DY + 3];
#pragma unroll
        for (int d = 0; d < DY + 3; ++d) acc[d] = 0.0;
        if (r < p.R)
            for (int q = p.region_run[r] + sl; q < p.region_run[r + 1]; q += lpr) {
                const double *src = p.part + (size_t)q * p.part_stride;
#pragma unroll
                for (int d = 0; d < DY + 3; ++d) acc[d] += __ldcg(src + d);
            }
        for (int o = lpr >> 1; o > 0; o >>= 1)
#pragma unroll
            for (int d = 0; d < DY + 3; ++d) acc[d] += __shfl_xor_sync(0xffffffffu, acc[d], o);
        if (r < p.R && sl == 0) bias_noise_region<DY>(p, r, acc);
    }
}

// ------------------------------------------------------------------------------------------------
// Tile pipeline of the streaming kernels.  A CTA walks its contiguous sample range in tiles of
// kTile = 256 threads x kS samples; the inputs of a tile (x, y, latent mean g, latent variance h) are
// brought to shared memory by bulk asynchronous copies (TMA, cp.async.bulk) that complete on an mbarrier,
// kStages tiles ahead of the arithmetic, so no thread ever waits on a global load and no registers are
// spent on prefetching.  Inside a tile every thread works on kS samples at once: the region coefficients
// are read from shared memory once per basis function for all kS samples and the kS sine recurrences
// are independent dependency chains for the FP64 pipe.
// ------------------------------------------------------------------------------------------------
constexpr int kS = 4;
constexpr int kTile = kThreads * kS;
constexpr int kStages = 3;
constexpr int kThreadsB = 256;              // phase B block size, kSB samples per thread (same tile)
constexpr int kSB = kTile / kThreadsB;

template <int DY, bool NEED_Y, bool NEED_G, bool NEED_H>
struct TileLayout {
    static constexpr int kX = 0;
    static constexpr int kH = kTile;
    static constexpr int kY = kH + (NEED_H ? kTile : 0);
    static constexpr int kG = kY + (NEED_Y ? kTile * DY : 0);
    static constexpr int kDoubles = kG + (NEED_G ? kTile * DY : 0);
    static_assert((DY * 8) % 16 == 0, "rows of y / g must be multiples of 16 bytes for the bulk copies");
};

// One thread arms the barrier of a stage and issues the copies of `cnt` samples starting at `start`.
template <int DY, bool NEED_Y, bool NEED_G, bool NEED_H>
__device__ __forceinline__ void issue_tile(const StreamArgs &p, double *stage, uint64_t *bar, int64_t start, int cnt) {
    using L = TileLayout<DY, NEED_Y, NEED_G, NEED_H>;
    const int even = cnt & ~1;   // 8-byte rows: bulk copies move multiples of 16 bytes, an odd tail goes by hand
    uint32_t bytes = (uint32_t)even * 8u * (NEED_H ? 2u : 1u) + (uint32_t)cnt * DY * 8u * ((NEED_Y ? 1u : 0u) + (NEED_G ? 1u : 0u));
    if (cnt & 1) {
        stage[L::kX + cnt - 1] = p.x[start + cnt - 1];
        if (NEED_H) stage[L::kH + cnt - 1] = p.h[start + cnt - 1];
    }
    mbar_arrive_expect_tx(bar, bytes);
    if (even) {
        bulk_g2s(stage + L::kX, p.x + start, (uint32_t)even * 8u, bar);
        if (NEED_H) bulk_g2s(stage + L::kH, p.h + start, (uint32_t)even * 8u, bar);
    }
    if (NEED_Y) bulk_g2s(stage + L::kY, p.y + start * DY, (uint32_t)cnt * DY * 8u, bar);
    if (NEED_G) bulk_g2s(stage + L::kG, p.g + start * DY, (uint32_t)cnt * DY * 8u, bar);
}

// Lane 0 of warp 0 feeds the pipeline: before it starts tile t it issues every tile up to t + kStages - 1
// whose stage has been released by all compute warps (non-blocking probe of the stage's "empty" barrier) and
// blocks only for tile t itself.  No warp ever waits at a CTA-wide barrier between tiles, so the warps drift
// apart by up to kStages - 1 tiles and the latency-bound parts of one warp (sincospi, epilogue) overlap the
// FMA streams of the others.
template <int DY, bool NEED_Y, bool NEED_G, bool NEED_H>
__device__ __forceinline__ void refill(const StreamArgs &p, double *stages, uint64_t *full_bar, uint64_t *empty_bar, int &next_issue,
                                       int t, int n_tiles, int64_t c0, int64_t c1) {
    using L = TileLayout<DY, NEED_Y, NEED_G, NEED_H>;
    while (next_issue < n_tiles && next_issue < t + kStages) {
        const int stage = next_issue % kStages;
        if (next_issue >= kStages) {
            const uint32_t parity = (uint32_t)(((next_issue / kStages) - 1) & 1);
            if (next_issue == t)
                mbar_wait(&empty_bar[stage], parity);
            else if (!mbar_test(&empty_bar[stage], parity))
                break;
        }
        const int64_t start = c0 + (int64_t)next_issue * kTile;
        const int cnt = (int)((c1 - start < kTile) ? c1 - start : kTile);
        issue_tile<DY, NEED_Y, NEED_G, NEED_H>(p, stages + stage * L::kDoubles, &full_bar[stage], start, cnt);
        ++next_issue;
    }
}

// ------------------------------------------------------------------------------------------------
// Phase A: T[i][d] = sum_n phi_i(n) r_d(n),  r = y - (fbar + b + Phi A_old^T)
//   INFER  : targets are the layer's own prediction Phi A_old^T + (b_old + fbar)   (ci, j > 0;
//            LatentOutputs.py:25-40 via MRGP.py:577) instead of the observations (LatentOutputs.py:6-18)
//   LATENT : the layer has coarser layers below it (fbar = g + parent bias); layer 0 has fbar == 0.
// y_tilde_i = T_i + (sum_n phi_i^2) a_i reproduces Posteriors.py:61-78 (the penalty over k != i) with
// one pass over the samples instead of M.  The basis is generated twice per sample (once for Phi A^T,
// once for Phi^T r) instead of being kept in registers: 30 extra FMAs buy kS samples in flight.
// ------------------------------------------------------------------------------------------------
template <int DY, int M, int SB, bool INFER, bool LATENT>
__device__ __forceinline__ void phase_a_block(double (&T)[M * DY], const double *st, int k0, int lo_rel, int hi_rel,
                                              const double *sA, double inv2L, double rs, const double (&b)[DY],
                                              const double (&pb)[DY]) {
    using L = TileLayout<DY, !INFER, LATENT, false>;
    asm volatile("" ::: "memory");   // keep the region coefficients in shared memory, not in registers
    double f1[SB], c2[SB], f[SB], fm[SB], e[SB][DY], r[SB][DY];
    bool act[SB];
#pragma unroll
    for (int q = 0; q < SB; ++q) {
        const int idx = (k0 + q) * kThreads + threadIdx.x;
        act[q] = idx >= lo_rel && idx < hi_rel;
        const double x = act[q] ? st[L::kX + idx] : 0.0;
        basis_seed(x, inv2L, act[q] ? rs : 0.0, f1[q], c2[q]);
        f[q] = f1[q];
        fm[q] = 0.0;
#pragma unroll
        for (int d = 0; d < DY; ++d) e[q][d] = 0.0;
    }
#pragma unroll 5
    for (int i = 0; i < M; ++i) {
        double a[DY];
#pragma unroll
        for (int d = 0; d < DY; ++d) a[d] = sA[i * DY + d];
#pragma unroll
        for (int q = 0; q < SB; ++q) {
#pragma unroll
            for (int d = 0; d < DY; ++d) e[q][d] = fma(f[q], a[d], e[q][d]);
            const double fn = fma(c2[q], f[q], -fm[q]);
            fm[q] = f[q];
            f[q] = fn;
        }
    }
    asm volatile("" ::: "memory");   // read the targets / latent mean only now (register pressure)
#pragma unroll
    for (int q = 0; q < SB; ++q) {
        const int idx = (k0 + q) * kThreads + threadIdx.x;
#pragma unroll
        for (int d = 0; d < DY; ++d) {
            const double g = (LATENT && act[q]) ? st[L::kG + idx * DY + d] : 0.0;
            const double yv = (!INFER && act[q]) ? st[L::kY + idx * DY + d] : 0.0;
            const double fb = LATENT ? g + pb[d] : 0.0;   // fbar
            const double target = INFER ? e[q][d] + (b[d] + fb) : yv;
            r[q][d] = target - ((fb + b[d]) + e[q][d]);
        }
        f[q] = f1[q];
        fm[q] = 0.0;
    }
#pragma unroll
    for (int i = 0; i < M; ++i) {
#pragma unroll
        for (int q = 0; q < SB; ++q) {
#pragma unroll
            for (int d = 0; d < DY; ++d) T[i * DY + d] = fma(f[q], r[q][d], T[i * DY + d]);
            const double fn = fma(c2[q], f[q], -fm[q]);
            fm[q] = f[q];
            f[q] = fn;
        }
    }
}

template <int DY, int M, bool INFER, bool LATENT>
__global__ void __launch_bounds__(kThreads, 1) k_phase_a(StreamArgs p) {
    using L = TileLayout<DY, !INFER, LATENT, false>;
    constexpr int NCW = kThreads / 32;
    extern __shared__ __align__(128) double dsm[];
    double *stages = dsm;
    double *red = dsm + kStages * L::kDoubles;
    __shared__ double sA_all[NCW][M * DY];   // region coefficients, one private copy per warp
    __shared__ __align__(8) uint64_t full_bar[kStages];
    __shared__ __align__(8) uint64_t empty_bar[kStages];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t c0 = p.sample_begin + (int64_t)blockIdx.x * p.cta_quantum;
    const int64_t c1 = (c0 + p.cta_quantum < p.n_samples) ? c0 + p.cta_quantum : p.n_samples;
    const int n_tiles = (c1 > c0) ? (int)((c1 - c0 + kTile - 1) / kTile) : 0;
    ts_begin(p.ts, p.layer * 4 + 0);
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], NCW);
        }
        mbar_fence_init();
    }
    __syncthreads();
    int next_issue = 0;
    double *sA = sA_all[warp];
    double T[M * DY];
#pragma unroll
    for (int i = 0; i < M * DY; ++i) T[i] = 0.0;
    int s = p.cta_seg[blockIdx.x];
    const int s_end = p.cta_seg[blockIdx.x + 1];
    int loaded = -1;
    double inv2L = 0.0, rs = 0.0, b[DY], pb[DY];
#pragma unroll
    for (int d = 0; d < DY; ++d) b[d] = pb[d] = 0.0;
    Segment sg;
    if (s < s_end) sg = p.segs[s];
    for (int t = 0; t < n_tiles; ++t) {
        const int stage = t % kStages;
        const double *st = stages + stage * L::kDoubles;
        if (tid == 0) refill<DY, !INFER, LATENT, false>(p, stages, full_bar, empty_bar, next_issue, t, n_tiles, c0, c1);
        mbar_wait(&full_bar[stage], (uint32_t)((t / kStages) & 1));
        const int64_t tile_lo = c0 + (int64_t)t * kTile;
        const int64_t tile_hi = (tile_lo + kTile < c1) ? tile_lo + kTile : c1;
        int64_t pos = tile_lo;
        while (pos < tile_hi) {
            if (loaded != s) {
                __syncwarp();
                for (int q = lane; q < M * DY; q += 32) sA[q] = q < p.n_basis * DY ? p.A[(size_t)sg.region * (p.n_basis * DY) + q] : 0.0;
                inv2L = p.inv2L[sg.region];
                rs = p.rsqrtL[sg.region];
#pragma unroll
                for (int d = 0; d < DY; ++d) {
                    b[d] = p.bias[(size_t)sg.region * DY + d];
                    pb[d] = LATENT ? p.pbias[(size_t)sg.parent * DY + d] : 0.0;
                }
                __syncwarp();
                loaded = s;
            }
            const int64_t seg_end = sg.start + sg.len;
            const int64_t hi = (seg_end < tile_hi) ? seg_end : tile_hi;
            // 256-sample sub-blocks of the tile that intersect [pos, hi)
            int ka = (int)((pos - tile_lo) / kThreads);
            const int kb = (int)((hi - 1 - tile_lo) / kThreads);
            while (ka <= kb) {
                const int left = kb - ka + 1;
                if (left >= 3) {   // (three sub-blocks run as four with the last one masked: the small blocks are latency-bound)
                    phase_a_block<DY, M, 4, INFER, LATENT>(T, st, ka, (int)(pos - tile_lo), (int)(hi - tile_lo), sA, inv2L, rs, b, pb);
                    ka += 4;
                } else if (left >= 2) {
                    phase_a_block<DY, M, 2, INFER, LATENT>(T, st, ka, (int)(pos - tile_lo), (int)(hi - tile_lo), sA, inv2L, rs, b, pb);
                    ka += 2;
                } else {
                    phase_a_block<DY, M, 1, INFER, LATENT>(T, st, ka, (int)(pos - tile_lo), (int)(hi - tile_lo), sA, inv2L, rs, b, pb);
                    ka += 1;
                }
            }
            pos = hi;
            if (hi == seg_end) {
                if (sg.flush) {
                    block_reduce_store<M * DY, true>(T, red, p.part + (size_t)sg.run * p.part_stride);
#pragma unroll
                    for (int i = 0; i < M * DY; ++i) T[i] = 0.0;
                }
                ++s;
                if (s < s_end) sg = p.segs[s];
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);   // this warp is done with the stage
    }
    ts_end(p.ts, p.layer * 4 + 0);
}

// ------------------------------------------------------------------------------------------------
// Sufficient statistics of the observations for layer 0 of the fused ci sweep (csrc/chain.cu): per run
//     c[i][d] = sum_n phi_i(n) y_d(n),   sum_n y_d(n),   sum_n |y(n)|^2
// One pass over (x, y) per data set: 24 B and 3 M + 22 + 5 FP64 operations per sample (the basis once, no
// coefficients).  Same tile pipeline and segment / run plan as phase A; partial layout [c (M*DY) | sum y (DY) | sum |y|^2].
// ------------------------------------------------------------------------------------------------
template <int DY, int M, int SB>
__device__ __forceinline__ void ystats_block(double (&T)[M * DY + DY + 1], const double *st, int k0, int lo_rel, int hi_rel, double inv2L,
                                             double rs) {
    using L = TileLayout<DY, true, false, false>;
    double c2[SB], f[SB], fm[SB], yv[SB][DY];
#pragma unroll
    for (int q = 0; q < SB; ++q) {
        const int idx = (k0 + q) * kThreads + threadIdx.x;
        const bool act = idx >= lo_rel && idx < hi_rel;
        const double x = act ? st[L::kX + idx] : 0.0;
        basis_seed(x, inv2L, act ? rs : 0.0, f[q], c2[q]);
        fm[q] = 0.0;
        double rr = 0.0;
#pragma unroll
        for (int d = 0; d < DY; ++d) {
            yv[q][d] = act ? st[L::kY + idx * DY + d] : 0.0;
            T[M * DY + d] += yv[q][d];
            rr = fma(yv[q][d], yv[q][d], rr);
        }
        T[M * DY + DY] += rr;
    }
#pragma unroll
    for (int i = 0; i < M; ++i) {
#pragma unroll
        for (int q = 0; q < SB; ++q) {
#pragma unroll
            for (int d = 0; d < DY; ++d) T[i * DY + d] = fma(f[q], yv[q][d], T[i * DY + d]);
            const double fn = fma(c2[q], f[q], -fm[q]);
            fm[q] = f[q];
            f[q] = fn;
        }
    }
}

template <int NS, int NU>
__device__ __forceinline__ void reduce_ystats_region(double (*sm)[64], int r, const int32_t *region_run, const double *part, int part_stride, int M,
                                                     int MP, int DY, double *yc, double *ysum);

template <int DY, int M>
__global__ void __launch_bounds__(kThreads, 1) k_ystats(StreamArgs p) {
    using L = TileLayout<DY, true, false, false>;
    constexpr int NCW = kThreads / 32, NV = M * DY + DY + 1;
    extern __shared__ __align__(128) double dsm[];
    double *stages = dsm;
    double *red = dsm + kStages * L::kDoubles;
    __shared__ __align__(8) uint64_t full_bar[kStages];
    __shared__ __align__(8) uint64_t empty_bar[kStages];
    const int tid = threadIdx.x, lane = tid & 31;
    const int64_t c0 = p.sample_begin + (int64_t)blockIdx.x * p.cta_quantum;
    const int64_t c1 = (c0 + p.cta_quantum < p.n_samples) ? c0 + p.cta_quantum : p.n_samples;
    const int n_tiles = (c1 > c0) ? (int)((c1 - c0 + kTile - 1) / kTile) : 0;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], NCW);
        }
        mbar_fence_init();
    }
    __syncthreads();
    int next_issue = 0;
    double T[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) T[i] = 0.0;
    int s = p.cta_seg[blockIdx.x];
    const int s_end = p.cta_seg[blockIdx.x + 1];
    int loaded = -1;
    double inv2L = 0.0, rs = 0.0;
    Segment sg;
    if (s < s_end) sg = p.segs[s];
    for (int t = 0; t < n_tiles; ++t) {
        const int stage = t % kStages;
        const double *st = stages + stage * L::kDoubles;
        if (tid == 0) refill<DY, true, false, false>(p, stages, full_bar, empty_bar, next_issue, t, n_tiles, c0, c1);
        mbar_wait(&full_bar[stage], (uint32_t)((t / kStages) & 1));
        const int64_t tile_lo = c0 + (int64_t)t * kTile;
        const int64_t tile_hi = (tile_lo + kTile < c1) ? tile_lo + kTile : c1;
        int64_t pos = tile_lo;
        while (pos < tile_hi) {
            if (loaded != s) {
                inv2L = p.inv2L[sg.region];
                rs = p.rsqrtL[sg.region];
                loaded = s;
            }
            const int64_t seg_end = sg.start + sg.len;
            const int64_t hi = (seg_end < tile_hi) ? seg_end : tile_hi;
            int ka = (int)((pos - tile_lo) / kThreads);
            const int kb = (int)((hi - 1 - tile_lo) / kThreads);
            while (ka <= kb) {
                const int left = kb - ka + 1;
                if (left >= 3) {
                    ystats_block<DY, M, 4>(T, st, ka, (int)(pos - tile_lo), (int)(hi - tile_lo), inv2L, rs);
                    ka += 4;
                } else if (left >= 2) {
                    ystats_block<DY, M, 2>(T, st, ka, (int)(pos - tile_lo), (int)(hi - tile_lo), inv2L, rs);
                    ka += 2;
                } else {
                    ystats_block<DY, M, 1>(T, st, ka, (int)(pos - tile_lo), (int)(hi - tile_lo), inv2L, rs);
                    ka += 1;
                }
            }
            pos = hi;
            if (hi == seg_end) {
                if (sg.flush) {
                    block_reduce_store<NV, true>(T, red, p.part + (size_t)sg.run * p.part_stride);
#pragma unroll
                    for (int i = 0; i < NV; ++i) T[i] = 0.0;
                }
                ++s;
                if (s < s_end) sg = p.segs[s];
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);
    }
    // ---- tail: the last CTA to finish sums the run partials into the statistics of the regions (fixed order) ----
    if (!p.fuse_tail) return;
    __shared__ int sLast;
    __shared__ double sred[kThreads / 64][64];
    __syncthreads();
    if (tid == 0) sLast = (atom_add_acq_rel_gpu(p.done_counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (sLast) {
        for (int r = 0; r < p.R; ++r)
            reduce_ystats_region<kThreads / 64, 40>(sred, r, p.region_run, p.part, p.part_stride, p.n_basis, M, DY, p.yc_out, p.ysum_out);
        if (tid == 0) *p.done_counter = 0u;
    }
}

// yc[r][i][d], ysum[r][0..DY] = sums over the region's runs of the k_ystats partials (fixed order).
// (MP: the padded number of basis functions the partials were written for.)  1024 threads: value = tid % 64 (chunks of
// 64 values), 16 slices over the runs with their loads in flight together, combined in slice order.
template <int NS, int NU>
__device__ __forceinline__ void reduce_ystats_region(double (*sm)[64], int r, const int32_t *region_run, const double *part, int part_stride, int M,
                                                     int MP, int DY, double *yc, double *ysum) {
    const int nv = MP * DY + DY + 1, lane64 = threadIdx.x & 63, slice = threadIdx.x >> 6;
    const int q_end = region_run[r + 1];
    for (int v0 = 0; v0 < nv; v0 += 64) {
        const int v = v0 + lane64;
        double s = 0.0;
        if (v < nv)
            for (int q = region_run[r] + slice; q < q_end; q += NS * NU) {
                double t[NU];
#pragma unroll
                for (int u = 0; u < NU; ++u) t[u] = q + NS * u < q_end ? __ldcg(part + (size_t)(q + NS * u) * part_stride + v) : 0.0;
#pragma unroll
                for (int u = 0; u < NU; ++u) s += t[u];
            }
        sm[slice][lane64] = s;
        __syncthreads();
        if (slice == 0 && v < nv && !(v >= M * DY && v < MP * DY)) {
            double t = 0.0;
#pragma unroll
            for (int k = 0; k < NS; ++k) t += sm[k][lane64];
            if (v < M * DY)
                yc[(size_t)r * M * DY + v] = t;
            else
                ysum[(size_t)r * 4 + (v - MP * DY)] = t;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024) k_reduce_ystats(const int32_t *region_run, const double *part, int part_stride, int R, int M, int MP, int DY,
                                                        double *yc, double *ysum) {
    __shared__ double sm[16][64];
    reduce_ystats_region<16, 4>(sm, blockIdx.x, region_run, part, part_stride, M, MP, DY, yc, ysum);
}

// ------------------------------------------------------------------------------------------------
// Phase B: residual statistics with the NEW coefficients, fused with the propagation of the latent
// mean / variance to the next layer (Posteriors.py:81-148, Stats.py:126-157):
//   r = target - Phi A_new^T - fbar;   partial = [sum r_d, sum |r|^2, sum fvar, sum_n sum_i phi_i^2 cm2_i]
//   g <- fbar + Phi A_new^T,  h <- fvar + sum_i phi_i^2 cm2_i      (PROPAGATE; the layer's own bias and
//   bias variance are added by the next layer when it reads g, h, because they are not known yet).
// ------------------------------------------------------------------------------------------------
template <int DY, int M, int SB, int NT, bool INFER, bool LATENT, bool PROPAGATE>
__device__ __forceinline__ void phase_b_block(double (&acc)[DY + 3], const StreamArgs &p, const double *st, int k0, int64_t tile_lo,
                                              int lo_rel, int hi_rel, const double *sAn, const double *sAo, const double *sC,
                                              double inv2L, double rs, double pbv, const double (&b)[DY], const double (&pb)[DY]) {
    using L = TileLayout<DY, !INFER, LATENT, LATENT>;
    asm volatile("" ::: "memory");
    double c2[SB], f[SB], fm[SB], en[SB][DY], eo[SB][DY], v[SB];
    bool act[SB];
#pragma unroll
    for (int q = 0; q < SB; ++q) {
        const int idx = (k0 + q) * NT + threadIdx.x;
        act[q] = idx >= lo_rel && idx < hi_rel;
        const double x = act[q] ? st[L::kX + idx] : 0.0;
        basis_seed(x, inv2L, act[q] ? rs : 0.0, f[q], c2[q]);
        fm[q] = 0.0;
        v[q] = 0.0;
#pragma unroll
        for (int d = 0; d < DY; ++d) en[q][d] = eo[q][d] = 0.0;
    }
#pragma unroll 5
    for (int i = 0; i < M; ++i) {
        double an[DY], ao[DY];
#pragma unroll
        for (int d = 0; d < DY; ++d) {
            an[d] = sAn[i * DY + d];
            ao[d] = INFER ? sAo[i * DY + d] : 0.0;
        }
        const double c = sC[i];
#pragma unroll
        for (int q = 0; q < SB; ++q) {
#pragma unroll
            for (int d = 0; d < DY; ++d) {
                en[q][d] = fma(f[q], an[d], en[q][d]);
                if (INFER) eo[q][d] = fma(f[q], ao[d], eo[q][d]);
            }
            v[q] = fma(f[q] * c, f[q], v[q]);
            const double fn = fma(c2[q], f[q], -fm[q]);
            fm[q] = f[q];
            f[q] = fn;
        }
    }
#pragma unroll
    for (int q = 0; q < SB; ++q) {
        if (act[q]) {
            const int idx = (k0 + q) * NT + threadIdx.x;
            const int64_t n = tile_lo + idx;
            const double fv = LATENT ? st[L::kH + idx] + pbv : 0.0;
            double rr = 0.0;
#pragma unroll
            for (int d = 0; d < DY; ++d) {
                const double fb = LATENT ? st[L::kG + idx * DY + d] + pb[d] : 0.0;
                const double target = INFER ? eo[q][d] + (b[d] + fb) : st[L::kY + idx * DY + d];
                const double r = (target - en[q][d]) - fb;
                acc[d] += r;
                rr = fma(r, r, rr);
                if (PROPAGATE) p.g[n * DY + d] = fb + en[q][d];
            }
            acc[DY] += rr;
            acc[DY + 1] += fv;
            acc[DY + 2] += v[q];
            if (PROPAGATE) p.h[n] = fv + v[q];
        }
    }
}

template <int DY, int M, bool INFER, bool LATENT, bool PROPAGATE>
__global__ void __launch_bounds__(kThreadsB, 1) k_phase_b(StreamArgs p) {
    constexpr int NT = kThreadsB;
    constexpr int NCW = NT / 32;
    using L = TileLayout<DY, !INFER, LATENT, LATENT>;
    extern __shared__ __align__(128) double dsm[];
    double *stages = dsm;
    __shared__ double sAn_all[NCW][M * DY];        // region coefficients, one private copy per warp
    __shared__ double sAo_all[INFER ? NCW : 1][INFER ? M * DY : 1];
    __shared__ double sC_all[NCW][M];
    __shared__ double sRed[NCW * 8];
    __shared__ __align__(8) uint64_t full_bar[kStages];
    __shared__ __align__(8) uint64_t empty_bar[kStages];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (p.gate && *p.gate == 0u) return;   // uniform over the grid: the statistics of the fused sweep were good enough
    const int64_t c0 = p.sample_begin + (int64_t)blockIdx.x * p.cta_quantum;
    const int64_t c1 = (c0 + p.cta_quantum < p.n_samples) ? c0 + p.cta_quantum : p.n_samples;
    const int n_tiles = (c1 > c0) ? (int)((c1 - c0 + kTile - 1) / kTile) : 0;
    ts_begin(p.ts, p.layer * 4 + 2);
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], NCW);
        }
        mbar_fence_init();
    }
    __syncthreads();
    int next_issue = 0;
    double *sAn = sAn_all[warp];
    double *sAo = sAo_all[INFER ? warp : 0];
    double *sC = sC_all[warp];
    double acc[DY + 3];
#pragma unroll
    for (int i = 0; i < DY + 3; ++i) acc[i] = 0.0;
    int s = p.cta_seg[blockIdx.x];
    const int s_end = p.cta_seg[blockIdx.x + 1];
    int loaded = -1;
    double inv2L = 0.0, rs = 0.0, pbv = 0.0, b[DY], pb[DY];
#pragma unroll
    for (int d = 0; d < DY; ++d) b[d] = pb[d] = 0.0;
    Segment sg;
    if (s < s_end) sg = p.segs[s];
    for (int t = 0; t < n_tiles; ++t) {
        const int stage = t % kStages;
        const double *st = stages + stage * L::kDoubles;
        if (tid == 0) refill<DY, !INFER, LATENT, LATENT>(p, stages, full_bar, empty_bar, next_issue, t, n_tiles, c0, c1);
        mbar_wait(&full_bar[stage], (uint32_t)((t / kStages) & 1));
        const int64_t tile_lo = c0 + (int64_t)t * kTile;
        const int64_t tile_hi = (tile_lo + kTile < c1) ? tile_lo + kTile : c1;
        int64_t pos = tile_lo;
        while (pos < tile_hi) {
            if (loaded != s) {
                __syncwarp();
                for (int q = lane; q < M * DY; q += 32) {
                    const bool real = q < p.n_basis * DY;
                    sAn[q] = real ? p.A[(size_t)sg.region * (p.n_basis * DY) + q] : 0.0;
                    if (INFER) sAo[q] = real ? p.A_prev[(size_t)sg.region * (p.n_basis * DY) + q] : 0.0;
                }
                for (int q = lane; q < M; q += 32) sC[q] = q < p.n_basis ? p.cm2[(size_t)sg.region * p.n_basis + q] : 0.0;
                inv2L = p.inv2L[sg.region];
                rs = p.rsqrtL[sg.region];
                pbv = LATENT ? p.pbias_var[sg.parent] : 0.0;
#pragma unroll
                for (int d = 0; d < DY; ++d) {
                    b[d] = p.bias[(size_t)sg.region * DY + d];
                    pb[d] = LATENT ? p.pbias[(size_t)sg.parent * DY + d] : 0.0;
                }
                __syncwarp();
                loaded = s;
            }
            const int64_t seg_end = sg.start + sg.len;
            const int64_t hi = (seg_end < tile_hi) ? seg_end : tile_hi;
            int ka = (int)((pos - tile_lo) / NT);
            const int kb = (int)((hi - 1 - tile_lo) / NT);
            while (ka <= kb) {
                const int left = kb - ka + 1;
                if (kSB >= 4 && left >= 3) {
                    phase_b_block<DY, M, 4, NT, INFER, LATENT, PROPAGATE>(acc, p, st, ka, tile_lo, (int)(pos - tile_lo), (int)(hi - tile_lo), sAn, sAo, sC, inv2L, rs, pbv, b, pb);
                    ka += 4;
                } else if (left >= 2) {
                    phase_b_block<DY, M, 2, NT, INFER, LATENT, PROPAGATE>(acc, p, st, ka, tile_lo, (int)(pos - tile_lo), (int)(hi - tile_lo), sAn, sAo, sC, inv2L, rs, pbv, b, pb);
                    ka += 2;
                } else {
                    phase_b_block<DY, M, 1, NT, INFER, LATENT, PROPAGATE>(acc, p, st, ka, tile_lo, (int)(pos - tile_lo), (int)(hi - tile_lo), sAn, sAo, sC, inv2L, rs, pbv, b, pb);
                    ka += 1;
                }
            }
            pos = hi;
            if (hi == seg_end) {
                if (sg.flush) {
                    block_reduce_small<DY + 3, false, NT, true>(acc, sRed, p.part + (size_t)sg.run * p.part_stride);
#pragma unroll
                    for (int i = 0; i < DY + 3; ++i) acc[i] = 0.0;
                }
                ++s;
                if (s < s_end) sg = p.segs[s];
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);
    }
    // ---- tail: the last CTA to finish turns the run partials into the bias / noise posteriors --------
    if (!p.fuse_tail) {
        ts_end(p.ts, p.layer * 4 + 2);
        return;
    }
    __shared__ int sLast;
    compute_sync<NT>();
    if (tid == 0) sLast = (atom_add_acq_rel_gpu(p.done_counter, 1u) == gridDim.x - 1);
    compute_sync<NT>();
    if (sLast) {
        int lpr = 32;
        while (lpr > 1 && (NT / lpr) < p.R) lpr >>= 1;
        bias_noise_all<DY, NT>(p, lpr);
        if (tid == 0) *p.done_counter = 0u;
    }
    ts_end(p.ts, p.layer * 4 + 2);
}

// ------------------------------------------------------------------------------------------------
// per-region small kernels
// ------------------------------------------------------------------------------------------------
struct RegionArgs {
    int32_t R, M, DY, layer;
    int32_t mode;              // 0 ci, 1 fi
    int32_t infer;             // ci, layer > 0
    const int32_t *region_run; // (R + 1) run range of each region
    const int64_t *offsets;    // (R + 1)
    const double *part;        // partials of the preceding streaming kernel
    int32_t part_stride;
    // static
    double *L, *inv2L, *rsqrtL, *lam, *S, *d, *absx;
    // posterior / stats
    double *prec, *zeta, *ytil, *A, *A_prev, *m2, *cm2;
    double *noise_shape, *noise_scale, *noise_shape0, *noise_scale0, *noise_mean, *noise_log_mean;
    double *bias_prec, *bias_prec0, *bias_mean, *bias_mean0, *bias_var, *yvar, *sumsB;
    // shared (ci) or per-region (fi) axis / ARD
    double *axB, *axKappa, *axRho, *axLogC, *axCov, *ardShape, *ardScale, *ardMean, *ardLogMean;
    double *omega, *logOmegaHat, *omegaIters, *ardPartial, *omegaEta, *omegaWarm, *omegaK, *primeSk, *skTag, *wcontrib;
    double *primeB, *primeLogC, *primeShape, *primeScale;   // snapshot read by ARD / omega (ci)
    const double *priorB, *priorLogC, *priorShape, *priorScale;
    double *bcontrib;          // (R, M, 3) ci: 0.5 noise zeta ytil ytil^T
    double *rconst;            // (R, 8) ci: constants of the regions for the fused sweep, or null
    unsigned long long *chol_count;
    unsigned long long *ts;
    double fi_shape0_mix, fi_scale0_mix;   // sum_k (1/M) shape0_k, sum_k (1/M) scale0_k (Posteriors.py:293-295)
    // spectral density
    int32_t use_prior;
    double nu, ell, sf, interval_factor;
    int32_t L_given;
    int32_t zero_T;   // 1: Phi^T r is identically zero (inferred targets, see sweep_once): y_tilde = d a
};

// K3 + K2: L = factor max|x| (BasisInterval.py:15-16), 1/(2L), L^-1/2, lambda (KernelClass.py:36),
// S (KernelClass.py:80-90).  One warp per region.
__global__ void k_region_setup(RegionArgs a) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= a.R) return;
    double L;
    if (a.L_given) {
        L = a.L[r];
    } else {
        double m = 0.0;
        for (int q = a.region_run[r] + lane; q < a.region_run[r + 1]; q += 32) m = fmax(m, a.part[(size_t)q * a.part_stride]);
        m = warp_max(m);
        if (lane == 0) a.absx[r] = m;
        L = a.interval_factor * m;
    }
    if (lane == 0) {
        a.L[r] = L;
        a.inv2L[r] = 0.5 / L;
        a.rsqrtL[r] = 1.0 / sqrt(L);
    }
    for (int i = lane; i < a.M; i += 32) {
        const double w = (kPi * (double)(i + 1)) / (2.0 * L);
        const double lam = w * w;
        a.lam[(size_t)r * a.M + i] = lam;
        a.S[(size_t)r * a.M + i] = a.use_prior ? matern_spectral(lam, a.nu, a.ell, a.sf) : 1.0;
    }
}

// d[r][i] = sum over the region's runs of the phi^2 partials (Posteriors.py:41).
__global__ void k_reduce_d(RegionArgs a) {
    const int r = blockIdx.x;
    for (int i = threadIdx.x; i < a.M; i += blockDim.x) {
        double s = 0.0;
        for (int q = a.region_run[r]; q < a.region_run[r + 1]; ++q) s += a.part[(size_t)q * a.part_stride + i];
        a.d[(size_t)r * a.M + i] = s;
    }
}

// Sum the phase-A partials of region r for value t (= i*DY + d), `slices` threads per value.
// Block of 128 threads laid out as (slice, value) with value fastest; NVAL = M*DY <= 96 -> up to 1 slice
// per 128 threads; for regions with many runs (coarse layers) the kernel is launched with 1024 threads
// so that 8+ slices share the run loop.
template <int DY>
__global__ void __launch_bounds__(512) k_reduce_scale(RegionArgs a) {
    extern __shared__ double sm[];   // [slices][NV] + ytil[NV]
    const int r = blockIdx.x;
    const int M = a.M, NV = M * DY;
    const int nval = (NV + 31) & ~31;
    const int slices = blockDim.x / nval;
    const int v = threadIdx.x % nval, sl = threadIdx.x / nval;
    double acc = 0.0;
    if (v < NV && sl < slices)
        for (int q = a.region_run[r] + sl; q < a.region_run[r + 1]; q += slices) acc += a.part[(size_t)q * a.part_stride + v];
    if (sl < slices) sm[sl * nval + v] = acc;
    __syncthreads();
    double *ytil_s = sm + slices * nval;
    if (threadIdx.x < NV) {
        double t = 0.0;
        for (int q = 0; q < slices; ++q) t += sm[q * nval + threadIdx.x];
        const int i = threadIdx.x / DY;
        // y_tilde_i = Phi_i^T r + (sum phi_i^2) a_i   (Posteriors.py:61-78)
        const double yt = t + a.d[(size_t)r * M + i] * a.A[(size_t)r * NV + threadIdx.x];
        ytil_s[threadIdx.x] = yt;
        a.ytil[(size_t)r * NV + threadIdx.x] = yt;
    }
    __syncthreads();
    if (threadIdx.x < M) {
        const int i = threadIdx.x;
        const size_t ri = (size_t)r * M + i;
        const double noise = a.noise_mean[r];
        const double ard = (a.mode == 0) ? a.ardMean[i] : a.ardMean[ri];
        // Posteriors.py:40-42 / :304-306
        const double prec = ard / a.S[ri] + noise * a.d[ri];
        const double zeta = noise / prec;
        a.prec[ri] = prec;
        a.zeta[ri] = zeta;
        const double w = 0.5 * noise * zeta;
        static_assert(DY == 2, "dy == 2 only");
        const double y0 = ytil_s[i * DY], y1 = ytil_s[i * DY + 1];
        if (a.mode == 0) {
            // contribution to B_i, summed over regions by k_axis_shared (Posteriors.py:507-517)
            a.bcontrib[ri * 3 + 0] = w * (y0 * y0);
            a.bcontrib[ri * 3 + 1] = w * (y0 * y1);
            a.bcontrib[ri * 3 + 2] = w * (y1 * y1);
        } else {
            // fi: the prior B is the untouched zero prior, omega == 1/M (Posteriors.py:253-285)
            Bingham2 bg;
            bingham2(0.0 + w * (y0 * y0), 0.0 + w * (y0 * y1), 0.0 + w * (y1 * y1), bg);
            atomicAdd(a.chol_count, (unsigned long long)bg.n_chol);
            a.axB[ri * 4 + 0] = bg.b[0];
            a.axB[ri * 4 + 1] = bg.b[1];
            a.axB[ri * 4 + 2] = bg.b[1];
            a.axB[ri * 4 + 3] = bg.b[2];
            a.axKappa[ri * 2 + 0] = bg.kappa[0];
            a.axKappa[ri * 2 + 1] = bg.kappa[1];
            a.axRho[ri * 2 + 0] = bg.rho[0];
            a.axRho[ri * 2 + 1] = bg.rho[1];
            a.axLogC[ri] = bg.logc;
            a.axCov[ri * 4 + 0] = bg.cov[0];
            a.axCov[ri * 4 + 1] = bg.cov[1];
            a.axCov[ri * 4 + 2] = bg.cov[1];
            a.axCov[ri * 4 + 3] = bg.cov[2];
            // Stats.py:257-290
            const double cy0 = bg.cov[0] * y0 + bg.cov[1] * y1, cy1 = bg.cov[1] * y0 + bg.cov[2] * y1;
            a.A_prev[ri * DY + 0] = a.A[ri * DY + 0];
            a.A_prev[ri * DY + 1] = a.A[ri * DY + 1];
            a.A[ri * DY + 0] = zeta * cy0;
            a.A[ri * DY + 1] = zeta * cy1;
            const double z2 = zeta * zeta;
            const double m2 = 1.0 / prec + z2 * (y0 * cy0 + y1 * cy1);
            const double ccy0 = bg.cov[0] * cy0 + bg.cov[1] * cy1, ccy1 = bg.cov[1] * cy0 + bg.cov[2] * cy1;
            const double cm2 = 1.0 / prec + z2 * (y0 * (cy0 - ccy0) + y1 * (cy1 - ccy1));
            a.m2[ri] = m2;
            a.cm2[ri] = cm2;
            // Posteriors.py:288-295, Stats.py:251-255
            const double shape = a.fi_shape0_mix + 0.5 * (double)a.R;
            const double scale = a.fi_scale0_mix + 0.5 * (m2 / a.S[ri]);
            a.ardShape[ri] = shape;
            a.ardScale[ri] = scale;
            a.ardMean[ri] = shape / scale;
            a.ardLogMean[ri] = digamma(shape) - log(scale);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// ci mid-step (the work is latency-bound: a few dependent global loads per item, so it is spread over many SMs
// instead of a few fat CTAs):
//   k_mid1  P1-finish per (region, basis) item: run partials -> y_tilde, precision, zeta (Posteriors.py:35-78) and
//           per-CTA sums over the regions of the item's contribution to B_i (Posteriors.py:507-517) and of the two
//           terms that make sum_l m2/S linear in the axis covariance (ARD update, Posteriors.py:533-541);
//   k_ard   (side stream, critical chain) sums those partials, mixes in the previous posterior, runs the PD guard and
//           the Bingham update (P2, S1: Posteriors.py:497-530, Stats.py:375-382), the ARD update and the log
//           omega_hat table; k_scale_warp / k_scale then solve for omega;
//   k_mid2  (main stream, beside k_ard) re-derives the same axis update per CTA and finishes S2 for its regions:
//           a, m2, cm2 (Stats.py:67-100).
// `lpi` lanes (power of two) share the run loop of one item on coarse layers where a region has many runs.
// ------------------------------------------------------------------------------------------------
constexpr int kMidThreads = 256;

template <int DY>
__global__ void __launch_bounds__(kMidThreads) k_mid1(RegionArgs a, int lpi, int regions_per_cta) {
    static_assert(DY == 2, "dy == 2 only");
    extern __shared__ double sm[];   // contrib[32 * M * 4], contribW[32 * M * 4], sums[NVP], sumsW[NVWP]
    const int M = a.M, tid = threadIdx.x, NV = M * 3, NVP = (NV + 31) & ~31;   // NVP: padded length of a B-sum vector
    const int NVW = M * 4, NVWP = (NVW + 31) & ~31;                                // ... of the ARD-sum vector
    double *sContrib = sm, *sContribW = sm + 32 * M * 4, *sSum = sContribW + 32 * M * 4, *sSumW = sSum + NVP;
    ts_begin(a.ts, a.layer * 4 + 1);
    for (int t = tid; t < NVP; t += kMidThreads) sSum[t] = 0.0;
    for (int t = tid; t < NVWP; t += kMidThreads) sSumW[t] = 0.0;
    __syncthreads();
    const int r0 = blockIdx.x * regions_per_cta;
    const int r1 = (r0 + regions_per_cta < a.R) ? r0 + regions_per_cta : a.R;
    const int groups = kMidThreads / lpi, grp = tid / lpi, sl = tid % lpi;
    for (int cb = r0; cb < r1; cb += 32) {
        const int nreg = (cb + 32 < r1) ? 32 : r1 - cb;
        const int nitems = nreg * M;
        for (int base = 0; base < nitems; base += groups) {
            const int it = base + grp;
            const bool valid = it < nitems;
            const int l = cb + (valid ? it / M : 0), i = valid ? it % M : 0;
            double t0 = 0.0, t1 = 0.0;
            if (valid && !a.zero_T)
                for (int q = a.region_run[l] + sl; q < a.region_run[l + 1]; q += lpi) {
                    const double2 v = *reinterpret_cast<const double2 *>(a.part + (size_t)q * a.part_stride + i * 2);
                    t0 += v.x;
                    t1 += v.y;
                }
            for (int o = lpi >> 1; o > 0; o >>= 1) {
                t0 += __shfl_xor_sync(0xffffffffu, t0, o);
                t1 += __shfl_xor_sync(0xffffffffu, t1, o);
            }
            if (valid && sl == 0) {
                const size_t ri = (size_t)l * M + i;
                const double dsum = a.d[ri];
                const double y0 = t0 + dsum * a.A[ri * 2 + 0], y1 = t1 + dsum * a.A[ri * 2 + 1];   // Posteriors.py:61-78
                const double noise = a.noise_mean[l];
                const double prec = a.ardMean[i] / a.S[ri] + noise * dsum;                       // Posteriors.py:40-42
                const double zeta = noise / prec;
                a.ytil[ri * 2 + 0] = y0;
                a.ytil[ri * 2 + 1] = y1;
                a.prec[ri] = prec;
                a.zeta[ri] = zeta;
                const double w = 0.5 * noise * zeta;                                             // Posteriors.py:507-517
                sContrib[it * 4 + 0] = w * (y0 * y0);
                sContrib[it * 4 + 1] = w * (y0 * y1);
                sContrib[it * 4 + 2] = w * (y1 * y1);
                // sum_l m2_li / S_li of the ARD update (Posteriors.py:533-541) is linear in the axis covariance C_i that
                // the Bingham update is about to produce: m2 = 1/prec + zeta^2 tr(y y^T C) (Stats.py:67-100), so
                // sum_l m2/S = sum_l 1/(prec S) + tr((sum_l zeta^2 y y^T / S) C_i): the region sums are taken here
                const double is = 1.0 / a.S[ri], z2s = zeta * zeta * is;
                sContribW[it * 4 + 0] = is / prec;
                sContribW[it * 4 + 1] = z2s * (y0 * y0);
                sContribW[it * 4 + 2] = z2s * (y0 * y1);
                sContribW[it * 4 + 3] = z2s * (y1 * y1);
            }
        }
        __syncthreads();
        // sum over the regions of the chunk: one thread per value, regions in order (a serial chain of <= 32 adds is
        // shorter than the rounds of warp reductions it replaces: the kernel sits on the critical chain of the sweep)
        for (int vv = tid; vv < NV + NVW; vv += kMidThreads) {
            double t = 0.0;
            if (vv < NV) {
                const int i = vv / 3, c = vv % 3;
                for (int k = 0; k < nreg; ++k) t += sContrib[(k * M + i) * 4 + c];
                sSum[vv] += t;
            } else {
                const int w = vv - NV;
                for (int k = 0; k < nreg; ++k) t += sContribW[k * M * 4 + w];
                sSumW[w] += t;
            }
        }
        __syncthreads();
    }
    for (int t = tid; t < NVP; t += kMidThreads) a.bcontrib[(size_t)blockIdx.x * NVP + t] = sSum[t];   // per-CTA partials
    for (int t = tid; t < NVWP; t += kMidThreads) a.wcontrib[(size_t)blockIdx.x * NVWP + t] = sSumW[t];
    if (blockIdx.x == 0) {   // snapshot of the previous posterior (MRGP.py:575 / :581): k_mid2 and k_omega read it
        const bool first = (a.layer == 0);
        for (int t = tid; t < M * 4; t += kMidThreads) a.primeB[t] = first ? a.priorB[t] : a.axB[t];
        for (int t = tid; t < M; t += kMidThreads) {
            a.primeLogC[t] = first ? a.priorLogC[t] : a.axLogC[t];
            a.primeShape[t] = first ? a.priorShape[t] : a.ardShape[t];
            a.primeScale[t] = first ? a.priorScale[t] : a.ardScale[t];
        }
    }
    ts_end(a.ts, a.layer * 4 + 1);
}

// Sum of the per-CTA partial vectors of k_mid1 (length NVP each) into sData, in two steps so that the caller can
// issue its other global loads while these are in flight: load_b_partials puts up to 16 partials per thread into
// registers (`halves` slices of CTAs per value), reduce_b_partials adds them in a fixed tree.  k_mid2 and k_ard both
// use 256 threads, so both form bit-identical sums.
struct BPartials {
    double p[16];
    double tail;
};

__device__ __forceinline__ void load_b_partials(const double *bcontrib, int nb, int NVP, BPartials &r) {
    const int tid = threadIdx.x, nt = blockDim.x;      // NVP <= nt (M <= 85)
    const int halves = (nt / NVP >= 2) ? 2 : 1;
    const int v = tid % NVP, half = tid / NVP;
    r.tail = 0.0;
#pragma unroll
    for (int u = 0; u < 16; ++u) {
        const int q = half + u * halves;
        r.p[u] = (half < halves && q < nb) ? __ldcg(bcontrib + (size_t)q * NVP + v) : 0.0;
    }
    if (half < halves)
        for (int q = half + 16 * halves; q < nb; q += halves) r.tail += __ldcg(bcontrib + (size_t)q * NVP + v);
}

__device__ __forceinline__ void reduce_b_partials(BPartials &r, int NVP, double *sData, double *sHalf) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int halves = (nt / NVP >= 2) ? 2 : 1;
    const int v = tid % NVP, half = tid / NVP;
#pragma unroll
    for (int w = 8; w > 0; w >>= 1)
#pragma unroll
        for (int u = 0; u < w; ++u) r.p[u] += r.p[u + w];
    if (half < halves) sHalf[half * NVP + v] = r.p[0] + r.tail;
    __syncthreads();
    if (tid < NVP) sData[tid] = sHalf[tid] + (halves > 1 ? sHalf[NVP + tid] : 0.0);
}

// Second half of the ci mid-step.  Every CTA re-derives the axis update from the per-CTA partial sums of k_mid1
// (a few microseconds of redundant work instead of a grid-wide hand-off), then finishes S2 for its regions.
template <int DY>
__global__ void __launch_bounds__(kMidThreads) k_mid2(RegionArgs a, int regions_per_cta, int n_partials) {
    static_assert(DY == 2, "dy == 2 only");
    extern __shared__ double sm[];
    const int M = a.M, tid = threadIdx.x, NV = M * 3, NVP = (NV + 31) & ~31;
    (void)NV;
    ts_begin(a.ts, a.layer * 4 + 1);
    const int r0 = blockIdx.x * regions_per_cta;
    const int r1 = (r0 + regions_per_cta < a.R) ? r0 + regions_per_cta : a.R;
    double *sOmega = sm, *sPB = sOmega + M * M, *sData = sPB + 4 * M;
    double *sCovOut = sm + ((33 * M > M * M + 4 * M + 3 * NVP) ? 33 * M : M * M + 4 * M + 3 * NVP);
    BPartials bp;
    load_b_partials(a.bcontrib, n_partials, NVP, bp);      // in flight together with the staging loads below
    for (int t = tid; t < M * M; t += kMidThreads) sOmega[t] = a.omega[t];
    for (int t = tid; t < M * 4; t += kMidThreads) sPB[t] = a.primeB[t];
    reduce_b_partials(bp, NVP, sData, sData + NVP);
    __syncthreads();
    if (tid < M) {
        const int i = tid;
        double b00 = 0.0, b01 = 0.0, b11 = 0.0;
        for (int k = 0; k < M; ++k) {
            const double w = sOmega[i * M + k];
            b00 += w * sPB[k * 4 + 0];
            b01 += w * sPB[k * 4 + 1];
            b11 += w * sPB[k * 4 + 3];
        }
        Bingham2 bg;
        bingham2(b00 + sData[i * 3 + 0], b01 + sData[i * 3 + 1], b11 + sData[i * 3 + 2], bg);
        sCovOut[i * 4 + 0] = bg.cov[0];
        sCovOut[i * 4 + 1] = bg.cov[1];
        sCovOut[i * 4 + 2] = bg.cov[1];
        sCovOut[i * 4 + 3] = bg.cov[2];
    }
    __syncthreads();
    // ---- S2 per item with the new axis covariance: a, m2, cm2 (Stats.py:67-100).  (The axis state itself and the
    //      ARD update are written by k_ard, which derives the same update on the side stream.) ---------------------
    double *sCov = sCovOut;
    for (int cb = r0; cb < r1; cb += 32) {
        const int nreg = (cb + 32 < r1) ? 32 : r1 - cb;
        const int nitems = nreg * M;
        for (int it = tid; it < nitems; it += kMidThreads) {
            const int l = cb + it / M, i = it % M;
            const size_t ri = (size_t)l * M + i;
            const double c00 = sCov[i * 4 + 0], c01 = sCov[i * 4 + 1], c11 = sCov[i * 4 + 3];
            const double y0 = a.ytil[ri * 2], y1 = a.ytil[ri * 2 + 1];
            const double zeta = a.zeta[ri], prec = a.prec[ri];
            const double cy0 = c00 * y0 + c01 * y1, cy1 = c01 * y0 + c11 * y1;
            a.A_prev[ri * 2 + 0] = a.A[ri * 2 + 0];
            a.A_prev[ri * 2 + 1] = a.A[ri * 2 + 1];
            a.A[ri * 2 + 0] = zeta * cy0;
            a.A[ri * 2 + 1] = zeta * cy1;
            const double z2 = zeta * zeta;
            const double ccy0 = c00 * cy0 + c01 * cy1, ccy1 = c01 * cy0 + c11 * cy1;
            a.m2[ri] = 1.0 / prec + z2 * (y0 * cy0 + y1 * cy1);
            a.cm2[ri] = 1.0 / prec + z2 * (y0 * (cy0 - ccy0) + y1 * (cy1 - ccy1));
        }
    }
    ts_end(a.ts, a.layer * 4 + 1);
}

// ci, side stream, the critical chain of the sweep: shared axis update from the region sums of k_mid1 (P2, S1),
// ARD posterior and moments (Posteriors.py:533-541, Stats.py:385-388), the log omega_hat table (Stats.py:405-412)
// with its shifts and exponentials (k_ard, one block); then the doubly-stochastic scaling omega
// (Stats.py:413-420) by the Sinkhorn / Newton scheme of omega_solve_serial (mrgp_math.cuh): k_scale_warp (one
// warp, registers) for M <= 32, k_scale (one block, shared memory) otherwise.
constexpr int kOmegaThreads = 256;

__host__ __device__ inline size_t omega_smem_doubles(int M) { return (size_t)3 * M * M + 24 * M + 8 + 3 * ((3 * M + 31) & ~31) + 4 * M; }

__global__ void __launch_bounds__(kOmegaThreads) k_ard(RegionArgs a, int n_partials) {
    extern __shared__ double sm[];
    const int M = a.M, tid = threadIdx.x;
    constexpr int NW = kOmegaThreads / 32;
    double *P = sm, *s_mean = P + M * M, *s_lmean = s_mean + M, *s_k = s_lmean + M, *s_shape = s_k + M, *s_scale = s_shape + M;
    double *s_B = s_scale + M, *s_C = s_B + 4 * M, *s_part = s_C + 4 * M;   // s_part: NW x M
    const int NVP = (3 * M + 31) & ~31, NVWP = (4 * M + 31) & ~31;
    double *s_data = s_part + NW * M, *s_half = s_data + NVP, *s_w = s_half + 2 * NVP;   // B sums, scratch, ARD sums
    ts_begin(a.ts, a.layer * 4 + 3);
    // one wave of global loads: the per-CTA sums of k_mid1 (data part of B: same code as k_mid2, same bits; ARD sums:
    // one value per thread, k_mid1 runs at most 32 CTAs) go to registers while every other input is staged in
    // shared memory
    BPartials bp;
    load_b_partials(a.bcontrib, n_partials, NVP, bp);
    double pw[32];
    {
        const int t = tid < 4 * M ? tid : 0;
#pragma unroll
        for (int u = 0; u < 32; ++u) pw[u] = (tid < 4 * M && u < n_partials) ? __ldcg(a.wcontrib + (size_t)u * NVWP + t) : 0.0;
    }
    for (int t = tid; t < M * M; t += kOmegaThreads) P[t] = a.omega[t];   // the OLD omega mixes the previous posterior
    for (int t = tid; t < 4 * M; t += kOmegaThreads) s_B[t] = a.primeB[t];
    {
        // the k-only terms of the table, -logC' + shape' log scale' - lgamma(shape'), were prepared off the critical
        // chain: by k_init_shared for layer 0 (its "previous posterior" is the prior) and by the second warp of the
        // previous layer's k_scale_warp for the others; they are computed here only if that did not happen (block
        // solver, per-phase calls in an unusual order, state set from the host)
        const int slot = a.layer == 0 ? 2 : (a.layer & 1);
        const bool have_sk = a.skTag[slot] == (double)a.layer;
        for (int t = tid; t < M; t += kOmegaThreads) {
            const double shp = a.primeShape[t], scp = a.primeScale[t];
            s_shape[t] = shp;
            s_scale[t] = scp;
            s_k[t] = have_sk ? a.primeSk[slot * 64 + t] : -a.primeLogC[t] + shp * log(scp) - lgamma(shp);
        }
    }
#pragma unroll
    for (int w = 16; w > 0; w >>= 1)
#pragma unroll
        for (int u = 0; u < w; ++u) pw[u] += pw[u + w];
    if (tid < 4 * M) s_w[tid] = pw[0];
    reduce_b_partials(bp, NVP, s_data, s_half);
    __syncthreads();
    // the shared axis update (P2, P2a-c, S1: Posteriors.py:497-530, Stats.py:375-382), exactly as every CTA of
    // k_mid2 derives it for its own use; this kernel owns the stored axis state
    if (tid < M) {
        const int i = tid;
        double b00 = 0.0, b01 = 0.0, b11 = 0.0;
        for (int k = 0; k < M; ++k) {
            const double w = P[i * M + k];
            b00 += w * s_B[k * 4 + 0];
            b01 += w * s_B[k * 4 + 1];
            b11 += w * s_B[k * 4 + 3];
        }
        Bingham2 bg;
        bingham2(b00 + s_data[i * 3 + 0], b01 + s_data[i * 3 + 1], b11 + s_data[i * 3 + 2], bg);
        s_C[i * 4 + 0] = bg.cov[0];
        s_C[i * 4 + 1] = bg.cov[1];
        s_C[i * 4 + 2] = bg.cov[1];
        s_C[i * 4 + 3] = bg.cov[2];
        atomicAdd(a.chol_count, (unsigned long long)bg.n_chol);
        a.axB[i * 4 + 0] = bg.b[0];
        a.axB[i * 4 + 1] = bg.b[1];
        a.axB[i * 4 + 2] = bg.b[1];
        a.axB[i * 4 + 3] = bg.b[2];
        a.axKappa[i * 2 + 0] = bg.kappa[0];
        a.axKappa[i * 2 + 1] = bg.kappa[1];
        a.axRho[i * 2 + 0] = bg.rho[0];
        a.axRho[i * 2 + 1] = bg.rho[1];
        a.axLogC[i] = bg.logc;
        a.axCov[i * 4 + 0] = bg.cov[0];
        a.axCov[i * 4 + 1] = bg.cov[1];
        a.axCov[i * 4 + 2] = bg.cov[1];
        a.axCov[i * 4 + 3] = bg.cov[2];
        // sum_l m2_li / S_li = sum_l 1/(prec S) + tr((sum_l zeta^2 y y^T / S) C_i)
        const double beta2 = s_w[i * 4 + 0] + (s_w[i * 4 + 1] * bg.cov[0] + 2.0 * s_w[i * 4 + 2] * bg.cov[1] + s_w[i * 4 + 3] * bg.cov[2]);
        // ARD update of the same basis function in the same thread (no barrier: its sums do not depend on the axis
        // update and fill the latency of the chain above)
        double sh = 0.0, sc = 0.0;
        for (int k = 0; k < M; ++k) {
            const double w = P[i * M + k];
            sh += w * s_shape[k];
            sc += w * s_scale[k];
        }
        const double shape = sh + 0.5 * (double)a.R;
        const double scale = sc + 0.5 * beta2;
        a.ardShape[i] = shape;
        a.ardScale[i] = scale;
        const double mean = shape / scale, lmean = digamma(shape) - log(scale);
        a.ardMean[i] = mean;
        a.ardLogMean[i] = lmean;
        s_mean[i] = mean;
        s_lmean[i] = lmean;
    }
    __syncthreads();
    for (int t = tid; t < M * M; t += kOmegaThreads) {
        const int i = t / M, k = t % M;
        const double *C = s_C + i * 4, *B = s_B + k * 4;
        const double tr = C[0] * B[0] + C[1] * B[2] + C[2] * B[1] + C[3] * B[3];   // trace(C_i B'_k)
        const double lw = tr + s_k[k] + (s_shape[k] - 1.0) * s_lmean[i] - s_scale[k] * s_mean[i];
        a.logOmegaHat[t] = lw;
        P[t] = lw;                      // the old omega is no longer needed
    }
    // head of the scaling solve, done here by the whole block: row shift, column shift, exponentials.  The solve
    // (one warp, k_scale_warp) starts from the table K = exp(lw - rowmax - colmax), stored column-major, and the
    // column shifts (row shifts cancel in the row normalisation).  One thread per row, then one per column: a serial
    // chain of M maxima is shorter than the rounds of warp reductions it replaces.
    __syncthreads();
    double *s_rowmax = s_part, *s_colmax = s_part + M;   // the partial sums are no longer needed
    if (tid < M) {
        double mx = -INFINITY;
        for (int k = 0; k < M; ++k) mx = fmax(mx, P[tid * M + k]);
        s_rowmax[tid] = mx;
    }
    __syncthreads();
    if (tid < M) {
        double mx = -INFINITY;
        for (int i = 0; i < M; ++i) mx = fmax(mx, P[i * M + tid] - s_rowmax[i]);
        s_colmax[tid] = mx;
        a.omegaK[64 * 64 + tid] = mx;
    }
    __syncthreads();
    for (int t = tid; t < M * M; t += kOmegaThreads) {
        const int k = t / M, i = t % M;        // column-major output: coalesced stores
        a.omegaK[t] = exp((P[i * M + k] - s_rowmax[i]) - s_colmax[k]);
    }
    ts_dbg(a.ts, a.layer, 0, false);   // debug slots: [0] = (k_ard begin, k_ard end)
    ts_dbg(a.ts, a.layer, 0, true);
}


// Second kernel of the side stream: the doubly-stochastic scaling of exp(log omega_hat) (Stats.py:413-420).
__global__ void __launch_bounds__(kOmegaThreads) k_scale(RegionArgs a) {
    extern __shared__ double sm[];
    const int M = a.M, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = kOmegaThreads / 32;
    double *K = sm, *P = K + M * M, *S = P + M * M, *v = S + M * M, *c = v + M, *rhs = c + M, *dinv = rhs + M;
    double *yv = dinv + M, *xv = yv + M, *cshift = xv + M, *red = cshift + M;
    for (int t = tid; t < M * M; t += kOmegaThreads) K[t] = a.logOmegaHat[t];
    __syncthreads();
    for (int i = warp; i < M; i += NW) {
        double mx = -INFINITY;
        for (int k = lane; k < M; k += 32) mx = fmax(mx, K[i * M + k]);
        mx = warp_max(mx);
        for (int k = lane; k < M; k += 32) K[i * M + k] -= mx;
    }
    __syncthreads();
    for (int k = warp; k < M; k += NW) {
        double mx = -INFINITY;
        for (int i = lane; i < M; i += 32) mx = fmax(mx, K[i * M + k]);
        mx = warp_max(mx);
        for (int i = lane; i < M; i += 32) K[i * M + k] = exp(K[i * M + k] - mx);
        if (lane == 0) cshift[k] = mx;   // column shift (row shifts cancel in the row normalisation)
    }
    // warm start: the log column scalings of the previous sweep's solve for this layer (stored relative to
    // the un-shifted table, so that they do not depend on the shifts) seed the iteration
    const bool warm = a.omegaWarm[a.layer] > 0.5;
    __syncthreads();
    if (tid < M) {
        const double eta = a.omegaEta[a.layer * 64 + tid] + cshift[tid];
        v[tid] = (warm && isfinite(eta)) ? exp(fmax(-600.0, fmin(600.0, eta))) : 1.0;
    }
    __syncthreads();
    int iters = 0;
    double err_prev = INFINITY;
    int last = kOmegaNone;
    for (int it = 0; it < kOmegaWarmup + kOmegaMaxNewton; ++it) {
        ++iters;
        for (int i = warp; i < M; i += NW) {
            double s = 0.0;
            for (int k = lane; k < M; k += 32) s = fma(K[i * M + k], v[k], s);
            s = warp_sum(s);
            const double u = 1.0 / s;
            for (int k = lane; k < M; k += 32) P[i * M + k] = K[i * M + k] * v[k] * u;
        }
        __syncthreads();
        for (int k = warp; k < M; k += NW) {
            double s = 0.0;
            for (int i = lane; i < M; i += 32) s += P[i * M + k];
            s = warp_sum(s);
            if (lane == 0) c[k] = s;
        }
        __syncthreads();
        if (warp == 0) {
            double e = 0.0;
            for (int k = lane; k < M; k += 32) e = fmax(e, fabs(c[k] - 1.0));
            e = warp_max(e);
            if (lane == 0) red[0] = e;
        }
        __syncthreads();
        const double err = red[0];
        if (err < kOmegaTol) break;
        if (!isfinite(err)) {   // a bad (warm) start or an overshooting Newton step: start again from the shifts alone
            if (tid < M) v[tid] = 1.0;
            err_prev = INFINITY;
            last = kOmegaNone;
            __syncthreads();
            continue;
        }
        if (!omega_take_newton(err, err_prev, last)) {
            if (tid < M) v[tid] = fmax(1e-280, fmin(1e280, v[tid] / c[tid]));   // Sinkhorn column step
            err_prev = err;
            last = kOmegaSinkhorn;
            __syncthreads();
            continue;
        }
        err_prev = err;
        last = kOmegaNewton;
        for (int k = warp; k < M; k += NW)
            for (int m = lane; m <= k; m += 32) {
                double s0 = 0.0, s1 = 0.0;
                int i = 0;
                for (; i + 1 < M; i += 2) {
                    s0 = fma(P[i * M + k], P[i * M + m], s0);
                    s1 = fma(P[(i + 1) * M + k], P[(i + 1) * M + m], s1);
                }
                if (i < M) s0 = fma(P[i * M + k], P[i * M + m], s0);
                S[k * M + m] = ((k == m) ? c[k] : 0.0) - (s0 + s1) + 1.0 / (double)M;
            }
        if (tid < M) rhs[tid] = 1.0 - c[tid];
        __syncthreads();
        for (int j = 0; j < M; ++j) {   // Cholesky, lower triangle in place, diagonal untouched, 1/l_jj aside
            const double di = rsqrt(S[j * M + j]);
            if (tid > j && tid < M) S[tid * M + j] *= di;
            if (tid == 0) dinv[j] = di;
            __syncthreads();
            for (int r = j + 1 + (tid >> 4); r < M; r += 16)
                for (int q = j + 1 + (tid & 15); q <= r; q += 16) S[r * M + q] = fma(-S[r * M + j], S[q * M + j], S[r * M + q]);
            __syncthreads();
        }
        for (int j = 0; j < M; ++j) {   // L y = rhs
            const double yj = rhs[j] * dinv[j];
            if (tid > j && tid < M) rhs[tid] -= S[tid * M + j] * yj;
            if (tid == j) yv[j] = yj;
            __syncthreads();
        }
        for (int j = M - 1; j >= 0; --j) {   // L^T x = y
            const double xj = yv[j] * dinv[j];
            if (tid < j) yv[tid] -= S[j * M + tid] * xj;
            if (tid == j) xv[j] = xj;
            __syncthreads();
        }
        if (tid < M) v[tid] = fmax(1e-280, fmin(1e280, v[tid] * exp(fmax(-30.0, fmin(30.0, xv[tid])))));
        __syncthreads();
    }
    // last resort: plain Sinkhorn sweeps (see omega_solve_serial); on model tables the loop exits at its first test
    for (int it = 0; it < kOmegaFallbackSweeps; ++it) {
        for (int i = warp; i < M; i += NW) {
            double s = 0.0;
            for (int k = lane; k < M; k += 32) s = fma(K[i * M + k], v[k], s);
            s = warp_sum(s);
            const double u = 1.0 / s;
            for (int k = lane; k < M; k += 32) P[i * M + k] = K[i * M + k] * v[k] * u;
        }
        __syncthreads();
        for (int k = warp; k < M; k += NW) {
            double s = 0.0;
            for (int i = lane; i < M; i += 32) s += P[i * M + k];
            s = warp_sum(s);
            if (lane == 0) c[k] = s;
        }
        __syncthreads();
        if (warp == 0) {
            double e = 0.0;
            for (int k = lane; k < M; k += 32) e = fmax(e, fabs(c[k] - 1.0));
            e = warp_max(e);
            if (lane == 0) red[0] = e;
        }
        __syncthreads();
        const double err = red[0];
        if (err < kOmegaTol || !isfinite(err)) break;
        ++iters;
        if (tid < M) v[tid] = fmax(1e-280, fmin(1e280, v[tid] / c[tid]));
        __syncthreads();
    }
    for (int t = tid; t < M * M; t += kOmegaThreads) a.omega[t] = P[t];
    if (tid < M) a.omegaEta[a.layer * 64 + tid] = log(v[tid]) - cshift[tid];
    if (tid == 0) {
        a.omegaIters[a.layer] = (double)iters;
        a.omegaWarm[a.layer] = 1.0;
    }
    ts_end(a.ts, a.layer * 4 + 3);
}

// Dense per-region sums of the run partials (multi-GPU exchange buffer, SURVEY.md §8e): out[r][v] = sum over the
// local runs of region r (zero for regions without local samples); MAX = true for the max|x| partials.
template <bool MAX>
__global__ void k_region_sums(const int32_t *region_run, const double *part, int part_stride, int nv, int R, double *out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= R * part_stride) return;
    const int r = t / part_stride, v = t % part_stride;
    double acc = 0.0;
    if (v < nv)
        for (int q = region_run[r]; q < region_run[r + 1]; ++q) {
            const double x = part[(size_t)q * part_stride + v];
            acc = MAX ? fmax(acc, x) : acc + x;
        }
    out[(size_t)r * part_stride + v] = acc;   // padding columns are kept at zero
}

// The same solve for M <= 32 in ONE warp, matrices resident in registers: lane i owns row i of the kernel table
// (and of the Newton matrix), every loop over the M columns is unrolled, the only communication is warp
// shuffles plus two transposes through shared memory per Newton step.  No block barriers: a Newton step costs
// about a sixth of the block version's (which spends its time in 120 __syncthreads per step).  Same iteration
// (shifts, warm start, Sinkhorn warm-up, Newton on the log column scalings, cold restart, fallback sweeps) and
// same tolerances as k_scale / omega_solve_serial.
template <int M>
struct OmegaWarp {
    static constexpr int LD = 34;   // even: 16-byte aligned rows for the paired loads; 34 * 8 B rows are conflict-free
    // Row-normalised table P = diag(u) K diag(v) (rows in registers), its transpose in shared memory (T[k][i] =
    // P[i][k]) and, on lane k, column k (Q) with its sum c.  Returns max |c - 1| (NaN if any entry is NaN).
    static __device__ __forceinline__ double eval(const double (&K)[M], double (&P)[M], double (&Q)[M], double v, double &c,
                                                  double *T, bool row, int lane) {
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int k = 0; k < M; k += 2) {
            P[k] = K[k] * __shfl_sync(0xffffffffu, v, k);
            P[k + 1] = K[k + 1] * __shfl_sync(0xffffffffu, v, k + 1);
            s0 += P[k];
            s1 += P[k + 1];
        }
        const double u = row ? 1.0 / (s0 + s1) : 0.0;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < M; ++k) {
            P[k] *= u;
            T[k * LD + lane] = P[k];
        }
        __syncwarp();
        double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
        const double2 *col = reinterpret_cast<const double2 *>(T + (row ? lane : 0) * LD);
#pragma unroll
        for (int i = 0; i < M; i += 2) {
            const double2 t = col[i >> 1];
            Q[i] = t.x;
            Q[i + 1] = t.y;
            if (i & 2) {
                c2 += t.x;
                c3 += t.y;
            } else {
                c0 += t.x;
                c1 += t.y;
            }
        }
        c = (c0 + c1) + (c2 + c3);
        double e = row ? fabs(c - 1.0) : 0.0;
        const bool bad = !(e == e);
        e = warp_max(e);
        return __any_sync(0xffffffffu, bad) ? NAN : e;
    }
};

template <int M>
__global__ void __launch_bounds__(64, 1) k_scale_warp(RegionArgs a) {
    static_assert(M <= 32 && (M & 1) == 0, "one lane per row, columns in pairs");
    using W = OmegaWarp<M>;
    constexpr int LD = W::LD;
    __shared__ __align__(16) double T[M * LD];
    if (threadIdx.x >= 32) {
        // second warp, beside the solve: the posterior k_ard has just written is the "previous posterior" of the next
        // layer; the k-only terms of that layer's log omega_hat table (one lgamma per basis function) are ready before
        // its k_mid1 / k_ard need them
        const int i = threadIdx.x - 32, slot = (a.layer + 1) & 1;
        if (i < M) {
            const double shp = a.ardShape[i];
            a.primeSk[slot * 64 + i] = -a.axLogC[i] + shp * log(a.ardScale[i]) - lgamma(shp);
        }
        __syncwarp();
        if (i == 0) a.skTag[slot] = (double)(a.layer + 1);
        return;
    }
    const int lane = threadIdx.x;
    const bool row = lane < M;
    double K[M], P[M], Q[M];
    ts_dbg(a.ts, a.layer, 1, false);   // debug slots: [1] = prologue, [2] = iteration
#pragma unroll
    for (int k = 0; k < M; ++k) K[k] = row ? a.omegaK[k * M + lane] : 0.0;
    const double cshift = row ? a.omegaK[64 * 64 + lane] : 0.0;
    // warm start: the log column scalings of the previous sweep's solve for this layer (stored relative to the
    // un-shifted table, so that they do not depend on the shifts) seed the iteration
    const bool warm = a.omegaWarm[a.layer] > 0.5;
    double v = 1.0;
    if (row) {
        const double eta = a.omegaEta[a.layer * 64 + lane] + cshift;
        v = (warm && isfinite(eta)) ? exp(fmax(-600.0, fmin(600.0, eta))) : 1.0;
    }
    int iters = 0;
    double err_prev = INFINITY, c = 1.0;
    int last = kOmegaNone;
    ts_dbg(a.ts, a.layer, 1, true);
    ts_dbg(a.ts, a.layer, 2, false);
    for (int it = 0; it < kOmegaWarmup + kOmegaMaxNewton; ++it) {
        ++iters;
        const double err = W::eval(K, P, Q, v, c, T, row, lane);
        if (err < kOmegaTol) break;
        if (!isfinite(err)) {   // a bad (warm) start or an overshooting Newton step: start again from the shifts alone
            v = 1.0;
            err_prev = INFINITY;
            last = kOmegaNone;
            continue;
        }
        if (!omega_take_newton(err, err_prev, last)) {
            if (row) v = fmax(1e-280, fmin(1e280, v / c));   // Sinkhorn column step
            err_prev = err;
            last = kOmegaSinkhorn;
            continue;
        }
        err_prev = err;
        last = kOmegaNewton;
        // ---- Newton matrix: lane j builds row j of diag(c) - P^T P + 1/M from its column Q and the transposed table
        double H[M];
#pragma unroll
        for (int k = 0; k < M; k += 2) {
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            const double2 *r0 = reinterpret_cast<const double2 *>(T + k * LD);
            const double2 *r1 = reinterpret_cast<const double2 *>(T + (k + 1) * LD);
#pragma unroll
            for (int i = 0; i < M; i += 2) {
                const double2 t0 = r0[i >> 1], t1 = r1[i >> 1];
                a0 = fma(Q[i], t0.x, a0);
                a1 = fma(Q[i + 1], t0.y, a1);
                a2 = fma(Q[i], t1.x, a2);
                a3 = fma(Q[i + 1], t1.y, a3);
            }
            H[k] = ((lane == k) ? c : 0.0) - (a0 + a1) + 1.0 / (double)M;
            H[k + 1] = ((lane == k + 1) ? c : 0.0) - (a2 + a3) + 1.0 / (double)M;
        }
        // ---- Cholesky (right-looking, lane = row) fused with the forward substitution; the next pivot is formed
        //      first in every step (one shuffle) so that its reciprocal square root overlaps the rank-1 update
        double rhs = 1.0 - c, y = 0.0, dinv = 0.0;
        double piv = __shfl_sync(0xffffffffu, H[0], 0);
        double *colbuf = T;                                           // the transposed table is no longer needed
        __syncwarp();
#pragma unroll
        for (int k = 0; k < M; ++k) {
            const double di = rsqrt(piv);
            H[k] *= di;                                               // l_ik for lanes i >= k (l_kk on lane k)
            double *cb = colbuf + (k & 1) * 32;                       // two buffers: no barrier between the steps
            cb[lane] = H[k];
            if (k + 1 < M)   // the next pivot only needs its own row: h_jj - l_jk^2 on lane j = k + 1
                piv = __shfl_sync(0xffffffffu, fma(-H[k], H[k], H[k + 1]), k + 1);
            const double yk = __shfl_sync(0xffffffffu, rhs, k) * di;
            if (lane == k) {
                dinv = di;
                y = yk;
            }
            if (lane > k) rhs = fma(-H[k], yk, rhs);
            __syncwarp();
#pragma unroll
            for (int j = k + 1; j < M; ++j) H[j] = fma(-H[k], cb[j], H[j]);   // broadcast loads of l_jk
        }
        // ---- L^T x = y with the transposed factor: lane i reads l_ki, k > i, from shared memory -------------------
        __syncwarp();
#pragma unroll
        for (int k = 0; k < M; ++k) T[k * LD + lane] = H[k];          // T[k][i] = l_ik (valid for i >= k)
        __syncwarp();
        {
            const double2 *lt = reinterpret_cast<const double2 *>(T + (row ? lane : 0) * LD);
#pragma unroll
            for (int k = 0; k < M; k += 2) {
                const double2 t = lt[k >> 1];
                Q[k] = t.x;                                           // l_k,lane
                Q[k + 1] = t.y;
            }
        }
        double x = 0.0;
#pragma unroll
        for (int k = M - 1; k >= 0; --k) {
            const double xk = __shfl_sync(0xffffffffu, y, k) * __shfl_sync(0xffffffffu, dinv, k);
            if (lane == k) x = xk;
            if (lane < k) y = fma(-Q[k], xk, y);
        }
        if (row) v = fmax(1e-280, fmin(1e280, v * exp(fmax(-30.0, fmin(30.0, x)))));
    }
    ts_dbg(a.ts, a.layer, 2, true);
    // last resort: plain Sinkhorn sweeps (see omega_solve_serial); on model tables the loop exits at its first test
    for (int it = 0; it < kOmegaFallbackSweeps; ++it) {
        const double err = W::eval(K, P, Q, v, c, T, row, lane);
        if (err < kOmegaTol || !isfinite(err)) break;
        ++iters;
        if (row) v = fmax(1e-280, fmin(1e280, v / c));
    }
    if (row) {
#pragma unroll
        for (int k = 0; k < M; ++k) a.omega[lane * M + k] = P[k];
        a.omegaEta[a.layer * 64 + lane] = log(v) - cshift;
    }
    if (lane == 0) {
        a.omegaIters[a.layer] = (double)iters;
        a.omegaWarm[a.layer] = 1.0;
    }
    ts_end(a.ts, a.layer * 4 + 3);
}

// ------------------------------------------------------------------------------------------------
// Multi-GPU exchange over peer memory (NVLink / NVSwitch; SURVEY.md §8e).  Every rank keeps a small arena that
// its peers have mapped (CUDA IPC).  One exchange = (1) the dense per-region sums of the local run partials are
// written into the local arena, (2) the rank stores the next sequence number into its slot of every peer's flag
// array (st.release.sys), (3) a reduce kernel waits until every peer's number has arrived and sums, per region,
// the arenas of exactly the ranks whose sample chunk overlaps the region, in rank order - every rank forms the
// same sum in the same order, so the replicated small-matrix state stays bit-identical across ranks.  The arena
// has three slots used round-robin by exchange number: when a rank writes exchange e it has waited for every
// peer's signal e - 1, which a peer sends after it finished reading exchange e - 2 (stream order), so only the
// slots of e - 1 and e can be in use by a peer - never slot (e mod 3) of exchange e - 3.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxRanks = 16;
constexpr int kCommSlots = 3;

struct CommArgs {
    int32_t rank, world;
    const double *arena[kMaxRanks];            // arena base of every rank (own entry: the local pointer)
    unsigned long long *flags[kMaxRanks];      // flags[p][src]: last sequence number rank src has published to rank p
    unsigned long long *seq;                   // local: sequence number of the last exchange
    unsigned int *err;                         // local: set when a wait timed out
    unsigned long long slot_doubles;           // arena slot e mod kCommSlots starts at (e mod kCommSlots) * slot_doubles
    int64_t bounds[kMaxRanks + 1];             // rank q owns the samples [bounds[q], bounds[q + 1])
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ double ld_relaxed_sys(const double *p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Dense per-region sums of the local run partials into the arena, one block per region (threads = value x
// run slice), and - by the block that finishes last - the publication: the next sequence number is release-stored
// into this rank's slot of every peer's flag array.
template <bool MAX>
__global__ void __launch_bounds__(256) k_comm_sums_signal(CommArgs c, const int32_t *region_run, const double *part, int stride, int nv,
                                                          double *out, unsigned int *counter) {
    __shared__ double sm[256];
    __shared__ int sLast;
    const int r = blockIdx.x, tid = threadIdx.x;
    out += ((*c.seq + 1ull) % kCommSlots) * c.slot_doubles;   // the exchange this kernel publishes
    const int slices = 256 / stride > 0 ? 256 / stride : 1;
    const int v = tid % stride, sl = tid / stride;
    double acc = 0.0;
    if (sl < slices && v < nv)
        for (int q = region_run[r] + sl; q < region_run[r + 1]; q += slices) {
            const double x = __ldcg(part + (size_t)q * stride + v);
            acc = MAX ? fmax(acc, x) : acc + x;
        }
    sm[tid] = acc;
    __syncthreads();
    if (tid < stride) {
        double t = sm[tid];
        for (int k = 1; k < slices; ++k) t = MAX ? fmax(t, sm[k * stride + tid]) : t + sm[k * stride + tid];
        out[(size_t)r * stride + tid] = t;      // padding columns are kept at zero
    }
    __syncthreads();
    if (tid == 0) sLast = (atom_add_acq_rel_gpu(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!sLast) return;
    if (tid == 0) {
        *counter = 0u;
        sm[0] = 0.0;
        *c.seq = *c.seq + 1ull;
    }
    __syncthreads();
    __threadfence_system();
    if (tid < c.world) st_release_sys(c.flags[tid] + c.rank, *c.seq);
}

constexpr unsigned long long kCommTimeoutNs = 15000000000ull;   // a lost peer must not hang the GPU

// out[r][v] = sum (or max) over the ranks that own samples of region r of their arena entries.
template <bool MAX>
__global__ void __launch_bounds__(256) k_comm_reduce(CommArgs c, const int64_t *offsets, int R, int stride, int nv,
                                                     double *out) {
    __shared__ int ok;
    if (threadIdx.x < 32) {
        const unsigned long long want = *c.seq;
        bool good = *reinterpret_cast<volatile unsigned int *>(c.err) == 0u;   // one time-out ends all later waits
        if (good && (int)threadIdx.x < c.world && (int)threadIdx.x != c.rank) {
            const unsigned long long *f = c.flags[c.rank] + threadIdx.x;
            const unsigned long long t0 = global_ns();
            while (ld_acquire_sys(f) < want) {
                if (global_ns() - t0 > kCommTimeoutNs) {
                    good = false;
                    atomicExch(c.err, 1u);
                    break;
                }
                __nanosleep(64);
            }
        }
        good = __all_sync(0xffffffffu, good);
        if (threadIdx.x == 0) ok = good ? 1 : 0;
    }
    __syncthreads();
    if (!ok) return;
    const size_t slot_offset = (size_t)((*c.seq % kCommSlots) * c.slot_doubles);
    const int total = R * stride;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
        const int r = t / stride, v = t - r * stride;
        double acc = 0.0;
        const int64_t lo = offsets[r], hi = offsets[r + 1];
        if (v < nv && hi > lo) {
            int q0 = 0, q1 = c.world - 1;
            while (c.bounds[q0 + 1] <= lo) ++q0;
            while (c.bounds[q1] >= hi) --q1;
            for (int q = q0; q <= q1; ++q) {
                const double x = ld_relaxed_sys(c.arena[q] + slot_offset + t);
                acc = MAX ? fmax(acc, x) : acc + x;
            }
        }
        out[t] = acc;
    }
}

// Standalone bias / noise update (per-phase ABI entry; the sweep uses the fused tail of phase B).
template <int DY>
__global__ void __launch_bounds__(kThreadsB) k_bias_noise(StreamArgs p) {
    int lpr = 32;
    while (lpr > 1 && (kThreadsB / lpr) < p.R) lpr >>= 1;
    bias_noise_all<DY, kThreadsB>(p, lpr, blockIdx.x, gridDim.x);
}

// Shared noise and / or shared bias (noise_region_specific / bias_region_specific False, MRGP.py:27-28): the three
// other variants of Posteriors.py:81-211 (ci) and 345-475 (fi), from the per-region sums [sum r_d, sum |r|^2,
// sum f_var, sum phi^2 cm2] left in sumsB.  A shared posterior is stored once per region (all entries equal), so
// every consumer - P1, the ELBO (whose terms the reference also adds once per region, MRGP.py:426-475), prediction -
// reads it as before.  y_var is multiplied by the region's sample count except where the reference does not
// (Posteriors.py:138, 422).  One block; sums over the regions in a fixed order.
template <int DY>
__global__ void __launch_bounds__(256) k_bias_noise_shared(StreamArgs p) {
    __shared__ double red[256];
    __shared__ double sh[DY + 4];
    const int tid = threadIdx.x, R = p.R;
    auto block_sum = [&](double v) {
        red[tid] = v;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (tid < o) red[tid] += red[tid + o];
            __syncthreads();
        }
        const double t = red[0];
        __syncthreads();
        return t;
    };
    const double n_all = (double)(p.offsets[R] - p.offsets[0]);
    // ---- bias (Posteriors.py:81-110 / 345-374) --------------------------------------------------------------
    if (!p.bias_rs) {
        double S[DY];
        for (int d = 0; d < DY; ++d) {
            double v = 0.0;
            for (int r = tid; r < R; r += 256) v += p.sumsB[(size_t)r * (DY + 3) + d];
            S[d] = block_sum(v);
        }
        if (tid == 0) {
            const double bp0 = p.bias_prec0[0], bp = bp0 + n_all;
            double t3 = 0.0, t4 = 0.0;
            for (int d = 0; d < DY; ++d) {
                const double m0 = p.bias_mean0[d], m = (1.0 / bp) * (m0 * bp0 + S[d]);
                sh[d] = m;
                t3 += m0 * m0;
                t4 += m * m;
            }
            sh[DY] = bp;
            sh[DY + 1] = bp0 * t3;
            sh[DY + 2] = bp * t4;
        }
        __syncthreads();
    }
    // ---- per region: bias posterior, the bracket of the noise scale -------------------------------------------
    const bool times_n = !p.noise_rs || (p.ci ? !p.bias_rs : p.bias_rs);
    double bracket_sum = 0.0;
    for (int r = tid; r < R; r += 256) {
        const double n = (double)(p.offsets[r + 1] - p.offsets[r]);
        const double *sums = p.sumsB + (size_t)r * (DY + 3);
        double bp, t3, t4;
        if (p.bias_rs) {
            const double bp0 = p.bias_prec0[r];
            bp = bp0 + n;
            t3 = t4 = 0.0;
            for (int d = 0; d < DY; ++d) {
                const double m0 = p.bias_mean0[(size_t)r * DY + d], m = (1.0 / bp) * (m0 * bp0 + sums[d]);
                p.bias_prev_out[(size_t)r * DY + d] = p.bias_mean_out[(size_t)r * DY + d];
                p.bias_mean_out[(size_t)r * DY + d] = m;
                t3 += m0 * m0;
                t4 += m * m;
            }
            t3 *= bp0;
            t4 *= bp;
        } else {
            bp = sh[DY];
            t3 = sh[DY + 1];
            t4 = sh[DY + 2];
            for (int d = 0; d < DY; ++d) {
                p.bias_prev_out[(size_t)r * DY + d] = p.bias_mean_out[(size_t)r * DY + d];
                p.bias_mean_out[(size_t)r * DY + d] = sh[d];
            }
        }
        p.bias_prec[r] = bp;
        p.bias_var[r] = 1.0 / bp;
        const double yvar = p.infer ? 1.0 / p.noise_mean[r] : 0.0;
        p.yvar[r] = yvar;
        const double yv = times_n ? yvar * n : yvar;
        double bracket;
        if (!p.noise_rs && !p.bias_rs)
            bracket = sums[DY] + sums[DY + 1] + sums[DY + 2] + yv;      // the bias terms enter once (Posteriors.py:189-211)
        else
            bracket = t3 - t4 + sums[DY] + sums[DY + 1] + sums[DY + 2] + yv;
        if (p.noise_rs) {
            const double shape = p.noise_shape0[r] + 0.5 * (double)DY * n;
            const double scale = p.noise_scale0[r] + 0.5 * bracket;
            p.noise_shape[r] = shape;
            p.noise_scale[r] = scale;
            p.noise_mean[r] = shape / scale;
            p.noise_log_mean[r] = digamma(shape) - log(scale);
        } else {
            bracket_sum += bracket;
        }
    }
    if (!p.noise_rs) {
        double total = block_sum(bracket_sum);
        if (!p.bias_rs) total += sh[DY + 1] - sh[DY + 2];
        const double shape = p.noise_shape0[0] + 0.5 * (double)DY * n_all;
        const double scale = p.noise_scale0[0] + 0.5 * total;
        const double mean = shape / scale, lmean = digamma(shape) - log(scale);
        for (int r = tid; r < R; r += 256) {
            p.noise_shape[r] = shape;
            p.noise_scale[r] = scale;
            p.noise_mean[r] = mean;
            p.noise_log_mean[r] = lmean;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// B1: per-region optimisation of the basis half-interval L (BasisInterval.py:18-134, ci mode, dx == 1).
// All regions of a layer run the bounded Brent minimiser of SciPy's fminbound in lock-step (the reference calls
// scipy.optimize.fminbound(h, lo, hi) per region, BasisInterval.py:85-90; `_minimize_scalar_bounded`, xatol 1e-5,
// maxfun 500, is transcribed step for step in k_brent_step because the returned L sits within xatol of a bracket
// edge and only identical steps reproduce it, SURVEY.md App. D).  One iteration = one streaming evaluation of the
// data part of the objective for every region at its own trial L (k_interval_objective) + one small kernel that
// adds the prior part, consumes the value and proposes the next trial point.
//   h(L) = 1/2 noise sum_n [ sum_i (2|a_i|^2 + cm2_i) phi_i(n; L)^2 + (Phi(L) A^T)_n . (4 (b + fbar_n) - 2 y_n) ]
//          + 1/2 sum_i (log S_i(L) - 1/2 ard_mean_i m2_i / S_i(L))                       (BasisInterval.py:94-134)
// with the NEW a, m2, cm2, b, noise of the layer step and y the targets of the step (for inferred targets the
// layer's own prediction with the OLD coefficients and the OLD interval, LatentOutputs.py:25-49).
// ------------------------------------------------------------------------------------------------
struct BrentState {   // one per region, SoA in the workspace: field f of region r at st[f * R + r]
    enum { A = 0, B, FULC, NFC, XF, RAT, E, X, FX, FFULC, FNFC, XM, TOL1, TOL2, NUM, DONE, NFIELDS };
};

struct IntervalArgs {
    StreamArgs s;
    const double *trial_inv2L, *trial_rsqrtL;   // (R) trial interval of every region
    const double *w;                             // (R, M) 2 |a_i|^2 + cm2_i
    const double *bias_old;                      // (R, DY) bias used by the targets of the step
};

template <int DY, int M, bool INFER, bool LATENT>
__global__ void __launch_bounds__(kThreads) k_interval_objective(IntervalArgs q) {
    const StreamArgs &p = q.s;
    __shared__ double sA[M * DY], sAo[INFER ? M * DY : 1], sW[M], sScal[4 + 3 * DY], sRed[64];
    const int tid = threadIdx.x;
    double acc[1] = {0.0};
    const int s0 = p.cta_seg[blockIdx.x], s1 = p.cta_seg[blockIdx.x + 1];
    for (int s = s0; s < s1; ++s) {
        const Segment sg = p.segs[s];
        __syncthreads();
        if (tid < M * DY) {
            const bool real = tid < p.n_basis * DY;
            sA[tid] = real ? p.A[(size_t)sg.region * (p.n_basis * DY) + tid] : 0.0;
            if (INFER) sAo[tid] = real ? p.A_prev[(size_t)sg.region * (p.n_basis * DY) + tid] : 0.0;
        }
        if (tid < M) sW[tid] = tid < p.n_basis ? q.w[(size_t)sg.region * p.n_basis + tid] : 0.0;
        if (tid == 0) {
            sScal[0] = q.trial_inv2L[sg.region];
            sScal[1] = q.trial_rsqrtL[sg.region];
            sScal[2] = p.inv2L[sg.region];
            sScal[3] = p.rsqrtL[sg.region];
        }
        if (tid < DY) {
            sScal[4 + tid] = p.bias[(size_t)sg.region * DY + tid];                      // new bias
            sScal[4 + DY + tid] = q.bias_old[(size_t)sg.region * DY + tid];             // bias of the targets
            sScal[4 + 2 * DY + tid] = LATENT ? p.pbias[(size_t)sg.parent * DY + tid] : 0.0;
        }
        __syncthreads();
        const double ti2L = sScal[0], trs = sScal[1], oi2L = sScal[2], ors = sScal[3];
        const int64_t end = sg.start + sg.len;
        for (int64_t n = sg.start + tid; n < end; n += kThreads) {
            asm volatile("" ::: "memory");
            const double x = p.x[n];
            double f1, c2;
            basis_seed(x, ti2L, trs, f1, c2);
            double fm = 0.0, f = f1, e[DY], qv = 0.0;
#pragma unroll
            for (int d = 0; d < DY; ++d) e[d] = 0.0;
#pragma unroll 5
            for (int i = 0; i < M; ++i) {
#pragma unroll
                for (int d = 0; d < DY; ++d) e[d] = fma(f, sA[i * DY + d], e[d]);
                qv = fma(f * sW[i], f, qv);
                const double fn = fma(c2, f, -fm);
                fm = f;
                f = fn;
            }
            double eo[DY];
#pragma unroll
            for (int d = 0; d < DY; ++d) eo[d] = 0.0;
            if (INFER) {
                basis_seed(x, oi2L, ors, f1, c2);
                fm = 0.0;
                f = f1;
#pragma unroll 5
                for (int i = 0; i < M; ++i) {
#pragma unroll
                    for (int d = 0; d < DY; ++d) eo[d] = fma(f, sAo[i * DY + d], eo[d]);
                    const double fn = fma(c2, f, -fm);
                    fm = f;
                    f = fn;
                }
            }
            double dot = 0.0;
#pragma unroll
            for (int d = 0; d < DY; ++d) {
                const double fb = LATENT ? p.g[n * DY + d] + sScal[4 + 2 * DY + d] : 0.0;
                const double y = INFER ? eo[d] + (sScal[4 + DY + d] + fb) : p.y[n * DY + d];
                dot = fma(e[d], 4.0 * (sScal[4 + d] + fb) - 2.0 * y, dot);
            }
            acc[0] += qv + dot;
        }
        if (sg.flush) {
            block_reduce_small<1, false>(acc, sRed, p.part + (size_t)sg.run * p.part_stride);
            acc[0] = 0.0;
        }
    }
}

// Lower bound under adaptive intervals (MRGP.py:535-569 after MRGP.py:632-641): the data term is evaluated with the
// RE-LEARNT basis of the layer while its targets were inferred with the basis of the beginning of the step
// (LatentOutputs.py:20-49).  One pass per adaptive layer, after the rebuild and before the propagation:
//   r = target - Phi_new A^T - fbar,  target = Phi_old A_prev^T + b_old + fbar (or y on layer 0);
//   partial = [sum r_d, sum |r|^2, sum f_var, sum_i phi_new,i^2 cm2_i]   -> per-region sums for k_elbo.
template <int DY, int M, bool INFER, bool LATENT>
__global__ void __launch_bounds__(kThreads) k_adaptive_elbo_sums(IntervalArgs q) {
    const StreamArgs &p = q.s;
    __shared__ double sA[M * DY], sAo[INFER ? M * DY : 1], sW[M], sScal[5 + 3 * DY], sRed[64];
    const int tid = threadIdx.x;
    double acc[DY + 3];
#pragma unroll
    for (int d = 0; d < DY + 3; ++d) acc[d] = 0.0;
    const int s0 = p.cta_seg[blockIdx.x], s1 = p.cta_seg[blockIdx.x + 1];
    for (int s = s0; s < s1; ++s) {
        const Segment sg = p.segs[s];
        __syncthreads();
        if (tid < M * DY) {
            const bool real = tid < p.n_basis * DY;
            sA[tid] = real ? p.A[(size_t)sg.region * (p.n_basis * DY) + tid] : 0.0;
            if (INFER) sAo[tid] = real ? p.A_prev[(size_t)sg.region * (p.n_basis * DY) + tid] : 0.0;
        }
        if (tid < M) sW[tid] = tid < p.n_basis ? p.cm2[(size_t)sg.region * p.n_basis + tid] : 0.0;
        if (tid == 0) {
            sScal[0] = p.inv2L[sg.region];              // re-learnt interval
            sScal[1] = p.rsqrtL[sg.region];
            sScal[2] = q.trial_inv2L[sg.region];        // here: the interval of the beginning of the step
            sScal[3] = q.trial_rsqrtL[sg.region];
            sScal[4] = LATENT ? p.pbias_var[sg.parent] : 0.0;
        }
        if (tid < DY) {
            sScal[5 + tid] = q.bias_old[(size_t)sg.region * DY + tid];             // bias of the targets
            sScal[5 + DY + tid] = LATENT ? p.pbias[(size_t)sg.parent * DY + tid] : 0.0;
        }
        __syncthreads();
        const double ni2L = sScal[0], nrs = sScal[1], oi2L = sScal[2], ors = sScal[3], pbv = sScal[4];
        const int64_t end = sg.start + sg.len;
        for (int64_t n = sg.start + tid; n < end; n += kThreads) {
            asm volatile("" ::: "memory");
            const double x = p.x[n];
            double f1, c2;
            basis_seed(x, ni2L, nrs, f1, c2);
            double fm = 0.0, f = f1, e[DY], v = 0.0;
#pragma unroll
            for (int d = 0; d < DY; ++d) e[d] = 0.0;
#pragma unroll 5
            for (int i = 0; i < M; ++i) {
#pragma unroll
                for (int d = 0; d < DY; ++d) e[d] = fma(f, sA[i * DY + d], e[d]);
                v = fma(f * sW[i], f, v);
                const double fn = fma(c2, f, -fm);
                fm = f;
                f = fn;
            }
            double eo[DY];
#pragma unroll
            for (int d = 0; d < DY; ++d) eo[d] = 0.0;
            if (INFER) {
                basis_seed(x, oi2L, ors, f1, c2);
                fm = 0.0;
                f = f1;
#pragma unroll 5
                for (int i = 0; i < M; ++i) {
#pragma unroll
                    for (int d = 0; d < DY; ++d) eo[d] = fma(f, sAo[i * DY + d], eo[d]);
                    const double fn = fma(c2, f, -fm);
                    fm = f;
                    f = fn;
                }
            }
            double rr = 0.0;
#pragma unroll
            for (int d = 0; d < DY; ++d) {
                const double fb = LATENT ? p.g[n * DY + d] + sScal[5 + DY + d] : 0.0;
                const double target = INFER ? eo[d] + (sScal[5 + d] + fb) : p.y[n * DY + d];
                const double r = (target - e[d]) - fb;
                acc[d] += r;
                rr = fma(r, r, rr);
            }
            acc[DY] += rr;
            acc[DY + 1] += LATENT ? p.h[n] + pbv : 0.0;
            acc[DY + 2] += v;
        }
        if (sg.flush) {
            block_reduce_small<DY + 3, false>(acc, sRed, p.part + (size_t)sg.run * p.part_stride);
#pragma unroll
            for (int d = 0; d < DY + 3; ++d) acc[d] = 0.0;
        }
    }
}

struct BrentArgs {
    int32_t R, M, first;          // first: 1 = the value just computed is f(x0) of the initial point
    const int32_t *region_run;
    const double *part;
    int32_t part_stride;
    double *st;                   // BrentState fields
    double *trial_inv2L, *trial_rsqrtL;
    const double *noise_mean, *ard_mean, *m2;   // (R), (M), (R, M)
    int32_t use_prior;
    double nu, ell, sf, xatol;
    int32_t maxfun;
};

// One warp per region.  Step-exact transcription of scipy.optimize._optimize._minimize_scalar_bounded (SciPy 1.18.1),
// required for parity (SURVEY.md App. D).  That routine is
//   Copyright (c) 2001-2002 Enthought, Inc. 2003, SciPy Developers.  All rights reserved.
//   Redistribution and use in source and binary forms, with or without modification, are permitted provided that the
//   following conditions are met: 1. Redistributions of source code must retain the above copyright notice, this
//   list of conditions and the following disclaimer.  2. Redistributions in binary form must reproduce the above
//   copyright notice, this list of conditions and the following disclaimer in the documentation and/or other
//   materials provided with the distribution.  3. Neither the name of the copyright holder nor the names of its
//   contributors may be used to endorse or promote products derived from this software without specific prior
//   written permission.
//   THIS SOFTWARE IS PROVIDED BY THE COPYRIGHT HOLDERS AND CONTRIBUTORS "AS IS" AND ANY EXPRESS OR IMPLIED WARRANTIES,
//   INCLUDING, BUT NOT LIMITED TO, THE IMPLIED WARRANTIES OF MERCHANTABILITY AND FITNESS FOR A PARTICULAR PURPOSE ARE
//   DISCLAIMED.  IN NO EVENT SHALL THE COPYRIGHT OWNER OR CONTRIBUTORS BE LIABLE FOR ANY DIRECT, INDIRECT, INCIDENTAL,
//   SPECIAL, EXEMPLARY, OR CONSEQUENTIAL DAMAGES (INCLUDING, BUT NOT LIMITED TO, PROCUREMENT OF SUBSTITUTE GOODS OR
//   SERVICES; LOSS OF USE, DATA, OR PROFITS; OR BUSINESS INTERRUPTION) HOWEVER CAUSED AND ON ANY THEORY OF LIABILITY,
//   WHETHER IN CONTRACT, STRICT LIABILITY, OR TORT (INCLUDING NEGLIGENCE OR OTHERWISE) ARISING IN ANY WAY OUT OF THE
//   USE OF THIS SOFTWARE, EVEN IF ADVISED OF THE POSSIBILITY OF SUCH DAMAGE.                    (BSD 3-clause, SciPy)
__global__ void k_brent_step(BrentArgs a) {
    using B = BrentState;
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= a.R) return;
    double *st = a.st;
    const int R = a.R;
#define ST(f) st[(size_t)(B::f) * R + r]
    if (ST(DONE) != 0.0) return;
    const double x = ST(X);
    // ---- objective at the trial point: data part from the run partials, prior part here --------------------------
    double data = 0.0;
    for (int q = a.region_run[r] + lane; q < a.region_run[r + 1]; q += 32) data += a.part[(size_t)q * a.part_stride];
    data = warp_sum(data);
    double prior = 0.0;
    if (a.use_prior)
        for (int i = lane; i < a.M; i += 32) {
            const double w = (kPi * (double)(i + 1)) / (2.0 * x);
            const double S = matern_spectral(w * w + 0.0, a.nu, a.ell, a.sf);   // lambda_penalty == 0 for dx == 1
            prior += log(S) - 0.5 * (a.ard_mean[i] * a.m2[(size_t)r * a.M + i]) / S;
        }
    prior = warp_sum(prior);
    const double ll = -0.5 * a.noise_mean[r] * data;
    const double fval = a.use_prior ? -(ll + -0.5 * prior) : -ll;
    if (lane != 0) return;
    const double sqrt_eps = sqrt(2.2e-16);
    const double golden_mean = 0.5 * (3.0 - sqrt(5.0));
    double av = ST(A), bv = ST(B), fulc = ST(FULC), nfc = ST(NFC), xf = ST(XF), rat = ST(RAT), e = ST(E);
    double fx = ST(FX), ffulc = ST(FFULC), fnfc = ST(FNFC), xm = ST(XM), tol1 = ST(TOL1), tol2 = ST(TOL2);
    double num = ST(NUM);
    if (a.first) {
        fx = fval;
        num = 1.0;
        ffulc = fnfc = fx;
        xm = 0.5 * (av + bv);
        tol1 = sqrt_eps * fabs(xf) + a.xatol / 3.0;
        tol2 = 2.0 * tol1;
    } else {
        const double fu = fval;
        num += 1.0;
        if (fu <= fx) {
            if (x >= xf)
                av = xf;
            else
                bv = xf;
            fulc = nfc;
            ffulc = fnfc;
            nfc = xf;
            fnfc = fx;
            xf = x;
            fx = fu;
        } else {
            if (x < xf)
                av = x;
            else
                bv = x;
            if ((fu <= fnfc) || (nfc == xf)) {
                fulc = nfc;
                ffulc = fnfc;
                nfc = x;
                fnfc = fu;
            } else if ((fu <= ffulc) || (fulc == xf) || (fulc == nfc)) {
                fulc = x;
                ffulc = fu;
            }
        }
        xm = 0.5 * (av + bv);
        tol1 = sqrt_eps * fabs(xf) + a.xatol / 3.0;
        tol2 = 2.0 * tol1;
        if (num >= (double)a.maxfun) ST(DONE) = 1.0;
    }
    double xn = x;
    if (ST(DONE) == 0.0) {
        if (!(fabs(xf - xm) > (tol2 - 0.5 * (bv - av)))) {
            ST(DONE) = 1.0;   // while-condition false: converged, xf is the answer
        } else {
            bool golden = true;
            if (fabs(e) > tol1) {   // parabolic fit
                golden = false;
                double rr = (xf - nfc) * (fx - ffulc);
                double qq = (xf - fulc) * (fx - fnfc);
                double pp = (xf - fulc) * qq - (xf - nfc) * rr;
                qq = 2.0 * (qq - rr);
                if (qq > 0.0) pp = -pp;
                qq = fabs(qq);
                rr = e;
                e = rat;
                if ((fabs(pp) < fabs(0.5 * qq * rr)) && (pp > qq * (av - xf)) && (pp < qq * (bv - xf))) {
                    rat = (pp + 0.0) / qq;
                    xn = xf + rat;
                    if (((xn - av) < tol2) || ((bv - xn) < tol2)) {
                        const double d = xm - xf;
                        const double si = (d > 0.0 ? 1.0 : (d < 0.0 ? -1.0 : 0.0)) + (d == 0.0 ? 1.0 : 0.0);
                        rat = tol1 * si;
                    }
                } else {
                    golden = true;
                }
            }
            if (golden) {
                e = (xf >= xm) ? av - xf : bv - xf;
                rat = golden_mean * e;
            }
            const double si = (rat > 0.0 ? 1.0 : (rat < 0.0 ? -1.0 : 0.0)) + (rat == 0.0 ? 1.0 : 0.0);
            xn = xf + si * fmax(fabs(rat), tol1);
        }
    }
    ST(A) = av;
    ST(B) = bv;
    ST(FULC) = fulc;
    ST(NFC) = nfc;
    ST(XF) = xf;
    ST(RAT) = rat;
    ST(E) = e;
    ST(X) = xn;
    ST(FX) = fx;
    ST(FFULC) = ffulc;
    ST(FNFC) = fnfc;
    ST(XM) = xm;
    ST(TOL1) = tol1;
    ST(TOL2) = tol2;
    ST(NUM) = num;
    a.trial_inv2L[r] = 0.5 / xn;
    a.trial_rsqrtL[r] = 1.0 / sqrt(xn);
#undef ST
}

// Bracket and first trial point of every region (BasisInterval.py:77-84 and the head of the minimiser); also
// w = 2 |a_i|^2 + cm2_i.  absx = max|x| of the region.
__global__ void k_brent_start(BrentArgs a, const double *absx, double f_lo, double f_hi, const double *A, const double *cm2, double *w) {
    using B = BrentState;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int R = a.R, M = a.M;
    if (t < R * M) w[t] = 2.0 * (A[(size_t)t * 2] * A[(size_t)t * 2] + A[(size_t)t * 2 + 1] * A[(size_t)t * 2 + 1]) + cm2[t];
    if (t >= R) return;
    const int r = t;
    const double lo = absx[r] * f_lo;
    double hi = fmin((double)M, lo * f_hi);
    if (hi < lo) hi = lo * f_hi;
    const double golden_mean = 0.5 * (3.0 - sqrt(5.0));
    const double fulc = lo + golden_mean * (hi - lo);
    double *st = a.st;
#define ST(f) st[(size_t)(B::f) * R + r]
    ST(A) = lo;
    ST(B) = hi;
    ST(FULC) = fulc;
    ST(NFC) = fulc;
    ST(XF) = fulc;
    ST(RAT) = 0.0;
    ST(E) = 0.0;
    ST(X) = fulc;
    ST(FX) = 0.0;
    ST(FFULC) = 0.0;
    ST(FNFC) = 0.0;
    ST(XM) = 0.0;
    ST(TOL1) = 0.0;
    ST(TOL2) = 0.0;
    ST(NUM) = 0.0;
    ST(DONE) = 0.0;
#undef ST
    a.trial_inv2L[r] = 0.5 / fulc;
    a.trial_rsqrtL[r] = 1.0 / sqrt(fulc);
}

// The optimum of every region becomes its interval; counts the regions that did not converge.
__global__ void k_brent_finish(BrentArgs a, double *L, unsigned long long *not_converged) {
    using B = BrentState;
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.R) return;
    L[r] = a.st[(size_t)B::XF * a.R + r];
    if (a.st[(size_t)B::DONE * a.R + r] == 0.0) atomicAdd(not_converged, 1ull);
}

// ------------------------------------------------------------------------------------------------
// prediction and latent export (not on the sweep path): region found by binary search on offsets
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int find_region(const int64_t *off, int R, int64_t n) {
    int lo = 0, hi = R;   // off[lo] <= n < off[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (off[mid] <= n)
            lo = mid;
        else
            hi = mid;
    }
    return lo;
}

struct EvalLayer {
    const int64_t *offsets;   // region offsets used to assign sample positions to regions
    const double *inv2L, *rsqrtL, *A, *cm2, *bias, *bias_var, *noise_mean;
    int32_t R;
};

constexpr int kMaxLayers = 24;
struct EvalArgs {
    EvalLayer layer[kMaxLayers];
    int32_t n_layers;
    int32_t M;
    int64_t n;
    const double *x;
    double *out_mean;   // (n, DY) or null
    double *out_var;    // (n) or null
    int32_t single_region;   // 1: every point uses region 0 of layer 0 (MRGP.py:726-755, 833-861)
};

// out_mean = sum_j (Phi_j A_j^T + b_j), out_var = sum_j (bias_var_j + sum_i phi_i^2 cm2_ji) over the
// given layers (MRGP.py:782-803; Stats.py:126-157 when used to export the latent functions).
template <int DY>
__global__ void k_eval_layers(EvalArgs a) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= a.n) return;
    const double x = a.x[n];
    double mean[DY], var = 0.0;
#pragma unroll
    for (int d = 0; d < DY; ++d) mean[d] = 0.0;
    for (int j = 0; j < a.n_layers; ++j) {
        const EvalLayer &ly = a.layer[j];
        const int r = a.single_region ? 0 : find_region(ly.offsets, ly.R, n);
        double f1, c2;
        basis_seed(x, ly.inv2L[r], ly.rsqrtL[r], f1, c2);
        double fm = 0.0, f = f1, e[DY], v = 0.0;
#pragma unroll
        for (int d = 0; d < DY; ++d) e[d] = 0.0;
        const double *A = ly.A + (size_t)r * a.M * DY;
        const double *C = ly.cm2 + (size_t)r * a.M;
        for (int i = 0; i < a.M; ++i) {
#pragma unroll
            for (int d = 0; d < DY; ++d) e[d] = fma(f, A[i * DY + d], e[d]);
            v = fma(f * C[i], f, v);
            const double fn = fma(c2, f, -fm);
            fm = f;
            f = fn;
        }
#pragma unroll
        for (int d = 0; d < DY; ++d) mean[d] += ly.bias[(size_t)r * DY + d] + e[d];
        var += ly.bias_var[r] + v;
    }
    if (a.out_mean)
#pragma unroll
        for (int d = 0; d < DY; ++d) a.out_mean[n * DY + d] = mean[d];
    if (a.out_var) a.out_var[n] = var;
}

// Pull a byte range into L2 (one prefetch per 128-byte line, nothing waits on it).
__global__ void k_prefetch_l2(const char *base, size_t lines) {
    for (size_t l = (size_t)blockIdx.x * blockDim.x + threadIdx.x; l < lines; l += (size_t)gridDim.x * blockDim.x)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + l * 128));
}

// ------------------------------------------------------------------------------------------------
// Closed-form statistics of the ci layers above the first (static intervals).
//
// Such a layer regresses on targets inferred from its own posterior, y = Phi A_old + b_old + fbar
// (LatentOutputs.py:20-49), so every per-sample quantity the P4 / P5 statistics add up (Posteriors.py:81-93,
// 132-148) is a polynomial in the region's coefficients with basis-only weights:
//     r_n = y_n - Phi_n A_new - fbar_n = Phi_n (A_old - A_new) + b_old
//     sum_n r_d   = sum_i s_i dA_id + n b_old,d                                   s_i  = sum_n phi_i(n)
//     sum_n |r|^2 = sum_d dA_d^T G dA_d + 2 b_old . (s^T dA) + n |b_old|^2         G    = Phi^T Phi
//     sum_n fvar  = sum_{jp<j} (n bias_var_jp,anc + sum_i cm2_jp,anc,i D_jp,i)     D_jp = sum_n phi^jp_i(n)^2
//     sum_n sum_i phi_i^2 cm2_i = sum_i d_i cm2_i
// (for regions nested in the coarser layer jp; in general the last sum runs over the pieces region x coarser
// region, each with its own anc and D, see PieceTable).  s, G and D depend on
// x and the basis intervals only: they are built once (k_build_gram, k_build_ancD) and the layer's statistics
// become O(R M^2) work instead of a pass over the samples.  With the non-informative initialisation dA == 0 and
// b_old == 0 exactly (the layers are inert, SURVEY.md §8c) and the first two sums are exact zeros in both forms.
// ------------------------------------------------------------------------------------------------
constexpr int kGramRows = 128;

template <int M>
__global__ void __launch_bounds__(256) k_build_gram(const double *x, const int64_t *offsets, const double *inv2L, const double *rsqrtL,
                                                    int splits, double *partial /* [blocks][NP + M] */) {
    constexpr int NP = M * (M + 1) / 2, NQ = (NP + 255) / 256;
    constexpr int kRows = M > 40 ? 96 : kGramRows;   // 48 KB of static shared memory
    __shared__ double sPhi[kRows][M + 1];
    __shared__ unsigned char sI[NP], sK[NP];
    const int tid = threadIdx.x, blk = blockIdx.x, c = blk / splits, sp = blk % splits;
    for (int p = tid; p < NP; p += 256) {   // pair p = (i, k), i <= k, rows of the upper triangle one after the other
        int i = 0, rem = p;
        while (rem >= M - i) {
            rem -= M - i;
            ++i;
        }
        sI[p] = (unsigned char)i;
        sK[p] = (unsigned char)(i + rem);
    }
    const int64_t lo = offsets[c], hi = offsets[c + 1];
    const int64_t per = (hi - lo + splits - 1) / splits;
    const int64_t a = lo + sp * per, b = (a + per < hi) ? a + per : hi;
    const double i2 = inv2L[c], rs = rsqrtL[c];
    double acc[NQ], sacc = 0.0;
#pragma unroll
    for (int q = 0; q < NQ; ++q) acc[q] = 0.0;
    __syncthreads();
    for (int64_t base = a; base < b; base += kRows) {
        if (tid < kRows) {
            const int64_t n = base + tid;
            if (n < b) {
                double f1, c2;
                basis_seed(x[n], i2, rs, f1, c2);
                double fm = 0.0, f = f1;
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    sPhi[tid][i] = f;
                    const double fn = fma(c2, f, -fm);
                    fm = f;
                    f = fn;
                }
            } else {
#pragma unroll
                for (int i = 0; i < M; ++i) sPhi[tid][i] = 0.0;
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const int p = tid + q * 256;
            if (p < NP) {
                const int i = sI[p], k = sK[p];
                double t0 = 0.0, t1 = 0.0;
#pragma unroll 8
                for (int r = 0; r < kRows; r += 2) {
                    t0 = fma(sPhi[r][i], sPhi[r][k], t0);
                    t1 = fma(sPhi[r + 1][i], sPhi[r + 1][k], t1);
                }
                acc[q] += t0 + t1;
            }
        }
        if (tid < M) {
            double t = 0.0;
            for (int r = 0; r < kRows; ++r) t += sPhi[r][tid];
            sacc += t;
        }
        __syncthreads();
    }
    double *out = partial + (size_t)blk * (NP + M);
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        const int p = tid + q * 256;
        if (p < NP) out[p] = acc[q];
    }
    if (tid < M) out[NP + tid] = sacc;
}

// G[c][i][k] (full, symmetric) and s[c][i] from the split partials, summed in split order.
// (MP: the padded number of basis functions of the partials; entries of the padding are dropped.)
__global__ void k_reduce_gram(const double *partial, int splits, int R, int M, int MP, double *G, double *s) {
    const int NP = MP * (MP + 1) / 2;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= R * (NP + MP)) return;
    const int c = t / (NP + MP), p = t % (NP + MP);
    int i = 0, k = 0;
    if (p >= NP) {
        if (p - NP >= M) return;
    } else {
        int rem = p;
        while (rem >= MP - i) {
            rem -= MP - i;
            ++i;
        }
        k = i + rem;
        if (k >= M) return;
    }
    double acc = 0.0;
    for (int sp = 0; sp < splits; ++sp) acc += partial[((size_t)c * splits + sp) * (NP + MP) + p];
    if (p >= NP) {
        s[(size_t)c * M + (p - NP)] = acc;
        return;
    }
    G[((size_t)c * M + i) * M + k] = acc;
    G[((size_t)c * M + k) * M + i] = acc;
}

// D[piece][i] = sum over the samples of the piece of the squared basis functions of its coarser layer.  A piece is
// the intersection of a region of the layer with a region of a coarser layer jp (regions need not be nested: the
// uniform index sets of the reference are not, IndexSetGenerator.py:25-42); blockIdx.x = (piece, split).
struct PieceTable {
    const int32_t *ptr;    // (n_anc, R + 1): pieces of (jp, region) are ptr[jp * (R + 1) + c] .. ptr[.. + 1]
    const int32_t *jp;     // (P) coarser layer of the piece
    const int32_t *anc;    // (P) region of that layer
    const int64_t *lo, *hi;   // (P) sample range
    int32_t P;
};

template <int M>
__global__ void __launch_bounds__(256) k_build_ancD(EvalArgs ea, const double *x, PieceTable pt, int splits, double *partial) {
    __shared__ double sW[8][M];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int blk = blockIdx.x, pc = blk / splits, sp = blk % splits;
    const EvalLayer &ly = ea.layer[pt.jp[pc]];
    const int anc = pt.anc[pc];
    const int64_t lo = pt.lo[pc], hi = pt.hi[pc];
    const double i2 = ly.inv2L[anc], rs = ly.rsqrtL[anc];
    const int64_t per = (hi - lo + splits - 1) / splits;
    const int64_t a = lo + sp * per, b = (a + per < hi) ? a + per : hi;
    double acc[M];
#pragma unroll
    for (int i = 0; i < M; ++i) acc[i] = 0.0;
    for (int64_t n = a + tid; n < b; n += 256) {
        double f1, c2;
        basis_seed(x[n], i2, rs, f1, c2);
        double fm = 0.0, f = f1;
#pragma unroll
        for (int i = 0; i < M; ++i) {
            acc[i] = fma(f, f, acc[i]);
            const double fn = fma(c2, f, -fm);
            fm = f;
            f = fn;
        }
    }
#pragma unroll
    for (int i = 0; i < M; ++i) {
        const double t = warp_sum(acc[i]);
        if (lane == 0) sW[warp][i] = t;
    }
    __syncthreads();
    if (tid < M) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sW[w][tid];
        partial[(size_t)blk * M + tid] = t;
    }
}

__global__ void k_reduce_ancD(const double *partial, int splits, int P, int M, int MP, double *D) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= P * M) return;
    const int i = t % M, pc = t / M;
    double acc = 0.0;
    for (int sp = 0; sp < splits; ++sp) acc += partial[((size_t)pc * splits + sp) * MP + i];
    D[t] = acc;
}

struct StatsBArgs {
    StreamArgs p;             // bias / noise fields of the layer
    EvalArgs anc;             // the coarser layers (cm2, bias_var, offsets)
    const double *s, *G, *D;  // invariants of the layer: (R, M), (R, M, M), (P, M)
    PieceTable pt;
    const double *A, *A_prev, *d, *cm2;
};

// One warp per region: the five sums of the header, then P4 / P5 / S5 for the region.
template <int DY>
__global__ void __launch_bounds__(256) k_stats_b(StatsBArgs q) {
    static_assert(DY == 2, "dy == 2 only");
    const StreamArgs &p = q.p;
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    ts_begin(p.ts, p.layer * 4 + 2);
    if (c < p.R) {
        const int M = q.anc.M;
        const double n = (double)(p.offsets[c + 1] - p.offsets[c]);
        // dA = A_old - A_new for this lane's basis functions (M <= 64: two per lane)
        double dA[2][2], sd0 = 0.0, sd1 = 0.0, dc = 0.0;
        bool any = false;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int i = lane + 32 * h;
            dA[h][0] = dA[h][1] = 0.0;
            if (i < M) {
                const size_t ri = (size_t)c * M + i;
                dA[h][0] = q.A_prev[ri * 2 + 0] - q.A[ri * 2 + 0];
                dA[h][1] = q.A_prev[ri * 2 + 1] - q.A[ri * 2 + 1];
                const double si = q.s[ri];
                sd0 = fma(si, dA[h][0], sd0);
                sd1 = fma(si, dA[h][1], sd1);
                dc = fma(q.d[ri], q.cm2[ri], dc);
                any = any || dA[h][0] != 0.0 || dA[h][1] != 0.0;
            }
        }
        sd0 = warp_sum(sd0);
        sd1 = warp_sum(sd1);
        dc = warp_sum(dc);
        double quad = 0.0;
        if (__any_sync(0xffffffffu, any)) {   // dA^T G dA, column i of the symmetric G per lane (coalesced rows)
            const double *G = q.G + (size_t)c * M * M;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int i = lane + 32 * h;
                double t0 = 0.0, t1 = 0.0;
                for (int k = 0; k < M; ++k) {
                    const double g = (i < M) ? G[(size_t)k * M + i] : 0.0;
                    const int src = k & 31;
                    const double a0 = __shfl_sync(0xffffffffu, (k < 32) ? dA[0][0] : dA[1][0], src);
                    const double a1 = __shfl_sync(0xffffffffu, (k < 32) ? dA[0][1] : dA[1][1], src);
                    t0 = fma(g, a0, t0);
                    t1 = fma(g, a1, t1);
                }
                quad += dA[h][0] * t0 + dA[h][1] * t1;
            }
            quad = warp_sum(quad);
        }
        double fv = 0.0;
        for (int jp = 0; jp < q.anc.n_layers; ++jp) {
            const EvalLayer &ly = q.anc.layer[jp];
            const int32_t *pp = q.pt.ptr + (size_t)jp * (p.R + 1) + c;
            for (int pc = pp[0]; pc < pp[1]; ++pc) {
                const int anc = q.pt.anc[pc];
                double t = 0.0;
                for (int i = lane; i < M; i += 32) t = fma(ly.cm2[(size_t)anc * M + i], q.D[(size_t)pc * M + i], t);
                fv += warp_sum(t) + (double)(q.pt.hi[pc] - q.pt.lo[pc]) * ly.bias_var[anc];
            }
        }
        if (lane == 0) {
            const double b0 = p.bias_mean_out[(size_t)c * 2 + 0], b1 = p.bias_mean_out[(size_t)c * 2 + 1];   // b_old
            double sums[DY + 3];
            sums[0] = sd0 + n * b0;
            sums[1] = sd1 + n * b1;
            sums[2] = quad + 2.0 * (b0 * sd0 + b1 * sd1) + n * (b0 * b0 + b1 * b1);
            sums[3] = fv;
            sums[4] = dc;
            bias_noise_region<DY>(p, c, sums);
        }
    }
    ts_end(p.ts, p.layer * 4 + 2);
}

// Index-set form of the predictive second moment (MRGP.py:863-932): per test point the sum over the layers of
//   sum_i phi_i^2 cm2_i + bias_var + n_test(region) / noise_mean + f_var(first test point of the region)
// where f_var is the latent variance of the coarser layers at that point (Stats.py:126-157; the reference adds
// `latent_f_var[l][0]`, the value of the region's FIRST sample, to every sample of the region, MRGP.py:929) and the
// squared-mean term of MRGP.py:928 vanishes identically (the targets are inferred from the same statistics).
template <int DY>
__device__ __forceinline__ double layer_var_at(const EvalLayer &ly, int M, int r, double x) {
    double f1, c2;
    basis_seed(x, ly.inv2L[r], ly.rsqrtL[r], f1, c2);
    double fm = 0.0, f = f1, v = 0.0;
    const double *Cm = ly.cm2 + (size_t)r * M;
    for (int i = 0; i < M; ++i) {
        v = fma(f * Cm[i], f, v);
        const double fn = fma(c2, f, -fm);
        fm = f;
        f = fn;
    }
    return v + ly.bias_var[r];
}

template <int DY>
__global__ void k_eval_var_indexed(EvalArgs a) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= a.n) return;
    const double x = a.x[n];
    double total = 0.0;
    for (int j = 0; j < a.n_layers; ++j) {
        const EvalLayer &ly = a.layer[j];
        const int r = find_region(ly.offsets, ly.R, n);
        const int64_t first = ly.offsets[r];
        total += layer_var_at<DY>(ly, a.M, r, x) + (double)(ly.offsets[r + 1] - first) / ly.noise_mean[r];
        const double xf = a.x[first];
        for (int jp = 0; jp < j; ++jp) {
            const EvalLayer &lp = a.layer[jp];
            total += layer_var_at<DY>(lp, a.M, find_region(lp.offsets, lp.R, first), xf);
        }
    }
    a.out_var[n] = total;
}

// ------------------------------------------------------------------------------------------------
// ELBO (MRGP.py:414-569), one block per layer.  prime == the shared prior for layer 0 and the CURRENT
// shared posterior for layers > 0 (alias at MRGP.py:379).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double block_sum_1024(double v, double *sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    v = warp_sum(v);
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    double t = 0.0;
    if (warp == 0) {
        t = (lane < (int)(blockDim.x >> 5)) ? sm[lane] : 0.0;
        t = warp_sum(t);
    }
    return t;   // valid in warp 0
}

// Grid (J, C): CTA (j, c) takes the regions [c kElboRegions, (c + 1) kElboRegions) of layer j (CTA (j, 0) also the terms
// of the shared posterior) and leaves six partial sums; the last CTA of a layer to finish adds the partials in chunk
// order (a fixed order: the bound is bit-reproducible).  One CTA per layer, as in round 1, walked the 512 regions x 30
// basis functions of the finest layer with 256 threads in a chain of dependent loads: 85 us after an L2 flush.
constexpr int kElboRegions = 32;
template <int DY>
__global__ void __launch_bounds__(256) k_elbo(const RegionArgs *layers, double *out /* (J, 6) */, double *part /* (J, C, 6) */,
                                              unsigned int *counter /* (J) */) {
    static_assert(DY == 2, "dy == 2 only");
    __shared__ double sm[32];
    __shared__ int sLast;
    const RegionArgs &a = layers[blockIdx.x];
    const int j = blockIdx.x, c = blockIdx.y, C = gridDim.y, M = a.M, R = a.R;
    const int r_lo = c * kElboRegions, r_hi = min(R, r_lo + kElboRegions);
    if (r_lo >= R) return;                                    // (not counted: the layer has ceil(R / kElboRegions) chunks)
    const int n_chunks = (R + kElboRegions - 1) / kElboRegions;
    const bool first = (j == 0);
    const double *pB = first ? a.priorB : a.axB;
    const double *pLogC = first ? a.priorLogC : a.axLogC;
    const double *pShape = first ? a.priorShape : a.ardShape;
    const double *pScale = first ? a.priorScale : a.ardScale;
    double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0, t4 = 0.0, t5 = 0.0;
    for (int r = r_lo + threadIdx.x; r < r_hi; r += blockDim.x) {
        const double n = (double)(a.offsets[r + 1] - a.offsets[r]);
        const double *sb = a.sumsB + (size_t)r * (DY + 3);
        double bb = 0.0, bs = 0.0, w0w0 = 0.0, ww0 = 0.0;
        for (int d = 0; d < DY; ++d) {
            const double b = a.bias_mean[(size_t)r * DY + d], b0 = a.bias_mean0[(size_t)r * DY + d];
            bb += b * b;
            bs += b * sb[d];
            w0w0 += b0 * b0;
            ww0 += b * b0;
        }
        // :535-569  sum |r - b|^2 = sum |r|^2 - 2 b . sum r + n |b|^2
        const double mean_term = sb[DY] - 2.0 * bs + n * bb;
        const double nlm = a.noise_log_mean[r], nm = a.noise_mean[r];
        t0 += mean_term + sb[DY + 1] + sb[DY + 2] + a.bias_var[r] + a.yvar[r] * n + 0.5 * DY * (nlm - kLog2Pi) * n;
        // :449-475
        const double tau = a.bias_prec[r], tau0 = a.bias_prec0[r];
        const double term1 = 1.0 / (tau * nm) + bb - 2.0 * ww0 + w0w0;
        t4 += (0.5 * DY * (log(tau0) + nlm - kLog2Pi) + 0.5 * tau0 * nm * term1) - (0.5 * DY * (log(tau) + nlm - kLog2Pi) - 0.5);
        // :426-447
        const double c0 = a.noise_shape0[r], d0 = a.noise_scale0[r], cc = a.noise_shape[r], d = a.noise_scale[r];
        t5 += (c0 * log(d0) - lgamma(c0) + (c0 - 1.0) * nlm - d0 * nm) - (cc * log(d) - lgamma(cc) + (cc - 1.0) * nlm - d * nm);
    }
    // :520-533
#pragma unroll 4
    for (int t = r_lo * M + threadIdx.x; t < r_hi * M; t += blockDim.x) {
        const int i = t % M;
        t1 += (0.5 * a.ardLogMean[i] / a.S[t] - 0.5 * a.ardMean[i] * a.m2[t] / a.S[t]) - (0.5 * log(a.prec[t]) - 0.5);
    }
    if (c == 0) {
        // :499-518 (element-wise product inside the trace -> diagonal entries only), :477-497
        for (int t = threadIdx.x; t < M * M; t += blockDim.x) {
            const int i = t / M, k = t % M;
            const double w = a.omega[t];
            t2 += w * (-pLogC[k] + a.axCov[i * 4 + 0] * pB[k * 4 + 0] + a.axCov[i * 4 + 3] * pB[k * 4 + 3]);
            t3 += w * (pShape[k] * log(pScale[k]) - lgamma(pShape[k]) + (pShape[k] - 1.0) * a.ardLogMean[i] - pScale[k] * a.ardMean[i]);
        }
        for (int i = threadIdx.x; i < M; i += blockDim.x) {
            t2 -= -a.axLogC[i] + a.axCov[i * 4 + 0] * a.axB[i * 4 + 0] + a.axCov[i * 4 + 3] * a.axB[i * 4 + 3];
            t3 -= a.ardShape[i] * log(a.ardScale[i]) - lgamma(a.ardShape[i]) + (a.ardShape[i] - 1.0) * a.ardLogMean[i] - a.ardScale[i] * a.ardMean[i];
        }
    }
    double vals[6] = {t0, t1, t2, t3, t4, t5};
    double *mine = part + ((size_t)j * C + c) * 6;
    for (int q = 0; q < 6; ++q) {
        const double s = block_sum_1024(vals[q], sm);
        if (threadIdx.x == 0) {
            mine[q] = s;
            if (n_chunks == 1) out[j * 6 + q] = s;
        }
    }
    if (n_chunks == 1) return;
    __syncthreads();
    if (threadIdx.x == 0) sLast = (atom_add_acq_rel_gpu(counter + j, 1u) == (unsigned)n_chunks - 1u);
    __syncthreads();
    if (sLast) {
        if (threadIdx.x < 6) {
            double s = 0.0;
            for (int k = 0; k < n_chunks; ++k) s += __ldcg(part + ((size_t)j * C + k) * 6 + threadIdx.x);
            out[j * 6 + threadIdx.x] = s;
        }
        if (threadIdx.x == 0) counter[j] = 0u;
    }
}

// ------------------------------------------------------------------------------------------------
// initialisation (Priors.py non-informative; Posteriors.py:10-30; Stats.py:8-62, 355-369)
// ------------------------------------------------------------------------------------------------
template <int DY>
__global__ void k_init_layer(RegionArgs a, double noise_var0, double ard_influence, double logc0, double rho0) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int M = a.M;
    if (t < a.R) {
        const int r = t;
        a.noise_shape0[r] = kEps;
        a.noise_scale0[r] = (kEps + 1.0) * noise_var0;
        a.noise_shape[r] = kEps;
        a.noise_scale[r] = (kEps + 1.0) * noise_var0;
        a.noise_mean[r] = kEps / ((kEps + 1.0) * noise_var0);
        a.noise_log_mean[r] = digamma(kEps) - log((kEps + 1.0) * noise_var0);
        a.bias_prec0[r] = kEps;
        a.bias_prec[r] = kEps;
        a.bias_var[r] = 1.0 / kEps;
        a.yvar[r] = 0.0;
        for (int d = 0; d < DY; ++d) {
            a.bias_mean0[(size_t)r * DY + d] = 0.0;
            a.bias_mean[(size_t)r * DY + d] = 0.0;
        }
        for (int d = 0; d < DY + 3; ++d) a.sumsB[(size_t)r * (DY + 3) + d] = 0.0;
        if (a.rconst) {   // what the fused sweep needs of the region besides its state (csrc/chain.cu, bias_noise_update)
            const double n = (double)(a.offsets[r + 1] - a.offsets[r]);
            double *rc = a.rconst + (size_t)r * 8;
            rc[0] = n;
            rc[1] = kEps;                                   // bias_prec0
            rc[2] = 0.0;                                    // bias_mean0
            rc[3] = 0.0;
            rc[4] = kEps;                                   // noise_shape0
            rc[5] = (kEps + 1.0) * noise_var0;              // noise_scale0
            rc[6] = digamma(kEps + 0.5 * (double)DY * n);   // psi(noise shape): the shape is c0 + dy n / 2 in every sweep
            rc[7] = 0.0;
        }
    }
    if (t < a.R * M) {
        a.prec[t] = 1.0 / a.S[t];
        a.zeta[t] = 0.0;
        a.m2[t] = 0.0;
        a.cm2[t] = 0.0;
        for (int d = 0; d < DY; ++d) {
            a.ytil[(size_t)t * DY + d] = 0.0;
            a.A[(size_t)t * DY + d] = 0.0;
            a.A_prev[(size_t)t * DY + d] = 0.0;
        }
        if (a.mode == 1) {
            for (int q = 0; q < DY * DY; ++q) {
                a.axB[(size_t)t * DY * DY + q] = 0.0;
                a.axCov[(size_t)t * DY * DY + q] = 0.0;
            }
            for (int d = 0; d < DY; ++d) {
                a.axKappa[(size_t)t * DY + d] = 0.0;
                a.axRho[(size_t)t * DY + d] = rho0;
            }
            a.axLogC[t] = logc0;
            a.ardShape[t] = kEps;
            a.ardScale[t] = kEps / ard_influence;
            a.ardMean[t] = kEps / (kEps / ard_influence);
            a.ardLogMean[t] = digamma(kEps) - log(kEps / ard_influence);
        }
    }
}

template <int DY>
__global__ void k_init_shared(RegionArgs a, double *priorB, double *priorLogC, double *priorShape, double *priorScale,
                              double ard_influence, double logc0, double rho0) {
    const int M = a.M;
    for (int t = threadIdx.x; t < M; t += blockDim.x) {
        for (int q = 0; q < DY * DY; ++q) {
            priorB[t * DY * DY + q] = 0.0;
            a.axB[t * DY * DY + q] = 0.0;
            a.axCov[t * DY * DY + q] = 0.0;
            a.primeB[t * DY * DY + q] = 0.0;
        }
        for (int d = 0; d < DY; ++d) {
            a.axKappa[t * DY + d] = 0.0;
            a.axRho[t * DY + d] = rho0;
        }
        priorLogC[t] = logc0;
        a.axLogC[t] = logc0;
        a.primeLogC[t] = logc0;
        priorShape[t] = kEps;
        priorScale[t] = kEps / ard_influence;
        a.ardShape[t] = kEps;
        a.ardScale[t] = kEps / ard_influence;
        a.primeShape[t] = kEps;
        a.primeScale[t] = kEps / ard_influence;
        a.ardMean[t] = kEps / (kEps / ard_influence);
        a.ardLogMean[t] = digamma(kEps) - log(kEps / ard_influence);
        a.primeSk[2 * 64 + t] = -logc0 + kEps * log(kEps / ard_influence) - lgamma(kEps);   // layer 0: the prior
    }
    if (threadIdx.x == 0) {
        a.skTag[0] = -1.0;
        a.skTag[1] = -1.0;
        a.skTag[2] = 0.0;
    }
    for (int t = threadIdx.x; t < M * M; t += blockDim.x) {
        a.omega[t] = 1.0 / (double)M;
        a.logOmegaHat[t] = 0.0;
    }
}

// ------------------------------------------------------------------------------------------------
// micro-benchmarks
// ------------------------------------------------------------------------------------------------

// Batched Cholesky (lower), one warp per n x n matrix (n <= 32): lane r owns row r; the pivot and the
// scaled column are broadcast with warp shuffles.  Mirrors LAPACK potrf's info convention.
__global__ void k_batched_cholesky(double *a, int n, int64_t batch, int32_t *info) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= batch) return;
    double *A = a + w * (int64_t)n * n;
    double row[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) row[c] = (lane < n && c < n && c <= lane) ? A[lane * n + c] : 0.0;
    int bad = 0;
#pragma unroll
    for (int k = 0; k < 32; ++k) {
        if (k < n) {
            double piv = __shfl_sync(0xffffffffu, row[k], k);
            if (!(piv > 0.0) && bad == 0) bad = k + 1;
            const double rp = (bad == 0) ? 1.0 / sqrt(piv) : 0.0;
            if (lane >= k) row[k] *= rp;   // column k of L
#pragma unroll
            for (int c = k + 1; c < 32; ++c) {
                const double lck = __shfl_sync(0xffffffffu, row[k], c);   // L[c][k]
                if (c < n && lane >= c) row[c] = fma(-row[k], lck, row[c]);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < 32; ++c)
        if (lane < n && c < n && c <= lane) A[lane * n + c] = row[c];
    if (lane == 0) info[w] = bad;
}

// Small matrices (n <= 8): one THREAD per matrix, the factor in registers (a warp per 2 x 2 matrix would leave 31 lanes
// idle; the PD guard of the model, SanityCheck.py:59-65, is this case with n = dy).  Same conventions as above.
template <int N>
__global__ void __launch_bounds__(256) k_batched_cholesky_small(double *a, int64_t batch, int32_t *info) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    double *A = a + b * (N * N);
    double L[N][N];
#pragma unroll
    for (int r = 0; r < N; ++r)
#pragma unroll
        for (int c = 0; c < N; ++c) L[r][c] = c <= r ? A[r * N + c] : 0.0;
    int bad = 0;
#pragma unroll
    for (int k = 0; k < N; ++k) {
        const double piv = L[k][k];
        if (!(piv > 0.0) && bad == 0) bad = k + 1;
        const double rp = bad == 0 ? rsqrt(piv) : 0.0;
#pragma unroll
        for (int r = k; r < N; ++r) L[r][k] *= rp;
#pragma unroll
        for (int c = k + 1; c < N; ++c)
#pragma unroll
            for (int r = c; r < N; ++r) L[r][c] = fma(-L[r][k], L[c][k], L[r][c]);
    }
#pragma unroll
    for (int r = 0; r < N; ++r)
#pragma unroll
        for (int c = 0; c <= r; ++c) A[r * N + c] = L[r][c];
    info[b] = bad;
}

__global__ void k_fp64_probe(int64_t iters, double *sink) {
    double a0 = 1.0 + threadIdx.x * 1e-9, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3;
    double a4 = a0 + 4e-3, a5 = a0 + 5e-3, a6 = a0 + 6e-3, a7 = a0 + 7e-3;
    const double m = 0.999999999, c = 1e-9;
    for (int64_t i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c);
        a1 = fma(a1, m, c);
        a2 = fma(a2, m, c);
        a3 = fma(a3, m, c);
        a4 = fma(a4, m, c);
        a5 = fma(a5, m, c);
        a6 = fma(a6, m, c);
        a7 = fma(a7, m, c);
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678) sink[0] = s;
}

}  // namespace mrgp
