// common.cuh -- context, workspace pool, error plumbing and the scalar quantizer shared by all
// GPFQ kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/gpfq.h"

#define GPFQ_DEAD_NORM 1e-16   // quantized_network.py:83
#define GPFQ_PERP_DOT 1e-10    // quantized_network.py:86

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct ConvPtrs {
    const float *const *Xp;   // device array of n_channels device pointers
    const float *const *Xqp;
};

struct AlphEntry {
    std::vector<char> blob;  // levels (fp64), the prefix offsets (int32), one equispaced flag per alphabet (int32)
    size_t off = 0;          // byte offset inside the WS_ALPH device buffer
};

// One set of timing events + the static part of the report per API call; a ring of them lets callers
// enqueue many GPFQ_NO_SYNC calls and read every call's stage times afterwards (gpfq_query_stats).
struct CallRecord {
    cudaEvent_t e[8] = {};
    bool rec[8] = {};
    int kind = 0;  // 0 dense Gram+sweep, 1 dense stream, 2 conv
    gpfq_stats st = {};
};
static constexpr int GPFQ_RING = 128;

struct gpfq_ctx {
    int device = 0;
    int sm_count = 148;
    size_t smem_optin = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaStream_t stream = nullptr;  // the one kernels launch on
    std::vector<CallRecord> ring;
    int64_t calls = 0;          // API calls begun so far
    CallRecord *cur = nullptr;  // record of the call in progress
    cudaEvent_t ev_copy[4] = {};
    cudaStream_t aux_stream[8] = {};   // residual-form sweep, up to 4 neuron groups: [g] the W part of group g's residual update,
                                       // [4 + g] the main chain of group g >= 1 (group 0 runs on `stream`)
    cudaEvent_t ev_chain[12] = {};     // ... [3 g] residuals sliced (main -> aux), [3 g + 1] W part landed (aux -> main), [3 g + 2] done
    std::string err = "";
    int launches = 0;
    int conv_variant = 0;         // 3x3 patch-Gram kernel: 0 TMA-staged / correlation form (default), 1 direct LDG, 2 generic,
                                  // 3 NHWC entry point: shared-memory planes kernel instead of the correlation form
    int corr_pack = 0;            // correlation form, images packed as virtual channels: 0 by shape, 1 always (tests), 2 never
    bool corr_direct_small = false;  // correlation form also on images below 128 pixels (tests)
    int corr_occ[2][9] = {};      // correlation-form kernels: resident CTAs per SM by [X~ == X][rows per band] (0: not queried yet)
    int corr_rb = 0;              // correlation-form conv Grams: rows per band (0: chosen per image height)
    int corr_strip_occ[2][2][3] = {};  // strip kernel: resident CTAs per SM by [X~ == X][rows per band 1 / 4][strip width 8 / 14 / 16]
    int corr_strip = 0;           // ... small images (W in {8, 14, 16, 28, 32, 56, 64}): 0 the strip kernel, 2 the band kernel
    bool stream_literal = false;  // streaming walk: reproduce the reference's fp32-rounded w*X products (set per call)
    int gram_variant = 0;         // Dense Gram stage: 0 auto, 1 fp64 DMMA (mma.sync), 2 int8 slices on tcgen05 (gram_i8.cu)
    int lowrank_variant = 0;      // sweep outer level: 0 auto, 1 Gram rows, 2 residual (low-rank) form
    int sweep_walk = 0;           // range walk of the Gram-row sweep: 0 auto, 1 tensor-core walk (sweep_tc.cu), 2 sweep_pipe / sweep_tile
    int sweep_i8 = 0;             // sweep contractions of the residual form: 0 auto, 1 int8 slices on tcgen05, 2 fp64 DMMA
    int i8_pairs_d = 0;           // int8 Gram: keep slice pairs with k + l <= this (0: the default of gram_i8.cu)
    const double *h_alph = nullptr;  // host copy of the current call's alphabets (levels back to back) and their offsets
    const int *h_koff = nullptr, *h_flags = nullptr;
    int64_t conv_part_bytes = 0;      // partial Gram workspace of the last conv call (gpfq_conv_partial_bytes)
    double *gram_only_out = nullptr;  // set for the duration of gpfq_conv_gram_nhwc: conv_finish hands the Grams out, no walk
    int last_gram_kernel = 0;     // what the last Dense Gram stage ran (1 DMMA, 2 int8 tcgen05)
    size_t i8_oom_bytes = 0;      // smallest int8-Gram workspace that failed to allocate (0: none yet)
    int rounding = GPFQ_ROUND_NEAREST;  // gpfq_set_rounding: the mode and its seeds (one per alphabet of a call)
    std::vector<uint64_t> seeds;
    const uint64_t *d_seeds = nullptr;  // the seeds of the call in progress on the device; nullptr: nearest rounding
    std::vector<double> l1;             // gpfq_set_l1_penalty: one lambda per alphabet of a call (empty: no penalty)
    const double *d_l1 = nullptr;       // the lambdas of the call in progress on the device; nullptr: no penalty
    // grow-only named workspaces
    DevBuf ws[50];
    DevBuf pinned[4];
    // alphabets already resident on the device (steady-state calls re-use them: no copy, no sync)
    std::vector<AlphEntry> alph_cache;
    size_t alph_used = 0;
};

enum WsSlot {
    WS_X = 0, WS_XQ, WS_W, WS_Q, WS_WT, WS_QT, WS_G1, WS_G2, WS_PART, WS_DT, WS_NRM, WS_ALPH,
    WS_U, WS_PTRS, WS_CG, WS_CPART, WS_PATCH_A, WS_PATCH_B, WS_ACT_A, WS_ACT_B, WS_QIDX, WS_MISC,
    WS_I8_SQ, WS_I8_SX, WS_I8_E, WS_I8_TILES, WS_LR_XD, WS_LR_XT, WS_LR_U, WS_CORR_B,
    WS_SL_W, WS_SL_XT, WS_SL_XQT, WS_SL_XQ, WS_SL_U, WS_SL_KQ, WS_SL_E,
    WS_TC_TAB, WS_TC_G2S, WS_TC_G1S, WS_TC_E, WS_TC_P, WS_TC_W, WS_TC_G1M, WS_SCALES, WS_UNIT_H, WS_SEEDS, WS_L1, WS_L1_LAMBDA
};

int gpfq_fail(gpfq_ctx *ctx, int code, const char *fmt, ...);
cudaError_t gpfq_record(gpfq_ctx *ctx, int which, cudaStream_t s);  // record timing event `which` of the current call
int gpfq_ws(gpfq_ctx *ctx, int slot, size_t bytes, void **out);         // device workspace
int gpfq_pinned(gpfq_ctx *ctx, int slot, size_t bytes, void **out);     // pinned host staging

#define CUDA_TRY(ctx, expr)                                                                    \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess)                                                                 \
            return gpfq_fail((ctx), _e == cudaErrorMemoryAllocation ? GPFQ_ERR_OOM : GPFQ_ERR_CUDA, \
                             "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

#define GPFQ_TRY(expr)                \
    do {                              \
        int _rc = (expr);             \
        if (_rc != GPFQ_OK) return _rc; \
    } while (0)

#define KERNEL_CHECK(ctx)                                                                     \
    do {                                                                                      \
        (ctx)->launches++;                                                                    \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess)                                                                \
            return gpfq_fail((ctx), GPFQ_ERR_CUDA, "kernel launch failed: %s (%s:%d)",        \
                             cudaGetErrorString(_e), __FILE__, __LINE__);                     \
    } while (0)

// Partial Gram workspace (WS_CPART) of the conv kernels for sizes without a kernel of their own: at most 1 GiB, reached
// through fewer column chunks / image chunks (conv_pick_chunks, gpfq_conv_layer_nhwc) unless one slot per channel exceeds it.
static constexpr int64_t CONV_PART_LIMIT = (int64_t)1 << 30;

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------------------------
// Scalar quantizer: alphabet[argmin_k |alphabet[k] - v|], first minimal index on ties
// (quantized_network.py:57).  Same fp64 subtraction/abs/compare as NumPy, so ties break alike.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double gpfq_bit_round(double v, const double *__restrict__ alph, int K) {
    double best = alph[0];
    double bd = fabs(__dsub_rn(best, v));
#pragma unroll 4
    for (int k = 1; k < K; ++k) {
        const double a = alph[k];
        const double d = fabs(__dsub_rn(a, v));
        if (d < bd) { bd = d; best = a; }
    }
    return best;
}

// out-of-line copy for the rarely taken branches of the fast paths (keeps their loop bodies small)
static __device__ __noinline__ double gpfq_bit_round_slow(double v, const double *__restrict__ alph, int K) {
    return gpfq_bit_round(v, alph, K);
}

// The same quantizer when the levels are ascending and equispaced (`rad * linspace(-1, 1, K)`, :396/:545 -- the host
// checks this per alphabet): |a_k - v| is unimodal in k, so the first minimal index of the full scan is the grid guess
// rint((v - a_0) / step) or one of its two neighbours (the guess is off by at most one, at a tie either side is in the
// window).  The three candidates are compared with the very same subtraction / abs / strict-less tests in ascending
// order, so ties still go to the lower index; indices clamped at the ends only repeat a level, which never wins a
// strict comparison against its own earlier copy.  Branch-free: this sits on the serial critical path of every walk.
// inv_step <= 0 (not equispaced) or a non-finite / huge argument: literal scan.
__device__ __forceinline__ double gpfq_bit_round_eq(double v, const double *__restrict__ alph, int K, double inv_step) {
    const double gpos = (v - alph[0]) * inv_step;
    if (!(inv_step > 0.0) || !(fabs(gpos) < 1e9)) return gpfq_bit_round_slow(v, alph, K);  // also NaN / inf arguments
    const int kr = __double2int_rn(gpos), hi = K - 1;
    const int i1 = min(max(kr, 0), hi), i0 = max(i1 - 1, 0), i2 = min(i1 + 1, hi);
    const double a0 = alph[i0], a1 = alph[i1], a2 = alph[i2];
    const double d0 = fabs(__dsub_rn(a0, v)), d1 = fabs(__dsub_rn(a1, v)), d2 = fabs(__dsub_rn(a2, v));
    double best = a0, bd = d0;
    if (d1 < bd) { bd = d1; best = a1; }
    if (d2 < bd) best = a2;
    return best;
}

// The same quantizer for the ternary alphabet {-a, 0, a} (bits = log2 3: the VGG16 and MNIST configurations): the literal
// three-level scan itself -- the same subtractions, absolute values and strict comparisons in ascending order, so every tie goes
// where _bit_round_parallel sends it -- with the levels in registers: no index arithmetic, no shared-memory loads on the
// serial chain of the walk (the windowed form above costs ~115 dependent cycles per step, this one ~25).
__device__ __forceinline__ double gpfq_bit_round_ternary(double v, double a) {
    const double dl = fabs(__dsub_rn(-a, v)), dm = fabs(__dsub_rn(0.0, v)), dh = fabs(__dsub_rn(a, v));
    double best = -a, bd = dl;
    if (dm < bd) { bd = dm; best = 0.0; }
    if (dh < bd) best = a;
    return best;
}
// a > 0 when the alphabet staged at `alph` is exactly {-a, 0, a}, else 0
__device__ __forceinline__ double gpfq_ternary_radius(const double *alph, int K) {
    return (K == 3 && alph[1] == 0.0 && alph[2] > 0.0 && alph[0] == -alph[2]) ? alph[2] : 0.0;
}

// inv_step of an alphabet staged in shared memory (flag from the host: 1 = ascending and equispaced)
__device__ __forceinline__ double gpfq_inv_step(const double *alph, int K, int equispaced) {
    return (equispaced && K >= 2) ? (double)(K - 1) / (alph[K - 1] - alph[0]) : 0.0;
}

// One greedy decision in Gram form (SURVEY.md App. A item 6):
//   nrm  = (double)(float)sqrt(G2[t,t])         (snrm2 result, quantized_network.py:83)
//   d    = <Xq_t, u_{t-1}>                       (:86)
//   num  = <Xq_t, u_{t-1} + w_t X_t>             (:89)
__device__ __forceinline__ double gpfq_decide(double nrm, double d, double num, double w,
                                              const double *__restrict__ alph, int K, double inv_step = 0.0) {
    if (nrm < GPFQ_DEAD_NORM) return 0.0;
    if (fabs(d) < GPFQ_PERP_DOT) return gpfq_bit_round_eq(w, alph, K, inv_step);
    return gpfq_bit_round_eq(num / (nrm * nrm), alph, K, inv_step);
}

// The same decision for the sweep's in-block walk, out of line (32 unrolled call sites share one copy) and with the
// division by nrm^2 done as a Markstein correction of num * RN(1/nrm^2): q0 = RN(num r), e = RN(num - q0 den) (exact,
// fma), v = RN(q0 + e r) is the correctly rounded quotient, i.e. bit-identical to num / den, while the reciprocal
// is computed once per direction instead of once per neuron and step.
static __device__ __noinline__ double gpfq_decide_rcp(double nrm, double rinv, double d, double num, double w,
                                               const double *__restrict__ alph, int K, double inv_step) {
    if (nrm < GPFQ_DEAD_NORM) return 0.0;
    double v = w;
    if (!(fabs(d) < GPFQ_PERP_DOT)) {
        const double den = nrm * nrm;
        const double q0 = num * rinv;
        const double e = fma(-q0, den, num);
        v = fma(e, rinv, q0);
    }
    return gpfq_bit_round_eq(v, alph, K, inv_step);
}

// ---------------------------------------------------------------------------------------------
// Per-unit (per-channel) alphabets: a unit with scale s uses the levels fl64(s * alph[k]), formed on the fly with one
// correctly rounded product per level (what NumPy's `rad_u * alphabet` gives for a scalar rad_u), so no level table per
// unit is staged.  s = 0 gives the all-zero alphabet; its inv_step is 0, so the literal scan decides and no division by
// the zero span happens.  The window of gpfq_bit_round_eq carries over: the scaled levels are ascending and as nearly
// equispaced as the base levels, and the three candidates are compared with the same tests in ascending order.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double gpfq_bit_round_s(double v, const double *__restrict__ alph, int K, double s) {
    double best = __dmul_rn(s, alph[0]);
    double bd = fabs(__dsub_rn(best, v));
#pragma unroll 4
    for (int k = 1; k < K; ++k) {
        const double a = __dmul_rn(s, alph[k]);
        const double d = fabs(__dsub_rn(a, v));
        if (d < bd) { bd = d; best = a; }
    }
    return best;
}

static __device__ __noinline__ double gpfq_bit_round_s_slow(double v, const double *__restrict__ alph, int K, double s) {
    return gpfq_bit_round_s(v, alph, K, s);
}

__device__ __forceinline__ double gpfq_bit_round_eq_s(double v, const double *__restrict__ alph, int K, double inv_step, double s) {
    const double gpos = (v - __dmul_rn(s, alph[0])) * inv_step;
    if (!(inv_step > 0.0) || !(fabs(gpos) < 1e9)) return gpfq_bit_round_s_slow(v, alph, K, s);
    const int kr = __double2int_rn(gpos), hi = K - 1;
    const int i1 = min(max(kr, 0), hi), i0 = max(i1 - 1, 0), i2 = min(i1 + 1, hi);
    const double a0 = __dmul_rn(s, alph[i0]), a1 = __dmul_rn(s, alph[i1]), a2 = __dmul_rn(s, alph[i2]);
    const double d0 = fabs(__dsub_rn(a0, v)), d1 = fabs(__dsub_rn(a1, v)), d2 = fabs(__dsub_rn(a2, v));
    double best = a0, bd = d0;
    if (d1 < bd) { bd = d1; best = a1; }
    if (d2 < bd) best = a2;
    return best;
}

// inv_step of the scaled levels of an equispaced base alphabet (0: literal scan), computed once per unit
__device__ __forceinline__ double gpfq_inv_step_s(const double *alph, int K, int equispaced, double s) {
    if (!equispaced || K < 2) return 0.0;
    const double span = __dsub_rn(__dmul_rn(s, alph[K - 1]), __dmul_rn(s, alph[0]));
    return (span > 0.0 && span < 1e300) ? (double)(K - 1) / span : 0.0;
}

// The scalar quantizer with the unit's own levels: SCALED = false is the base alphabet, unchanged
template <bool SCALED>
__device__ __forceinline__ double gpfq_round_unit(double v, const double *__restrict__ alph, int K, double inv_step, double s) {
    if (SCALED) return gpfq_bit_round_eq_s(v, alph, K, inv_step, s);
    return gpfq_bit_round_eq(v, alph, K, inv_step);
}

template <bool SCALED>
__device__ __forceinline__ double gpfq_decide_unit(double nrm, double d, double num, double w, const double *__restrict__ alph,
                                                   int K, double inv_step, double s) {
    if (nrm < GPFQ_DEAD_NORM) return 0.0;
    if (fabs(d) < GPFQ_PERP_DOT) return gpfq_round_unit<SCALED>(w, alph, K, inv_step, s);
    return gpfq_round_unit<SCALED>(num / (nrm * nrm), alph, K, inv_step, s);
}

// ---------------------------------------------------------------------------------------------
// Stochastic rounding (SPFQ, gpfq_set_rounding): unbiased rounding between the two levels that bracket the argument, with
// counter-based draws, so a decision depends only on (seed, unit, step) -- not on the shard, launch geometry or device.
//   draw(seed, u, t) = (splitmix64(splitmix64(seed ^ splitmix64(u)) ^ t) >> 11) * 2^-53      exact fp64 in [0, 1)
// A walk forms the unit key splitmix64(seed ^ splitmix64(u)) once; each step then costs one splitmix64, off the chain.
//   stoc_round(v, A, r): A[0] unless v > A[0] (NaN included); A[K-1] when v >= A[K-1]; else with k = max{i : A[i] <= v},
//                        p = (v - A[k]) / (A[k+1] - A[k]) (correctly rounded fp64), A[k+1] if r < p else A[k].
// A unit with a scale s uses the levels fl64(s * A[k]), as the nearest quantizer does.
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t gpfq_splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ uint64_t gpfq_unit_key(uint64_t seed, int64_t u) { return gpfq_splitmix64(seed ^ gpfq_splitmix64((uint64_t)u)); }
__device__ __forceinline__ double gpfq_draw(uint64_t key, int64_t t) {
    return (double)(gpfq_splitmix64(key ^ (uint64_t)t) >> 11) * 0x1p-53;
}

template <bool SCALED>
__device__ __forceinline__ double gpfq_level(const double *__restrict__ alph, int k, double s) {
    return SCALED ? __dmul_rn(s, alph[k]) : alph[k];
}
__device__ __forceinline__ double gpfq_stoc_pick(double v, double lo, double hi, double r) {
    return r < __ddiv_rn(__dsub_rn(v, lo), __dsub_rn(hi, lo)) ? hi : lo;
}

// the literal form: the bracketing interval by a downward scan (levels non-decreasing, checked by the host)
template <bool SCALED>
static __device__ __noinline__ double gpfq_stoc_round_scan(double v, const double *__restrict__ alph, int K, double s, double r) {
    const double a0 = gpfq_level<SCALED>(alph, 0, s);
    if (!(v > a0)) return a0;
    const double top = gpfq_level<SCALED>(alph, K - 1, s);
    if (v >= top) return top;
    int k = K - 2;
    while (gpfq_level<SCALED>(alph, k, s) > v) --k;   // stops at k = 0 at the latest: A[0] < v
    return gpfq_stoc_pick(v, gpfq_level<SCALED>(alph, k, s), gpfq_level<SCALED>(alph, k + 1, s), r);
}

// The same quantizer for an equispaced alphabet (inv_step > 0, as for gpfq_bit_round_eq): the grid position's integer part
// guesses k, and the guess is moved until A[k] <= v < A[k+1] holds, so k is the literal scan's (the guess is off by at most one
// for levels within 1 % of a step of the grid).  inv_step <= 0, a non-finite or huge argument: the scan.
template <bool SCALED>
__device__ __forceinline__ double gpfq_stoc_round_eq(double v, const double *__restrict__ alph, int K, double inv_step, double s,
                                                     double r) {
    const double a0 = gpfq_level<SCALED>(alph, 0, s);
    const double gpos = (v - a0) * inv_step;
    if (!(inv_step > 0.0) || !(fabs(gpos) < 1e9)) return gpfq_stoc_round_scan<SCALED>(v, alph, K, s, r);
    if (!(v > a0)) return a0;
    const double top = gpfq_level<SCALED>(alph, K - 1, s);
    if (v >= top) return top;
    int k = min(max((int)floor(gpos), 0), K - 2);
    while (k > 0 && gpfq_level<SCALED>(alph, k, s) > v) --k;
    while (k < K - 2 && gpfq_level<SCALED>(alph, k + 1, s) <= v) ++k;
    return gpfq_stoc_pick(v, gpfq_level<SCALED>(alph, k, s), gpfq_level<SCALED>(alph, k + 1, s), r);
}

// ... for the ternary alphabet {-a, 0, a} with the levels in registers: p = (v - (-a)) / (0 - (-a)) on (-a, 0), (v - 0) / (a - 0)
// on [0, a) -- the literal expressions, since v - (-a) = v + a and 0 - (-a) = a, v - 0 = v exactly
__device__ __forceinline__ double gpfq_stoc_round_ternary(double v, double a, double r) {
    if (!(v > -a)) return -a;
    if (v >= a) return a;
    if (v >= 0.0) return r < __ddiv_rn(v, a) ? a : 0.0;
    return r < __ddiv_rn(__dadd_rn(v, a), a) ? 0.0 : -a;
}

// One greedy step with stochastic rounding: the reference's guards, then stoc_round of w (:86 guard) or num / nrm^2
template <bool SCALED>
__device__ __forceinline__ double gpfq_decide_stoch(double nrm, double d, double num, double w, const double *__restrict__ alph,
                                                    int K, double inv_step, double s, double r) {
    if (nrm < GPFQ_DEAD_NORM) return 0.0;
    const double v = fabs(d) < GPFQ_PERP_DOT ? w : __ddiv_rn(num, nrm * nrm);
    return gpfq_stoc_round_eq<SCALED>(v, alph, K, inv_step, s, r);
}

// ---------------------------------------------------------------------------------------------
// Sparse GPFQ (gpfq_set_l1_penalty): an L1 penalty lambda per alphabet soft-thresholds the value of every greedy step before it
// is quantized.  tau = fl(lambda / fl(nrm^2)) depends only on the direction and the alphabet, so the walks form it off the chain
// (per tap, per block of directions, or in a table); the step is then
//   v' = 0 if |v| <= tau, else fl(v - copysign(tau, v))          (NaN stays NaN: the comparison is false)
// with v the reference's value (w for the :86 guard, num / nrm^2 otherwise).  tau = +0 (lambda = 0) gives v' = v up to the
// sign of a zero, which neither quantizer sees.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double gpfq_shrink(double v, double tau) {
    return fabs(v) <= tau ? 0.0 : __dsub_rn(v, copysign(tau, v));
}
__device__ __forceinline__ double gpfq_l1_tau(double lambda, double nrm) { return __ddiv_rn(lambda, __dmul_rn(nrm, nrm)); }

// One greedy step with the penalty: the reference's guards, the shrink, then nearest (STOCH = false) or stochastic rounding
template <bool SCALED, bool STOCH>
__device__ __forceinline__ double gpfq_decide_l1(double nrm, double d, double num, double w, const double *__restrict__ alph, int K,
                                                 double inv_step, double s, double r, double tau) {
    if (nrm < GPFQ_DEAD_NORM) return 0.0;
    const double v = gpfq_shrink(fabs(d) < GPFQ_PERP_DOT ? w : __ddiv_rn(num, nrm * nrm), tau);
    if (STOCH) return gpfq_stoc_round_eq<SCALED>(v, alph, K, inv_step, s, r);
    return gpfq_round_unit<SCALED>(v, alph, K, inv_step, s);
}

// The step of a walk: nearest rounding (STOCH = false: gpfq_decide_unit, unchanged) or stochastic with the draw r
// L1: the penalty's shrink with the step's tau
template <bool SCALED, bool STOCH, bool L1 = false>
__device__ __forceinline__ double gpfq_decide_any(double nrm, double d, double num, double w, const double *__restrict__ alph, int K,
                                                  double inv_step, double s, double r, double tau = 0.0) {
    if (L1) return gpfq_decide_l1<SCALED, STOCH>(nrm, d, num, w, alph, K, inv_step, s, r, tau);
    if (STOCH) return gpfq_decide_stoch<SCALED>(nrm, d, num, w, alph, K, inv_step, s, r);
    return gpfq_decide_unit<SCALED>(nrm, d, num, w, alph, K, inv_step, s);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
