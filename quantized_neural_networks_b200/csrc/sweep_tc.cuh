// sweep_tc.cuh -- host interface of the tensor-core range walk (sweep_tc.cu).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace stc {
constexpr int NB = 32;           // directions per block of the walk
constexpr int NT = 128;          // neurons per CTA = TMEM lanes = walker threads
constexpr int S = 5;             // digit slices of the Gram rows
constexpr int KB = 64;           // K bytes (= directions) per K block of the operand tiles
constexpr int MAX_R = 512;       // directions per range (the level-index tile of a range stays in shared memory)
constexpr int B_SLICE = NB * KB;         // one digit slice of one K block of a block's 32 Gram rows (2 KB)
constexpr int B_STAGE = S * B_SLICE;     // all slices of it: what one pipeline stage fetches (10 KB)

// What the walk of one block of 32 directions reads besides the residual dots: everything that depends on the directions
// only, laid out as the walker threads read it (one bulk copy per block).
struct TabA {
    double g2c[NB * NB];   // [t][u] = G2[t0 + u][t0 + t] for u > t (0 otherwise): what decision t does to the dots after it
    double g1dd[NB];       // G1[t][t]
    double rinv[NB];       // RN(1 / nrm^2), 0 for a dead direction (and for the padding beyond N0)
    double den[NB];        // nrm^2
    double ris[NB];        // rinv / (2 h): the decision argument in units of the alphabet's step
    double nrm[NB];        // (double)(float)sqrt(G2[t][t])   (the snrm2 result of quantized_network.py:83)
    double sc[NB];         // h 2^(e_t - 38): scale of the integer Q-term sums of direction t
    int32_t deadm[NB];     // 0x7ff00000 for a dead direction (masks the perpendicularity flag), else 0
    double qe;             // max over the block's directions t of 2^(e_t - 39) rinv_t: a neuron whose decisions in the range's earlier
                           // blocks sum to S = sum |k'_s| gets p moved by at most h S qe by the rounding of the Gram digit slices
    double qe_pad;         // (the bulk copy moves multiples of 16 bytes)
    int32_t ex[NB];        // e_t: the exponent of the digit slices of row t (a replay takes the exact Q terms from it)
};
}  // namespace stc

struct TcTables {
    const stc::TabA *tabs = nullptr;   // one per block of 32 directions (N0P / 32)
    const int8_t *g2s = nullptr;       // digit slices of G2[block rows][earlier directions of the block's range]:
                                       // [block][K block][slice][32 rows x 64 B, 64B-swizzled]
    int64_t R = 0;                     // directions per range
    const double *G2 = nullptr;        // the fp64 Gram rows the slices were made from (sweep_tc_prepare), for the replay
    int64_t ldg = 0;
    bool compact = false;
    CUtensorMap mapP, mapW;            // P (rowsP, N0P) fp64 and the neuron-major weights (rowsP, N0P) fp32 (sweep_tc_bind)
    int64_t rowsP = 0;
};

// Tables of every block (once per layer).  G(t, s) is read at G[t * ldg + s - (compact ? first direction of t's range : 0)]:
// the full (N0, N0) matrices of the Gram-row sweep or the compact block-diagonal tiles of the residual-form sweep.
int sweep_tc_prepare(gpfq_ctx *ctx, const double *G1, const double *G2, int64_t ldg, bool compact, int64_t N0, int64_t N0P, int64_t R,
                     double h, TcTables *out);
// Digit slices of the strictly lower part of every range's G1 tile (row t, K = range-local earlier directions), the B operand of
// the decision-independent product P_r = W_r strict_lower(G1_rr)^T (slgemm_i8): 5 x N0P x R int8 (sl_offset) + N0P exponents.
int sweep_tc_slice_g1_lower(gpfq_ctx *ctx, const double *G1, int64_t ldg, bool compact, int64_t N0, int64_t N0P, int64_t R, int32_t *e,
                            int8_t *slices);
// Walk of the directions [tb, te) of one range for nj neurons (one CTA per 128).
//   P   (nj, ldp) fp64: everything the directions before tb AND the weights of the range's own earlier directions contribute to the
//       residual dots, P[j][t]; the kernel adds the Q terms of the range itself (tcgen05, int8 level indices x Gram digit slices)
//   Wn  (nj, ldwn) fp32: the weights neuron-major (sweep_tc_weights)
//       both bound once per layer (sweep_tc_bind: rowsP x ldp allocations, rowsP a multiple of 128); this launch's neuron 0 is row row0
//   Kq  out: the decisions as int8 level indices k' = q / (a / 2) (sl_offset layout, krows rows, neuron 0 at row krow0)
int sweep_tc_bind(gpfq_ctx *ctx, TcTables *tab, const double *P, const float *Wn, int64_t rowsP, int64_t ldp);
//   a, levels, K: an alphabet on the symmetric grid (device levels, a = levels[K - 1]; alphabet_on_symmetric_grid); K == 3 runs the
//       ternary specialisation
//   scales (nullable, device, this launch's nj neurons): per-channel alphabets -- neuron j walks with fl(scales[j] levels[k]); the
//       tables must then be prepared with h = 1
//   u0: stochastic rounding (ctx->d_seeds set): this launch's neuron j draws as unit u0 + j
int sweep_tc_range(gpfq_ctx *ctx, const TcTables &tab, int64_t tb, int64_t te, int64_t row0, int64_t nj, int8_t *Kq, int64_t krows,
                   int64_t krow0, double a, const double *levels, int K, const double *scales = nullptr, int64_t u0 = 0);
// Wn[j][t] = W[t * ldw + wcol0 + j], (nj, N0P) fp32, zeros beyond N0
int sweep_tc_weights(gpfq_ctx *ctx, const float *W, int64_t ldw, int64_t wcol0, int64_t N0, int64_t N0P, int64_t nj, float *Wn);
// Q[t * ldq + col0 + j] = the level of index Kq[j][t] for t < N0, j < nj
int sweep_tc_q_from_kq(gpfq_ctx *ctx, const int8_t *Kq, int64_t krows, int64_t N0, int64_t nj, const double *levels, int K, double *Q,
                       int64_t ldq, int64_t col0, const double *scales = nullptr);
// Gram-row form of the sweep (full G1 / G2 in HBM): the strictly lower part of every range's G1 tile as a compact fp64 matrix
// (N0P, R) for the in-range W terms on the fp64 pipe; P[:, tb : tb + n] += Do; Qt[:, tb : te] from the level indices
int sweep_tc_mask_g1_lower(gpfq_ctx *ctx, const double *G1, int64_t ldg, int64_t N0, int64_t N0P, int64_t R, double *G1m);
int sweep_tc_add_outer(gpfq_ctx *ctx, double *P, int64_t ldp, const double *Do, int64_t ldd, int64_t nj, int64_t n);
int sweep_tc_qt_from_kq(gpfq_ctx *ctx, const int8_t *Kq, int64_t krows, int64_t tb, int64_t te, int64_t nj, const double *levels, int K,
                        double *Qt, int64_t ldq, const double *scales = nullptr);
// P[:, 0 : n] += part[0] + ... + part[ns - 1] (partials `stride` elements apart, row stride ldd): the K-split residual dots
int sweep_tc_add_partials(gpfq_ctx *ctx, double *P, int64_t ldp, const double *part, int ns, int64_t stride, int64_t ldd, int64_t nj,
                          int64_t n);
