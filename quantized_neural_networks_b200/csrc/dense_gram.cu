// dense_gram.cu -- Dense layer, Gram form: K1 Gram stage + K2 blocked triangular sweep.
//
// Replaces the N0-step loop of _quantize_neuron_parallel (quantized_network.py:117-119) for all
// neurons of a layer.  With G1[t,s] = <Xq_t, X_s>, G2[t,s] = <Xq_t, Xq_s> (fp64 accumulation of exact
// fp32 products) the residual dot of step t is
//     d_t = <Xq_t, u_{t-1}> = sum_{s<t} ( w_s G1[t,s] - q_s G2[t,s] )
// so q_t = Q( (d_t + w_t G1[t,t]) / fl32(sqrt(G2[t,t]))^2 ) with the two guards of :83-87 intact.
// The sweep walks ranges of directions: what the earlier ranges contribute to a range is one NT contraction
// (gemm_nt.cuh, two segments), then one persistent kernel walks the range's blocks of 32 directions for a tile of
// neurons (sweep_pipe_kernel / sweep_tile_kernel below, or the tensor-core walk of sweep_tc.cu).
#include <algorithm>

#include "gemm_nt.cuh"
#include "slgemm_i8.cuh"
#include "sweep_tc.cuh"

static constexpr int SWEEP_B = 32;
static constexpr int64_t SWEEP_OUTER = 512;  // directions per range of the two-level sweep

// Wt[j - j0][t] = (double) W[t*ldw + j]   (neuron-major copy of the shard, fp64)
__global__ void transpose_w_kernel(const float *__restrict__ W, int64_t ldw, int64_t N0, int64_t j0,
                                   int64_t nj, double *__restrict__ Wt) {
    __shared__ float tile[32][33];
    const int64_t tb = (int64_t)blockIdx.x * 32, jb = (int64_t)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t t = tb + r, j = jb + threadIdx.x;
        tile[r][threadIdx.x] = (t < N0 && j < nj) ? W[t * ldw + j0 + j] : 0.f;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t j = jb + r, t = tb + threadIdx.x;
        if (j < nj && t < N0) Wt[j * N0 + t] = (double)tile[threadIdx.x][r];
    }
}

// Q[t*ldq + j0 + j] = Qt[j][t]
__global__ void transpose_q_kernel(const double *__restrict__ Qt, int64_t N0, int64_t nj,
                                   double *__restrict__ Q, int64_t ldq, int64_t col0) {
    __shared__ double tile[32][33];
    const int64_t tb = (int64_t)blockIdx.x * 32, jb = (int64_t)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t j = jb + r, t = tb + threadIdx.x;
        tile[r][threadIdx.x] = (j < nj && t < N0) ? Qt[j * N0 + t] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t t = tb + r, j = jb + threadIdx.x;
        if (t < N0 && j < nj) Q[t * ldq + col0 + j] = tile[threadIdx.x][r];
    }
}

// ---------------------------------------------------------------------------------------------
// Persistent sweep: one CTA owns NT neurons and walks ALL direction blocks of a range for them -- one launch per
// range, no inter-CTA dependency (neurons are independent).  Per block of 32 directions:
//   panel   D[32 x NT] = G1[blk, :p] Wt[tile, :p]^T - G2[blk, :p] Qt[tile, :p]^T   on the fp64 tensor pipe
//           (DMMA.8x8x4; warp w owns direction rows 8(w&3).., K half w>>2), K streamed through a cp.async ring;
//           the Gram rows are shared by every CTA (L2), the W / Q panels are the CTA's own.  The last K chunk is the
//           strictly-lower part of the block's own G1 diagonal tile: everything the weights contribute to the
//           residual dots is known before the walk starts, only the q-terms are sequential;
//   walk    thread-per-neuron: d[32] in registers, 32 fully unrolled greedy steps -- decision (reciprocal + Markstein
//           correction, equispaced rounding window), then one DFMA per remaining direction (d -= q G2[t][tt], the
//           Gram column broadcast from shared memory).  Measured dependent latencies on B200 (tools/fp64_latency.cu):
//           DFMA 8.3, LDS.64 35, F2I+I2F 36 cycles, so a step is ~250 cycles; the other seven warps wait, which is
//           why two CTAs share an SM (launch bounds, <= 106 KB shared memory): one walks while the other contracts;
//   Q block -> shared memory -> Qt (neuron-major), read back by the later panels of this same CTA.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double gpfq_decide_rcp_inl(double nrm, double rinv, double d, double num, double w,
                                                      const double *__restrict__ alph, int K, double inv_step, double tern = 0.0) {
    if (nrm < GPFQ_DEAD_NORM) return 0.0;
    double v = w;
    if (!(fabs(d) < GPFQ_PERP_DOT)) {
        const double den = nrm * nrm;
        const double q0 = num * rinv;
        const double e = fma(-q0, den, num);
        v = fma(e, rinv, q0);
    }
    if (tern > 0.0) return gpfq_bit_round_ternary(v, tern);   // CTA-uniform: {-a, 0, a} with the levels in registers
    return gpfq_bit_round_eq(v, alph, K, inv_step);
}

// The same decision with the neuron's own levels fl64(s * alph[k]) (per-channel alphabets, common.cuh): inv_step and tern are
// the neuron's (tern = fl64(s * a) of a ternary base alphabet {-a, 0, a}, 0 otherwise).
template <bool SCALED>
__device__ __forceinline__ double gpfq_decide_rcp_unit(double nrm, double rinv, double d, double num, double w,
                                                       const double *__restrict__ alph, int K, double inv_step, double tern,
                                                       double s) {
    if (!SCALED) return gpfq_decide_rcp_inl(nrm, rinv, d, num, w, alph, K, inv_step, tern);
    if (nrm < GPFQ_DEAD_NORM) return 0.0;
    double v = w;
    if (!(fabs(d) < GPFQ_PERP_DOT)) {
        const double den = nrm * nrm;
        const double q0 = num * rinv;
        const double e = fma(-q0, den, num);
        v = fma(e, rinv, q0);
    }
    if (tern > 0.0) return gpfq_bit_round_ternary(v, tern);
    return gpfq_bit_round_eq_s(v, alph, K, inv_step, s);
}

// The same step with stochastic rounding (r = the step's draw): the argument is formed exactly as above (the Markstein quotient is
// the correctly rounded num / nrm^2), then stoc_round between the bracketing levels (common.cuh)
template <bool SCALED>
__device__ __forceinline__ double gpfq_decide_rcp_stoch(double nrm, double rinv, double d, double num, double w,
                                                        const double *__restrict__ alph, int K, double inv_step, double tern,
                                                        double s, double r) {
    if (nrm < GPFQ_DEAD_NORM) return 0.0;
    double v = w;
    if (!(fabs(d) < GPFQ_PERP_DOT)) {
        const double den = nrm * nrm;
        const double q0 = num * rinv;
        const double e = fma(-q0, den, num);
        v = fma(e, rinv, q0);
    }
    if (tern > 0.0) return gpfq_stoc_round_ternary(v, tern, r);
    return gpfq_stoc_round_eq<SCALED>(v, alph, K, inv_step, s, r);
}

// The step with the L1 penalty (common.cuh): the same argument, shrunk by the direction's tau, then nearest (STOCH = false) or
// stochastic rounding
template <bool SCALED, bool STOCH>
__device__ __forceinline__ double gpfq_decide_rcp_l1(double nrm, double rinv, double d, double num, double w,
                                                     const double *__restrict__ alph, int K, double inv_step, double tern, double s,
                                                     double r, double tau) {
    if (nrm < GPFQ_DEAD_NORM) return 0.0;
    double v = w;
    if (!(fabs(d) < GPFQ_PERP_DOT)) {
        const double den = nrm * nrm;
        const double q0 = num * rinv;
        const double e = fma(-q0, den, num);
        v = fma(e, rinv, q0);
    }
    v = gpfq_shrink(v, tau);
    if (STOCH) {
        if (tern > 0.0) return gpfq_stoc_round_ternary(v, tern, r);
        return gpfq_stoc_round_eq<SCALED>(v, alph, K, inv_step, s, r);
    }
    if (tern > 0.0) return gpfq_bit_round_ternary(v, tern);
    return gpfq_round_unit<SCALED>(v, alph, K, inv_step, s);
}

// Per-neuron scale, inv_step and ternary radius of neuron jt + j (SCALED; else the alphabet's own)
template <bool SCALED>
__device__ __forceinline__ void sweep_unit_levels(const double *__restrict__ scales, int64_t idx, bool live,
                                                  const double *alph, int K, int flag, double inv_step, double tern,
                                                  double *sc, double *inv_u, double *tern_u) {
    if (!SCALED) { *sc = 1.0; *inv_u = inv_step; *tern_u = tern; return; }
    const double s = live ? scales[idx] : 0.0;
    *sc = s;
    *inv_u = gpfq_inv_step_s(alph, K, flag, s);
    *tern_u = __dmul_rn(s, tern);
}

template <int NT>
struct SweepCfg {
    // K chunk per pipeline stage: 64 earlier directions (one barrier per chunk: fewer, fatter steps on the latency-bound
    // in-range panel) where two CTAs still fit an SM, 32 for the 32-neuron tile
    static constexpr int B = SWEEP_B, KC = NT == 32 ? 32 : 64, LD = KC + 4, STAGES = 3, THREADS = 256;
    static constexpr size_t SMEM = sizeof(double) * ((size_t)STAGES * B * LD + (size_t)STAGES * NT * LD + 2 * B * (B + 1) +
                                                     2 * B * (NT + 1) + 2 * NT * (B + 1) + 3 * B + GPFQ_MAX_K);
    // (2 B x (B+1) is the G2 diagonal tile plus B rows of zeros: the walk reads 31 entries below the diagonal at every
    //  step, whatever the step)
};

// SCALED: neuron j of alphabet a walks with the levels scales[a * nj + j] * alphabet (per-channel alphabets).
// STOCH: stochastic rounding, neuron j with unit id u0 + j and seed seeds[a], direction t with step id t.
// L1: the penalty lambdas[a]; each walker lane forms tau of one direction of the block, broadcast by a shuffle at its step.
template <int NT, bool ALIGNED, bool SCALED = false, bool STOCH = false, bool L1 = false>
__global__ void __launch_bounds__(256, 2)
sweep_tile_kernel(const double *__restrict__ G1, const double *__restrict__ G2, int64_t ldg, int64_t N0,
                  const double *__restrict__ Wt, double *__restrict__ Qt, int64_t nj,
                  const double *__restrict__ alphabets, const int *__restrict__ Koff,
                  const int *__restrict__ Flags, int64_t t_begin, int64_t t_end, const double *__restrict__ Dt,
                  int64_t ldd, const double *__restrict__ scales = nullptr, const uint64_t *__restrict__ seeds = nullptr,
                  int64_t u0 = 0, const double *__restrict__ lambdas = nullptr) {
    // Directions [t_begin, t_end) (t_begin a multiple of 32).  Dt (nullable): (n_alph, nj, ldd) contributions of the
    // directions before t_begin, from one large NT contraction on the host side (two-level blocking).
    using Cfg = SweepCfg<NT>;
    constexpr int B = Cfg::B, KC = Cfg::KC, LD = Cfg::LD, STAGES = Cfg::STAGES, THREADS = Cfg::THREADS, NA = NT / 8;
    constexpr int GCH = B * (KC / 2) / THREADS;                          // 16-byte chunks of the Gram tile per thread (2)
    constexpr int WCH = (NT * (KC / 2) + THREADS - 1) / THREADS;         // ... of the W / Q tile per thread (2, 1, 1)
    constexpr int DPT = B * B / THREADS;                                 // diagonal-tile entries per thread (4)
    constexpr int WPT = (NT * B + THREADS - 1) / THREADS;                // W-block entries per thread (4, 2, 1)
    extern __shared__ __align__(16) unsigned char sweep_smem[];
    double *gst = reinterpret_cast<double *>(sweep_smem);   // STAGES x B x LD   (Gram rows of the block)
    double *wst = gst + STAGES * B * LD;                    // STAGES x NT x LD  (W or Q panel of the tile)
    double *g2d = wst + STAGES * NT * LD;                   // 2B x (B+1): G2 diagonal tile, then B rows of zeros
    double *dsm = g2d + 2 * B * (B + 1);                    // 2 x B x (NT+1): one partial per K-half warp group
    double *wblk = dsm + 2 * B * (NT + 1);                  // NT x (B+1)
    double *qblk = wblk + NT * (B + 1);                     // NT x (B+1)
    double *nrm = qblk + NT * (B + 1);                      // B
    double *rinv = nrm + B;                                 // B: RN(1 / nrm^2)
    double *g1dd = rinv + B;                                // B: G1[t][t]
    double *alph = g1dd + B;                                // GPFQ_MAX_K

    const int a = blockIdx.y;
    const int K = Koff[a + 1] - Koff[a];
    const int64_t jt = (int64_t)blockIdx.x * NT;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, grp = lane >> 2, tig = lane & 3;
    const int strip = warp & 3, khalf = warp >> 2;  // direction rows 8*strip.., k-steps [16*khalf, 16*khalf + 16)
    double *Qa = Qt + (int64_t)a * nj * N0;
    for (int e = tid; e < K; e += THREADS) alph[e] = alphabets[Koff[a] + e];
    for (int e = tid; e < B * (B + 1); e += THREADS) g2d[B * (B + 1) + e] = 0.0;
    __syncthreads();
    const double inv_step = gpfq_inv_step(alph, K, Flags[a]);
    const double tern = gpfq_ternary_radius(alph, K);
    // the walker lanes' neuron levels (once per neuron, not per block)
    double sc, inv_u, tern_u;
    sweep_unit_levels<SCALED>(scales, (int64_t)a * nj + jt + (tid >> 2), tid < 4 * NT && jt + (tid >> 2) < nj, alph, K, Flags[a], inv_step,
                              tern, &sc, &inv_u, &tern_u);
    const uint64_t key = STOCH ? gpfq_unit_key(seeds[a], u0 + jt + (tid >> 2)) : 0;

    // this thread's 16-byte chunks of every W / Q tile (fixed for the whole walk)
    int w_off[WCH];
    const double *w_src[WCH], *q_src[WCH];
    int w_bytes[WCH];
#pragma unroll
    for (int i = 0; i < WCH; ++i) {
        const int idx = tid + i * THREADS, r = idx / (KC / 2), c = idx % (KC / 2);
        const bool in_tile = idx < NT * (KC / 2);
        const bool ok = in_tile && (jt + r < nj);
        w_off[i] = in_tile ? r * LD + c * 2 : -1;
        w_src[i] = Wt + (ok ? (jt + r) * N0 + c * 2 : 0);
        q_src[i] = Qa + (ok ? (jt + r) * N0 + c * 2 : 0);
        w_bytes[i] = ok ? 16 : 0;
    }

    const int nblk = (int)((t_end - t_begin + B - 1) / B);
    const double *Da = Dt ? Dt + (int64_t)a * nj * ldd : nullptr;
    for (int b = 0; b < nblk; ++b) {
        const int64_t t0 = t_begin + (int64_t)b * B;
        const int nb = (int)((t_end - t0) < B ? (t_end - t0) : B);
        // ---- the block's own operands: requested now, parked in registers while the panel runs
        double pg1[DPT], pg2[DPT], pw[WPT], pd[WPT];
#pragma unroll
        for (int i = 0; i < DPT; ++i) {
            const int e = tid + i * THREADS, r = e / B, c = e % B;
            const bool ok = r < nb && c <= r;
            pg1[i] = ok ? __ldg(G1 + (t0 + r) * ldg + t0 + c) : 0.0;
            pg2[i] = ok ? __ldg(G2 + (t0 + r) * ldg + t0 + c) : 0.0;
        }
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int e = tid + i * THREADS, j = e / B, t = e % B;
            const bool ok = e < NT * B && jt + j < nj && t < nb;
            pw[i] = ok ? __ldg(Wt + (jt + j) * N0 + t0 + t) : 0.0;
            pd[i] = (ok && Da) ? __ldg(Da + (jt + j) * ldd + (t0 - t_begin) + t) : 0.0;  // prior ranges
        }
        // ---- panel: contributions of the earlier blocks of this range
        int g_off[GCH], g_bytes[GCH];
        const double *g1_src[GCH], *g2_src[GCH];
#pragma unroll
        for (int i = 0; i < GCH; ++i) {
            const int idx = tid + i * THREADS, r = idx / (KC / 2), c = idx % (KC / 2);
            const bool ok = t0 + r < N0;
            g_off[i] = r * LD + c * 2;
            g1_src[i] = G1 + (ok ? (t0 + r) * ldg + c * 2 : 0);
            g2_src[i] = G2 + (ok ? (t0 + r) * ldg + c * 2 : 0);
            g_bytes[i] = ok ? 16 : 0;
        }
        double acc[NA][2];
#pragma unroll
        for (int i = 0; i < NA; ++i) acc[i][0] = acc[i][1] = 0.0;
        const int nck = (b * B + KC - 1) / KC;  // chunks per segment: the b * 32 earlier directions of this range
        const int total = 2 * nck;              // nck of (G1, W), then nck of (G2, Q)
        auto issue = [&](int it) {
            if (it < total) {
                const int seg = it >= nck;
                const int krel = (seg ? it - nck : it) * KC;   // first direction of the chunk, relative to t_begin
                const int64_t k0 = t_begin + krel;
                const int kleft = b * B - krel;                // directions of the chunk that exist (a multiple of 32)
                const int st = it % STAGES;
                if (ALIGNED) {
#pragma unroll
                    for (int i = 0; i < GCH; ++i) {
                        const bool in = ((tid + i * THREADS) % (KC / 2)) * 2 < kleft;
                        cp_async16(gst + st * B * LD + g_off[i], in ? (seg ? g2_src[i] : g1_src[i]) + k0 : G1, in ? g_bytes[i] : 0);
                    }
#pragma unroll
                    for (int i = 0; i < WCH; ++i)
                        if (w_off[i] >= 0) {
                            const bool in = ((tid + i * THREADS) % (KC / 2)) * 2 < kleft;
                            cp_async16(wst + st * NT * LD + w_off[i], in ? (seg ? q_src[i] : w_src[i]) + k0 : Wt, in ? w_bytes[i] : 0);
                        }
                } else {
                    load_tile<double, B, KC, THREADS, false>(gst + st * B * LD, seg ? G2 : G1, ldg, t0, N0, k0, t0);
                    load_tile<double, NT, KC, THREADS, false>(wst + st * NT * LD, seg ? Qa : Wt, N0, jt, nj, k0, t0);
                }
            }
            cp_async_commit();
        };
        auto contract = [&](const double *gs, const double *ws, bool neg) {
            const double *as = gs + (strip * 8 + grp) * LD + tig + khalf * (KC / 2);
            const double *bs = ws + grp * LD + tig + khalf * (KC / 2);
#pragma unroll
            for (int kk = 0; kk < KC / 2; kk += 4) {
                const double av = neg ? -as[kk] : as[kk];
#pragma unroll
                for (int i = 0; i < NA; ++i) dmma_m8n8k4(acc[i][0], acc[i][1], av, bs[i * 8 * LD + kk]);
            }
        };
        issue(0);
        issue(1);
        for (int it = 0; it < total; ++it) {
            cp_async_wait<1>();
            __syncthreads();  // chunk `it` landed for everyone; chunk it-1 fully consumed
            issue(it + 2);
            const int st = it % STAGES;
            contract(gst + st * B * LD, wst + st * NT * LD, it >= nck);
        }
        cp_async_wait<0>();
        __syncthreads();      // every warp is done with the ring: stage 0 takes the block's own (masked) tile
        // ---- stage the block's operands
#pragma unroll
        for (int i = 0; i < DPT; ++i) {
            const int e = tid + i * THREADS, r = e / B, c = e % B;
            g2d[r * (B + 1) + c] = pg2[i];
            gst[r * LD + c] = c < r ? pg1[i] : 0.0;   // strictly lower: what w_s (s < t, same block) adds to d_t
            if (KC > B) gst[r * LD + B + c] = 0.0;    // the block's own chunk is 32 directions wide: zero the rest
            if (c == r) {
                const double nv = r < nb ? (double)(float)sqrt(pg2[i]) : 0.0;
                nrm[r] = nv;
                rinv[r] = nv < GPFQ_DEAD_NORM ? 0.0 : 1.0 / (nv * nv);
                g1dd[r] = pg1[i];
            }
        }
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int e = tid + i * THREADS, j = e / B, t = e % B;
            if (e < NT * B) {
                wblk[j * (B + 1) + t] = pw[i];
                qblk[j * (B + 1) + t] = pd[i];
                wst[j * LD + t] = pw[i];
                if (KC > B) wst[j * LD + B + t] = 0.0;
            }
        }
        __syncthreads();
        contract(gst, wst, false);
#pragma unroll
        for (int i = 0; i < NA; ++i) {
            double *dp = dsm + khalf * B * (NT + 1) + (strip * 8 + grp) * (NT + 1) + i * 8 + tig * 2;
            dp[0] = acc[i][0];
            dp[1] = acc[i][1];
        }
        __syncthreads();
        // ---- the walk: FOUR lanes per neuron (lane = 4 j + r) take neuron jt + j through the block's 32 directions.
        // Lane r keeps the residual dots of directions = r (mod 4) in d[0..7]; a step broadcasts the current direction's
        // dot from its owner lane (one 64-bit shuffle), all four lanes take the same decision, and each applies the
        // q-term to its own eight directions -- 8 instead of 31 LDS + DFMA per lane and step on the serial path.
        // The loop over groups of four steps is ROLLED (unrolled it is 160 KB of straight-line code: instruction-fetch
        // bound); the register file shifts down one slot per group, folded into the group's last update, so the body
        // is the same for every group; rows 32..63 of the G2 tile are zeros.
        if (tid < 4 * NT) {
            const int j = tid >> 2, r = tid & 3;
            double d[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {  // prior ranges + the two K-halves of this range's panel, in fixed order
                const int t = 4 * i + r;
                d[i] = qblk[j * (B + 1) + t] + (dsm[t * (NT + 1) + j] + dsm[B * (NT + 1) + t * (NT + 1) + j]);
            }
            __syncwarp();  // every lane has read its prior-range values before the first q lands in qblk
            const double tau_l = L1 ? gpfq_l1_tau(lambdas[a], nrm[lane]) : 0.0;   // tau of direction `lane` of the block
            const double *wrow = wblk + j * (B + 1);
            double *qrow = qblk + j * (B + 1);
            const int ngrp = (nb + 3) >> 2;
#pragma unroll 1
            for (int g4 = 0; g4 < ngrp; ++g4) {
                const double *gbase = g2d + (4 * g4 + r) * (B + 1) + 4 * g4;  // G2[4 (g4 + i) + r][4 g4 + rr] at gbase[4 i (B+1) + rr]
#pragma unroll
                for (int rr = 0; rr < 4; ++rr) {
                    const int tt = 4 * g4 + rr;
                    const double d0 = __shfl_sync(0xffffffffu, d[0], (lane & ~3) + rr);
                    const double wv = wrow[tt];
                    const double num = fma(wv, g1dd[tt], d0);
                    double q = L1 ? gpfq_decide_rcp_l1<SCALED, STOCH>(nrm[tt], rinv[tt], d0, num, wv, alph, K, inv_u, tern_u, sc,
                                                                      STOCH ? gpfq_draw(key, t0 + tt) : 0.0,
                                                                      __shfl_sync(0xffffffffu, tau_l, tt))
                             : STOCH ? gpfq_decide_rcp_stoch<SCALED>(nrm[tt], rinv[tt], d0, num, wv, alph, K, inv_u, tern_u, sc,
                                                                     gpfq_draw(key, t0 + tt))
                                     : gpfq_decide_rcp_unit<SCALED>(nrm[tt], rinv[tt], d0, num, wv, alph, K, inv_u, tern_u, sc);
                    if (tt >= nb) q = 0.0;  // past the end of a partial block: no decision, no update
                    if (r == rr && tt < nb) qrow[tt] = q;
                    if (rr < 3) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) d[i] = fma(-gbase[4 * i * (B + 1) + rr], q, d[i]);
                    } else {  // last step of the group: slot 0 is spent in every lane, shift down while updating
#pragma unroll
                        for (int i = 0; i < 7; ++i) d[i] = fma(-gbase[4 * (i + 1) * (B + 1) + rr], q, d[i + 1]);
                        d[7] = 0.0;
                    }
                }
            }
        }
        __syncthreads();
        for (int e = tid; e < NT * B; e += THREADS) {
            const int j = e / B, t = e % B;
            if (jt + j < nj && t < nb) Qa[(jt + j) * N0 + t0 + t] = qblk[j * (B + 1) + t];
        }
        __syncthreads();  // Q block visible to this CTA's later panel loads
    }
}

// ---------------------------------------------------------------------------------------------
// Pipelined range walk: the same work as sweep_tile_kernel, but the panel of block b + 1 is contracted WHILE block b is being
// walked.  In sweep_tile_kernel a block costs panel + walk back to back (measured 12.9 us per block of 32 directions, of
// which the serial walk is 6 us); here four warps (the "contractors") prepare block b + 1 -- the contributions of every
// direction whose decision is already known, i.e. the W terms of all earlier directions of the range and the Q terms of
// blocks <= b - 1 -- underneath the walk of block b by the walker warps (4 lanes per neuron, as before), and only ONE
// 32-direction chunk, G2[block b + 1, block b] x Q_b, remains between two walks.  Two working sets (block operands, prior
// dots, decisions) alternate between the roles; named barriers hand them over:
//   READY[s]      contractors -> walkers: set s holds block b's operands and residual dots
//   WALK_DONE[s]  walkers -> contractors: the decisions of block b are in set s (and in Qt)
// One CTA per SM (up to 200 KB of shared memory); the host uses it when every CTA of the launch is resident at once.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void named_bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;\n" ::"r"(id), "r"(count) : "memory"); }

template <int NT>
struct PipeCfg {
    // K chunks of 64 directions through a cp.async ring, four deep where shared memory allows (three chunks in flight: the
    // contractors are bound by the L2 latency of their chunk loads, and late blocks of a range have up to 15 chunks to get through
    // while one block is walked)
    static constexpr int B = SWEEP_B, KC = 64, LD = KC + 4, STAGES = NT == 32 ? 3 : 4, THREADS = 256, CT = 128;
    static constexpr int SET = 2 * B * (B + 1) + 2 * NT * (B + 1) + B * (NT + 1) + 3 * B;   // doubles per working set
    static constexpr size_t SMEM = sizeof(double) * ((size_t)STAGES * (B + NT) * LD + 2 * SET + GPFQ_MAX_K);
};

template <int NT, bool SCALED = false, bool STOCH = false, bool L1 = false>
__global__ void __launch_bounds__(256, 1)
sweep_pipe_kernel(const double *__restrict__ G1, const double *__restrict__ G2, int64_t ldg, int64_t N0,
                  const double *__restrict__ Wt, double *__restrict__ Qt, int64_t nj, const double *__restrict__ alphabets,
                  const int *__restrict__ Koff, const int *__restrict__ Flags, int64_t t_begin, int64_t t_end,
                  const double *__restrict__ Dt, int64_t ldd, const double *__restrict__ scales = nullptr,
                  const uint64_t *__restrict__ seeds = nullptr, int64_t u0 = 0, const double *__restrict__ lambdas = nullptr) {
    using Cfg = PipeCfg<NT>;
    constexpr int B = Cfg::B, KC = Cfg::KC, LD = Cfg::LD, STAGES = Cfg::STAGES, CT = Cfg::CT, NA = NT / 8, NW = 4 * NT;
    constexpr int BAR_C = 1, BAR_READY = 2, BAR_WALK_DONE = 4, BAR_Q_STORED = 6, HANDOVER = NW + CT;
    extern __shared__ __align__(16) unsigned char sweep_smem[];
    double *gst = reinterpret_cast<double *>(sweep_smem);   // STAGES x B x LD   (Gram rows of the block being prepared)
    double *wst = gst + STAGES * B * LD;                    // STAGES x NT x LD  (W or Q panel of the tile)
    double *sets = wst + STAGES * NT * LD;                  // 2 working sets
    double *alph = sets + 2 * Cfg::SET;
    auto g2d_of = [&](int s) { return sets + s * Cfg::SET; };                  // 2B x (B+1): G2 diagonal tile, then B rows of zeros
    auto wblk_of = [&](int s) { return g2d_of(s) + 2 * B * (B + 1); };         // NT x (B+1)
    auto qblk_of = [&](int s) { return wblk_of(s) + NT * (B + 1); };           // NT x (B+1): prior dots in, decisions out
    auto dsm_of = [&](int s) { return qblk_of(s) + NT * (B + 1); };            // B x (NT+1): this range's part of the dots
    auto nrm_of = [&](int s) { return dsm_of(s) + B * (NT + 1); };             // B, then rinv (B), then G1[t][t] (B)

    const int a = blockIdx.y;
    const int K = Koff[a + 1] - Koff[a];
    const int64_t jt = (int64_t)blockIdx.x * NT;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    double *Qa = Qt + (int64_t)a * nj * N0;
    for (int e = tid; e < K; e += 256) alph[e] = alphabets[Koff[a] + e];
    for (int e = tid; e < 2 * B * (B + 1); e += 256) g2d_of(e / (B * (B + 1)))[B * (B + 1) + e % (B * (B + 1))] = 0.0;
    __syncthreads();
    const double inv_step = gpfq_inv_step(alph, K, Flags[a]);
    const double tern = gpfq_ternary_radius(alph, K);
    const int nblk = (int)((t_end - t_begin + B - 1) / B);
    const double *Da = Dt ? Dt + (int64_t)a * nj * ldd : nullptr;

    if (warp >= 4) {
        // =============================== contractors ===============================
        const int ct = tid - 128, cw = warp - 4, grp = lane >> 2, tig = lane & 3;
        constexpr int GCH = B * (KC / 2) / CT;                      // 16-byte pieces of a Gram chunk per thread (8)
        constexpr int WCH = (NT * (KC / 2) + CT - 1) / CT;          // ... of a W / Q chunk per thread (2, 4, 8)
        constexpr int DPT = B * B / CT;                             // diagonal-tile entries per thread (8)
        constexpr int WPT = (NT * B + CT - 1) / CT;                 // W-block entries per thread (2, 4, 8)
        int w_off[WCH], w_bytes[WCH];
        const double *w_src[WCH], *q_src[WCH];
#pragma unroll
        for (int i = 0; i < WCH; ++i) {
            const int idx = ct + i * CT, r = idx / (KC / 2), c = idx % (KC / 2);
            const bool in_tile = idx < NT * (KC / 2);
            const bool ok = in_tile && (jt + r < nj);
            w_off[i] = in_tile ? r * LD + c * 2 : -1;
            w_src[i] = Wt + (ok ? (jt + r) * N0 + c * 2 : 0);
            q_src[i] = Qa + (ok ? (jt + r) * N0 + c * 2 : 0);
            w_bytes[i] = ok ? 16 : 0;
        }
        for (int b = 0; b < nblk; ++b) {
            const int s = b & 1;
            const int64_t t0 = t_begin + (int64_t)b * B;
            const int nb = (int)((t_end - t0) < B ? (t_end - t0) : B);
            if (b > 0) named_bar_sync(BAR_C, CT);   // every contractor is done with ring slots 0 / 1 of the previous block
            // the early panel reads the decisions of blocks <= b-2 from Qt: block b-2's have been stored (long ago: its walk ended
            // before block b-1 was even handed over)
            if (b >= 2) named_bar_sync(BAR_Q_STORED + (s & 1), HANDOVER);
            // ---- the block's own operands and its G2 tile against the previous block: requested now, parked in registers
            double pg1[DPT], pg2[DPT], pgp[DPT], pw[WPT], pd[WPT];
#pragma unroll
            for (int i = 0; i < DPT; ++i) {
                const int e = ct + i * CT, r = e / B, c = e % B;
                const bool ok = r < nb && c <= r;
                pg1[i] = ok ? __ldg(G1 + (t0 + r) * ldg + t0 + c) : 0.0;
                pg2[i] = ok ? __ldg(G2 + (t0 + r) * ldg + t0 + c) : 0.0;
                pgp[i] = (b > 0 && r < nb) ? __ldg(G2 + (t0 + r) * ldg + t0 - B + c) : 0.0;
            }
#pragma unroll
            for (int i = 0; i < WPT; ++i) {
                const int e = ct + i * CT, j = e / B, t = e % B;
                const bool ok = e < NT * B && jt + j < nj && t < nb;
                pw[i] = ok ? __ldg(Wt + (jt + j) * N0 + t0 + t) : 0.0;
                pd[i] = (ok && Da) ? __ldg(Da + (jt + j) * ldd + (t0 - t_begin) + t) : 0.0;  // prior ranges
            }
            // ---- early panel: W terms of blocks 0 .. b-1, Q terms of blocks 0 .. b-2 (block b-1 is being walked right now)
            int g_off[GCH], g_bytes[GCH];
            const double *g1_src[GCH], *g2_src[GCH];
#pragma unroll
            for (int i = 0; i < GCH; ++i) {
                const int idx = ct + i * CT, r = idx / (KC / 2), c = idx % (KC / 2);
                const bool ok = t0 + r < N0;
                g_off[i] = r * LD + c * 2;
                g1_src[i] = G1 + (ok ? (t0 + r) * ldg + c * 2 : 0);
                g2_src[i] = G2 + (ok ? (t0 + r) * ldg + c * 2 : 0);
                g_bytes[i] = ok ? 16 : 0;
            }
            double acc[NA][2];
#pragma unroll
            for (int i = 0; i < NA; ++i) acc[i][0] = acc[i][1] = 0.0;
            const int n1 = b * B, n2 = b > 0 ? (b - 1) * B : 0;
            const int nck1 = (n1 + KC - 1) / KC, nck2 = (n2 + KC - 1) / KC, total = nck1 + nck2;
            auto issue = [&](int it) {
                if (it < total) {
                    const int seg = it >= nck1;
                    const int krel = (seg ? it - nck1 : it) * KC;
                    const int64_t k0 = t_begin + krel;
                    const int kleft = (seg ? n2 : n1) - krel;      // directions of the chunk that exist (a multiple of 32)
                    const int st = it % STAGES;
#pragma unroll
                    for (int i = 0; i < GCH; ++i) {
                        const bool in = ((ct + i * CT) % (KC / 2)) * 2 < kleft;
                        cp_async16(gst + st * B * LD + g_off[i], in ? (seg ? g2_src[i] : g1_src[i]) + k0 : G1, in ? g_bytes[i] : 0);
                    }
#pragma unroll
                    for (int i = 0; i < WCH; ++i)
                        if (w_off[i] >= 0) {
                            const bool in = ((ct + i * CT) % (KC / 2)) * 2 < kleft;
                            cp_async16(wst + st * NT * LD + w_off[i], in ? (seg ? q_src[i] : w_src[i]) + k0 : Wt, in ? w_bytes[i] : 0);
                        }
                }
                cp_async_commit();
            };
            auto contract = [&](const double *gs, const double *ws, bool neg, int kmax) {
                const double *as = gs + (cw * 8 + grp) * LD + tig;
                const double *bs = ws + grp * LD + tig;
#pragma unroll 4
                for (int kk = 0; kk < kmax; kk += 4) {
                    const double av = neg ? -as[kk] : as[kk];
#pragma unroll
                    for (int i = 0; i < NA; ++i) dmma_m8n8k4(acc[i][0], acc[i][1], av, bs[i * 8 * LD + kk]);
                }
            };
#pragma unroll
            for (int p = 0; p < STAGES - 1; ++p) issue(p);
            for (int it = 0; it < total; ++it) {
                cp_async_wait<STAGES - 2>();
                named_bar_sync(BAR_C, CT);  // chunk `it` landed for every contractor; chunk it-1 fully consumed
                issue(it + STAGES - 1);
                const int st = it % STAGES;
                contract(gst + st * B * LD, wst + st * NT * LD, it >= nck1, KC);
            }
            cp_async_wait<0>();
            named_bar_sync(BAR_C, CT);      // the ring is idle: slot 0 takes the block's own (masked) tile, slot 1 the tile
                                            // against the previous block
            // ---- working set s (its last reader, the walk of block b-2, is over: WALK_DONE of b-2 was awaited while
            //      preparing block b-1) and the two register-parked tiles
            double *g2d = g2d_of(s), *wblk = wblk_of(s), *qblk = qblk_of(s), *nrm = nrm_of(s), *rinv = nrm + B, *g1dd = rinv + B;
            double *gst1 = gst + B * LD, *wst1 = wst + NT * LD;
#pragma unroll
            for (int i = 0; i < DPT; ++i) {
                const int e = ct + i * CT, r = e / B, c = e % B;
                g2d[r * (B + 1) + c] = pg2[i];
                gst[r * LD + c] = c < r ? pg1[i] : 0.0;   // strictly lower: what w_s (s < t, same block) adds to d_t
                gst1[r * LD + c] = pgp[i];
                if (c == r) {
                    const double nv = r < nb ? (double)(float)sqrt(pg2[i]) : 0.0;
                    nrm[r] = nv;
                    rinv[r] = nv < GPFQ_DEAD_NORM ? 0.0 : 1.0 / (nv * nv);
                    g1dd[r] = pg1[i];
                }
            }
#pragma unroll
            for (int i = 0; i < WPT; ++i) {
                const int e = ct + i * CT, j = e / B, t = e % B;
                if (e < NT * B) {
                    wblk[j * (B + 1) + t] = pw[i];
                    qblk[j * (B + 1) + t] = pd[i];
                    wst[j * LD + t] = pw[i];
                }
            }
            named_bar_sync(BAR_C, CT);
            contract(gst, wst, false, B);
            if (b > 0) {
                named_bar_sync(BAR_WALK_DONE + (s ^ 1), HANDOVER);   // block b-1 is walked: its decisions sit in the other set
                const double *qprev = qblk_of(s ^ 1);
#pragma unroll
                for (int i = 0; i < WPT; ++i) {
                    const int e = ct + i * CT, j = e / B, t = e % B;
                    if (e < NT * B) wst1[j * LD + t] = qprev[j * (B + 1) + t];
                }
                named_bar_sync(BAR_C, CT);
                contract(gst1, wst1, true, B);
            }
            double *dsm = dsm_of(s);
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                double *dp = dsm + (cw * 8 + grp) * (NT + 1) + i * 8 + tig * 2;
                dp[0] = acc[i][0];
                dp[1] = acc[i][1];
            }
            __threadfence_block();
            named_bar_arrive(BAR_READY + s, HANDOVER);
        }
    } else if (tid < NW) {
        // =============================== walkers: FOUR lanes per neuron (lane = 4 j + r) ===============================
        const int j = tid >> 2, r = tid & 3;
        double sc, inv_u, tern_u;
        sweep_unit_levels<SCALED>(scales, (int64_t)a * nj + jt + j, jt + j < nj, alph, K, Flags[a], inv_step, tern, &sc, &inv_u,
                                  &tern_u);
        const uint64_t key = STOCH ? gpfq_unit_key(seeds[a], u0 + jt + j) : 0;
        for (int b = 0; b < nblk; ++b) {
            const int s = b & 1;
            const int64_t t0 = t_begin + (int64_t)b * B;
            const int nb = (int)((t_end - t0) < B ? (t_end - t0) : B);
            named_bar_sync(BAR_READY + s, HANDOVER);
            const double *g2d = g2d_of(s), *wrow = wblk_of(s) + j * (B + 1), *dsm = dsm_of(s), *nrm = nrm_of(s), *rinv = nrm + B, *g1dd = rinv + B;
            double *qrow = qblk_of(s) + j * (B + 1);
            double d[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {  // prior ranges + this range's panel
                const int t = 4 * i + r;
                d[i] = qrow[t] + dsm[t * (NT + 1) + j];
            }
            __syncwarp();  // every lane has read its prior-range values before the first q lands in qblk
            const double tau_l = L1 ? gpfq_l1_tau(lambdas[a], nrm[lane]) : 0.0;   // tau of direction `lane` of the block
            const int ngrp = (nb + 3) >> 2;
#pragma unroll 1
            for (int g4 = 0; g4 < ngrp; ++g4) {
                const double *gbase = g2d + (4 * g4 + r) * (B + 1) + 4 * g4;  // G2[4 (g4 + i) + r][4 g4 + rr] at gbase[4 i (B+1) + rr]
#pragma unroll
                for (int rr = 0; rr < 4; ++rr) {
                    const int tt = 4 * g4 + rr;
                    const double d0 = __shfl_sync(0xffffffffu, d[0], (lane & ~3) + rr);
                    const double wv = wrow[tt];
                    const double num = fma(wv, g1dd[tt], d0);
                    double q = L1 ? gpfq_decide_rcp_l1<SCALED, STOCH>(nrm[tt], rinv[tt], d0, num, wv, alph, K, inv_u, tern_u, sc,
                                                                      STOCH ? gpfq_draw(key, t0 + tt) : 0.0,
                                                                      __shfl_sync(0xffffffffu, tau_l, tt))
                             : STOCH ? gpfq_decide_rcp_stoch<SCALED>(nrm[tt], rinv[tt], d0, num, wv, alph, K, inv_u, tern_u, sc,
                                                                     gpfq_draw(key, t0 + tt))
                                     : gpfq_decide_rcp_unit<SCALED>(nrm[tt], rinv[tt], d0, num, wv, alph, K, inv_u, tern_u, sc);
                    if (tt >= nb) q = 0.0;  // past the end of a partial block: no decision, no update
                    if (r == rr && tt < nb) qrow[tt] = q;
                    if (rr < 3) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) d[i] = fma(-gbase[4 * i * (B + 1) + rr], q, d[i]);
                    } else {  // last step of the group: slot 0 is spent in every lane, shift down while updating
#pragma unroll
                        for (int i = 0; i < 7; ++i) d[i] = fma(-gbase[4 * (i + 1) * (B + 1) + rr], q, d[i + 1]);
                        d[7] = 0.0;
                    }
                }
            }
            // ---- hand the decisions over (they sit in qblk of this set) before anything else: the contractors only need them in
            // shared memory for the one chunk that separates this walk from the next
            __threadfence_block();
            named_bar_arrive(BAR_WALK_DONE + s, HANDOVER);
            // ---- this lane's own decisions (directions = r mod 4) go out to Qt, for later ranges and the result.
            // qblk of this set is rewritten only after the contractors have seen Q_STORED of this block (two blocks on).
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int tt = 4 * i + r;
                if (jt + j < nj && tt < nb) Qa[(jt + j) * N0 + t0 + tt] = qrow[tt];
            }
            if (b + 2 < nblk) {   // somebody will wait for it
                __threadfence_block();
                named_bar_arrive(BAR_Q_STORED + s, HANDOVER);
            }
        }
    }
}

template <int NT>
static int launch_sweep_pipe(gpfq_ctx *ctx, const double *G1, const double *G2, int64_t ldg, int64_t N0, const double *Wt,
                             double *Qt, int64_t nj, const double *d_alph, const int *d_koff, const int *d_flags,
                             int n_alph, int64_t t_begin, int64_t t_end, const double *Dt, int64_t ldd, const double *scales,
                             int64_t u0) {
    const size_t smem = PipeCfg<NT>::SMEM;
    dim3 grid((unsigned)ceil_div64(nj, NT), (unsigned)n_alph);
    const uint64_t *seeds = ctx->d_seeds;
    const double *lambdas = ctx->d_l1;
    auto k = seeds ? (scales ? sweep_pipe_kernel<NT, true, true> : sweep_pipe_kernel<NT, false, true>)
                   : (scales ? sweep_pipe_kernel<NT, true> : sweep_pipe_kernel<NT, false>);
    if (lambdas)
        k = seeds ? (scales ? sweep_pipe_kernel<NT, true, true, true> : sweep_pipe_kernel<NT, false, true, true>)
                  : (scales ? sweep_pipe_kernel<NT, true, false, true> : sweep_pipe_kernel<NT, false, false, true>);
    CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, 256, smem, ctx->stream>>>(G1, G2, ldg, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, t_begin, t_end, Dt, ldd, scales, seeds, u0,
                                        lambdas);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

template <int NT>
static int launch_sweep_tile(gpfq_ctx *ctx, const double *G1, const double *G2, int64_t ldg, int64_t N0, const double *Wt,
                             double *Qt, int64_t nj, const double *d_alph, const int *d_koff, const int *d_flags,
                             int n_alph, int64_t t_begin, int64_t t_end, const double *Dt, int64_t ldd, const double *scales,
                             int64_t u0) {
    const size_t smem = SweepCfg<NT>::SMEM;
    dim3 grid((unsigned)ceil_div64(nj, NT), (unsigned)n_alph);
    const bool aligned = (N0 % 2 == 0) && (ldg % 2 == 0) && ((uintptr_t)G1 % 16 == 0) && ((uintptr_t)G2 % 16 == 0) &&
                         ((uintptr_t)Wt % 16 == 0) && ((uintptr_t)Qt % 16 == 0) && ((nj * N0) % 2 == 0);
    const uint64_t *seeds = ctx->d_seeds;
    const double *lambdas = ctx->d_l1;
    auto k = seeds ? (aligned ? (scales ? sweep_tile_kernel<NT, true, true, true> : sweep_tile_kernel<NT, true, false, true>)
                              : (scales ? sweep_tile_kernel<NT, false, true, true> : sweep_tile_kernel<NT, false, false, true>))
                   : (aligned ? (scales ? sweep_tile_kernel<NT, true, true> : sweep_tile_kernel<NT, true, false>)
                              : (scales ? sweep_tile_kernel<NT, false, true> : sweep_tile_kernel<NT, false, false>));
    if (lambdas)
        k = seeds ? (aligned ? (scales ? sweep_tile_kernel<NT, true, true, true, true> : sweep_tile_kernel<NT, true, false, true, true>)
                             : (scales ? sweep_tile_kernel<NT, false, true, true, true> : sweep_tile_kernel<NT, false, false, true, true>))
                  : (aligned ? (scales ? sweep_tile_kernel<NT, true, true, false, true> : sweep_tile_kernel<NT, true, false, false, true>)
                             : (scales ? sweep_tile_kernel<NT, false, true, false, true> : sweep_tile_kernel<NT, false, false, false, true>));
    CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, 256, smem, ctx->stream>>>(G1, G2, ldg, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, t_begin, t_end, Dt, ldd, scales, seeds, u0,
                                        lambdas);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int pick_splits(gpfq_ctx *ctx, int64_t N0, int64_t m, int BM, int BN, int BK) {
    const int64_t tm = ceil_div64(N0, BM), tn = ceil_div64(N0, BN);
    int64_t tiles = 0;  // tiles touching the lower triangle
    for (int64_t i = 0; i < tm; ++i)
        for (int64_t jn = 0; jn < tn; ++jn)
            if (jn * BN <= i * BM + BM - 1) ++tiles;
    const int64_t target = 2LL * ctx->sm_count * 2;  // two CTAs per SM, two waves
    int64_t s = ceil_div64(target, tiles > 0 ? tiles : 1);
    const int64_t max_by_k = m / (8 * BK) > 0 ? m / (8 * BK) : 1;  // at least 8 k-tiles per split
    if (s > max_by_k) s = max_by_k;
    if (s > 32) s = 32;
    while (s > 1 && (size_t)s * N0 * N0 * sizeof(double) > ((size_t)2 << 30)) --s;
    return (int)(s < 1 ? 1 : s);
}

// G = A B^T over the sample axis, lower triangle (+ diagonal tiles).  A, B: (N0, m) fp32 device.
static int gram_stage(gpfq_ctx *ctx, const float *A, const float *B, int64_t ld, int64_t N0, int64_t m,
                      double *G) {
    constexpr int BM = 128, BN = 64, BK = 32;
    const int nsplit = pick_splits(ctx, N0, m, BM, BN, BK);
    GemmArgs g = {};
    g.seg[0] = {A, B, ld, ld, m, 1.0};
    g.nseg = 1;
    g.M = g.N = N0;
    g.ldc = N0;
    g.nsplit = nsplit;
    g.lower_only = 1;
    if (nsplit == 1) {
        g.C = G;
        g.split_stride = 0;
        GPFQ_TRY((launch_gemm_nt<float, BM, BN, BK>(ctx, g, 1)));
    } else {
        double *part = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_PART, (size_t)nsplit * N0 * N0 * sizeof(double), (void **)&part));
        g.C = part;
        g.split_stride = N0 * N0;
        GPFQ_TRY((launch_gemm_nt<float, BM, BN, BK>(ctx, g, 1)));
        const int64_t n = N0 * N0;
        int blocks = (int)(ceil_div64(n, 256) < 4096 ? ceil_div64(n, 256) : 4096);
        reduce_splits_kernel<<<blocks, 256, 0, ctx->stream>>>(part, nsplit, N0 * N0, G, n);
        KERNEL_CHECK(ctx);
    }
    return GPFQ_OK;
}

// Which kernel computes the Dense Grams: the int8-slice tcgen05 kernel (gram_i8.cu) when the layer is large enough
// to feed it and its slice workspace fits, else the fp64 DMMA contraction above.  ctx->gram_variant forces one.
size_t gram_i8_workspace_bytes(gpfq_ctx *, int64_t, int64_t, bool);
int gram_i8_stage(gpfq_ctx *, const float *, const float *, int64_t, int64_t, int64_t, double *, double *);

bool dense_gram_uses_i8(gpfq_ctx *ctx, int64_t N0, int64_t m, bool same) {
    if (ctx->gram_variant == 1) return false;
    if (N0 > 65000 || m >= ((int64_t)1 << 31) - 256) return false;
    if (ctx->gram_variant != 2 && (N0 < 256 || m < 1024)) return false;
    // an earlier call of this size or smaller ran out of device memory for the slices: do not try again
    return ctx->i8_oom_bytes == 0 || gram_i8_workspace_bytes(ctx, N0, m, same) < ctx->i8_oom_bytes;
}

int dense_gram_only(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m, double *G1,
                    double *G2) {
    const bool same = G1 == G2;
    if (dense_gram_uses_i8(ctx, N0, m, same)) {
        ctx->last_gram_kernel = 2;
        const int rc = gram_i8_stage(ctx, same ? Xq : X, Xq, ldx, N0, m, G1, G2);
        if (rc != GPFQ_ERR_OOM) return rc;
        ctx->i8_oom_bytes = gram_i8_workspace_bytes(ctx, N0, m, same);  // workspaces are allocated before any launch
        ctx->err.clear();
    }
    ctx->last_gram_kernel = 1;
    GPFQ_TRY(gram_stage(ctx, Xq, Xq, ldx, N0, m, G2));
    if (!same) GPFQ_TRY(gram_stage(ctx, Xq, X, ldx, N0, m, G1));
    return GPFQ_OK;
}

// ---------------------------------------------------------------------------------------------
// Low-rank form of the outer level (m << N0, e.g. VGG16 fc1: N0 = 25088, m = 1504).
// What the directions before a range contribute to it is  D[t] = <X~_t, u>  with the residual
//     u = sum_{s < range} (w_s X_s - q_s X~_s)   (m numbers per neuron)   -- quantized_network.py:119 itself,
// so instead of contracting Gram rows over ALL earlier directions (2 R tb nj MACs per range, N0^2 nj in total) the
// residuals U (nj x m, fp64) are carried along:   U += W_range X_range - Q_range X~_range   (2 R m nj MACs),
// D_range = U X~_range^T (R m nj MACs): 3 m N0 nj in total, and only the block-diagonal R x R Gram tiles are ever
// computed.  Same exact-product numerics as the Gram form; the range walk (sweep_tile_kernel) is unchanged.
// ---------------------------------------------------------------------------------------------
// Xd[t][i] = (double) X[t][i]  and  Xt[i][t] = (double) X[t][i]
__global__ void widen_transpose_kernel(const float *__restrict__ X, int64_t ldx, int64_t N0, int64_t m,
                                       double *__restrict__ Xd, double *__restrict__ Xt) {
    __shared__ float tile[32][33];
    const int64_t ib = (int64_t)blockIdx.x * 32, tb = (int64_t)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t t = tb + r, i = ib + threadIdx.x;
        const float v = (t < N0 && i < m) ? X[t * ldx + i] : 0.f;
        tile[r][threadIdx.x] = v;
        if (t < N0 && i < m) Xd[t * m + i] = (double)v;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t i = ib + r, t = tb + threadIdx.x;
        if (i < m && t < N0) Xt[i * N0 + t] = (double)tile[threadIdx.x][r];
    }
}

static bool dense_uses_lowrank(gpfq_ctx *ctx, int64_t N0, int64_t m, int64_t nj, int n_alph, bool same, bool i8_ok) {
    if (ctx->lowrank_variant == 1) return false;
    if (ctx->lowrank_variant >= 2) return N0 > 64;
    if (!i8_ok) return 3 * m < N0 && N0 >= 4096 && nj >= 256;   // fp64 (DMMA) contractions: the measured rule of round 1
    // int8-slice contractions (slgemm_i8.cu) and the tensor-core range walk (sweep_tc.cu).  Both forms calibrated on this pool's B200
    // (tools/dense_methods.py, profiles/dense_methods_r2.md):
    //   carried residuals  39 slice-pair products of nj x m x N0 at an effective 1.08e15 int8 op/s (the kernels are bound by their
    //                      operand stream from L2 and per-CTA latency, not by the tensor pipe) + 0.265 us per direction for the
    //                      chain update -> slicing -> dots -> walk of every range (~135 us per 512 directions, whatever nj)
    //   Gram rows          N0^2 nj fp64 MACs at 1.2e13 /s (DMMA contraction) + 0.1 us per direction (walk) + the full tcgen05
    //                      Gram stage (15 pairs)
    // m > N0 (config 4's 4096 x 4096 at m = 5000: 6.9 against 8.5 ms) only with thousands of neurons to amortise the chain.
    if (N0 < 1024 || nj < 64) return false;
    if (m > N0 && (nj < 2048 || m > 2 * N0)) return false;
    // few samples against many directions (VGG16's fc layers, also one rank's shard of them: 125 neurons of fc3 measured 2.26 ms by
    // Gram rows -- the full Gram stage at m = 1504 runs far below the rate assumed here -- against ~1.4 ms in the residual form)
    if (2 * m <= N0 && N0 >= 4096) return true;
    const double grams = same ? 1.0 : 2.0;
    const double t_lr = 7.2e-14 * nj * (double)m * N0 + 0.265e-6 * N0 + 0.1e-3;
    const double t_gr = (double)N0 * N0 * nj / 1.2e13 + 0.1e-6 * N0 + grams * 15.0 * (double)N0 * N0 * m / 2.2e15 + 0.3e-3;
    return t_lr < t_gr;
}

static int64_t pick_range_length(gpfq_ctx *ctx, int64_t nj, int n_alph) {
    // R: a multiple of the contraction's 64-column tile that fills whole rounds of CTA slots (two CTAs per SM)
    const int64_t slots = 2LL * ctx->sm_count, tiles_m = ceil_div64(nj, 128) * n_alph;
    int64_t R = SWEEP_OUTER;
    if (tiles_m * 8 >= ctx->sm_count) {
        double best = 0.0;
        for (int64_t n = 5; n <= 12; ++n) {
            const int64_t tiles = tiles_m * n;
            const double eff = (double)tiles / (double)(ceil_div64(tiles, slots) * slots) - 0.004 * (double)llabs(n - 8);
            if (eff > best) { best = eff; R = 64 * n; }
        }
    }
    return R;
}

static int dispatch_sweep_tile(gpfq_ctx *ctx, int NT, const double *G1, const double *G2, int64_t ldg, int64_t N0,
                               const double *Wt, double *Qt, int64_t nj, const double *d_alph, const int *d_koff,
                               const int *d_flags, int n_alph, int64_t tb, int64_t te, const double *Dp, int64_t R,
                               const double *scales, int64_t u0) {
    // The pipelined walk (one CTA per SM) when its 16-byte copies are possible and every CTA of the launch is resident at
    // once; the narrowest neuron tile that allows it.
    const bool aligned = (N0 % 2 == 0) && (ldg % 2 == 0) && ((uintptr_t)G1 % 16 == 0) && ((uintptr_t)G2 % 16 == 0) &&
                         ((uintptr_t)Wt % 16 == 0) && ((uintptr_t)Qt % 16 == 0) && ((nj * N0) % 2 == 0);
    if (aligned) {
        const int64_t sms = ctx->sm_count;
        if (ceil_div64(nj, 8) * n_alph <= sms)
            return launch_sweep_pipe<8>(ctx, G1, G2, ldg, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, n_alph, tb, te, Dp, R, scales, u0);
        if (ceil_div64(nj, 16) * n_alph <= sms)
            return launch_sweep_pipe<16>(ctx, G1, G2, ldg, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, n_alph, tb, te, Dp, R, scales, u0);
        if (ceil_div64(nj, 32) * n_alph <= sms)
            return launch_sweep_pipe<32>(ctx, G1, G2, ldg, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, n_alph, tb, te, Dp, R, scales, u0);
    }
    if (NT == 32) return launch_sweep_tile<32>(ctx, G1, G2, ldg, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, n_alph, tb, te, Dp, R, scales, u0);
    if (NT == 16) return launch_sweep_tile<16>(ctx, G1, G2, ldg, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, n_alph, tb, te, Dp, R, scales, u0);
    return launch_sweep_tile<8>(ctx, G1, G2, ldg, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, n_alph, tb, te, Dp, R, scales, u0);
}

// Sweep with the low-rank outer level.  Wt (nj, N0) is ready; Qt (n_alph, nj, N0) receives the result.  scales (nullable):
// (n_alph, nj) per-neuron scales.
static int dense_lowrank_sweep(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m,
                               const double *Wt, double *Qt, int64_t nj, const double *d_alph, const int *d_koff,
                               const int *d_flags, int n_alph, int NT, const double *scales, int64_t u0) {
    const bool same = (Xq == X);
    cudaStream_t st = ctx->stream;
    const int64_t R = pick_range_length(ctx, nj, n_alph);
    double *Xd = nullptr, *Xt = nullptr, *Xqd = nullptr, *Xqt = nullptr, *Ut = nullptr, *Gc1 = nullptr, *Gc2 = nullptr, *Do = nullptr;
    const size_t xbytes = (size_t)N0 * m * sizeof(double);
    GPFQ_TRY(gpfq_ws(ctx, WS_LR_XD, xbytes * (same ? 1 : 2), (void **)&Xd));
    GPFQ_TRY(gpfq_ws(ctx, WS_LR_XT, xbytes * (same ? 1 : 2), (void **)&Xt));
    Xqd = same ? Xd : Xd + (size_t)N0 * m;
    Xqt = same ? Xt : Xt + (size_t)N0 * m;
    GPFQ_TRY(gpfq_ws(ctx, WS_LR_U, (size_t)n_alph * nj * m * sizeof(double), (void **)&Ut));
    GPFQ_TRY(gpfq_ws(ctx, WS_G2, (size_t)N0 * R * sizeof(double), (void **)&Gc2));
    if (same) Gc1 = Gc2;
    else GPFQ_TRY(gpfq_ws(ctx, WS_G1, (size_t)N0 * R * sizeof(double), (void **)&Gc1));
    GPFQ_TRY(gpfq_ws(ctx, WS_DT, (size_t)n_alph * nj * R * sizeof(double), (void **)&Do));

    CUDA_TRY(ctx, gpfq_record(ctx, 2, st));
    {
        dim3 grid((unsigned)ceil_div64(m, 32), (unsigned)ceil_div64(N0, 32));
        widen_transpose_kernel<<<grid, dim3(32, 8), 0, st>>>(X, ldx, N0, m, Xd, Xt);
        KERNEL_CHECK(ctx);
        if (!same) {
            widen_transpose_kernel<<<grid, dim3(32, 8), 0, st>>>(Xq, ldx, N0, m, Xqd, Xqt);
            KERNEL_CHECK(ctx);
        }
    }
    // block-diagonal Gram tiles, compact: Gc[t][s - tb(t)], row stride R (exact fp32 x fp32 products, fp64 sums).  All full
    // ranges go down as the batches of ONE launch per Gram (a 512 x 512 lower triangle alone is ~20 CTAs), a ragged last
    // range as one more.
    const int64_t nfull = N0 / R;
    for (int which = 0; which < (same ? 1 : 2); ++which) {
        for (int64_t b0 = 0; b0 < nfull; b0 += 65535) {
            const int64_t nb = std::min<int64_t>(65535, nfull - b0), tb = b0 * R;
            GemmArgs g = {};
            g.seg[0] = {Xq + tb * ldx, (which ? X : Xq) + tb * ldx, ldx, ldx, m, 1.0};
            g.nseg = 1;
            g.M = g.N = R;
            g.C = (which ? Gc1 : Gc2) + tb * R;
            g.ldc = R;
            g.nsplit = 1;
            g.lower_only = 1;
            g.batch_strideA0 = R * ldx;
            g.batch_strideB = R * ldx;
            g.batch_strideC = R * R;
            GPFQ_TRY((launch_gemm_nt<float, 128, 64, 32>(ctx, g, (int)nb)));
        }
        if (nfull * R < N0) {
            const int64_t tb = nfull * R;
            GemmArgs g = {};
            g.seg[0] = {Xq + tb * ldx, (which ? X : Xq) + tb * ldx, ldx, ldx, m, 1.0};
            g.nseg = 1;
            g.M = g.N = N0 - tb;
            g.C = (which ? Gc1 : Gc2) + tb * R;
            g.ldc = R;
            g.nsplit = 1;
            g.lower_only = 1;
            GPFQ_TRY((launch_gemm_nt<float, 128, 64, 32>(ctx, g, 1)));
        }
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 3, st));
    CUDA_TRY(ctx, cudaMemsetAsync(Ut, 0, (size_t)n_alph * nj * m * sizeof(double), st));
    cudaStream_t side = ctx->copy_stream;
    if (n_alph == 1 && nj >= 2048 && ctx->lowrank_variant != 3) {   // measured: 512 neurons run faster as one chain
        // Two independent half-problems on two streams: neurons are independent, so while one half sits in the
        // latency-bound walk of a range (one CTA per neuron tile, DMMA pipe idle) the other half's contractions run,
        // and vice versa -- the hardware interleaves the two chains, nothing else synchronises them.
        const int64_t half = ceil_div64(ceil_div64(nj, 2), 128) * 128;
        const int64_t one = nj * R;
        const int64_t tiles_h = ceil_div64(half, 128) * ceil_div64(R, 64);
        int64_t ns = tiles_h >= ctx->sm_count ? 1 : ctx->sm_count / tiles_h;
        ns = std::min<int64_t>(std::min<int64_t>(ns, 8), std::max<int64_t>(1, m / 256));
        double *Dpart = nullptr;
        if (ns > 1) GPFQ_TRY(gpfq_ws(ctx, WS_PART, (size_t)ns * one * sizeof(double), (void **)&Dpart));
        auto chain = [&](cudaStream_t on, int64_t j_lo, int64_t njh) -> int {
            cudaStream_t keep = ctx->stream;
            ctx->stream = on;
            int rc = GPFQ_OK;
            for (int64_t tb = 0, pb = 0; tb < N0 && rc == GPFQ_OK; pb = tb, tb += R) {
                const int64_t te = tb + R < N0 ? tb + R : N0;
                if (tb > 0) {
                    GemmArgs g = {};   // U += W[pb:tb] X[pb:tb] - Q[pb:tb] X~[pb:tb]
                    g.seg[0] = {Wt + j_lo * N0 + pb, Xt + pb, N0, N0, tb - pb, 1.0};
                    g.seg[1] = {Qt + j_lo * N0 + pb, Xqt + pb, N0, N0, tb - pb, -1.0};
                    g.nseg = 2;
                    g.M = njh;
                    g.N = m;
                    g.C = Ut + j_lo * m;
                    g.ldc = m;
                    g.nsplit = 1;
                    g.accumulate = 1;
                    rc = launch_gemm_nt<double, 128, 64, 16>(ctx, g, 1);
                    if (rc != GPFQ_OK) break;
                    GemmArgs d = {};   // D[range] = U X~[range]^T
                    d.seg[0] = {Ut + j_lo * m, Xqd + tb * m, m, m, m, 1.0};
                    d.nseg = 1;
                    d.M = njh;
                    d.N = te - tb;
                    d.C = Do + j_lo * R;
                    d.ldc = R;
                    d.nsplit = 1;
                    if (ns > 1) {
                        d.C = Dpart + j_lo * R;
                        d.nsplit = (int)ns;
                        d.split_stride = one;
                        rc = launch_gemm_nt<double, 128, 64, 16>(ctx, d, 1);
                        if (rc != GPFQ_OK) break;
                        const int blocks = (int)std::min<int64_t>(ceil_div64(njh * R, 256), 4096);
                        reduce_splits_kernel<<<blocks, 256, 0, on>>>(Dpart + j_lo * R, (int)ns, one, Do + j_lo * R, njh * R);
                        ctx->launches++;
                        if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) {
                            rc = gpfq_fail(ctx, GPFQ_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e), __FILE__, __LINE__);
                            break;
                        }
                    } else {
                        rc = launch_gemm_nt<double, 128, 64, 16>(ctx, d, 1);
                        if (rc != GPFQ_OK) break;
                    }
                }
                rc = dispatch_sweep_tile(ctx, NT, Gc1 - tb, Gc2 - tb, R, N0, Wt + j_lo * N0, Qt + j_lo * N0, njh, d_alph, d_koff,
                                         d_flags, 1, tb, te, tb > 0 ? Do + j_lo * R : nullptr, R, scales ? scales + j_lo : nullptr,
                                         u0 + j_lo);
            }
            ctx->stream = keep;
            return rc;
        };
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[0], st));          // Gram tiles, widened inputs and U = 0 are ready
        CUDA_TRY(ctx, cudaStreamWaitEvent(side, ctx->ev_copy[0], 0));
        GPFQ_TRY(chain(st, 0, half));
        GPFQ_TRY(chain(side, half, nj - half));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[1], side));
        CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_copy[1], 0));
        return GPFQ_OK;
    }
    // One chain (several alphabets, or few neurons).  The W part of the residual update, U += W[range] X[range], does not depend on the range's decisions: it runs on the
    // side stream WHILE the range is walked (the walk is a latency-bound chain on one CTA per neuron tile and leaves the
    // DMMA pipe idle); only the Q part, U -= Q[range] X~[range], waits for the walk.  Order on U: D(range) reads it, then the
    // W part (side stream, after D), then the Q part (main stream, after the walk and the W part) -- events 0 / 1.
    auto residual_update = [&](int64_t lo, int64_t hi, bool w_part, cudaStream_t on) -> int {
        GemmArgs g = {};
        if (w_part) g.seg[0] = {Wt + lo, Xt + lo, N0, N0, hi - lo, 1.0};
        else g.seg[0] = {Qt + lo, Xqt + lo, N0, N0, hi - lo, -1.0};
        g.nseg = 1;
        g.M = nj;
        g.N = m;
        g.C = Ut;
        g.ldc = m;
        g.nsplit = 1;
        g.accumulate = 1;
        g.batch_strideA0 = w_part ? 0 : nj * N0;   // W is shared by the alphabets of a batch, Q is per alphabet
        g.batch_strideC = nj * m;
        cudaStream_t keep = ctx->stream;
        ctx->stream = on;
        const int rc = launch_gemm_nt<double, 128, 64, 16>(ctx, g, n_alph);
        ctx->stream = keep;
        return rc;
    };
    for (int64_t tb = 0, pb = 0; tb < N0; pb = tb, tb += R) {
        const int64_t te = tb + R < N0 ? tb + R : N0;
        if (tb > 0) {
            // U -= Q[pb:tb] X~[pb:tb], after the W part of the same range (side stream) has landed
            CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_copy[1], 0));
            GPFQ_TRY(residual_update(pb, tb, false, st));
            {   // D[range] = U X~[range]^T
                GemmArgs g = {};
                g.seg[0] = {Ut, Xqd + tb * m, m, m, m, 1.0};
                g.nseg = 1;
                g.M = nj;
                g.N = te - tb;
                g.C = Do;
                g.ldc = R;
                g.nsplit = 1;
                g.batch_strideA0 = nj * m;
                g.batch_strideC = nj * R;
                // few neurons (one rank of a multi-GPU job): split the samples so that every SM gets a CTA; fixed-order sum
                const int64_t tiles = ceil_div64(nj, 128) * n_alph * ceil_div64(te - tb, 64);
                int64_t ns = tiles >= ctx->sm_count ? 1 : ctx->sm_count / tiles;
                ns = std::min<int64_t>(std::min<int64_t>(ns, 8), std::max<int64_t>(1, m / 256));
                if (ns > 1) {
                    const size_t one = (size_t)n_alph * nj * R;
                    double *Dpart = nullptr;
                    GPFQ_TRY(gpfq_ws(ctx, WS_PART, (size_t)ns * one * sizeof(double), (void **)&Dpart));
                    g.C = Dpart;
                    g.nsplit = (int)ns;
                    g.split_stride = (int64_t)one;
                    GPFQ_TRY((launch_gemm_nt<double, 128, 64, 16>(ctx, g, n_alph)));
                    const int blocks = (int)std::min<int64_t>(ceil_div64((int64_t)one, 256), 4096);
                    reduce_splits_kernel<<<blocks, 256, 0, ctx->stream>>>(Dpart, (int)ns, (int64_t)one, Do, (int64_t)one);
                    KERNEL_CHECK(ctx);
                } else {
                    GPFQ_TRY((launch_gemm_nt<double, 128, 64, 16>(ctx, g, n_alph)));
                }
            }
        }
        if (te < N0) {   // the W part of THIS range for the ranges after it: side stream, once D(range) has read U
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[0], st));
            CUDA_TRY(ctx, cudaStreamWaitEvent(side, ctx->ev_copy[0], 0));
            GPFQ_TRY(residual_update(tb, te, true, side));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[1], side));
        }
        // the compact tiles are addressed like the full matrices: column s of row t lives at Gc[t * R + (s - tb)]
        GPFQ_TRY(dispatch_sweep_tile(ctx, NT, Gc1 - tb, Gc2 - tb, R, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, n_alph, tb, te,
                                     tb > 0 ? Do : nullptr, R, scales, u0));
    }
    return GPFQ_OK;
}

// ---------------------------------------------------------------------------------------------
// The same residual-form sweep with its contractions on the 5th-generation tensor cores (slgemm_i8.cu): X, X~ and W as five
// int8 digit slices each (sliced ONCE per layer; X^T / X~^T with one exponent per sample, X~ and W with one per row), the
// decisions of a range as ONE slice of level indices k' = q / h (alphabets on the symmetric grid: q = h k', |k'| <= K - 1,
// the literal 0 of a dead direction is k' = 0), the fp64 residuals U re-sliced after every range.  Per range:
//     U += W_r X_r  (19 slice pairs, dropped terms < 2^-46 of 2^(eW + eX) per direction)  -  h K'_r X~_r  (5 pairs, exact)
//     D_r = U X~_r^T (15 pairs, < 2^-38 of 2^(eU + eX~) per sample: ~1e-11 of the decision argument, as the tcgen05 Gram)
// every slice-pair sum is an exact integer in TMEM, the fp64 combination has a fixed order: bit-reproducible.
// ---------------------------------------------------------------------------------------------
// The gate of sweep_tc_kernel and of the int8 residual form: an alphabet whose levels lie on the symmetric grid
// a_k = -a + k 2a / (K - 1), a = a[K-1] > 0.  Both decide on that grid (the rounded grid position for K > 3, the thresholds +-a/2
// for K = 3) and carry the range's decisions as h k' with h = a / (K - 1); only the output values are looked up from the real
// levels.  So the levels must sit on the grid more tightly than the walk's flag windows resolve: a level delta off the grid
// moves a decision threshold by at most delta, and an unflagged decision is literal only while that shift stays well inside
// the window -- 2^-30 of a step for K > 3 (>= 2^-36 a for K <= 128), ~2^-20 relative for K = 3.  delta <= 2^-40 a keeps the
// shift below 1/16 of the window, and the h k' residual within 2^-40 a of the real one per direction (below what the int8
// contractions drop).  `c * median|W| * linspace(-1, 1, K)` is off the grid by a few ulp and passes.  Two levels must be exact:
// for odd K the middle one is 0.0, since the level index k' = 0 is also the literal 0 of a dead direction and is written out
// as 0.0 (stc_q_from_kq_kernel: a middle level of 1e-14 a, inside the tolerance, would come out as 0.0, not as a level); and
// K = 3 is decided with exact comparisons against +-a / 2, so its ends must be exact negatives (gpfq_ternary_radius).
// Anything else -- levels within the 1 % equispaced window but off the grid, an asymmetric or non-uniform alphabet -- walks
// with sweep_pipe / sweep_tile and the fp64 residual form, which compare the real levels.
static bool alphabet_on_symmetric_grid(const double *a, int K, int flag, double *h) {
    if (!flag || K < 2 || K - 1 > 127 || !(a[K - 1] > 0.0)) return false;
    const double top = a[K - 1];
    if (K % 2 == 1 && a[K / 2] != 0.0) return false;
    if (K == 3) {
        if (a[0] != -top) return false;
    } else {
        const double step = 2.0 * top / (double)(K - 1), tol = 0x1p-40 * top;
        for (int k = 0; k < K; ++k)
            if (!(fabs(a[k] - (-top + k * step)) <= tol)) return false;
    }
    *h = top / (double)(K - 1);
    return true;
}

static bool dense_lowrank_uses_i8(gpfq_ctx *ctx, int64_t N0, int64_t m, int64_t nj, int n_alph, double *h) {
    if (ctx->sweep_i8 == 2 || n_alph != 1 || !ctx->h_alph || !ctx->h_koff || !ctx->h_flags) return false;
    if (m > 204 * 128 || N0 >= ((int64_t)1 << 30)) return false;   // one K chunk of the s32 accumulators
    return alphabet_on_symmetric_grid(ctx->h_alph + ctx->h_koff[0], ctx->h_koff[1] - ctx->h_koff[0], ctx->h_flags[0], h);
}

// The int8 residual form slices X^T / X~^T with ONE exponent per sample over all N0 directions, and the range's G1 rows with one per
// row.  A direction whose norm is far below the largest entries of its samples therefore reaches U, P and D_r through fewer bits:
// its decision argument moves by up to ~2^-39 N0 (max-sample norm / ||x~_t||) of a step, and no replay can recover what the slices
// dropped.  So the layer takes the int8 contractions only while sqrt(sum_i colmax_i^2) -- the norm of the per-sample maxima over
// X and X~, which bounds every direction's norm -- stays within LOWRANK_I8_SPREAD times the smallest live ||x~_t||.  ReLU
// activations of similar norms sit near 6 (4.2 / 0.71 for N0 = 25088); direction norms spread over 10^+-1 give ~600.
// A layer past the gate walks with the fp64 contractions of dense_lowrank_sweep.
static constexpr double LOWRANK_I8_SPREAD = 64.0;

__global__ void __launch_bounds__(256) spread_colmax_kernel(const float *__restrict__ X, int64_t ldx, int64_t N0, int64_t m,
                                                            int *__restrict__ colmax, int rows_per_cta) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= m) return;
    const int64_t t0 = (int64_t)blockIdx.y * rows_per_cta, t1 = min(N0, t0 + rows_per_cta);
    float mx = 0.f;
    for (int64_t t = t0; t < t1; ++t) mx = fmaxf(mx, fabsf(X[t * ldx + i]));
    atomicMax(colmax + i, __float_as_int(mx));   // non-negative floats order like their bit patterns
}

// one warp per direction: the least ||x~_t||^2 over the live directions (fp32(sqrt) >= GPFQ_DEAD_NORM), as fp64 bits
__global__ void __launch_bounds__(256) spread_min_norm_kernel(const float *__restrict__ Xq, int64_t ldx, int64_t N0, int64_t m,
                                                              unsigned long long *__restrict__ minn2) {
    const int64_t t = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (t >= N0) return;
    double n2 = 0.0;
    for (int64_t i = lane; i < m; i += 32) {
        const double x = (double)Xq[t * ldx + i];
        n2 = fma(x, x, n2);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n2 += __shfl_xor_sync(0xffffffffu, n2, o);
    if (lane == 0 && !((double)(float)sqrt(n2) < GPFQ_DEAD_NORM)) atomicMin(minn2, (unsigned long long)__double_as_longlong(n2));
}

__global__ void __launch_bounds__(256) spread_gate_kernel(const int *__restrict__ colmax, int64_t m,
                                                          const unsigned long long *__restrict__ minn2, int *__restrict__ wide) {
    __shared__ double red[8];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < m; i += 256) {
        const double c = (double)__int_as_float(colmax[i]);
        s = fma(c, c, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) s += red[w];
        const double mn = __longlong_as_double((long long)*minn2);   // +inf when every direction is dead
        *wide = !(s <= LOWRANK_I8_SPREAD * LOWRANK_I8_SPREAD * mn);  // (NaN / Inf in the inputs: wide)
    }
}

// *ok = the layer passes the spread gate above.  One 4-byte read-back: the choice of form is made on the host.
static int lowrank_i8_spread_ok(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m, bool *ok) {
    cudaStream_t st = ctx->stream;
    unsigned char *ws = nullptr;
    const size_t cm_bytes = (size_t)ceil_div64(m, 64) * 64 * sizeof(int);
    GPFQ_TRY(gpfq_ws(ctx, WS_MISC, cm_bytes + 16, (void **)&ws));
    int *colmax = reinterpret_cast<int *>(ws);
    unsigned long long *minn2 = reinterpret_cast<unsigned long long *>(ws + cm_bytes);
    int *wide = reinterpret_cast<int *>(ws + cm_bytes + 8);
    CUDA_TRY(ctx, cudaMemsetAsync(colmax, 0, cm_bytes, st));
    CUDA_TRY(ctx, cudaMemsetAsync(minn2, 0x7f, 8, st));   // 0x7f7f7f7f7f7f7f7f: a huge finite double
    const int rows_per_cta = 256;
    const dim3 g((unsigned)ceil_div64(m, 256), (unsigned)ceil_div64(N0, rows_per_cta));
    spread_colmax_kernel<<<g, 256, 0, st>>>(X, ldx, N0, m, colmax, rows_per_cta);
    KERNEL_CHECK(ctx);
    if (Xq != X) {
        spread_colmax_kernel<<<g, 256, 0, st>>>(Xq, ldx, N0, m, colmax, rows_per_cta);
        KERNEL_CHECK(ctx);
    }
    spread_min_norm_kernel<<<(unsigned)ceil_div64(N0, 8), 256, 0, st>>>(Xq, ldx, N0, m, minn2);
    KERNEL_CHECK(ctx);
    spread_gate_kernel<<<1, 256, 0, st>>>(colmax, m, minn2, wide);
    KERNEL_CHECK(ctx);
    int h_wide = 1;
    CUDA_TRY(ctx, cudaMemcpyAsync(&h_wide, wide, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    *ok = h_wide == 0;
    return GPFQ_OK;
}

// h_j = fl(s_j a) / (K - 1): the level step of neuron j with per-channel alphabets, computed as sweep_tc_kernel computes it
__global__ void unit_steps_kernel(const double *__restrict__ scales, int64_t nj, int64_t njP, double a, int K, double *__restrict__ hrow) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < njP) hrow[j] = j < nj ? __dmul_rn(scales[j], a) / (double)(K - 1) : 0.0;
}

// d_scales (nullable): (nj) per-neuron scales (per-channel alphabets): the walk applies each neuron's own step, and the Q part of the
// residual update becomes -diag(h) K'_r X~_r (a per-row multiplier in the slgemm_i8_kernel epilogue); the W part and D_r are unchanged.
static int dense_lowrank_sweep_i8(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m,
                                  const double *Wt, int64_t nj, const double *d_alph, double h, gpfq_stats *stats, const float *W,
                                  int64_t ldw, int64_t j0, double *Qd, int64_t ldq, int64_t col0, const double *d_scales, int64_t u0) {
    const bool same = (Xq == X);
    cudaStream_t st = ctx->stream, side = ctx->copy_stream;
    int64_t R = pick_range_length(ctx, nj, 1);
    R = std::max<int64_t>(128, R / 128 * 128);      // K blocks of the update are 128 directions
    R = std::min<int64_t>(R, stc::MAX_R);           // the tensor-core walk keeps a range's level indices in shared memory
    // Ternary alphabets: the tensor-core range walk (sweep_tc.cu) -- the W terms of every range as ONE batched product before the
    // sweep, the Q terms inside the walk kernel, one thread per neuron
    const int K_levels = ctx->h_koff[1] - ctx->h_koff[0];
    const double a_top = ctx->h_alph[ctx->h_koff[0] + K_levels - 1];
    const double *d_levels = d_alph;   // one alphabet per call on this path: its levels start the device array
    const int64_t N0P = ceil_div64(N0, R) * R, mP = ceil_div64(m, 128) * 128, njP = ceil_div64(nj, 128) * 128;   // whole ranges
    constexpr int S = 5;
    int8_t *sW = nullptr, *sXT = nullptr, *sXqT = nullptr, *sXq = nullptr, *sU = nullptr, *sKq = nullptr;
    int32_t *e = nullptr;
    double *Ut = nullptr, *Gc1 = nullptr, *Gc2 = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_SL_W, (size_t)S * njP * N0P, (void **)&sW));
    GPFQ_TRY(gpfq_ws(ctx, WS_SL_XT, (size_t)S * mP * N0P, (void **)&sXT));
    if (same) sXqT = sXT;
    else GPFQ_TRY(gpfq_ws(ctx, WS_SL_XQT, (size_t)S * mP * N0P, (void **)&sXqT));
    GPFQ_TRY(gpfq_ws(ctx, WS_SL_XQ, (size_t)S * N0P * mP, (void **)&sXq));
    GPFQ_TRY(gpfq_ws(ctx, WS_SL_U, (size_t)S * njP * mP, (void **)&sU));
    GPFQ_TRY(gpfq_ws(ctx, WS_SL_KQ, (size_t)njP * N0P, (void **)&sKq));
    GPFQ_TRY(gpfq_ws(ctx, WS_SL_E, (size_t)(2 * njP + N0P + 3 * mP + 16) * sizeof(int32_t), (void **)&e));
    int32_t *eW = e, *eU = eW + njP, *eXq = eU + njP, *eXT = eXq + N0P;   // X^T and X~^T share their per-sample exponents
    int *scratch = eXT + mP;
    GPFQ_TRY(gpfq_ws(ctx, WS_LR_U, (size_t)nj * m * sizeof(double), (void **)&Ut));
    double *hrow = nullptr;   // per-neuron steps (per-channel alphabets), padded to njP rows
    if (d_scales) {
        GPFQ_TRY(gpfq_ws(ctx, WS_UNIT_H, (size_t)njP * sizeof(double), (void **)&hrow));
        unit_steps_kernel<<<(unsigned)ceil_div64(njP, 256), 256, 0, st>>>(d_scales, nj, njP, a_top, K_levels, hrow);
        KERNEL_CHECK(ctx);
    }
    const double h_q = d_scales ? 1.0 : h;   // the walk's tables and the Q part: h itself, or 1 with the steps applied per neuron
    const size_t gc_bytes = (size_t)ceil_div64(N0, R) * R * R * sizeof(double);
    GPFQ_TRY(gpfq_ws(ctx, WS_G2, gc_bytes, (void **)&Gc2));
    if (same) Gc1 = Gc2;
    else GPFQ_TRY(gpfq_ws(ctx, WS_G1, gc_bytes, (void **)&Gc1));
    constexpr int D_DOTS_GRAM = 6;

    CUDA_TRY(ctx, gpfq_record(ctx, 2, st));
    // slicing, once per layer
    GPFQ_TRY(sl_rowsplit<float>(ctx, Xq, ldx, N0, m, eXq, sXq, N0P, mP, 0, N0P));
    SlOperand oXqB;
    GPFQ_TRY(sl_make_operand(ctx, &oXqB, sXq, N0P, mP, S, eXq, 0, true));
    GPFQ_TRY(sl_transsplit(ctx, X, same ? nullptr : Xq, ldx, N0, m, eXT, scratch, sXT, sXqT, mP, N0P));
    GPFQ_TRY(sl_rowsplit<double>(ctx, Wt, N0, nj, N0, eW, sW, njP, N0P, 0, njP));
    // block-diagonal Gram tiles, compact: Gc[t][s - tb(t)], row stride R -- on tcgen05 as well (15 slice pairs over the m
    // samples, as the Dense Gram stage of gram_i8.cu: dropped terms ~2e-11 of |X~_t||X_s|): every range is one batch of one launch
    {
        int8_t *sXr = nullptr, *sXqA = sXq;
        int32_t *eXr = eXq;
        if (!same) {
            GPFQ_TRY(gpfq_ws(ctx, WS_I8_SX, (size_t)S * N0P * mP, (void **)&sXr));
            GPFQ_TRY(gpfq_ws(ctx, WS_I8_E, (size_t)N0P * sizeof(int32_t), (void **)&eXr));
            GPFQ_TRY(sl_rowsplit<float>(ctx, X, ldx, N0, m, eXr, sXr, N0P, mP, 0, N0P));
        }
        SlOperand oXqA, oXrB;
        GPFQ_TRY(sl_make_operand(ctx, &oXqA, sXqA, N0P, mP, S, eXq, 0, false));
        GPFQ_TRY(sl_make_operand(ctx, &oXrB, same ? sXq : sXr, N0P, mP, S, eXr, 0, true));
        const int nrange = (int)ceil_div64(N0, R);
        // rows / columns beyond N0 of the last range are zero slices: their (unused) outputs are zeros; Gc holds nrange * R rows
        for (int which = 0; which < (same ? 1 : 2); ++which) {
            SlProduct gp = {&oXqA, which ? &oXrB : &oXqB, 0, 0, 0, mP, D_DOTS_GRAM, 1.0};
            GPFQ_TRY(slgemm_i8(ctx, &gp, 1, which ? Gc1 : Gc2, R, R, R, false, nrange, R, R * R, true));
        }
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 3, st));
    CUDA_TRY(ctx, cudaMemsetAsync(Ut, 0, (size_t)nj * m * sizeof(double), st));
    CUDA_TRY(ctx, cudaMemsetAsync(sKq, 0, (size_t)njP * N0P, st));   // padding rows / directions of the index slice stay zero
    SlOperand oW, oXT, oXqT, oXq, oU, oKq;
    GPFQ_TRY(sl_make_operand(ctx, &oW, sW, njP, N0P, S, eW, 0, false));
    TcTables tct;
    double *Dsplit = nullptr;   // K-split partials of the residual dots (few neurons)
    if (ceil_div64(nj, 128) * (R / 64) * 3 <= ctx->sm_count) GPFQ_TRY(gpfq_ws(ctx, WS_PART, (size_t)6 * njP * R * sizeof(double), (void **)&Dsplit));
    double *Pd = nullptr;   // (nj, N0P): per range the W terms of the range itself, then + D_r (what the earlier ranges contribute)
    float *Wn = nullptr;    // (nj, N0P): the weights neuron-major, fp32
    {
        GPFQ_TRY(gpfq_ws(ctx, WS_TC_W, (size_t)njP * N0P * sizeof(float), (void **)&Wn));   // (rows >= nj: never written, never used)
        GPFQ_TRY(sweep_tc_weights(ctx, W, ldw, j0, N0, N0P, nj, Wn));
        int8_t *sG1 = nullptr;
        int32_t *eG1 = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_TC_G1S, (size_t)S * N0P * R, (void **)&sG1));
        GPFQ_TRY(gpfq_ws(ctx, WS_TC_E, (size_t)N0P * sizeof(int32_t), (void **)&eG1));
        GPFQ_TRY(gpfq_ws(ctx, WS_TC_P, (size_t)njP * N0P * sizeof(double), (void **)&Pd));
        GPFQ_TRY(sweep_tc_prepare(ctx, Gc1, Gc2, R, true, N0, N0P, R, h_q, &tct));
        GPFQ_TRY(sweep_tc_bind(ctx, &tct, Pd, Wn, njP, N0P));
        GPFQ_TRY(sweep_tc_slice_g1_lower(ctx, Gc1, R, true, N0, N0P, R, eG1, sG1));
        SlOperand oG1;
        GPFQ_TRY(sl_make_operand(ctx, &oG1, sG1, N0P, R, S, eG1, 0, true));
        // P[:, range r] = W[:, range r] strict_lower(G1_rr)^T for every range: the batches of one launch (19 slice pairs; column
        // tile tj of a range needs the K blocks 0 .. tj only)
        SlProduct pp = {&oW, &oG1, 0, 0, 0, R, 7, 1.0, 0};
        SlBatch pb;
        pb.n = (int)(N0P / R);
        pb.a_k = R;
        pb.b_rows = R;
        pb.c = R;
        pb.ktri = true;
        GPFQ_TRY(slgemm_i8_ex(ctx, &pp, 1, Pd, N0P, nj, R, false, pb));
    }
    GPFQ_TRY(sl_make_operand(ctx, &oXT, sXT, mP, N0P, S, eXT, 0, true));
    GPFQ_TRY(sl_make_operand(ctx, &oXqT, sXqT, mP, N0P, S, eXT, 0, true));
    GPFQ_TRY(sl_make_operand(ctx, &oXq, sXq, N0P, mP, S, eXq, 0, true));
    GPFQ_TRY(sl_make_operand(ctx, &oU, sU, njP, mP, S, eU, 0, false));
    GPFQ_TRY(sl_make_operand(ctx, &oKq, sKq, njP, N0P, 1, nullptr, 6, false));   // single digit b: value = b 2^(e - 6) = b
    const int D_UPDATE = 7, D_DOTS = 6;

    // One chain per group of neurons.  On the critical path of a range stay only what needs the previous range's decisions:
    // the Q part of the residual update (5 exact slice pairs), the re-slicing of U, the residual dots D_r and the walk.  The W
    // part of the update, U += W_r X_r (19 pairs), depends on no decision: it runs on the group's aux stream as soon as U has
    // been sliced for D_r, underneath D_r and the walk of range r.  Order on U (fixed, so the fp64 sums are reproducible):
    //   slice(r) | W part of r (aux) | Q part of r (main, after the walk and after the W part) | slice(r + 1) ...
    auto chain = [&](int g, cudaStream_t on, int64_t j_lo, int64_t njh) -> int {
        cudaStream_t keep = ctx->stream, aux = ctx->aux_stream[g];
        cudaEvent_t ev_sliced = ctx->ev_chain[3 * g], ev_wpart = ctx->ev_chain[3 * g + 1];
        int rc = GPFQ_OK;
        const int64_t rows_h = ceil_div64(njh, 128) * 128;
        // measured (VGG16 fc1 / fc2): with thousands of neurons the sweep is bound by the SUM of its contraction launches -- W and Q
        // part as ONE two-product launch (25.5 vs 27.3 ms); a shard of a few hundred neurons is bound by the LATENCY of the
        // chain -- W part off it, on the aux stream (11.0 vs 11.6 ms)
        const bool merged = nj >= 2048;
        auto cu = [&](cudaError_t e) { if (e != cudaSuccess && rc == GPFQ_OK) rc = gpfq_fail(ctx, GPFQ_ERR_CUDA, "%s", cudaGetErrorString(e)); };
        for (int64_t tb = 0, pb = 0; tb < N0 && rc == GPFQ_OK; pb = tb, tb += R) {
            const int64_t te = tb + R < N0 ? tb + R : N0;
            ctx->stream = on;
            if (tb > 0) {
                const int64_t Kp = ceil_div64(tb - pb, 128) * 128;   // the walk of [pb, tb) left its level indices in sKq
                if (merged) {   // U += W_r X_r - h K'_r X~_r as ONE launch of two products (same B-row exponents)
                    SlProduct up[2] = {{&oW, &oXT, j_lo, 0, pb, Kp, D_UPDATE, 1.0}, {&oKq, &oXqT, j_lo, 0, pb, Kp, 6, -h_q, -1, hrow}};
                    rc = slgemm_i8(ctx, up, 2, Ut + j_lo * m, m, njh, m, true);
                } else {
                    cu(cudaStreamWaitEvent(on, ev_wpart, 0));
                    SlProduct qp = {&oKq, &oXqT, j_lo, 0, pb, Kp, 6, -h_q, -1, hrow};
                    rc = slgemm_i8(ctx, &qp, 1, Ut + j_lo * m, m, njh, m, true);          // U -= h K'_r X~_r
                }
                if (rc != GPFQ_OK) break;
                rc = sl_rowsplit<double>(ctx, Ut + j_lo * m, m, njh, m, eU, sU, njP, mP, j_lo, rows_h);
                if (rc != GPFQ_OK) break;
            }
            if (!merged) cu(cudaEventRecord(ev_sliced, on));
            if (tb > 0) {
                SlProduct dp = {&oU, &oXq, j_lo, tb, 0, mP, D_DOTS, 1.0};
                // few neurons (one rank's shard): the residual dots are a handful of tiles with a long K loop -- split the samples
                // over batches so that every SM gets a tile, fixed-order sum of the partials afterwards
                const int64_t dtiles = ceil_div64(njh, 128) * ceil_div64(te - tb, 64);
                int ns = 1;
                for (int c : {6, 4, 3})   // (two-way splits measured slower than none: fc3's 1000 neurons 1.64 -> 1.76 ms)
                    if (ns == 1 && dtiles * c <= ctx->sm_count && (mP / 64) % c == 0 && mP / c >= 256) ns = c;
                if (ns > 1 && Dsplit) {
                    SlBatch sb;
                    sb.n = ns;
                    sb.a_k = sb.b_k = mP / ns;
                    sb.c = njP * R;
                    SlProduct dps = {&oU, &oXq, j_lo, tb, 0, mP / ns, D_DOTS, 1.0, 0};
                    rc = slgemm_i8_ex(ctx, &dps, 1, Dsplit + j_lo * R, R, njh, te - tb, false, sb);
                    if (rc == GPFQ_OK)
                        rc = sweep_tc_add_partials(ctx, Pd + j_lo * N0P + tb, N0P, Dsplit + j_lo * R, ns, njP * R, R, njh, te - tb);
                } else rc = slgemm_i8(ctx, &dp, 1, Pd + j_lo * N0P + tb, N0P, njh, te - tb, true);   // P_r += U X~_r^T
                if (rc != GPFQ_OK) break;
            }
            if (te < N0 && !merged) {   // the W part of THIS range, for the ranges after it
                const int64_t Kp = ceil_div64(te - tb, 128) * 128;
                cu(cudaStreamWaitEvent(aux, ev_sliced, 0));
                ctx->stream = aux;
                SlProduct wp = {&oW, &oXT, j_lo, 0, tb, Kp, D_UPDATE, 1.0};
                rc = slgemm_i8(ctx, &wp, 1, Ut + j_lo * m, m, njh, m, true);          // U += W_r X_r
                cu(cudaEventRecord(ev_wpart, aux));
                ctx->stream = on;
                if (rc != GPFQ_OK) break;
            }
            rc = sweep_tc_range(ctx, tct, tb, te, j_lo, njh, sKq, njP, j_lo, a_top, d_levels, K_levels,   // {-a, 0, a}: h = a / 2
                                d_scales ? d_scales + j_lo : nullptr, u0 + j_lo);
        }
        ctx->stream = keep;
        return rc;
    };
    if (stats) {
        stats->flops_algorithmic = 2LL * (19 + 5 + 15) * nj * m * N0;   // int8 operations of the 39 slice-pair products
        stats->reserved |= 1 | 2;   // int8-slice contractions, ranges walked by sweep_tc_kernel
    }
    int G = nj >= 4096 ? 4 : (nj >= 2048 ? 2 : 1);
    if (ctx->lowrank_variant == 3) G = 1;
    while (G > 1 && ceil_div64(nj, G) < 256) G >>= 1;
    if (G > 1) {
        // Independent groups of neurons, one chain each on its own stream: while one group sits in the latency-bound walk of a
        // range (which is given few SMs: 128 neurons per CTA) the contractions of the other groups have the rest of the chip.
        const int64_t gs = ceil_div64(ceil_div64(nj, G), 128) * 128;
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[0], st));
        int rc = GPFQ_OK;
        for (int g = 0; g < G && rc == GPFQ_OK; ++g) {
            const int64_t j_lo = g * gs, njh = std::min<int64_t>(gs, nj - j_lo);
            if (njh <= 0) break;
            cudaStream_t on = g ? ctx->aux_stream[4 + g] : st;
            if (g) CUDA_TRY(ctx, cudaStreamWaitEvent(on, ctx->ev_copy[0], 0));
            rc = chain(g, on, j_lo, njh);
            if (g) {
                CUDA_TRY(ctx, cudaEventRecord(ctx->ev_chain[3 * g + 2], on));
                CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_chain[3 * g + 2], 0));
            }
        }
        if (rc != GPFQ_OK) return rc;
    } else {
        GPFQ_TRY(chain(0, st, 0, nj));
    }
    // the tensor-core walk leaves level indices only: the layer's fp64 values are made from them here
    GPFQ_TRY(sweep_tc_q_from_kq(ctx, sKq, njP, N0, nj, d_levels, K_levels, Qd, ldq, col0, d_scales));
    return GPFQ_OK;
}

// Dense layer by Gram + sweep.  All pointers are device pointers.
//   Qd: (n_alph, N0, ldq) fp64 device output, columns col0..col0+nj-1 written.
//   d_scales (nullable): (n_alph, nj) per-neuron scales of the shard (per-channel alphabets): every walk applies each neuron's own
//   levels, the same kernels run as for the per-layer call (DESIGN.md 5.5).
int dense_gram_path(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m,
                    const float *W, int64_t ldw, int64_t j0, int64_t nj, const double *d_alph,
                    const int *d_koff, const int *d_flags, int n_alph, double *Qd, int64_t ldq, int64_t col0,
                    gpfq_stats *st, const double *G1_pre, const double *G2_pre, const double *d_scales, int64_t u0) {
    // G2_pre != NULL: the Gram stage already ran elsewhere (sample-split over the ranks of a job and all-reduced,
    // gpfq_dense_layer_from_gram); X / Xq / m are then unused and the sweep starts from the given (N0, N0) matrices.
    const bool pre = (G2_pre != nullptr);
    const bool same = pre ? (G1_pre == nullptr || G1_pre == G2_pre) : (Xq == X);
    double *G1 = nullptr, *G2 = nullptr, *Wt = nullptr, *Qt = nullptr;
    double h_step = 0.0;
    // Stochastic rounding (ctx->d_seeds): every walk below takes it; the shard's first neuron has unit id u0
    bool i8_sweep = !pre && dense_lowrank_uses_i8(ctx, N0, m, nj, n_alph, &h_step);
    const bool lowrank = !pre && dense_uses_lowrank(ctx, N0, m, nj, n_alph, same, i8_sweep);
    // sweep_i8 = 0: the int8 contractions only for layers within the spread gate (lowrank_i8_spread_ok); 1 forces them
    if (lowrank && i8_sweep && ctx->sweep_i8 == 0) GPFQ_TRY(lowrank_i8_spread_ok(ctx, X, Xq, ldx, N0, m, &i8_sweep));
    // Neurons per CTA of the range walk: the narrowest tile that still fits every CTA on the chip at once (two per SM, so
    // that one CTA's serial walk overlaps another's contraction).
    const int64_t slots = 2LL * ctx->sm_count;
    const int NT = ceil_div64(nj, 8) * n_alph <= slots ? 8 : (ceil_div64(nj, 16) * n_alph <= slots ? 16 : 32);
    GPFQ_TRY(gpfq_ws(ctx, WS_WT, (size_t)nj * N0 * sizeof(double), (void **)&Wt));
    // Qt (neuron-major decisions): every form but the int8 residual form, whose walk leaves level indices only
    if (!(lowrank && i8_sweep)) GPFQ_TRY(gpfq_ws(ctx, WS_QT, (size_t)n_alph * nj * N0 * sizeof(double), (void **)&Qt));
    {
        dim3 grid((unsigned)ceil_div64(N0, 32), (unsigned)ceil_div64(nj, 32));
        transpose_w_kernel<<<grid, dim3(32, 8), 0, ctx->stream>>>(W, ldw, N0, j0, nj, Wt);
        KERNEL_CHECK(ctx);
    }
    if (lowrank) {
        if (i8_sweep) {   // writes Qd itself
            GPFQ_TRY(dense_lowrank_sweep_i8(ctx, X, Xq, ldx, N0, m, Wt, nj, d_alph, h_step, st, W, ldw, j0, Qd, ldq, col0, d_scales, u0));
        } else {
            GPFQ_TRY(dense_lowrank_sweep(ctx, X, Xq, ldx, N0, m, Wt, Qt, nj, d_alph, d_koff, d_flags, n_alph, NT, d_scales, u0));
            for (int a = 0; a < n_alph; ++a) {
                dim3 grid((unsigned)ceil_div64(N0, 32), (unsigned)ceil_div64(nj, 32));
                transpose_q_kernel<<<grid, dim3(32, 8), 0, ctx->stream>>>(Qt + (int64_t)a * nj * N0, N0, nj,
                                                                          Qd + (int64_t)a * N0 * ldq, ldq, col0);
                KERNEL_CHECK(ctx);
            }
        }
        CUDA_TRY(ctx, gpfq_record(ctx, 4, ctx->stream));
        if (st) {
            st->method = GPFQ_METHOD_GRAM >> 4;
            st->gram_kernel = 3;
            if (!i8_sweep) st->flops_algorithmic = 6 * m * N0 * nj * n_alph;
            st->bytes_algorithmic = (same ? 1 : 2) * 4 * N0 * m;
        }
        return GPFQ_OK;
    }
    if (pre) {
        G2 = const_cast<double *>(G2_pre);  // read-only below
        G1 = same ? G2 : const_cast<double *>(G1_pre);
    } else {
        GPFQ_TRY(gpfq_ws(ctx, WS_G2, (size_t)N0 * N0 * sizeof(double), (void **)&G2));
        if (same) G1 = G2;
        else GPFQ_TRY(gpfq_ws(ctx, WS_G1, (size_t)N0 * N0 * sizeof(double), (void **)&G1));
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 2, ctx->stream));
    if (!pre) GPFQ_TRY(dense_gram_only(ctx, X, Xq, ldx, N0, m, G1, G2));
    else ctx->last_gram_kernel = 0;
    CUDA_TRY(ctx, gpfq_record(ctx, 3, ctx->stream));

    // Two-level blocking: directions in ranges of R; what the earlier ranges contribute to a range is ONE large NT
    // contraction (all SMs, split over neurons x directions, and over K when that is too few tiles), the
    // persistent neuron-tile kernel then walks the range.
    const int64_t tiles_m = ceil_div64(nj, 128) * n_alph;
    int64_t R = pick_range_length(ctx, nj, n_alph);
    double *Do = nullptr, *Dpart = nullptr;
    // One alphabet on the symmetric grid (alphabet_on_symmetric_grid): the tensor-core range walk (sweep_tc.cu).  P = (what the
    // earlier ranges contribute: the Gram-row contraction below) + (the W terms of the range itself: one batched product on the
    // fp64 pipe up front).
    double h_tc = 0.0;
    // (measured, profiles/dense_methods_r2.md: below ~2048 directions the few extra launches of the preparation cost more than the
    //  walk saves -- MNIST's layers 0.65 -> 0.73 ms -- so those keep sweep_pipe_kernel; sweep_walk = 1 forces the new walk)
    const bool use_tc = n_alph == 1 && ctx->sweep_walk != 2 && (N0 >= 2048 || ctx->sweep_walk == 1) && ctx->h_alph && ctx->h_koff &&
                        ctx->h_flags && N0 < ((int64_t)1 << 30) &&
                        alphabet_on_symmetric_grid(ctx->h_alph + ctx->h_koff[0], ctx->h_koff[1] - ctx->h_koff[0], ctx->h_flags[0], &h_tc);
    TcTables tct;
    double *Pd = nullptr, *G1m = nullptr;
    float *Wn = nullptr;
    int8_t *sKq = nullptr;
    int64_t N0P = 0, njP = 0;
    const int K_levels = use_tc ? ctx->h_koff[1] - ctx->h_koff[0] : 0;
    const double a_top = use_tc ? ctx->h_alph[ctx->h_koff[0] + K_levels - 1] : 0.0;
    if (use_tc) {
        R = std::min<int64_t>(R, stc::MAX_R);
        N0P = ceil_div64(N0, R) * R;
        njP = ceil_div64(nj, 128) * 128;
        GPFQ_TRY(gpfq_ws(ctx, WS_TC_P, (size_t)njP * N0P * sizeof(double), (void **)&Pd));
        GPFQ_TRY(gpfq_ws(ctx, WS_TC_W, (size_t)njP * N0P * sizeof(float), (void **)&Wn));
        GPFQ_TRY(gpfq_ws(ctx, WS_TC_G1M, (size_t)N0P * R * sizeof(double), (void **)&G1m));
        GPFQ_TRY(gpfq_ws(ctx, WS_SL_KQ, (size_t)njP * N0P, (void **)&sKq));
        CUDA_TRY(ctx, cudaMemsetAsync(Pd, 0, (size_t)njP * N0P * sizeof(double), ctx->stream));
        GPFQ_TRY(sweep_tc_weights(ctx, W, ldw, j0, N0, N0P, nj, Wn));
        GPFQ_TRY(sweep_tc_prepare(ctx, G1, G2, N0, false, N0, N0P, R, d_scales ? 1.0 : h_tc, &tct));   // scaled: steps per walker
        GPFQ_TRY(sweep_tc_bind(ctx, &tct, Pd, Wn, njP, N0P));
        GPFQ_TRY(sweep_tc_mask_g1_lower(ctx, G1, N0, N0, N0P, R, G1m));
        const int64_t nfull = N0 / R;
        GemmArgs g = {};   // P[:, range] = Wt[:, range] strict_lower(G1[range, range])^T, every full range a batch
        g.seg[0] = {Wt, G1m, N0, R, R, 1.0};
        g.nseg = 1;
        g.M = nj;
        g.N = R;
        g.C = Pd;
        g.ldc = N0P;
        g.nsplit = 1;
        g.batch_strideA0 = R;
        g.batch_strideB = R * R;
        g.batch_strideC = R;
        for (int64_t b0 = 0; b0 < nfull; b0 += 65535) {
            GemmArgs gb = g;
            gb.seg[0].A = Wt + b0 * R;
            gb.seg[0].B = G1m + b0 * R * R;
            gb.C = Pd + b0 * R;
            GPFQ_TRY((launch_gemm_nt<double, 128, 64, 16>(ctx, gb, (int)std::min<int64_t>(65535, nfull - b0))));
        }
        if (nfull * R < N0) {   // the ragged last range
            const int64_t tb = nfull * R;
            GemmArgs gl = g;
            gl.seg[0] = {Wt + tb, G1m + tb * R, N0, R, N0 - tb, 1.0};
            gl.N = N0 - tb;
            gl.C = Pd + tb;
            GPFQ_TRY((launch_gemm_nt<double, 128, 64, 16>(ctx, gl, 1)));
        }
    }
    if (N0 > R) GPFQ_TRY(gpfq_ws(ctx, WS_DT, (size_t)n_alph * nj * R * sizeof(double), (void **)&Do));
    for (int64_t tb = 0; tb < N0; tb += R) {
        const int64_t te = tb + R < N0 ? tb + R : N0;
        if (tb > 0) {
            GemmArgs g = {};
            g.seg[0] = {Wt, G1 + tb * N0, N0, N0, tb, 1.0};
            g.seg[1] = {Qt, G2 + tb * N0, N0, N0, tb, -1.0};
            g.nseg = 2;
            g.M = nj;
            g.N = te - tb;
            g.C = Do;
            g.ldc = R;
            g.nsplit = 1;
            g.batch_strideA1 = nj * N0;
            g.batch_strideC = nj * R;
            // few neurons: split K (the earlier directions) so that every SM gets a CTA; fixed-order reduction
            const int64_t tiles = tiles_m * ceil_div64(te - tb, 64);
            int64_t ns = tiles >= ctx->sm_count ? 1 : ctx->sm_count / tiles;
            ns = std::min<int64_t>(std::min<int64_t>(ns, 16), std::max<int64_t>(1, tb / 128));
            if (ns > 1) {
                const size_t one = (size_t)n_alph * nj * R;
                GPFQ_TRY(gpfq_ws(ctx, WS_PART, (size_t)ns * one * sizeof(double), (void **)&Dpart));
                g.C = Dpart;
                g.nsplit = (int)ns;
                g.split_stride = (int64_t)one;
                GPFQ_TRY((launch_gemm_nt<double, 128, 64, 16>(ctx, g, n_alph)));
                int blocks = (int)std::min<int64_t>(ceil_div64((int64_t)one, 256), 4096);
                reduce_splits_kernel<<<blocks, 256, 0, ctx->stream>>>(Dpart, (int)ns, (int64_t)one, Do, (int64_t)one);
                KERNEL_CHECK(ctx);
            } else {
                GPFQ_TRY((launch_gemm_nt<double, 128, 64, 16>(ctx, g, n_alph)));
            }
        }
        if (use_tc) {
            if (tb > 0) GPFQ_TRY(sweep_tc_add_outer(ctx, Pd + tb, N0P, Do, R, nj, te - tb));
            GPFQ_TRY(sweep_tc_range(ctx, tct, tb, te, 0, nj, sKq, njP, 0, a_top, d_alph, K_levels, d_scales, u0));
            GPFQ_TRY(sweep_tc_qt_from_kq(ctx, sKq, njP, tb, te, nj, d_alph, K_levels, Qt, N0, d_scales));
        } else {
            GPFQ_TRY(dispatch_sweep_tile(ctx, NT, G1, G2, N0, N0, Wt, Qt, nj, d_alph, d_koff, d_flags, n_alph, tb, te,
                                         tb > 0 ? Do : nullptr, R, d_scales, u0));
        }
    }
    for (int a = 0; a < n_alph; ++a) {
        dim3 grid((unsigned)ceil_div64(N0, 32), (unsigned)ceil_div64(nj, 32));
        transpose_q_kernel<<<grid, dim3(32, 8), 0, ctx->stream>>>(Qt + (int64_t)a * nj * N0, N0, nj,
                                                                  Qd + (int64_t)a * N0 * ldq, ldq, col0);
        KERNEL_CHECK(ctx);
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 4, ctx->stream));
    if (st) {
        st->method = GPFQ_METHOD_GRAM >> 4;
        st->gram_kernel = ctx->last_gram_kernel;
        if (use_tc) st->reserved |= 2;   // ranges walked by sweep_tc_kernel
        st->flops_algorithmic = pre ? 2 * N0 * N0 * nj * n_alph : (same ? 1 : 2) * m * N0 * (N0 + 1);  // lower triangles
        st->bytes_algorithmic = (pre ? 0 : (same ? 1 : 2) * 4 * N0 * m) + (same ? 1 : 2) * 8 * N0 * N0;
    }
    return GPFQ_OK;
}
