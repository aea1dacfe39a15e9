// dense_stream.cu -- Dense layer, streaming form (K3): the literal residual walk of
// _quantize_neuron_parallel (quantized_network.py:113-121) with the residual u kept on chip.
//
// One CTA walks J neurons through all N0 directions.  u (fp64, J x m) lives in shared memory (or an
// L2-resident global scratch when m is too long); every step streams the rows X_t, Xq_t once
// (coalesced) and
//   * applies the pending update of step t-1:  u += fl32(w X_{t-1}) - q Xq_{t-1}        (:119)
//   * accumulates  d = <Xq_t, u>  and  s = <Xq_t, u + fl32(w_t X_t)>                      (:86, :89)
// in one pass, then reduces across the CTA in a fixed order and takes the decision (:83-89).
// The arithmetic follows the reference's dtype ladder exactly (fp32 product w*X, fp64 everything
// else, no contraction in the update), so this kernel is the parity anchor of the library.
#include "common.cuh"

static constexpr int STREAM_T = 512;

// nrm[t] = (double)(float)sqrt(sum_i Xq[t][i]^2)  -- what scipy.linalg.norm(float32 row) returns (snrm2)
// g1d[t] = <Xq_t, X_t> (exact fp32 x fp32 products, fp64 sum): the w_t-term of step t in the exact-product walk
__global__ void __launch_bounds__(256) row_norms_kernel(const float *__restrict__ X, const float *__restrict__ Xq,
                                                        int64_t ldx, int64_t m, double *__restrict__ nrm,
                                                        double *__restrict__ g1d) {
    __shared__ double red[2][8];
    const float *rq = Xq + (int64_t)blockIdx.x * ldx, *rx = X + (int64_t)blockIdx.x * ldx;
    double s = 0.0, g = 0.0;
    for (int64_t i = threadIdx.x; i < m; i += 256) {
        const double v = (double)rq[i];
        s = fma(v, v, s);
        g = fma(v, (double)rx[i], g);
    }
    s = warp_sum(s);
    g = warp_sum(g);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = g; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0, gt = 0.0;
        for (int w = 0; w < 8; ++w) { tot += red[0][w]; gt += red[1][w]; }
        nrm[blockIdx.x] = (double)(float)sqrt(tot);
        g1d[blockIdx.x] = gt;
    }
}

// SCALED: neuron jb + j of the shard walks with the levels scales[jb + j] * alphabet (common.cuh)
// STOCH: stochastic rounding with the seed *seed, unit id u0 + jb + j (the global neuron), step id t
// L1: the penalty's shrink with tau[t] (row_norms_l1_kernel)
template <int J, bool SCALED = false, bool STOCH = false, bool L1 = false>
__global__ void __launch_bounds__(STREAM_T)
dense_stream_kernel(const float *__restrict__ X, const float *__restrict__ Xq, int64_t ldx, int64_t N0,
                    int64_t m, const float *__restrict__ W, int64_t ldw, int64_t j0, int64_t nj,
                    const double *__restrict__ nrm, const double *__restrict__ alphabet, int K,
                    double *__restrict__ Q, int64_t ldq, int64_t col0, double *__restrict__ u_scratch,
                    int u_in_smem, const double *__restrict__ scales = nullptr, const uint64_t *__restrict__ seed = nullptr,
                    int64_t u0 = 0, const double *__restrict__ tau = nullptr) {
    extern __shared__ __align__(16) unsigned char stream_smem[];
    constexpr int NW = STREAM_T / 32;
    __shared__ double red[NW][2 * J];
    __shared__ double qsh[J];
    __shared__ double alph[GPFQ_MAX_K];

    const int64_t jb = (int64_t)blockIdx.x * J;
    double *u = u_in_smem ? reinterpret_cast<double *>(stream_smem)
                          : u_scratch + (int64_t)blockIdx.x * J * m;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    for (int e = tid; e < K; e += STREAM_T) alph[e] = alphabet[e];
    for (int64_t e = tid; e < (int64_t)J * m; e += STREAM_T) u[e] = 0.0;
    __syncthreads();
    const double sc = (SCALED && tid < J && jb + tid < nj) ? scales[jb + tid] : 0.0;
    const uint64_t key = (STOCH && tid < J) ? gpfq_unit_key(*seed, u0 + jb + tid) : 0;

    float wprev[J];
    double qprev[J];
#pragma unroll
    for (int j = 0; j < J; ++j) { wprev[j] = 0.f; qprev[j] = 0.0; }

    for (int64_t t = 0; t < N0; ++t) {
        float w[J];
#pragma unroll
        for (int j = 0; j < J; ++j) w[j] = (jb + j < nj) ? W[t * ldw + j0 + jb + j] : 0.f;
        const float *x = X + t * ldx, *xq = Xq + t * ldx;
        const float *xp = X + (t > 0 ? t - 1 : 0) * ldx, *xqp = Xq + (t > 0 ? t - 1 : 0) * ldx;
        double d[J], s[J];
#pragma unroll
        for (int j = 0; j < J; ++j) d[j] = s[j] = 0.0;

        for (int64_t i = tid; i < m; i += STREAM_T) {
            const float xv = x[i], xqv = xq[i];
            const double xqd = (double)xqv;
            float xpv = 0.f;
            double xqpd = 0.0;
            if (t > 0) { xpv = xp[i]; xqpd = (double)xqp[i]; }
#pragma unroll
            for (int j = 0; j < J; ++j) {
                double uj = u[(int64_t)j * m + i];
                if (t > 0) {
                    // u += w[t-1]*X_{t-1} - q[t-1]*Xq_{t-1}: fp32 product, fp64 product, sub, add (:119)
                    const double wx = (double)__fmul_rn(wprev[j], xpv);
                    const double qx = __dmul_rn(qprev[j], xqpd);
                    uj = __dadd_rn(uj, __dsub_rn(wx, qx));
                    u[(int64_t)j * m + i] = uj;
                }
                d[j] = fma(xqd, uj, d[j]);
                const double uw = __dadd_rn(uj, (double)__fmul_rn(w[j], xv));  // u + w*X  (:89)
                s[j] = fma(xqd, uw, s[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < J; ++j) {
            d[j] = warp_sum(d[j]);
            s[j] = warp_sum(s[j]);
        }
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < J; ++j) { red[warp][j] = d[j]; red[warp][J + j] = s[j]; }
        }
        __syncthreads();
        if (tid < J) {
            double dd = 0.0, ss = 0.0;
            for (int wv = 0; wv < NW; ++wv) { dd += red[wv][tid]; ss += red[wv][J + tid]; }
            const double q = L1       ? gpfq_decide_l1<SCALED, STOCH>(nrm[t], dd, ss, (double)w[tid], alph, K, 0.0, sc,
                                                                        STOCH ? gpfq_draw(key, t) : 0.0, tau[t])
                           : STOCH    ? gpfq_decide_stoch<SCALED>(nrm[t], dd, ss, (double)w[tid], alph, K, 0.0, sc, gpfq_draw(key, t))
                           : SCALED ? gpfq_decide_unit<true>(nrm[t], dd, ss, (double)w[tid], alph, K, 0.0, sc)
                                    : gpfq_decide(nrm[t], dd, ss, (double)w[tid], alph, K);
            qsh[tid] = q;
            if (jb + tid < nj) Q[t * ldq + col0 + jb + tid] = q;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < J; ++j) { wprev[j] = w[j]; qprev[j] = qsh[j]; }
    }
}

// ---------------------------------------------------------------------------------------------
// Register-resident walk (m <= STREAM_T * 16).  One CTA walks J neurons; thread `tid` owns EPV groups of four
// consecutive samples (i = (v*STREAM_T + tid)*4 + c) of every one of them, so the residual never leaves the
// register file and a step costs no shared-memory or global traffic beyond the two rows X_t, Xq_t (LDG.128),
// which are requested one step ahead (they do not depend on the decision).  Per step:
//   convert the rows of step t to fp64 once; reuse the fp32 registers for the loads of step t+1
//   d_j = <Xq_t, u_j>                                  (:86)    one DFMA per sample and neuron
//   LITERAL: s_j = <Xq_t, u_j + fl32(w_j X_t)>         (:89)    the reference's dtype ladder, mul/sub/add unfused
//   else   : s_j = d_j + w_j <Xq_t, X_t>                         exact fp32 x fp32 products (the Gram form's numerics;
//                                                                <Xq_t, X_t> comes from row_norms_kernel)
//   reduction: one transposing butterfly per warp for all values, per-warp partials to shared memory, barrier,
//   warp 0 sums the 16 partials of every value by a fixed shuffle tree and decides, barrier, broadcast
//   u_j += fl32(w_j X_t) - q_j Xq_t   (:119)   [non-LITERAL: two DFMAs on the exact products]
// ---------------------------------------------------------------------------------------------
template <int V>
__device__ __forceinline__ void warp_reduce_multi(double (&vals)[V], int lane) {
    // V a power of two <= 32.  Afterwards vals[0] of lane l holds the warp total of value index
    // idx(l) = the top log2(V) bits of l (bit 4 first); the summation tree is fixed.
    int n = V;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        if (n > 1) {
            n >>= 1;
            const bool hi = (lane & off) != 0;
#pragma unroll
            for (int i = 0; i < V / 2; ++i) {
                if (i < n) {
                    const double send = hi ? vals[i] : vals[i + n];
                    const double keep = hi ? vals[i + n] : vals[i];
                    vals[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                }
            }
        } else {
            vals[0] += __shfl_xor_sync(0xffffffffu, vals[0], off);
        }
    }
}

template <int V>
__device__ __forceinline__ int warp_reduce_index(int lane) {
    int idx = 0, n = V, bit = 16;
    while (n > 1) { idx = idx * 2 + ((lane & bit) ? 1 : 0); n >>= 1; bit >>= 1; }
    return idx;
}

template <int EPV, int J, bool LITERAL, bool VEC, bool SCALED = false, bool STOCH = false, bool L1 = false>
__global__ void __launch_bounds__(STREAM_T)
dense_stream_reg_kernel(const float *__restrict__ X, const float *__restrict__ Xq, int64_t ldx, int64_t N0,
                        int64_t m, const float *__restrict__ W, int64_t ldw, int64_t j0, int64_t nj,
                        const double *__restrict__ nrm, const double *__restrict__ g1d,
                        const double *__restrict__ alphabet, int K, int equispaced,
                        double *__restrict__ Q, int64_t ldq, int64_t col0, const double *__restrict__ scales = nullptr,
                        const uint64_t *__restrict__ seed = nullptr, int64_t u0 = 0, const double *__restrict__ tau = nullptr) {
    constexpr int NW = STREAM_T / 32, EPT = 4 * EPV;
    constexpr int V = LITERAL ? 2 * J : J;  // values reduced per step
    __shared__ double red[NW][V];
    __shared__ double qsh[J];
    __shared__ double alph[GPFQ_MAX_K];
    __shared__ double unit_s[SCALED ? 2 * J : 1];  // per neuron: scale, inv_step of its levels
    __shared__ uint64_t unit_key[STOCH ? J : 1];    // per neuron: the stochastic-rounding unit key (one per unit, not per step)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t jb = (int64_t)blockIdx.x * J;
    for (int e = tid; e < K; e += STREAM_T) alph[e] = alphabet[e];
    if (STOCH && tid < J) unit_key[tid] = gpfq_unit_key(*seed, u0 + jb + tid);
    if (SCALED && tid < J) {
        const double sc = jb + tid < nj ? scales[jb + tid] : 0.0;
        unit_s[tid] = sc;
        unit_s[J + tid] = gpfq_inv_step_s(alphabet, K, equispaced, sc);
    }

    double u[J][EPT];
#pragma unroll
    for (int j = 0; j < J; ++j)
#pragma unroll
        for (int e = 0; e < EPT; ++e) u[j][e] = 0.0;

    float cx[EPT], cq[EPT], w[J], wn[J];
    auto load_rows = [&](int64_t t) {
        const float *x = X + t * ldx, *xq = Xq + t * ldx;
#pragma unroll
        for (int v = 0; v < EPV; ++v) {
            const int64_t i = ((int64_t)v * STREAM_T + tid) * 4;
            if (VEC) {  // m % 4 == 0: a group of four is wholly inside or wholly outside
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
                if (i < m) {
                    a = __ldg(reinterpret_cast<const float4 *>(x + i));
                    b = __ldg(reinterpret_cast<const float4 *>(xq + i));
                }
                cx[4 * v] = a.x; cx[4 * v + 1] = a.y; cx[4 * v + 2] = a.z; cx[4 * v + 3] = a.w;
                cq[4 * v] = b.x; cq[4 * v + 1] = b.y; cq[4 * v + 2] = b.z; cq[4 * v + 3] = b.w;
            } else {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const bool ok = i + c < m;
                    cx[4 * v + c] = ok ? __ldg(x + i + c) : 0.f;
                    cq[4 * v + c] = ok ? __ldg(xq + i + c) : 0.f;
                }
            }
        }
    };
    auto load_w = [&](int64_t t, float *rw) {
#pragma unroll
        for (int j = 0; j < J; ++j) rw[j] = (jb + j < nj) ? __ldg(W + t * ldw + j0 + jb + j) : 0.f;
    };

    double nrm_t = nrm[0], g1_t = LITERAL ? 0.0 : g1d[0];
    load_rows(0);
    load_w(0, w);
    __syncthreads();  // alphabet staged
    const double inv_step = gpfq_inv_step(alph, K, equispaced);

    for (int64_t t = 0; t < N0; ++t) {
        // rows of step t -> fp64 (once); their fp32 registers then receive the rows of step t+1
        double xqd[EPT], xd[LITERAL ? 1 : EPT];
        float fx[LITERAL ? EPT : 1];
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            xqd[e] = (double)cq[e];
            if (LITERAL) fx[e] = cx[e];
            else xd[e] = (double)cx[e];
        }
        double nrm_n = 0.0, g1_n = 0.0;
        if (t + 1 < N0) {
            load_rows(t + 1);
            load_w(t + 1, wn);
            nrm_n = nrm[t + 1];
            if (!LITERAL) g1_n = g1d[t + 1];
        }
        double val[V];
        {
            double acc[2][V];  // even / odd samples feed two independent chains per value
#pragma unroll
            for (int v = 0; v < V; ++v) acc[0][v] = acc[1][v] = 0.0;
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
#pragma unroll
                for (int j = 0; j < J; ++j) {
                    acc[e & 1][j] = fma(xqd[e], u[j][e], acc[e & 1][j]);
                    if (LITERAL) {
                        const double uw = __dadd_rn(u[j][e], (double)__fmul_rn(w[j], fx[e]));  // u + w*X  (:89)
                        acc[e & 1][J + j] = fma(xqd[e], uw, acc[e & 1][J + j]);
                    }
                }
            }
#pragma unroll
            for (int v = 0; v < V; ++v) val[v] = acc[0][v] + acc[1][v];
        }
        warp_reduce_multi<V>(val, lane);
        if ((lane & (32 / V - 1)) == 0) red[warp][warp_reduce_index<V>(lane)] = val[0];
        __syncthreads();
        if (warp == 0) {
            // lane = 16 * (j & 1) + w: two neurons per pass, a 16-lane shuffle tree over the per-warp partials
#pragma unroll
            for (int jp = 0; jp < J; jp += 2) {
                const int j = jp + (lane >> 4), wv = lane & 15;
                const bool live = j < J;
                double dd = live ? red[wv][j] : 0.0;
                double ss = (LITERAL && live) ? red[wv][J + j] : 0.0;
#pragma unroll
                for (int off = 8; off >= 1; off >>= 1) {
                    dd += __shfl_xor_sync(0xffffffffu, dd, off);
                    if (LITERAL) ss += __shfl_xor_sync(0xffffffffu, ss, off);
                }
                if (live && wv == 0) {
                    float wj = w[0];
#pragma unroll
                    for (int jj = 1; jj < J; ++jj) wj = (j == jj) ? w[jj] : wj;
                    const double num = LITERAL ? ss : fma((double)wj, g1_t, dd);
                    const double q =
                        L1       ? gpfq_decide_l1<SCALED, STOCH>(nrm_t, dd, num, (double)wj, alph, K, SCALED ? unit_s[J + j] : inv_step,
                                                                 SCALED ? unit_s[j] : 1.0, STOCH ? gpfq_draw(unit_key[j], t) : 0.0, tau[t])
                      : STOCH    ? gpfq_decide_stoch<SCALED>(nrm_t, dd, num, (double)wj, alph, K, SCALED ? unit_s[J + j] : inv_step,
                                                             SCALED ? unit_s[j] : 1.0, gpfq_draw(unit_key[j], t))
                      : SCALED ? gpfq_decide_unit<true>(nrm_t, dd, num, (double)wj, alph, K, unit_s[J + j], unit_s[j])
                               : gpfq_decide(nrm_t, dd, num, (double)wj, alph, K, inv_step);
                    qsh[j] = q;
                    if (jb + j < nj) Q[t * ldq + col0 + jb + j] = q;
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < J; ++j) {
            const double qj = qsh[j];
            const double wd = (double)w[j];
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                if (LITERAL) {
                    // u += w[t]*X_t - q[t]*Xq_t: fp32 product, fp64 product, sub, add (:119)
                    const double wx = (double)__fmul_rn(w[j], fx[e]);
                    u[j][e] = __dadd_rn(u[j][e], __dsub_rn(wx, __dmul_rn(qj, xqd[e])));
                } else {
                    u[j][e] = fma(-qj, xqd[e], fma(wd, xd[e], u[j][e]));
                }
            }
        }
#pragma unroll
        for (int j = 0; j < J; ++j) w[j] = wn[j];
        nrm_t = nrm_n;
        g1_t = g1_n;
    }
}

template <int EPV, int J>
static int launch_stream_reg(gpfq_ctx *ctx, bool literal, bool vec, const float *X, const float *Xq, int64_t ldx,
                             int64_t N0, int64_t m, const float *W, int64_t ldw, int64_t j0, int64_t nj,
                             const double *nrm, const double *g1d, const double *d_alph, int K, int eq, double *Qd,
                             int64_t ldq, int64_t col0, const double *scales, const uint64_t *seed, int64_t u0, const double *tau) {
    const unsigned nblk = (unsigned)ceil_div64(nj, J);
#define LAUNCH(LIT, VEC, S, R, L) \
    dense_stream_reg_kernel<EPV, J, LIT, VEC, S, R, L><<<nblk, STREAM_T, 0, ctx->stream>>>(X, Xq, ldx, N0, m, W, ldw, j0, nj, nrm, \
                                                                                        g1d, d_alph, K, eq, Qd, ldq, col0, scales, seed, u0, tau)
#define LAUNCH_S(R, L)                                                                                 \
    if (scales) {                                                                                      \
        if (literal) { if (vec) LAUNCH(true, true, true, R, L); else LAUNCH(true, false, true, R, L); }  \
        else { if (vec) LAUNCH(false, true, true, R, L); else LAUNCH(false, false, true, R, L); }        \
    } else {                                                                                           \
        if (literal) { if (vec) LAUNCH(true, true, false, R, L); else LAUNCH(true, false, false, R, L); } \
        else { if (vec) LAUNCH(false, true, false, R, L); else LAUNCH(false, false, false, R, L); }      \
    }
    if (tau) { if (seed) { LAUNCH_S(true, true) } else { LAUNCH_S(false, true) } }
    else if (seed) { LAUNCH_S(true, false) } else { LAUNCH_S(false, false) }
#undef LAUNCH_S
#undef LAUNCH
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

// (EPV, J): EPV groups of four samples per thread, J neurons per CTA
static int dispatch_stream_reg(gpfq_ctx *ctx, int epv, int J, bool literal, bool vec, const float *X, const float *Xq,
                               int64_t ldx, int64_t N0, int64_t m, const float *W, int64_t ldw, int64_t j0, int64_t nj,
                               const double *nrm, const double *g1d, const double *d_alph, int K, int eq, double *Qd,
                               int64_t ldq, int64_t col0, const double *scales, const uint64_t *seed, int64_t u0, const double *tau) {
#define SR(E, JJ) \
    if (epv == E && J == JJ) \
        return launch_stream_reg<E, JJ>(ctx, literal, vec, X, Xq, ldx, N0, m, W, ldw, j0, nj, nrm, g1d, d_alph, K, eq, Qd, \
                                        ldq, col0, scales, seed, u0, tau);
    SR(1, 1) SR(1, 2) SR(1, 4)
    SR(2, 1) SR(2, 2)
    SR(3, 1) SR(3, 2)
    SR(4, 1)
#undef SR
    return gpfq_fail(ctx, GPFQ_ERR_ARG, "no streaming kernel for EPV=%d J=%d", epv, J);
}

template <int J>
static int launch_stream(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m,
                         const float *W, int64_t ldw, int64_t j0, int64_t nj, const double *nrm,
                         const double *d_alph, int K, double *Qd, int64_t ldq, int64_t col0, const double *scales,
                         const uint64_t *seed, int64_t u0, const double *tau) {
    const int64_t nblk = ceil_div64(nj, J);
    const size_t need = (size_t)J * m * sizeof(double);
    const size_t static_smem = 8192;  // red/qsh/alph, generous
    const bool in_smem = need + static_smem <= ctx->smem_optin;
    double *scratch = nullptr;
    if (!in_smem) GPFQ_TRY(gpfq_ws(ctx, WS_U, (size_t)nblk * need, (void **)&scratch));
    auto k = seed ? (scales ? dense_stream_kernel<J, true, true> : dense_stream_kernel<J, false, true>)
                  : (scales ? dense_stream_kernel<J, true> : dense_stream_kernel<J, false>);
    if (tau)
        k = seed ? (scales ? dense_stream_kernel<J, true, true, true> : dense_stream_kernel<J, false, true, true>)
                 : (scales ? dense_stream_kernel<J, true, false, true> : dense_stream_kernel<J, false, false, true>);
    if (in_smem)
        CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
    k<<<(unsigned)nblk, STREAM_T, in_smem ? need : 0, ctx->stream>>>(X, Xq, ldx, N0, m, W, ldw, j0, nj, nrm,
                                                                   d_alph, K, Qd, ldq, col0, scratch,
                                                                   in_smem ? 1 : 0, scales, seed, u0, tau);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

// Dense layer by the streaming walk.  Device pointers.  Alphabets are walked one after another
// (each needs its own residual); Qd: (n_alph, N0, ldq).  d_scales (nullable): (n_alph, nj) per-neuron scales of the shard.
// The same norms and, for the L1 penalty (common.cuh), tau[a * N0 + t] = lambda_a / nrm_t^2 for each of the call's n_alph
// penalties: one table per alphabet, built in the same pass so that the walks read tau instead of dividing per step
__global__ void __launch_bounds__(256) row_norms_l1_kernel(const float *__restrict__ X, const float *__restrict__ Xq,
                                                           int64_t ldx, int64_t m, double *__restrict__ nrm,
                                                           double *__restrict__ g1d, const double *__restrict__ lambdas,
                                                           int n_alph, int64_t N0, double *__restrict__ tau) {
    __shared__ double red[2][8];
    const float *rq = Xq + (int64_t)blockIdx.x * ldx, *rx = X + (int64_t)blockIdx.x * ldx;
    double s = 0.0, g = 0.0;
    for (int64_t i = threadIdx.x; i < m; i += 256) {
        const double v = (double)rq[i];
        s = fma(v, v, s);
        g = fma(v, (double)rx[i], g);
    }
    s = warp_sum(s);
    g = warp_sum(g);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = g; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0, gt = 0.0;
        for (int w = 0; w < 8; ++w) { tot += red[0][w]; gt += red[1][w]; }
        const double nv = (double)(float)sqrt(tot);
        nrm[blockIdx.x] = nv;
        g1d[blockIdx.x] = gt;
        for (int a = 0; a < n_alph; ++a) tau[(int64_t)a * N0 + blockIdx.x] = gpfq_l1_tau(lambdas[a], nv);
    }
}

// Stochastic rounding (ctx->d_seeds): the shard's first neuron has unit id u0.  L1 penalty (ctx->d_l1): tau from a table.
int dense_stream_path(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m,
                      const float *W, int64_t ldw, int64_t j0, int64_t nj, const double *d_alph,
                      const int *h_koff, const int *h_flags, int n_alph, double *Qd, int64_t ldq, int64_t col0,
                      gpfq_stats *st, const double *d_scales, int64_t u0) {
    double *nrm = nullptr, *tau = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_NRM, (size_t)2 * N0 * sizeof(double), (void **)&nrm));
    double *g1d = nrm + N0;
    if (ctx->d_l1) GPFQ_TRY(gpfq_ws(ctx, WS_L1, (size_t)n_alph * N0 * sizeof(double), (void **)&tau));
    CUDA_TRY(ctx, gpfq_record(ctx, 2, ctx->stream));
    if (tau) row_norms_l1_kernel<<<(unsigned)N0, 256, 0, ctx->stream>>>(X, Xq, ldx, m, nrm, g1d, ctx->d_l1, n_alph, N0, tau);
    else row_norms_kernel<<<(unsigned)N0, 256, 0, ctx->stream>>>(X, Xq, ldx, m, nrm, g1d);
    KERNEL_CHECK(ctx);
    const bool literal = ctx->stream_literal;
    if (m <= (int64_t)STREAM_T * 16) {
        // register-resident residual: EPV groups of four samples per thread, J neurons per CTA
        const int epv = (int)ceil_div64(m, STREAM_T * 4);
        const int jmax = epv == 1 ? 4 : (epv <= 3 ? 2 : 1);
        int J = 1;
        while (J * 2 <= jmax && ceil_div64(nj, J * 2) >= ctx->sm_count) J *= 2;
        const bool vec = (m % 4 == 0) && (ldx % 4 == 0) && ((uintptr_t)X % 16 == 0) && ((uintptr_t)Xq % 16 == 0);
        for (int a = 0; a < n_alph; ++a) {
            const double *al = d_alph + h_koff[a];
            const int K = h_koff[a + 1] - h_koff[a];
            GPFQ_TRY(dispatch_stream_reg(ctx, epv, J, literal, vec, X, Xq, ldx, N0, m, W, ldw, j0, nj, nrm, g1d, al, K,
                                         h_flags[a], Qd + (int64_t)a * N0 * ldq, ldq, col0, d_scales ? d_scales + a * nj : nullptr,
                                         ctx->d_seeds ? ctx->d_seeds + a : nullptr, u0, tau ? tau + a * N0 : nullptr));
        }
    } else {
        // long sample axis: residual in shared memory (or an L2-resident scratch), literal arithmetic
        const size_t per_neuron = (size_t)m * sizeof(double);
        int J = 1;
        while (J < 4 && ceil_div64(nj, J * 2) >= ctx->sm_count && (size_t)(J * 2) * per_neuron + 8192 <= ctx->smem_optin)
            J *= 2;
        for (int a = 0; a < n_alph; ++a) {
            const double *al = d_alph + h_koff[a];
            const int K = h_koff[a + 1] - h_koff[a];
            double *Qa = Qd + (int64_t)a * N0 * ldq;
            const double *sa = d_scales ? d_scales + a * nj : nullptr;
            const uint64_t *sd = ctx->d_seeds ? ctx->d_seeds + a : nullptr;
            const double *ta = tau ? tau + a * N0 : nullptr;
            if (J == 4) GPFQ_TRY(launch_stream<4>(ctx, X, Xq, ldx, N0, m, W, ldw, j0, nj, nrm, al, K, Qa, ldq, col0, sa, sd, u0, ta));
            else if (J == 2) GPFQ_TRY(launch_stream<2>(ctx, X, Xq, ldx, N0, m, W, ldw, j0, nj, nrm, al, K, Qa, ldq, col0, sa, sd, u0, ta));
            else GPFQ_TRY(launch_stream<1>(ctx, X, Xq, ldx, N0, m, W, ldw, j0, nj, nrm, al, K, Qa, ldq, col0, sa, sd, u0, ta));
        }
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 3, ctx->stream));
    if (st) {
        st->method = GPFQ_METHOD_STREAM >> 4;
        st->flops_algorithmic = 6 * m * N0 * nj * n_alph;
        st->bytes_algorithmic = 8 * N0 * m + 12 * N0 * nj;
    }
    return GPFQ_OK;
}
