// conv.cu -- Conv2D / DepthwiseConv2D channels (K4): many channels per launch.
//
// Replaces the channel loop of _quantize_conv2D_layer_parallel_jit (quantized_network.py:844-860) and
// the per-filter pool of _quantize_channel_parallel_jit (:706-718), whose workers run the kk = kh*kw
// step walk of _quantize_filter2D_parallel_jit (:219-228).  kk is tiny (9 for 3x3) and n_patches is
// huge, so each channel is a pure HBM stream of its two (kk, n_patches) patch matrices:
//   stage 1  conv_gram_kernel     per channel G1 = Xq X^T (kk x kk), G2 = Xq Xq^T (lower), fp64
//                                 accumulation of exact fp32 products, per-CTA partials
//   stage 2  conv_finalize_kernel fixed-order sum of the partials (deterministic)
//   stage 3  conv_sweep_kernel    one thread per (channel, filter): the kk-step walk in registers
// Stages 1 and 3 have kernels of their own for kk in {1, 2, 3, 4, 6, 9}; every other kk <= 128 (5 x 5, 7 x 7, 11 x 11, ...)
// takes conv_gramx_kernel (DMMA tiles for a runtime kk) and conv_walkx_kernel (one warp per filter).
// Also here: the on-device single-channel im2col that serves gpfq_conv_layer_nhwc (the reference's
// _build_patch_array :729-809 / tf.image.extract_patches :158-172) and the MSQ baseline.
#include "common.cuh"

static constexpr int CONV_BLOCK = 256;
static constexpr int CONV_MAXKK = 9;

// ---- stage 1 ---------------------------------------------------------------------------------
// Thread group G (of NG) owns the Gram rows t = G, G+NG, ...; every group sweeps all columns of the
// CTA's chunk, so the 81+45 fp64 accumulators of a 3x3 channel are split over two thread groups.
template <int KK, bool SAME, int NG, int G>
__device__ __forceinline__ void conv_gram_body(const float *__restrict__ X, const float *__restrict__ Xq,
                                               int64_t n, int64_t c_beg, int64_t c_end, int tg, int gt,
                                               double *__restrict__ red) {
    constexpr int NR = (KK - G + NG - 1) / NG;
    double a1[NR][KK], a2[NR][KK];
#pragma unroll
    for (int r = 0; r < NR; ++r)
#pragma unroll
        for (int s = 0; s < KK; ++s) a1[r][s] = a2[r][s] = 0.0;

    float cx[KK], cq[KK];
    int64_t p = c_beg + tg;
    if (p < c_end) {
#pragma unroll
        for (int s = 0; s < KK; ++s) {
            cq[s] = __ldg(Xq + (int64_t)s * n + p);
            if (!SAME) cx[s] = __ldg(X + (int64_t)s * n + p);
        }
    }
    for (; p < c_end; p += gt) {
        float nx[KK], nq[KK];
        const int64_t pn = p + gt;
        if (pn < c_end) {
#pragma unroll
            for (int s = 0; s < KK; ++s) {
                nq[s] = __ldg(Xq + (int64_t)s * n + pn);
                if (!SAME) nx[s] = __ldg(X + (int64_t)s * n + pn);
            }
        }
        double xd[KK], qd[KK];
#pragma unroll
        for (int s = 0; s < KK; ++s) {
            qd[s] = (double)cq[s];
            if (!SAME) xd[s] = (double)cx[s];
        }
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int t = G + r * NG;
#pragma unroll
            for (int s = 0; s < KK; ++s) {
                if (!SAME) a1[r][s] = fma(qd[t], xd[s], a1[r][s]);
                if (s <= t) a2[r][s] = fma(qd[t], qd[s], a2[r][s]);
            }
        }
#pragma unroll
        for (int s = 0; s < KK; ++s) {
            cq[s] = nq[s];
            if (!SAME) cx[s] = nx[s];
        }
    }
    // fixed-order reduction: lanes (xor butterfly), then warps of this group in index order
    const int lane = threadIdx.x & 31, wig = tg >> 5, nwg = gt >> 5;
    double *myred = red + (size_t)(G * nwg + wig) * (2 * KK * KK);
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const int t = G + r * NG;
#pragma unroll
        for (int s = 0; s < KK; ++s) {
            if (!SAME) {
                const double v = warp_sum(a1[r][s]);
                if (lane == 0) myred[t * KK + s] = v;
            }
            if (s <= t) {
                const double v = warp_sum(a2[r][s]);
                if (lane == 0) myred[KK * KK + t * KK + s] = v;
            }
        }
    }
}

// partial: (n_channels, n_chunks, 2*KK*KK)
template <int KK, bool SAME, int NG>
__global__ void __launch_bounds__(CONV_BLOCK, 1)
conv_gram_kernel(ConvPtrs ptrs, int64_t n, int64_t chunk_cols, double *__restrict__ partial, int slots) {
    __shared__ double red[(CONV_BLOCK / 32) * 2 * KK * KK];
    const int ch = blockIdx.y, chunk = blockIdx.x;
    const float *X = ptrs.Xp[ch];
    const float *Xq = SAME ? X : ptrs.Xqp[ch];
    const int64_t c_beg = (int64_t)chunk * chunk_cols;
    const int64_t c_end = (c_beg + chunk_cols < n) ? c_beg + chunk_cols : n;
    double *out = partial + ((size_t)ch * slots + chunk) * (2 * KK * KK);
    constexpr int GT = CONV_BLOCK / NG;
    const int g = threadIdx.x / GT, tg = threadIdx.x % GT;
    if (NG == 1) {
        conv_gram_body<KK, SAME, 1, 0>(X, Xq, n, c_beg, c_end, tg, GT, red);
    } else {
        if (g == 0) conv_gram_body<KK, SAME, NG, 0>(X, Xq, n, c_beg, c_end, tg, GT, red);
        else conv_gram_body<KK, SAME, NG, (NG > 1 ? 1 : 0)>(X, Xq, n, c_beg, c_end, tg, GT, red);
    }
    __syncthreads();
    // entry (t, s) was accumulated by group t % NG; sum that group's warps in index order
    constexpr int NWG = GT / 32;
    for (int e = threadIdx.x; e < 2 * KK * KK; e += CONV_BLOCK) {
        const int which = e / (KK * KK), t = (e % (KK * KK)) / KK, s = e % KK;
        if ((which == 0 && SAME) || (which == 1 && s > t)) continue;
        const int og = t % NG;
        double tot = 0.0;
        for (int w = 0; w < NWG; ++w) tot += red[(size_t)(og * NWG + w) * (2 * KK * KK) + e];
        out[e] = tot;
    }
}

// ---- stage 1, 3x3 fast path ---------------------------------------------------------------------
// KK = 9 on the fp64 tensor pipe.  Lane l = (g, k) = (l >> 2, l & 3) owns patch row g of four columns per
// step (a float4 per row per 16 columns, so every request is a run of full 32-byte sectors).  The 8 x 8
// corners of G1 = Xq X^T and G2 = Xq Xq^T are one DMMA.8x8x4 each per 4 columns (the A fragment of Xq
// rows 0..7 is also the B fragment of G2); the ninth row / column (26 entries) are five DFMAs per lane.
// Per column: 168 fp64-pipe slots for 126 useful products and 32 F2F (XU pipe), ~100 registers, no
// shared-memory staging -- occupancy (16 warps/SM, 8 LDG.128 in flight per lane) covers the HBM latency.
// Needs n % 4 == 0 and 16-byte aligned patch matrices; everything else takes the generic kernel above.
__device__ __forceinline__ float4 ldg_stream4(const float *p) { return __ldcs(reinterpret_cast<const float4 *>(p)); }

__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

struct Gram9Acc {
    double g1[2], g2[2];  // C fragments: G[g][2k], G[g][2k+1]
    double a1, a2, a3, a4, a5;  // G1[g][8], G1[8][g], G2[8][g], G1[8][8], G2[8][8] (partial over this lane's columns)
};

template <bool SAME>
__device__ __forceinline__ void gram9_step(Gram9Acc &acc, float q, float x, float q8, float x8) {
    const double qd = (double)q, q8d = (double)q8;
    dmma884(acc.g2[0], acc.g2[1], qd, qd);
    acc.a3 = fma(q8d, qd, acc.a3);
    acc.a5 = fma(q8d, q8d, acc.a5);
    if (!SAME) {
        const double xd = (double)x, x8d = (double)x8;
        dmma884(acc.g1[0], acc.g1[1], qd, xd);
        acc.a1 = fma(qd, x8d, acc.a1);
        acc.a2 = fma(q8d, xd, acc.a2);
        acc.a4 = fma(q8d, x8d, acc.a4);
    }
}

// The same step with the ninth row already in fp64 (the TMA kernel converts that row once per warp, not once per lane).
template <bool SAME>
__device__ __forceinline__ void gram9_step_d(Gram9Acc &acc, float q, float x, double q8d, double x8d) {
    const double qd = (double)q;
    dmma884(acc.g2[0], acc.g2[1], qd, qd);
    acc.a3 = fma(q8d, qd, acc.a3);
    acc.a5 = fma(q8d, q8d, acc.a5);
    if (!SAME) {
        const double xd = (double)x;
        dmma884(acc.g1[0], acc.g1[1], qd, xd);
        acc.a1 = fma(qd, x8d, acc.a1);
        acc.a2 = fma(q8d, xd, acc.a2);
        acc.a4 = fma(q8d, x8d, acc.a4);
    }
}

// Fragments -> one 2*81-entry partial [G1 | G2] in shared memory (lower triangle of G2 valid).
template <bool SAME>
__device__ __forceinline__ void gram9_store(Gram9Acc &acc, double *r, int g, int k) {
    constexpr int KK = 9;
    // the ninth row / column: sum this lane group's four column phases (fixed butterfly order)
    double *edge[5] = {&acc.a1, &acc.a2, &acc.a3, &acc.a4, &acc.a5};
#pragma unroll
    for (int e = 0; e < 5; ++e) {
        double v = *edge[e];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        *edge[e] = v;
    }
    if (!SAME) {
        r[g * KK + 2 * k] = acc.g1[0];
        r[g * KK + 2 * k + 1] = acc.g1[1];
    }
    r[KK * KK + g * KK + 2 * k] = acc.g2[0];
    r[KK * KK + g * KK + 2 * k + 1] = acc.g2[1];
    if (k == 0) {
        if (!SAME) {
            r[g * KK + 8] = acc.a1;
            r[8 * KK + g] = acc.a2;
        }
        r[KK * KK + 8 * KK + g] = acc.a3;
        r[KK * KK + g * KK + 8] = 0.0;  // above the diagonal, never read
        if (g == 0) {
            if (!SAME) r[8 * KK + 8] = acc.a4;
            r[KK * KK + 8 * KK + 8] = acc.a5;
        }
    }
}

template <bool SAME>
__global__ void __launch_bounds__(CONV_BLOCK, 2)
conv_gram9_dmma_kernel(ConvPtrs ptrs, int64_t n, int64_t chunk_cols, double *__restrict__ partial, int slots) {
    constexpr int KK = 9, NW = CONV_BLOCK / 32, SZ = 2 * KK * KK;
    __shared__ double red[NW][SZ];
    const int ch = blockIdx.y, chunk = blockIdx.x;
    const float *X = ptrs.Xp[ch];
    const float *Xq = SAME ? X : ptrs.Xqp[ch];
    const int64_t c_beg = (int64_t)chunk * chunk_cols;
    const int64_t c_end = (c_beg + chunk_cols < n) ? c_beg + chunk_cols : n;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, k = lane & 3;
    const float *qrow = Xq + (int64_t)g * n, *q8row = Xq + (int64_t)8 * n;
    const float *xrow = X + (int64_t)g * n, *x8row = X + (int64_t)8 * n;

    Gram9Acc acc = {};
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 q[2], x[2], q8[2], x8[2];
    auto load = [&](int64_t base, float4 *lq, float4 *lx, float4 *lq8, float4 *lx8) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int64_t c = base + 16 * u + 4 * k;
            const bool ok = c < c_end;  // n % 4 == 0: a float4 is wholly inside or wholly outside
            lq[u] = ok ? ldg_stream4(qrow + c) : z4;
            lq8[u] = ok ? ldg_stream4(q8row + c) : z4;
            if (!SAME) {
                lx[u] = ok ? ldg_stream4(xrow + c) : z4;
                lx8[u] = ok ? ldg_stream4(x8row + c) : z4;
            }
        }
    };
    auto compute = [&](const float4 *lq, const float4 *lx, const float4 *lq8, const float4 *lx8) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            gram9_step<SAME>(acc, lq[u].x, lx[u].x, lq8[u].x, lx8[u].x);
            gram9_step<SAME>(acc, lq[u].y, lx[u].y, lq8[u].y, lx8[u].y);
            gram9_step<SAME>(acc, lq[u].z, lx[u].z, lq8[u].z, lx8[u].z);
            gram9_step<SAME>(acc, lq[u].w, lx[u].w, lq8[u].w, lx8[u].w);
        }
    };
    // two register buffers in ping-pong: the loads of the next 32 columns are in flight while the current 32 are
    // multiplied (out-of-range loads return zeros, which add nothing)
    float4 p[2], px[2], p8[2], px8[2];
    constexpr int64_t S = NW * 32;
    int64_t base = c_beg + (int64_t)warp * 32;
    load(base, q, x, q8, x8);
    for (; base < c_end; base += 2 * S) {
        load(base + S, p, px, p8, px8);
        compute(q, x, q8, x8);
        load(base + 2 * S, q, x, q8, x8);
        compute(p, px, p8, px8);
    }
    gram9_store<SAME>(acc, red[warp], g, k);
    __syncthreads();
    double *out = partial + ((size_t)ch * slots + chunk) * SZ;
    for (int e = threadIdx.x; e < SZ; e += CONV_BLOCK) {
        if (SAME && e < KK * KK) continue;
        double tot = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) tot += red[w][e];  // warps in index order
        out[e] = tot;
    }
}

// ---- stage 1, 3x3 fast path with TMA staging ------------------------------------------------------
// Same arithmetic and lane mapping as conv_gram9_dmma_kernel, but the patch rows reach the SM as bulk
// async copies (cp.async.bulk = UBLKCP, completion on an mbarrier) into a ring of shared-memory stages,
// issued by a dedicated producer warp: the bytes in flight (4 of 5 stages of 18 rows x 512 columns,
// ~150 KB per SM) no longer live in registers, so 16 consumer warps keep the fp64 pipe fed while the
// whole HBM latency is covered.  Each consumer warp owns a fixed 32-column slice of every stage, so the
// summation order is fixed.  Row pitch is COLS + 16 floats: lane groups g and g+1 then start 16 banks
// apart and the LDS.128 fragments are conflict free.
namespace tma9 {
constexpr int CWARPS = 24;                 // consumer warps
constexpr int COLS = CWARPS * 32;          // columns per stage
constexpr int PITCH = COLS + 16;           // floats
constexpr int STAGES = 3;
constexpr int THREADS = (CWARPS + 1) * 32;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n.reg .pred p;\nWAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
}  // namespace tma9

template <bool SAME>
__global__ void __launch_bounds__(tma9::THREADS, 1)
conv_gram9_tma_kernel(ConvPtrs ptrs, int64_t n, int64_t chunk_cols, double *__restrict__ partial, int slots) {
    using namespace tma9;
    constexpr int KK = 9, SZ = 2 * KK * KK, ROWS = SAME ? KK : 2 * KK;
    constexpr int STAGE_FLOATS = ROWS * PITCH;
    extern __shared__ __align__(128) unsigned char tma9_smem[];
    float *stages = reinterpret_cast<float *>(tma9_smem);                                     // STAGES x ROWS x PITCH
    double *red = reinterpret_cast<double *>(tma9_smem + (size_t)STAGES * STAGE_FLOATS * 4);  // CWARPS x SZ
    uint64_t *full = reinterpret_cast<uint64_t *>(red + CWARPS * SZ);
    uint64_t *empty = full + STAGES;

    const int ch = blockIdx.y, chunk = blockIdx.x;
    const float *X = ptrs.Xp[ch];
    const float *Xq = SAME ? X : ptrs.Xqp[ch];
    const int64_t c_beg = (int64_t)chunk * chunk_cols;
    const int64_t c_end = (c_beg + chunk_cols < n) ? c_beg + chunk_cols : n;
    const int n_iter = (int)((c_end - c_beg + COLS - 1) / COLS);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], CWARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();

    if (warp == CWARPS) {
        // ---- producer: one lane streams the rows of every stage
        if (lane == 0) {
            for (int it = 0; it < n_iter; ++it) {
                const int s = it % STAGES;
                if (it >= STAGES) mbar_wait(&empty[s], ((it / STAGES) - 1) & 1);
                const int64_t c0 = c_beg + (int64_t)it * COLS;
                const int64_t cols = (c_end - c0 < COLS) ? c_end - c0 : COLS;
                const uint32_t bytes = (uint32_t)cols * 4u;
                mbar_expect_tx(&full[s], bytes * ROWS);
                float *dst = stages + (size_t)s * STAGE_FLOATS;
#pragma unroll 1
                for (int r = 0; r < KK; ++r) {
                    bulk_g2s(dst + r * PITCH, Xq + (int64_t)r * n + c0, bytes, &full[s]);
                    if (!SAME) bulk_g2s(dst + (KK + r) * PITCH, X + (int64_t)r * n + c0, bytes, &full[s]);
                }
            }
        }
        return;
    }

    // ---- consumers
    const int g = lane >> 2, k = lane & 3;
    Gram9Acc acc = {};
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    // The ninth row (tap 8) is needed by all eight row-lanes of a column: every lane converts ONE column of it per stage
    // and parks the fp64 values in the warp's (still unused) reduction slot, instead of 8 redundant F2F per value --
    // 18 instead of 32 conversions per lane and stage on the quarter-rate XU pipe.
    double *r8 = red + warp * SZ;  // [0, 32): Xq tap 8, [32, 64): X tap 8, fp64
    for (int it = 0; it < n_iter; ++it) {
        const int s = it % STAGES;
        mbar_wait(&full[s], (it / STAGES) & 1);
        const float *st = stages + (size_t)s * STAGE_FLOATS;
        const int64_t valid = c_end - (c_beg + (int64_t)it * COLS);  // columns present in this stage (multiple of 4)
        float4 q[2], x[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int c = warp * 32 + 16 * u + 4 * k;
            const bool ok = c < valid;
            q[u] = ok ? *reinterpret_cast<const float4 *>(st + g * PITCH + c) : z4;
            if (!SAME) x[u] = ok ? *reinterpret_cast<const float4 *>(st + (KK + g) * PITCH + c) : z4;
        }
        {
            const int c8 = warp * 32 + lane;
            const bool ok8 = c8 < valid;
            r8[lane] = ok8 ? (double)st[8 * PITCH + c8] : 0.0;
            if (!SAME) r8[32 + lane] = ok8 ? (double)st[(KK + 8) * PITCH + c8] : 0.0;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);  // the slice is in registers: hand the stage back
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const double2 qa = *reinterpret_cast<const double2 *>(r8 + 16 * u + 4 * k);
            const double2 qb = *reinterpret_cast<const double2 *>(r8 + 16 * u + 4 * k + 2);
            double2 xa = make_double2(0.0, 0.0), xb = xa;
            if (!SAME) {
                xa = *reinterpret_cast<const double2 *>(r8 + 32 + 16 * u + 4 * k);
                xb = *reinterpret_cast<const double2 *>(r8 + 32 + 16 * u + 4 * k + 2);
            }
            gram9_step_d<SAME>(acc, q[u].x, x[u].x, qa.x, xa.x);
            gram9_step_d<SAME>(acc, q[u].y, x[u].y, qa.y, xa.y);
            gram9_step_d<SAME>(acc, q[u].z, x[u].z, qb.x, xb.x);
            gram9_step_d<SAME>(acc, q[u].w, x[u].w, qb.y, xb.y);
        }
        __syncwarp();  // every lane has read the parked row before the next stage overwrites it
    }
    gram9_store<SAME>(acc, red + warp * SZ, g, k);
    // consumer-only barrier (the producer warp has left)
    asm volatile("bar.sync 1, %0;\n" ::"r"(CWARPS * 32));
    double *out = partial + ((size_t)ch * slots + chunk) * SZ;
    for (int e = threadIdx.x; e < SZ; e += CWARPS * 32) {
        if (SAME && e < KK * KK) continue;
        double tot = 0.0;
#pragma unroll
        for (int w = 0; w < CWARPS; ++w) tot += red[w * SZ + e];  // warps in index order
        out[e] = tot;
    }
}

// ---- stage 1, 3x3 / stride 1 straight from the NHWC activations --------------------------------------
// The patch matrix of a 3x3 stride-1 convolution is nine shifted views of the (zero-padded) channel image, so
// it never has to exist: a CTA stages a band of rows of CG = 8 channels of one image in shared memory as
// per-channel planes (pitch P, halo included), and warp w runs the DMMA/DFMA Gram of conv_gram9_* for channel
// w with its operands read from the plane at (row + r_g, col + c_g).  Lane (g, k) takes output columns
// col4 + k of four "cells" of four columns per step, so the 32 lanes of an LDS touch a 3 x 6 window per
// cell: neighbouring lanes hit the same word (broadcast) and a pitch with P mod 32 in [8, 12] keeps the three
// rows on disjoint banks.  HBM traffic drops from 72 to 8 bytes per patch column and channel; the kernel is
// bound by the fp64 pipe (168 slots per column).  Output widths that are not a multiple of four take a ragged last
// cell (its extra lanes contribute zeros).  Geometry outside 3x3 / stride 1 / rate 1 goes through im2col_kernel + the
// patch kernels.
namespace nhwc9 {
constexpr int CG = 8;              // channels per CTA = consumer warps
constexpr int THREADS = CG * 32;
constexpr int MAX_PLANE = 1664;    // floats per plane: 2 matrices x 8 channels x 6.5 KB = 104 KB -> two CTAs per SM
}  // namespace nhwc9

struct Nhwc9Geom {
    int H, W, Ho, Wo, pt, pl;      // input size, output size, top / left padding (SAME: 1, VALID: 0)
    int P, BR;                     // plane pitch (floats), output rows per band
    int64_t C;                     // channels of the activation tensor
    int64_t c_first;               // first channel handled by blockIdx.y == 0
    int n_ch;                      // channels handled by this launch
    int64_t img0, n_img;           // image range of this launch
    int imgs_per_cta;
};

template <bool SAME>
__global__ void __launch_bounds__(nhwc9::THREADS, 2)
conv_gram9_nhwc_kernel(const float *__restrict__ act, const float *__restrict__ actq, Nhwc9Geom gm,
                       double *__restrict__ partial, int slots) {
    using namespace nhwc9;
    constexpr int KK = 9, SZ = 2 * KK * KK;
    extern __shared__ __align__(16) float nhwc9_smem[];
    const int plane = (gm.BR + 2) * gm.P;
    float *planes_q = nhwc9_smem;                    // CG planes of Xq
    float *planes_x = SAME ? planes_q : planes_q + CG * plane;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, k = lane & 3;
    const int r_g = g / 3, c_g = g % 3;
    const int64_t ch0 = gm.c_first + (int64_t)blockIdx.y * CG;          // first channel of this CTA
    const int nch_cta = (gm.n_ch - (int)blockIdx.y * CG) < CG ? (gm.n_ch - (int)blockIdx.y * CG) : CG;
    const int64_t ia = gm.img0 + (int64_t)blockIdx.x * gm.imgs_per_cta;
    const int64_t ib = (ia + gm.imgs_per_cta < gm.img0 + gm.n_img) ? ia + gm.imgs_per_cta : gm.img0 + gm.n_img;
    const int cells_per_row = (gm.Wo + 3) >> 2, Wp = cells_per_row * 4 + 2;  // a ragged last cell reads zero-filled columns
    const bool vec4 = (gm.C % 4 == 0) && (ch0 % 4 == 0) && (nch_cta == CG);

    Gram9Acc acc = {};
    for (int64_t img = ia; img < ib; ++img) {
        const float *ai = act + img * (int64_t)gm.H * gm.W * gm.C;
        const float *aq = SAME ? ai : actq + img * (int64_t)gm.H * gm.W * gm.C;
        for (int i0 = 0; i0 < gm.Ho; i0 += gm.BR) {
            const int br = (gm.Ho - i0) < gm.BR ? (gm.Ho - i0) : gm.BR;
            __syncthreads();  // the previous band has been consumed
            // ---- stage rows [i0 - pt, i0 - pt + br + 2) x cols [-pl, Wo + 2 - pl) of CG channels, zero outside the image
            const int npix = (br + 2) * Wp;
            if (vec4) {
                for (int e = tid; e < npix * 2; e += THREADS) {
                    const int quad = e & 1, pix = e >> 1;
                    const int rr = pix / Wp, cc = pix - rr * Wp;
                    const int iy = i0 - gm.pt + rr, ix = cc - gm.pl;
                    float4 vq = make_float4(0.f, 0.f, 0.f, 0.f), vx = vq;
                    if (iy >= 0 && iy < gm.H && ix >= 0 && ix < gm.W) {
                        const int64_t off = ((int64_t)iy * gm.W + ix) * gm.C + ch0 + quad * 4;
                        vq = __ldg(reinterpret_cast<const float4 *>(aq + off));
                        if (!SAME) vx = __ldg(reinterpret_cast<const float4 *>(ai + off));
                    }
                    float *dq = planes_q + (quad * 4) * plane + rr * gm.P + cc;
                    dq[0] = vq.x; dq[plane] = vq.y; dq[2 * plane] = vq.z; dq[3 * plane] = vq.w;
                    if (!SAME) {
                        float *dx = planes_x + (quad * 4) * plane + rr * gm.P + cc;
                        dx[0] = vx.x; dx[plane] = vx.y; dx[2 * plane] = vx.z; dx[3 * plane] = vx.w;
                    }
                }
            } else {
                for (int e = tid; e < npix * CG; e += THREADS) {
                    const int ch = e % CG, pix = e / CG;
                    const int rr = pix / Wp, cc = pix - rr * Wp;
                    const int iy = i0 - gm.pt + rr, ix = cc - gm.pl;
                    float vq = 0.f, vx = 0.f;
                    if (ch < nch_cta && iy >= 0 && iy < gm.H && ix >= 0 && ix < gm.W) {
                        const int64_t off = ((int64_t)iy * gm.W + ix) * gm.C + ch0 + ch;
                        vq = __ldg(aq + off);
                        if (!SAME) vx = __ldg(ai + off);
                    }
                    planes_q[ch * plane + rr * gm.P + cc] = vq;
                    if (!SAME) planes_x[ch * plane + rr * gm.P + cc] = vx;
                }
            }
            __syncthreads();
            if (warp >= nch_cta) continue;
            // ---- this warp's channel: four cells (16 output columns) per step
            const float *pq = planes_q + warp * plane, *px = planes_x + warp * plane;
            const int ncell = br * cells_per_row;
            int row = 0, cell = 0;  // (row, cell-in-row) of the step's first cell
            for (int f0 = 0; f0 < ncell; f0 += 4) {
                float q[4], x[4], q8[4], x8[4];
                int rw = row, cl = cell;
#pragma unroll
                for (int sgrp = 0; sgrp < 4; ++sgrp) {
                    const bool ok = f0 + sgrp < ncell && cl * 4 + k < gm.Wo;  // columns past Wo are not patches
                    const int base = rw * gm.P + cl * 4 + k;
                    q[sgrp] = ok ? pq[base + r_g * gm.P + c_g] : 0.f;
                    q8[sgrp] = ok ? pq[base + 2 * gm.P + 2] : 0.f;
                    if (!SAME) {
                        x[sgrp] = ok ? px[base + r_g * gm.P + c_g] : 0.f;
                        x8[sgrp] = ok ? px[base + 2 * gm.P + 2] : 0.f;
                    }
                    if (++cl == cells_per_row) { cl = 0; ++rw; }
                }
                row = rw; cell = cl;
#pragma unroll
                for (int sgrp = 0; sgrp < 4; ++sgrp) gram9_step<SAME>(acc, q[sgrp], x[sgrp], q8[sgrp], x8[sgrp]);
            }
        }
    }
    __syncthreads();
    double *red = reinterpret_cast<double *>(nhwc9_smem);  // the planes are dead: reuse them for the fragments
    if (warp < nch_cta) gram9_store<SAME>(acc, red + warp * SZ, g, k);
    __syncthreads();
    for (int e = tid; e < nch_cta * SZ; e += THREADS) {
        const int ch = e / SZ, idx = e % SZ;
        if (SAME && idx < KK * KK) continue;
        partial[(((size_t)blockIdx.y * CG + ch) * slots + blockIdx.x) * SZ + idx] = red[ch * SZ + idx];
    }
}

// ---- stage 1, any kk <= 128 on the fp64 tensor pipe ---------------------------------------------
// The sizes without a kernel above (5 x 5, 7 x 7, 11 x 11, 1 x 7, ...).  The kk patch rows are padded with zero rows to
// KP = 8 NB and cut into NB blocks of eight; the lower-triangular 8 x 8 tiles (I >= J) of G2 = Xq Xq^T and G1 = Xq X^T are one
// DMMA.8x8x4 each per four columns (exact fp32 products, fp64 sums: the Gram form of DESIGN section 3).  A CTA stages TC
// columns of Xq (and X) in shared memory, converted to fp64 once; the next stage's loads are in flight in registers while
// the current one is multiplied.  Warp (p, cg) owns the tiles of block rows p and NB-1-p (NB + 1 tiles per Gram, the A fragment
// of a row loaded once per four columns) over the four-column steps cg, cg + CG, ... of every stage; the CG column groups are
// added in index order at the end, so the summation order is fixed and the result bit-reproducible.  Padding rows are zero, so
// they add nothing; a tap that only ever reads padding has an exactly zero row.  Any n and any row alignment (scalar loads).
// Writes the partial layout of conv_gram_kernel: lower triangle + diagonal of G2, of G1 too (its upper triangle is written 0).
namespace gramx {
constexpr int MAX_KK = 128;
template <int NB>
struct Cfg {
    static constexpr int KP = 8 * NB;
    static constexpr int NP = (NB + 1) / 2;                  // block-row pairs
    static constexpr int CG = 8 / NP >= 1 ? 8 / NP : 1;      // column groups
    static constexpr int NW = NP * CG;                       // warps (5..8)
    static constexpr int NT = NW * 32;
    static constexpr int TC = 2048 / KP >= 256 ? 256 : 2048 / KP >= 128 ? 128 : 2048 / KP >= 64 ? 64 : 2048 / KP >= 32 ? 32 : 16;
    static constexpr int LTC = TC == 256 ? 8 : TC == 128 ? 7 : TC == 64 ? 6 : TC == 32 ? 5 : 4;
    static constexpr int PITCH = TC + 4;                     // doubles: lanes (g, k) of an LDS.64 half-warp on distinct banks
    static constexpr int MINB = NB == 1 ? 3 : NB <= 4 ? 2 : 1;   // CTAs per SM the registers allow without spills
    static_assert((TC / 4) % CG == 0, "every column group gets the same steps");
};
// dynamic shared memory: the fp64 stage, reused for the column-group sum (CG > 1)
template <int NB, bool SAME>
constexpr size_t smem_bytes() {
    using C = Cfg<NB>;
    const size_t stage = (size_t)(SAME ? 1 : 2) * C::KP * C::PITCH * sizeof(double);
    const size_t red = C::CG > 1 ? (size_t)2 * C::KP * C::KP * sizeof(double) : 0;
    return stage > red ? stage : red;
}
}  // namespace gramx

template <int NB, bool SAME>
__global__ void __launch_bounds__(gramx::Cfg<NB>::NT, gramx::Cfg<NB>::MINB)
conv_gramx_kernel(ConvPtrs ptrs, int64_t n, int kk, int64_t chunk_cols, double *__restrict__ partial, int slots) {
    using C = gramx::Cfg<NB>;
    constexpr int KP = C::KP, TC = C::TC, PITCH = C::PITCH, NT = C::NT, NMAT = SAME ? 1 : 2;
    constexpr int E = (NMAT * KP * TC + NT - 1) / NT;   // staged elements per thread and stage
    extern __shared__ __align__(16) double gramx_smem[];
    double *sq = gramx_smem;                            // KP x PITCH: Xq
    double *sx = SAME ? sq : sq + KP * PITCH;           // KP x PITCH: X
    const int ch = blockIdx.y, chunk = blockIdx.x;
    const float *X = ptrs.Xp[ch];
    const float *Xq = SAME ? X : ptrs.Xqp[ch];
    const int64_t c_beg = (int64_t)chunk * chunk_cols;
    const int64_t c_end = (c_beg + chunk_cols < n) ? c_beg + chunk_cols : n;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, k = lane & 3;
    const int p = warp % C::NP, cg = warp / C::NP;
    const int I1 = p, I2 = NB - 1 - p;
    const int real = NMAT * kk * TC;                    // staged elements of the kk real rows

    // padding rows kk .. KP-1 stay zero for the whole kernel
    for (int e = tid; e < NMAT * (KP - kk) * PITCH; e += NT) {
        const int m = e / ((KP - kk) * PITCH), rc = e % ((KP - kk) * PITCH);
        gramx_smem[m * KP * PITCH + kk * PITCH + rc] = 0.0;
    }
    float pre[E];
    auto load = [&](int64_t c0) {
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int e = tid + i * NT;
            const int c = e & (TC - 1), mr = e >> C::LTC;
            const int m = mr >= kk ? 1 : 0, r = mr - m * kk;
            const int64_t col = c0 + c;
            const float *src = m ? X : Xq;
            pre[i] = (e < real && col < c_end) ? __ldg(src + (int64_t)r * n + col) : 0.f;
        }
    };
    double acc2[NB + 1][2] = {}, acc1[NB + 1][2] = {};
    load(c_beg);
    for (int64_t c0 = c_beg; c0 < c_end; c0 += TC) {
        __syncthreads();  // the previous stage has been read
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int e = tid + i * NT;
            if (e < real) {
                const int c = e & (TC - 1), mr = e >> C::LTC;
                const int m = mr >= kk ? 1 : 0, r = mr - m * kk;
                gramx_smem[(m * KP + r) * PITCH + c] = (double)pre[i];
            }
        }
        __syncthreads();
        if (c0 + TC < c_end) load(c0 + TC);  // in flight while this stage is multiplied
        for (int ks = cg; ks < TC / 4; ks += C::CG) {
            const int col = 4 * ks + k;
            const double a1 = sq[(8 * I1 + g) * PITCH + col], a2 = sq[(8 * I2 + g) * PITCH + col];
#pragma unroll
            for (int j = 0; j <= NB; ++j) {
                // tile j: (I1, j) for j <= I1, else (I2, j - I1 - 1); the middle row of an odd NB has no second row
                const bool r1 = j <= I1;
                if (!r1 && I2 == I1) continue;
                const int J = r1 ? j : j - I1 - 1;
                const double a = r1 ? a1 : a2;
                dmma884(acc2[j][0], acc2[j][1], a, sq[(8 * J + g) * PITCH + col]);
                if (!SAME) dmma884(acc1[j][0], acc1[j][1], a, sx[(8 * J + g) * PITCH + col]);
            }
        }
    }

    double *out = partial + ((size_t)ch * slots + chunk) * (2 * kk * kk);
    // lane (g, k) of tile (I, J) holds entries (8 I + g, 8 J + 2 k + u), u = 0, 1
    auto tile_of = [&](int j, int &I, int &J) {
        const bool r1 = j <= I1;
        I = r1 ? I1 : I2;
        J = r1 ? j : j - I1 - 1;
        return r1 || I2 != I1;
    };
    if (!SAME)
        for (int e = tid; e < kk * kk; e += NT)
            if (e % kk > e / kk) out[e] = 0.0;  // upper triangle of G1: not computed
    if (C::CG == 1) {
#pragma unroll
        for (int j = 0; j <= NB; ++j) {
            int I, J;
            if (!tile_of(j, I, J)) continue;
            const int t = 8 * I + g;
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int s = 8 * J + 2 * k + u;
                if (t < kk && s <= t) {
                    out[kk * kk + t * kk + s] = acc2[j][u];
                    if (!SAME) out[t * kk + s] = acc1[j][u];
                }
            }
        }
        return;
    }
    // column groups in index order through shared memory: red[which][t][s], KP x KP each
    double *red = gramx_smem;
    for (int c = 0; c < C::CG; ++c) {
        __syncthreads();
        if (cg == c) {
#pragma unroll
            for (int j = 0; j <= NB; ++j) {
                int I, J;
                if (!tile_of(j, I, J)) continue;
                const int t = 8 * I + g;
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int s = 8 * J + 2 * k + u;
                    double *r2 = red + KP * KP + t * KP + s, *r1 = red + t * KP + s;
                    *r2 = c == 0 ? acc2[j][u] : *r2 + acc2[j][u];
                    if (!SAME) *r1 = c == 0 ? acc1[j][u] : *r1 + acc1[j][u];
                }
            }
        }
    }
    __syncthreads();
    for (int e = tid; e < kk * kk; e += NT) {
        const int t = e / kk, s = e % kk;
        if (s > t) continue;
        out[kk * kk + e] = red[KP * KP + t * KP + s];
        if (!SAME) out[e] = red[t * KP + s];
    }
}

// ---- stage 2 ---------------------------------------------------------------------------------
// gram: (n_channels, 2*kk*kk): [G1 | G2], lower triangle + diagonal of each valid.
__global__ void conv_finalize_kernel(const double *__restrict__ partial, int n_chunks, int kk, int same,
                                     double *__restrict__ gram) {
    const int ch = blockIdx.x, sz = 2 * kk * kk;
    for (int e = threadIdx.x; e < sz; e += blockDim.x) {
        const int which = e / (kk * kk), t = (e % (kk * kk)) / kk, s = e % kk;
        if (which == 1 && s > t) { gram[(size_t)ch * sz + e] = 0.0; continue; }
        const int src = (which == 0 && same) ? kk * kk + t * kk + s : e;
        if (which == 0 && same && s > t) { gram[(size_t)ch * sz + e] = 0.0; continue; }
        double tot = 0.0;
        for (int c = 0; c < n_chunks; ++c) tot += partial[((size_t)ch * n_chunks + c) * sz + src];
        gram[(size_t)ch * sz + e] = tot;
    }
}

// ---- stage 3 ---------------------------------------------------------------------------------
// One thread per (channel, filter, alphabet).  W/Q tap stride CF = Cg*F, where a group of Cg = C / groups input channels
// feeds Fg = F / groups filters.  Ungrouped (Cg = C, Fg = F): channel c, filter f at c*F + f.  GROUPED: channel c walks only
// the Fg filters of its group g = c / Cg, filter f < Fg at (c % Cg)*F + g*Fg + f -- the (kh, kw, C / groups, F) kernel of a
// grouped Conv2D, indexed in place.
template <bool GROUPED>
__device__ __forceinline__ int64_t conv_wq_offset(int64_t c, int64_t f, int64_t F, int64_t Cg, int64_t Fg) {
    return GROUPED ? (c % Cg) * F + (c / Cg) * Fg + f : c * F + f;
}

template <int KK, bool GROUPED>
__global__ void __launch_bounds__(128)
conv_sweep_kernel(const double *__restrict__ gram, const float *__restrict__ W, double *__restrict__ Q,
                  int64_t CF, int64_t F, int64_t c0, const double *__restrict__ alphabets,
                  const int *__restrict__ Koff, const int *__restrict__ Flags, int64_t q_alph_stride, int64_t Cg, int64_t Fg) {
    __shared__ double g1[KK * KK], g2[KK * KK], nrm[KK], alph[GPFQ_MAX_K];
    const int ch = blockIdx.y, a = blockIdx.z;
    const int K = Koff[a + 1] - Koff[a];
    for (int e = threadIdx.x; e < KK * KK; e += blockDim.x) {
        g1[e] = gram[(size_t)ch * 2 * KK * KK + e];
        g2[e] = gram[(size_t)ch * 2 * KK * KK + KK * KK + e];
    }
    for (int e = threadIdx.x; e < K; e += blockDim.x) alph[e] = alphabets[Koff[a] + e];
    __syncthreads();
    if (threadIdx.x < KK) nrm[threadIdx.x] = (double)(float)sqrt(g2[threadIdx.x * KK + threadIdx.x]);
    __syncthreads();
    const double inv_step = gpfq_inv_step(alph, K, Flags[a]);
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= (GROUPED ? Fg : F)) return;
    const int64_t base = conv_wq_offset<GROUPED>(c0 + ch, f, F, Cg, Fg);
    double w[KK], q[KK];
#pragma unroll
    for (int t = 0; t < KK; ++t) w[t] = (double)W[(int64_t)t * CF + base];
#pragma unroll
    for (int t = 0; t < KK; ++t) {
        double d = 0.0;
#pragma unroll
        for (int s = 0; s < KK; ++s)
            if (s < t) d += w[s] * g1[t * KK + s] - q[s] * g2[t * KK + s];
        const double num = fma(w[t], g1[t * KK + t], d);
        q[t] = gpfq_decide(nrm[t], d, num, w[t], alph, K, inv_step);
        Q[(int64_t)a * q_alph_stride + (int64_t)t * CF + base] = q[t];
    }
}

// The same walk for any kk <= 128: one warp per (channel, filter, alphabet).  The channel's lower triangles sit in shared
// memory packed by columns (column s holds rows s .. kk-1, so the lanes of one update read consecutive words).  Lane l holds the
// running dots d[t'] of the directions t' = l, l + 32, ...; after step t every later direction adds its term
// w_t G1[t', t] - q_t G2[t', t], so d[t'] is summed over s < t' in ascending s, as in conv_sweep_kernel.  The lane that owns t
// decides and q_t goes to the others by shuffle.
namespace walkx {
constexpr int MAXW = 16;  // warps (filters) per CTA
__host__ __device__ constexpr int col_off(int s, int kk) { return s * kk - s * (s - 1) / 2; }
}  // namespace walkx

template <bool GROUPED>
__global__ void __launch_bounds__(walkx::MAXW * 32)
conv_walkx_kernel(const double *__restrict__ gram, int kk, const float *__restrict__ W, double *__restrict__ Q, int64_t CF,
                  int64_t F, int64_t c0, const double *__restrict__ alphabets, const int *__restrict__ Koff,
                  const int *__restrict__ Flags, int64_t q_alph_stride, int64_t Cg, int64_t Fg) {
    extern __shared__ double walkx_smem[];
    const int tri = kk * (kk + 1) / 2;
    double *g1 = walkx_smem, *g2 = g1 + tri, *nrm = g2 + tri, *alph = nrm + kk;
    const int ch = blockIdx.y, a = blockIdx.z;
    const int K = Koff[a + 1] - Koff[a];
    const double *gc = gram + (size_t)ch * 2 * kk * kk;
    for (int e = threadIdx.x; e < kk * kk; e += blockDim.x) {
        const int t = e / kk, s = e % kk;
        if (s > t) continue;
        const int o = walkx::col_off(s, kk) + t - s;
        g1[o] = gc[e];
        g2[o] = gc[kk * kk + e];
    }
    for (int e = threadIdx.x; e < K; e += blockDim.x) alph[e] = alphabets[Koff[a] + e];
    __syncthreads();
    for (int t = threadIdx.x; t < kk; t += blockDim.x) nrm[t] = (double)(float)sqrt(g2[walkx::col_off(t, kk)]);
    __syncthreads();
    const double inv_step = gpfq_inv_step(alph, K, Flags[a]);
    const int lane = threadIdx.x & 31;
    const int64_t f = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (f >= (GROUPED ? Fg : F)) return;
    const int64_t base = conv_wq_offset<GROUPED>(c0 + ch, f, F, Cg, Fg);
    double *q_out = Q + (int64_t)a * q_alph_stride + base;
    double w[4], d[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int t = 32 * j + lane;
        w[j] = t < kk ? (double)W[(int64_t)t * CF + base] : 0.0;
        d[j] = 0.0;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (32 * j >= kk) break;
        const int o_end = kk - 32 * j < 32 ? kk - 32 * j : 32;
        for (int o = 0; o < o_end; ++o) {
            const int t = 32 * j + o;
            const int off = walkx::col_off(t, kk) - t;  // g[off + t'] = G[t', t]
            double qt = 0.0;
            if (lane == o) {
                const double num = fma(w[j], g1[off + t], d[j]);
                qt = gpfq_decide(nrm[t], d[j], num, w[j], alph, K, inv_step);
                q_out[(int64_t)t * CF] = qt;
            }
            qt = __shfl_sync(0xffffffffu, qt, o);
            const double wt = __shfl_sync(0xffffffffu, w[j], o);
#pragma unroll
            for (int j2 = j; j2 < 4; ++j2) {
                const int t2 = 32 * j2 + lane;
                if (t2 > t && t2 < kk) d[j2] += wt * g1[off + t2] - qt * g2[off + t2];
            }
        }
    }
}

// ---- on-device single-channel im2col (extract_patches semantics) ------------------------------
// out[ch]: (kh*kw, n_img*Ho*Wo), row r*kw+c, column (img*Ho + i)*Wo + j.
__global__ void im2col_kernel(const float *__restrict__ act, int64_t n_img, int H, int Wd, int64_t C,
                              int64_t c_first, int kh, int kw, int sh, int sw, int rh, int rw, int pt, int pl,
                              int Ho, int Wo, float *__restrict__ out, int64_t ch_stride) {
    const int ch = blockIdx.y;
    const int tap = blockIdx.z;
    const int r = tap / kw, cc = tap % kw;
    const int64_t n = n_img * Ho * Wo;
    float *dst = out + (size_t)ch * ch_stride + (size_t)tap * n;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(p % Wo);
        const int i = (int)((p / Wo) % Ho);
        const int64_t img = p / ((int64_t)Wo * Ho);
        const int y = i * sh + r * rh - pt, x = j * sw + cc * rw - pl;
        float v = 0.f;
        if (y >= 0 && y < H && x >= 0 && x < Wd) v = act[((img * H + y) * Wd + x) * C + c_first + ch];
        dst[p] = v;
    }
}

// ---- MSQ -------------------------------------------------------------------------------------
template <typename T>
__global__ void msq_kernel(const T *__restrict__ W, int64_t n, const double *__restrict__ alphabet, int K, int equispaced,
                           double *__restrict__ Q) {
    __shared__ double alph[GPFQ_MAX_K];
    for (int e = threadIdx.x; e < K; e += blockDim.x) alph[e] = alphabet[e];
    __syncthreads();
    const double inv_step = gpfq_inv_step(alph, K, equispaced);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        Q[i] = gpfq_bit_round_eq((double)W[i], alph, K, inv_step);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <int KK>
static int launch_conv_gram(gpfq_ctx *ctx, ConvPtrs ptrs, bool same, int64_t n, int n_ch, int n_chunks,
                            int64_t chunk_cols, double *partial, bool vec_ok, int slots) {
    dim3 grid((unsigned)n_chunks, (unsigned)n_ch);
    if (KK == 9 && vec_ok && (ctx->conv_variant == 0 || ctx->conv_variant == 3)) {
        using namespace tma9;
        constexpr size_t tail = (size_t)CWARPS * 2 * 81 * sizeof(double) + 2 * STAGES * sizeof(uint64_t);
        const size_t smem = (size_t)STAGES * (same ? 9 : 18) * PITCH * sizeof(float) + tail;
        if (same) {
            CUDA_TRY(ctx, cudaFuncSetAttribute(conv_gram9_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            conv_gram9_tma_kernel<true><<<grid, THREADS, smem, ctx->stream>>>(ptrs, n, chunk_cols, partial, slots);
        } else {
            CUDA_TRY(ctx, cudaFuncSetAttribute(conv_gram9_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            conv_gram9_tma_kernel<false><<<grid, THREADS, smem, ctx->stream>>>(ptrs, n, chunk_cols, partial, slots);
        }
        KERNEL_CHECK(ctx);
        return GPFQ_OK;
    }
    if (KK == 9 && vec_ok && ctx->conv_variant == 1) {
        if (same) conv_gram9_dmma_kernel<true><<<grid, CONV_BLOCK, 0, ctx->stream>>>(ptrs, n, chunk_cols, partial, slots);
        else conv_gram9_dmma_kernel<false><<<grid, CONV_BLOCK, 0, ctx->stream>>>(ptrs, n, chunk_cols, partial, slots);
        KERNEL_CHECK(ctx);
        return GPFQ_OK;
    }
    constexpr int NG = (KK >= 9) ? 2 : 1;
    if (same) conv_gram_kernel<KK, true, 1><<<grid, CONV_BLOCK, 0, ctx->stream>>>(ptrs, n, chunk_cols, partial, slots);
    else conv_gram_kernel<KK, false, NG><<<grid, CONV_BLOCK, 0, ctx->stream>>>(ptrs, n, chunk_cols, partial, slots);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

template <int NB, bool SAME>
static int launch_conv_gramx(gpfq_ctx *ctx, ConvPtrs ptrs, int64_t n, int kk, int n_ch, int n_chunks, int64_t chunk_cols,
                             double *partial, int slots) {
    constexpr size_t smem = gramx::smem_bytes<NB, SAME>();
    CUDA_TRY(ctx, cudaFuncSetAttribute(conv_gramx_kernel<NB, SAME>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    conv_gramx_kernel<NB, SAME><<<dim3((unsigned)n_chunks, (unsigned)n_ch), gramx::Cfg<NB>::NT, smem, ctx->stream>>>(
        ptrs, n, kk, chunk_cols, partial, slots);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

// kh * kw with a kernel of its own (conv_gram_kernel<KK> and friends, conv_sweep_kernel<KK>)
bool conv_specialised_kk(int kk) { return kk == 1 || kk == 2 || kk == 3 || kk == 4 || kk == 6 || kk == 9; }

// kh * kw with batched Gram and walk kernels: the specialised sizes above, every other size through conv_gramx_kernel /
// conv_walkx_kernel.  Larger kernels run one Dense problem per channel.
int conv_supported_kk(int kk) { return kk >= 1 && kk <= gramx::MAX_KK; }

// Column chunks per channel: grid = n_chunks x n_ch CTAs.  TMA kernel (kk == 9, vectorisable): one CTA per SM, whole
// waves of sm_count CTAs, chunks a multiple of the 512-column stage; the other kernels: two CTAs per SM.
// conv_gramx_kernel: chunks a multiple of its widest stage (256 columns); from 8 block rows (kk > 56) a column costs
// 72 DMMAs or more, so 1024-column chunks are already long enough.
int conv_pick_chunks(gpfq_ctx *ctx, int64_t n, int n_ch, int64_t *chunk_cols, int kk, bool vec_ok, int64_t part_rows) {
    const bool tma = (kk == 9 && vec_ok && (ctx->conv_variant == 0 || ctx->conv_variant == 3));
    const bool gx = !conv_specialised_kk(kk);
    const int64_t per_wave = tma ? ctx->sm_count : 2LL * ctx->sm_count;
    const int64_t min_cols = tma ? 32768 : (gx && kk > 56) ? 1024 : 4096, align = tma ? tma9::COLS : gx ? 256 : 128;
    int64_t waves = ((int64_t)n * n_ch) / (per_wave * min_cols);
    waves = waves < 1 ? 1 : (waves > 4 ? 4 : waves);
    int64_t want = (waves * per_wave) / n_ch;
    const int64_t max_chunks = ceil_div64(n, min_cols) > 0 ? ceil_div64(n, min_cols) : 1;
    if (want > max_chunks) want = max_chunks;
    if (gx) {
        // The partial workspace is part_rows (channels, times image chunks where those add slots; 0: n_ch) x n_chunks slots of
        // 2 kk^2 doubles, 256 KB at kk = 128.  Keep it within CONV_PART_LIMIT: fewer, longer column chunks when many channels
        // meet a large kernel (at least one chunk).
        const int64_t per_slot = (part_rows > 0 ? part_rows : n_ch) * 2 * kk * kk * (int64_t)sizeof(double);
        const int64_t cap = CONV_PART_LIMIT / per_slot;
        if (want > cap) want = cap;
    }
    if (want < 1) want = 1;
    int64_t cols = ceil_div64(n, want);
    cols = ceil_div64(cols, align) * align;
    *chunk_cols = cols;
    return (int)ceil_div64(n, cols);
}

// Gram partials of n_ch channels whose patch pointers (device) are in d_ptrs.
// `slots` = partial slots per channel (>= n_chunks; image-chunked callers interleave several launches), this launch
// fills slots [0, n_chunks) relative to `partial`.
int conv_gram_stage(gpfq_ctx *ctx, int kk, ConvPtrs d_ptrs, bool same, int64_t n, int n_ch, int n_chunks,
                    int64_t chunk_cols, double *partial, bool vec_ok, int slots) {
    switch (kk) {
        case 1: return launch_conv_gram<1>(ctx, d_ptrs, same, n, n_ch, n_chunks, chunk_cols, partial, vec_ok, slots);
        case 2: return launch_conv_gram<2>(ctx, d_ptrs, same, n, n_ch, n_chunks, chunk_cols, partial, vec_ok, slots);
        case 3: return launch_conv_gram<3>(ctx, d_ptrs, same, n, n_ch, n_chunks, chunk_cols, partial, vec_ok, slots);
        case 4: return launch_conv_gram<4>(ctx, d_ptrs, same, n, n_ch, n_chunks, chunk_cols, partial, vec_ok, slots);
        case 6: return launch_conv_gram<6>(ctx, d_ptrs, same, n, n_ch, n_chunks, chunk_cols, partial, vec_ok, slots);
        case 9: return launch_conv_gram<9>(ctx, d_ptrs, same, n, n_ch, n_chunks, chunk_cols, partial, vec_ok, slots);
    }
    if (!conv_supported_kk(kk)) return gpfq_fail(ctx, GPFQ_ERR_UNSUPPORTED, "conv kernel size kk=%d has no Gram kernel", kk);
#define GRAMX_CASE(NBV)                                                                                          \
    case NBV:                                                                                                    \
        return same ? launch_conv_gramx<NBV, true>(ctx, d_ptrs, n, kk, n_ch, n_chunks, chunk_cols, partial, slots) \
                    : launch_conv_gramx<NBV, false>(ctx, d_ptrs, n, kk, n_ch, n_chunks, chunk_cols, partial, slots);
    switch ((kk + 7) / 8) {
        GRAMX_CASE(1) GRAMX_CASE(2) GRAMX_CASE(3) GRAMX_CASE(4) GRAMX_CASE(5) GRAMX_CASE(6) GRAMX_CASE(7) GRAMX_CASE(8)
        GRAMX_CASE(9) GRAMX_CASE(10) GRAMX_CASE(11) GRAMX_CASE(12) GRAMX_CASE(13) GRAMX_CASE(14) GRAMX_CASE(15) GRAMX_CASE(16)
    }
#undef GRAMX_CASE
    return gpfq_fail(ctx, GPFQ_ERR_UNSUPPORTED, "conv kernel size kk=%d has no Gram kernel", kk);
}

int conv_finalize_stage(gpfq_ctx *ctx, const double *partial, int n_ch, int n_chunks, int kk, bool same,
                        double *gram) {
    conv_finalize_kernel<<<(unsigned)n_ch, 192, 0, ctx->stream>>>(partial, n_chunks, kk, same ? 1 : 0, gram);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

// W / Q: (kk, C / groups, F); channels c0 .. c0+n_ch-1 walk the F / groups filters of their group (groups = 1: all F).
int conv_sweep_stage(gpfq_ctx *ctx, int kk, const double *gram, const float *W, double *Q, int64_t C,
                     int64_t F, int64_t c0, int n_ch, const double *d_alph, const int *d_koff, const int *d_flags,
                     int n_alph, int64_t groups) {
    const int64_t Cg = C / groups, Fg = F / groups;
    const bool grouped = groups > 1;
    dim3 grid((unsigned)ceil_div64(Fg, 128), (unsigned)n_ch, (unsigned)n_alph);
    const int64_t CF = Cg * F, qs = (int64_t)kk * CF;
#define SWEEP_CASE(KKV)                                                                                                 \
    case KKV:                                                                                                           \
        if (grouped)                                                                                                    \
            conv_sweep_kernel<KKV, true><<<grid, 128, 0, ctx->stream>>>(gram, W, Q, CF, F, c0, d_alph, d_koff, d_flags, qs, Cg, Fg); \
        else                                                                                                            \
            conv_sweep_kernel<KKV, false><<<grid, 128, 0, ctx->stream>>>(gram, W, Q, CF, F, c0, d_alph, d_koff, d_flags, qs, Cg, Fg); \
        break;
    switch (kk) {
        SWEEP_CASE(1) SWEEP_CASE(2) SWEEP_CASE(3) SWEEP_CASE(4) SWEEP_CASE(6) SWEEP_CASE(9)
        default: {
            if (!conv_supported_kk(kk)) return gpfq_fail(ctx, GPFQ_ERR_UNSUPPORTED, "conv kernel size kk=%d has no walk kernel", kk);
            using namespace walkx;
            const int warps = Fg < MAXW ? (int)Fg : MAXW;
            const size_t smem = ((size_t)kk * (kk + 1) + kk + GPFQ_MAX_K) * sizeof(double);
            dim3 wgrid((unsigned)ceil_div64(Fg, warps), (unsigned)n_ch, (unsigned)n_alph);
            if (grouped) {
                CUDA_TRY(ctx, cudaFuncSetAttribute(conv_walkx_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                conv_walkx_kernel<true><<<wgrid, warps * 32, smem, ctx->stream>>>(gram, kk, W, Q, CF, F, c0, d_alph, d_koff, d_flags,
                                                                                 qs, Cg, Fg);
            } else {
                CUDA_TRY(ctx, cudaFuncSetAttribute(conv_walkx_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                conv_walkx_kernel<false><<<wgrid, warps * 32, smem, ctx->stream>>>(gram, kk, W, Q, CF, F, c0, d_alph, d_koff, d_flags,
                                                                                  qs, Cg, Fg);
            }
        }
    }
#undef SWEEP_CASE
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

int im2col_stage(gpfq_ctx *ctx, const float *act, int64_t n_img, int H, int Wd, int64_t C, int64_t c_first,
                 int n_ch, int kh, int kw, int sh, int sw, int rh, int rw, int pt, int pl, int Ho, int Wo,
                 float *out, int64_t ch_stride) {
    const int64_t n = n_img * Ho * Wo;
    int bx = (int)(ceil_div64(n, 256) < 2048 ? ceil_div64(n, 256) : 2048);
    dim3 grid((unsigned)bx, (unsigned)n_ch, (unsigned)(kh * kw));
    im2col_kernel<<<grid, 256, 0, ctx->stream>>>(act, n_img, H, Wd, C, c_first, kh, kw, sh, sw, rh, rw, pt, pl,
                                                 Ho, Wo, out, ch_stride);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

// Fused NHWC path: is this geometry eligible, and with which plane pitch / band height?
int nhwc9_plan(int kh, int kw, int sh, int sw, int rh, int rw, int Ho, int Wo, int *P_out, int *BR_out) {
    if (kh != 3 || kw != 3 || sh != 1 || sw != 1 || rh != 1 || rw != 1) return 0;
    int P = (Wo + 3) / 4 * 4 + 2;
    while (P % 32 < 8 || P % 32 > 12) ++P;  // three plane rows on disjoint banks for the 3 x 6 window reads
    int BR = nhwc9::MAX_PLANE / P - 2;
    if (BR > Ho) BR = Ho;
    if (BR < 4 && BR < Ho) return 0;         // very wide images: the halo would dominate
    *P_out = P;
    *BR_out = BR;
    return 1;
}

// Partial Grams of channels [c_first, c_first + n_ch) over images [img0, img0 + n_img): fills slots
// [0, n_slots) (relative to `partial`) of every channel; `slots` = total slots per channel.
int conv_gram9_nhwc_stage(gpfq_ctx *ctx, const float *act, const float *actq, bool same, int64_t img0, int64_t n_img,
                          int H, int Wd, int64_t C, int64_t c_first, int n_ch, int Ho, int Wo, int pt, int pl, int P,
                          int BR, int n_slots, double *partial, int slots) {
    using namespace nhwc9;
    Nhwc9Geom gm;
    gm.H = H; gm.W = Wd; gm.Ho = Ho; gm.Wo = Wo; gm.pt = pt; gm.pl = pl; gm.P = P; gm.BR = BR;
    gm.C = C; gm.c_first = c_first; gm.n_ch = n_ch; gm.img0 = img0; gm.n_img = n_img;
    gm.imgs_per_cta = (int)ceil_div64(n_img, n_slots);
    const size_t plane_bytes = (size_t)(BR + 2) * P * sizeof(float) * CG;
    size_t smem = plane_bytes * (same ? 1 : 2);
    const size_t red_bytes = (size_t)CG * 2 * 81 * sizeof(double);
    if (smem < red_bytes) smem = red_bytes;
    dim3 grid((unsigned)ceil_div64(n_img, gm.imgs_per_cta), (unsigned)ceil_div64(n_ch, CG));
    if (same) {
        CUDA_TRY(ctx, cudaFuncSetAttribute(conv_gram9_nhwc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        conv_gram9_nhwc_kernel<true><<<grid, THREADS, smem, ctx->stream>>>(act, act, gm, partial, slots);
    } else {
        CUDA_TRY(ctx, cudaFuncSetAttribute(conv_gram9_nhwc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        conv_gram9_nhwc_kernel<false><<<grid, THREADS, smem, ctx->stream>>>(act, actq, gm, partial, slots);
    }
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

int msq_stage(gpfq_ctx *ctx, const void *W, int is_f64, int64_t n, const double *d_alph, int K, int equispaced, double *Q) {
    int bx = (int)(ceil_div64(n, 256) < 1184 ? ceil_div64(n, 256) : 1184);
    if (bx < 1) bx = 1;
    if (is_f64) msq_kernel<double><<<bx, 256, 0, ctx->stream>>>((const double *)W, n, d_alph, K, equispaced, Q);
    else msq_kernel<float><<<bx, 256, 0, ctx->stream>>>((const float *)W, n, d_alph, K, equispaced, Q);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}
