// slgemm_i8.cu -- rectangular "NT" contraction  C (+)= sum_seg alpha_seg * A_seg B_seg^T  with fp64-class accuracy on the 5th-generation
// tensor cores: int8 digit slices (Ozaki scheme, as gram_i8.cu) + tcgen05.mma.kind::i8 into TMEM, operands by TMA.
//
// Used by the carried-residual (low-rank) form of the Dense sweep (dense_gram.cu): per range of directions
//     U += W_r X_r - Q_r X~_r          (nj x m, K = the range's directions;  quantized_network.py:119 for a whole range)
//     D_r = U X~_r^T                   (nj x R, K = the m samples;           the residual dots of :86/:89 for a whole range)
// which north_star (b) wants "folded in as small GEMMs" -- here they run on tcgen05 instead of the fp64 DMMA pipe.
//
// Operands are stored as S signed base-256 digit slices per value with one exponent per ROW (row = output row or column,
// K contiguous):   x[r][k] * 2^-e_r = sum_{s=1..S} b_s[r][k] 2^(2 - 8 s)   (b in [-128, 127]; rounding at 2^-(8S-2) of 2^e_r).
// Every slice pair with s_a + s_b = d accumulates EXACTLY into the s32 TMEM accumulator of its d (<= 5 pairs x K <= 26112);
// ALL d of a product are open at once -- a 128 x 64 output tile leaves room for eight 64-column accumulators in the 512 TMEM
// columns -- so a K block of every A slice and every B slice is fetched ONCE per stage and feeds all 15-19 pair MMAs, and the fp64 combination  sum_d S_d alpha 2^(4 - 8 d + eA_i + eB_j)  happens once per product,
// in registers (one output row per epilogue thread), in a fixed order: bit-reproducible.  C is touched once per tile.
//
// Kernel anatomy (one CTA per 128 x 64 output tile, one CTA per SM):
//   warp 0    producer: per stage one bulk copy (cp.async.bulk, UBLKCP) of 128 rows x 64 B per A slice and of 64 rows x 64 B per
//             B slice -- the slice tensors are stored K-block tiled and already 64B-swizzled (slgemm_i8.cuh), so a tile IS its
//             shared-memory image -- into a 3-stage mbarrier ring
//   warp 1    TMEM allocator + single-thread MMA issuer: 2 x tcgen05.mma.cta_group::1.kind::i8 (M128 N64 K32) per slice pair
//             and K block
//   warps 2-5 epilogue: per product tcgen05.ld of every accumulator -> fp64 fma into 64 register sums per thread; after the
//             last product the row is scaled by 2^eB and written (or added) to C
#include <algorithm>

#include "slgemm_i8.cuh"

namespace slg {
constexpr int TM = 128, TN = 64, BK = 64;    // output tile, K bytes per stage
constexpr int STAGES = 3;
constexpr int S = 5;                         // digit slices per sliced value
constexpr int P_BITS = 8 * S - 2;
constexpr int A_SLICE = TM * BK, B_SLICE = TN * BK;
constexpr int STAGE_BYTES = S * (A_SLICE + B_SLICE);
constexpr int THREADS = 192;
constexpr int MAX_PHASES = 8;                // 512 TMEM columns / TN
constexpr int OUT_PITCH = TN + 1;            // doubles: the epilogue's transposing tile (conflict-free row writes)
constexpr int KB_MAX = 408;                  // K blocks per call: 5 pairs * 408 * 64 * 128^2 < 2^31
constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */ + TN * sizeof(double);
}  // namespace slg

struct SlSeg {
    int SA, SB, D;          // slices of A / B; slice pairs with s_a + s_b <= D
    int a_row0, b_row0;     // first row of this product inside the A / B slice tensors (the tile offset is added)
    int k0, k0b, kblocks;   // first K byte of A / of B and K blocks of 64 bytes
    double alpha;
    const double *row_mul;  // per-row multiplier of alpha, indexed like the slice rows (nullptr: none; ROWMUL kernels only)
    const int32_t *eA;      // row exponents, indexed like the slice rows (nullptr: eA_const)
    int eA_const;
    const int8_t *A, *B;    // slice tensors (K-block tiled, pre-swizzled: sl_offset)
    int64_t rowsA, rowsB;   // their padded row counts
};

struct SlArgs {
    SlSeg seg[2];
    int nseg, tiles_n;
    const int32_t *eB;      // exponents of the B rows (= output columns), shared by the segments (nullptr: eB_const)
    int eB_const, b_row0;
    double *C;
    int64_t ldc;
    int M, N;               // valid rows / columns of C
    int accumulate, vec2;
    int batch_rows_a, batch_rows_b, batch_k0a, batch_k0b;   // blockIdx.y batches: A rows / B rows (and their exponents) / first K bytes advance
    int64_t batch_c;        // ... and C by batch_c elements
    int lower_only;         // skip tiles entirely above the diagonal (block-diagonal Gram tiles)
    int ktri;               // B strictly lower triangular in (row, K): column tile tj stops after K block tj
};

// K-major operand tile with 64-byte rows, SWIZZLE_64B: 8-row atoms of 512 B (SBO), LBO unused (1), descriptor version 1
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)4 << 61);
}

// Every slice pair (k, l), k + l = d <= D, of one K block, fully unrolled: descriptors are base + constant (the start address
// field holds bytes >> 4 and a stage never crosses the 14-bit field), the accumulator of d sits at TMEM column (d - 2) TN.
template <int SA, int SB, int D>
__device__ __forceinline__ void sl_issue_kblock(uint32_t tmem_base, uint64_t da, uint64_t db, uint32_t idesc, bool first) {
    using namespace slg;
#pragma unroll
    for (int d = 2; d <= D; ++d) {
        constexpr int dummy = 0;
        (void)dummy;
        const int k_lo = (d - SB) > 1 ? (d - SB) : 1, k_hi = SA < (d - 1) ? SA : (d - 1);
#pragma unroll
        for (int k = k_lo; k <= k_hi; ++k)
#pragma unroll
            for (int ks = 0; ks < BK / 32; ++ks)
                i8g::umma_i8(tmem_base + (uint32_t)((d - 2) * TN), da + (uint64_t)(((k - 1) * A_SLICE + ks * 32) >> 4),
                             db + (uint64_t)(((d - k - 1) * B_SLICE + ks * 32) >> 4), idesc,
                             (k == k_lo && ks == 0) ? (first ? 0u : 1u) : 1u);
    }
}

// ROWMUL: a segment with row_mul scales its rows by alpha * row_mul[row] (the per-neuron level step of the residual form's Q part
// with per-channel alphabets); the kernel without it is the one every other product uses.
template <bool ROWMUL>
__global__ void __launch_bounds__(slg::THREADS, 1)
slgemm_i8_kernel(const SlArgs args) {
    using namespace i8g;
    using namespace slg;
    extern __shared__ unsigned char sl_smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>(((uintptr_t)sl_smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + (size_t)STAGES * STAGE_BYTES);
    uint64_t *empty = full + STAGES;
    uint64_t *seg_full = empty + STAGES;    // the accumulators of the current segment are complete
    uint64_t *seg_empty = seg_full + 1;     // ... have been drained by the epilogue
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(seg_empty + 1);
    double *colscale = reinterpret_cast<double *>(smem + (size_t)STAGES * STAGE_BYTES + 256);   // [TN]: 2^eB of the tile's columns

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ti = blockIdx.x / args.tiles_n, tj = blockIdx.x % args.tiles_n;
    if (args.lower_only && tj * TN > ti * TM + TM - 1) return;
    const int brow_a = (int)blockIdx.y * args.batch_rows_a, brow_b = (int)blockIdx.y * args.batch_rows_b;   // batch offsets of the rows
    const int bk0a = (int)blockIdx.y * args.batch_k0a, bk0b = (int)blockIdx.y * args.batch_k0b;
    const int kcap = args.ktri ? tj + 1 : (1 << 30);

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(seg_full, 1);
        mbar_init(seg_empty, 4);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    if (warp >= 2 && threadIdx.x - 64 < TN) {
        const int c = threadIdx.x - 64;     // one column of the tile
        colscale[c] = ldexp(1.0, args.eB ? args.eB[args.b_row0 + brow_b + tj * TN + c] : args.eB_const);
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ---- producer: every slice of the A rows and of the B rows of one K block per stage, one bulk copy per slice
        if (lane == 0) {
            int iter = 0;
            for (int sg = 0; sg < args.nseg; ++sg) {
                const SlSeg &g = args.seg[sg];
                const uint32_t bytes = (uint32_t)(g.SA * A_SLICE + g.SB * B_SLICE);
                // slice s of K block kb of rows row0.. is ONE contiguous run of 128 (64) rows x 64 bytes
                const int8_t *pa = g.A + ((int64_t)((g.k0 + bk0a) / BK) * g.SA * g.rowsA + g.a_row0 + brow_a + ti * TM) * BK;
                const int8_t *pb = g.B + ((int64_t)((g.k0b + bk0b) / BK) * g.SB * g.rowsB + g.b_row0 + brow_b + tj * TN) * BK;
                const int kblocks = min(g.kblocks, kcap);
                const int64_t a_slice = g.rowsA * BK, b_slice = g.rowsB * BK;
                for (int kb = 0; kb < kblocks; ++kb, ++iter) {
                    const int s = iter % STAGES;
                    if (iter >= STAGES) mbar_wait(&empty[s], ((iter / STAGES) - 1) & 1);
                    unsigned char *a = smem + (size_t)s * STAGE_BYTES, *b = a + S * A_SLICE;
                    mbar_expect_tx(&full[s], bytes);
                    for (int sl = 0; sl < g.SA; ++sl) bulk_load(a + sl * A_SLICE, pa + ((int64_t)kb * g.SA + sl) * a_slice, A_SLICE, &full[s]);
                    for (int sl = 0; sl < g.SB; ++sl) bulk_load(b + sl * B_SLICE, pb + ((int64_t)kb * g.SB + sl) * b_slice, B_SLICE, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issuer: per K block every slice pair (k, l), k + l = d, into the accumulator of its d.  The whole warp runs the
        // (uniform) loops and waits; one elected lane issues.
        {
            // instruction descriptor: D = s32, A = B = signed 8-bit, both K-major, N = 64, M = 128
            const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
            int iter = 0;
            for (int sg = 0; sg < args.nseg; ++sg) {
                const SlSeg &g = args.seg[sg];
                if (sg > 0) {   // the epilogue must have drained the previous segment's accumulators
                    mbar_wait(seg_empty, (sg - 1) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                }
                const int mode = (g.SA == 5 && g.SB == 5 && g.D == 6) ? 1 : (g.SA == 5 && g.SB == 5 && g.D == 7) ? 2
                                 : (g.SA == 1 && g.SB == 5 && g.D == 6) ? 3 : 0;
                const int kblocks = min(g.kblocks, kcap);
                for (int kb = 0; kb < kblocks; ++kb, ++iter) {
                    const int s = iter % STAGES;
                    mbar_wait(&full[s], (iter / STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    const uint32_t a = smem_u32(smem + (size_t)s * STAGE_BYTES), b = a + S * A_SLICE;
                    const uint64_t da = umma_desc_sw64(a), db = umma_desc_sw64(b);
                    if (elect_one()) {
                        // the usual slice-pair sets as straight-line code (at 32 tensor-core cycles per M128 N64 K32 instruction the
                        // loop overhead of the generic form would be the bottleneck)
                        if (mode == 1) sl_issue_kblock<5, 5, 6>(tmem_base, da, db, idesc, kb == 0);
                        else if (mode == 2) sl_issue_kblock<5, 5, 7>(tmem_base, da, db, idesc, kb == 0);
                        else if (mode == 3) sl_issue_kblock<1, 5, 6>(tmem_base, da, db, idesc, kb == 0);
                        else
                            for (int d = 2; d <= g.D; ++d) {
                                const uint32_t tmem_d = tmem_base + (uint32_t)((d - 2) * TN);
                                const int k_lo = max(1, d - g.SB), k_hi = min(g.SA, d - 1);
                                for (int k = k_lo; k <= k_hi; ++k) {
                                    const uint32_t ak = a + (k - 1) * A_SLICE, bl = b + (d - k - 1) * B_SLICE;
#pragma unroll
                                    for (int ks = 0; ks < BK / 32; ++ks)
                                        umma_i8(tmem_d, umma_desc_sw64(ak + ks * 32), umma_desc_sw64(bl + ks * 32), idesc,
                                                (kb | (k - k_lo) | ks) ? 1u : 0u);
                                }
                            }
                        umma_commit(&empty[s]);  // the stage may be refilled once these MMAs have read it
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(seg_full);
                __syncwarp();
            }
        }
    } else {
        // ---- epilogue: TMEM lanes 32 * (warp % 4) .. + 31 are this warp's tile rows; one thread = one row, whose 64 fp64
        // sums stay in registers over all segments and phases:  sum_seg sum_d  S_d * alpha 2^(4 - 8 d + eA_row),  then 2^eB_col.
        const int quad = warp & 3;
        const int row_t = quad * 32 + lane;
        const uint32_t lane_field = (uint32_t)(quad * 32) << 16;
        double acc[TN];
#pragma unroll
        for (int i = 0; i < TN; ++i) acc[i] = 0.0;
        for (int sg = 0; sg < args.nseg; ++sg) {
            const SlSeg &g = args.seg[sg];
            const int ea = g.eA ? g.eA[g.a_row0 + brow_a + ti * TM + row_t] : g.eA_const;
            const double alpha = (ROWMUL && g.row_mul) ? g.alpha * g.row_mul[g.a_row0 + brow_a + ti * TM + row_t] : g.alpha;
            mbar_wait(seg_full, sg & 1);
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
#pragma unroll 1
            for (int d = 2; d <= g.D; ++d) {
                const double rs = ldexp(alpha, 4 - 8 * d + ea);
#pragma unroll
                for (int hf = 0; hf < TN / 32; ++hf) {
                    uint32_t v[32];
                    tmem_ld32(tmem_base + lane_field + (uint32_t)((d - 2) * TN + hf * 32), v);
#pragma unroll
                    for (int i = 0; i < 32; ++i) acc[hf * 32 + i] = fma((double)(int)v[i], rs, acc[hf * 32 + i]);
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(seg_empty);
        }
        // ---- the finished tile.  A thread holds one ROW; written straight out that is 32 scattered 16-byte accesses per
        // instruction (measured: 300 us per call on the read-modify-write of U).  The operand ring is idle by now (every MMA
        // of the CTA has completed), so each warp transposes its 32 rows through it and touches C in whole 256-byte runs.
        double *tr = reinterpret_cast<double *>(smem) + (size_t)quad * 32 * OUT_PITCH;
#pragma unroll
        for (int i = 0; i < TN; ++i) tr[lane * OUT_PITCH + i] = acc[i] * colscale[i];
        __syncwarp();
        const int64_t row0 = (int64_t)ti * TM + quad * 32, col0 = (int64_t)tj * TN;
        double *Cb = args.C + (int64_t)blockIdx.y * args.batch_c;
        // all loads of the read-modify-write first (64 independent requests in flight per lane), then the stores
        double old[32][TN / 32];
#pragma unroll
        for (int r = 0; r < 32; ++r)
#pragma unroll
            for (int hf = 0; hf < TN / 32; ++hf) {
                const int c = hf * 32 + lane;
                old[r][hf] = (args.accumulate && row0 + r < args.M && col0 + c < args.N) ? Cb[(row0 + r) * args.ldc + col0 + c] : 0.0;
            }
#pragma unroll
        for (int r = 0; r < 32; ++r)
#pragma unroll
            for (int hf = 0; hf < TN / 32; ++hf) {
                const int c = hf * 32 + lane;
                if (row0 + r < args.M && col0 + c < args.N) Cb[(row0 + r) * args.ldc + col0 + c] = old[r][hf] + tr[r * OUT_PITCH + c];
            }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512));
    }
}

// ---- slicing kernels ---------------------------------------------------------------------------------------------
// Row-wise: one CTA per (padded) row of a row-major matrix (fp32 or fp64 values): exponent of the row maximum, then the S
// digit slices of every value, 16 consecutive K positions per thread and step.  Rows >= rows and columns >= cols are zeros.
template <typename T>
__global__ void __launch_bounds__(256) sl_rowsplit_kernel(const T *__restrict__ X, int64_t ldx, int64_t rows, int64_t cols,
                                                          int32_t *__restrict__ e, int8_t *__restrict__ slices, int64_t rowsP,
                                                          int64_t colsP, int64_t row0) {
    using namespace slg;
    __shared__ double red[8];
    __shared__ int ex_s;
    const int64_t r = blockIdx.x;
    const T *row = X + r * ldx;
    double mx = 0.0;
    if (r < rows)
        for (int64_t i = threadIdx.x; i < cols; i += 256) mx = fmax(mx, fabs((double)row[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) mx = fmax(mx, red[w]);
        int ex = 0;
        if (mx > 0.0 && isfinite(mx)) frexp(mx, &ex);   // mx = f 2^ex, f in [0.5, 1)  =>  |x| < 2^ex
        e[row0 + r] = ex;
        ex_s = ex;
    }
    __syncthreads();
    const int ex = ex_s;
    for (int64_t i0 = (int64_t)threadIdx.x * 16; i0 < colsP; i0 += 256 * 16) {
        uint32_t packed[S][4];
#pragma unroll
        for (int k = 0; k < S; ++k) packed[k][0] = packed[k][1] = packed[k][2] = packed[k][3] = 0u;
        if (r < rows && i0 < cols) {
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const double x = (i0 + c < cols) ? (double)row[i0 + c] : 0.0;
                long long v = __double2ll_rn(ldexp(x, P_BITS - ex));   // |v| <= 2^38
#pragma unroll
                for (int k = S - 1; k >= 0; --k) {
                    const int dg = (int)((v + 128) & 255) - 128;       // balanced digit in [-128, 127]
                    v = (v - dg) >> 8;
                    packed[k][c >> 2] |= ((uint32_t)(dg & 0xff)) << (8 * (c & 3));
                }
            }
        }
#pragma unroll
        for (int k = 0; k < S; ++k)
            *reinterpret_cast<uint4 *>(slices + sl_offset(i0, k, row0 + r, rowsP, S)) =
                make_uint4(packed[k][0], packed[k][1], packed[k][2], packed[k][3]);
    }
}

// The same for short rows (colsP <= 32 * 16 * CH): one WARP per row, the row held in registers -- one pass over the data.
// (The residuals U are re-sliced after every range of the sweep: 2048 rows of 1504 doubles.)
template <typename T, int CH>
__global__ void __launch_bounds__(256) sl_rowsplit_warp_kernel(const T *__restrict__ X, int64_t ldx, int64_t rows, int64_t cols,
                                                               int32_t *__restrict__ e, int8_t *__restrict__ slices, int64_t rowsP,
                                                               int64_t colsP, int64_t row0, int64_t grid_rows) {
    using namespace slg;
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= grid_rows) return;
    const T *row = X + r * ldx;
    double v[CH][16];
    double mx = 0.0;
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
        const int64_t c0 = (int64_t)(ch * 32 + lane) * 16;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const double x = (r < rows && c0 + i < cols) ? (double)row[c0 + i] : 0.0;
            v[ch][i] = x;
            mx = fmax(mx, fabs(x));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    int ex = 0;
    if (mx > 0.0 && isfinite(mx)) frexp(mx, &ex);
    if (lane == 0) e[row0 + r] = ex;
    const double scale = ldexp(1.0, P_BITS - ex);
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
        const int64_t c0 = (int64_t)(ch * 32 + lane) * 16;
        if (c0 >= colsP) continue;
        uint32_t packed[S][4];
#pragma unroll
        for (int k = 0; k < S; ++k) packed[k][0] = packed[k][1] = packed[k][2] = packed[k][3] = 0u;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            long long q = __double2ll_rn(v[ch][c] * scale);
#pragma unroll
            for (int k = S - 1; k >= 0; --k) {
                const int dg = (int)((q + 128) & 255) - 128;
                q = (q - dg) >> 8;
                packed[k][c >> 2] |= ((uint32_t)(dg & 0xff)) << (8 * (c & 3));
            }
        }
#pragma unroll
        for (int k = 0; k < S; ++k)
            *reinterpret_cast<uint4 *>(slices + sl_offset(c0, k, row0 + r, rowsP, S)) =
                make_uint4(packed[k][0], packed[k][1], packed[k][2], packed[k][3]);
    }
}

// Column maxima of |X| (X: (N0, m) fp32): non-negative floats order like their bit patterns, so an integer atomicMax does it.
__global__ void __launch_bounds__(256) sl_colmax_kernel(const float *__restrict__ X, int64_t ldx, int64_t N0, int64_t m,
                                                        int *__restrict__ colmax, int rows_per_cta) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= m) return;
    const int64_t t0 = (int64_t)blockIdx.y * rows_per_cta, t1 = min(N0, t0 + rows_per_cta);
    float mx = 0.f;
    for (int64_t t = t0; t < t1; ++t) mx = fmaxf(mx, fabsf(X[t * ldx + i]));
    atomicMax(colmax + i, __float_as_int(mx));
}

__global__ void sl_exp_from_max_kernel(const int *__restrict__ colmax, int64_t n, int64_t nP, int32_t *__restrict__ e) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nP) return;
    int ex = 0;
    if (i < n) {
        const float mx = __int_as_float(colmax[i]);
        if (mx > 0.f && isfinite(mx)) frexpf(mx, &ex);
    }
    e[i] = ex;
}

// Transposed slicing: X (N0, m) fp32 -> slices (S, mP, N0P) of X^T (row = sample, K = direction), exponent per sample.
// Tile of 64 directions x 32 samples through shared memory; a thread then owns one sample and 16 consecutive directions.
__global__ void __launch_bounds__(128) sl_transsplit_kernel(const float *__restrict__ X, int64_t ldx, int64_t N0, int64_t m,
                                                            const int32_t *__restrict__ e, int8_t *__restrict__ slices, int64_t mP,
                                                            int64_t N0P) {
    using namespace slg;
    __shared__ float tile[64][33];
    const int64_t t0 = (int64_t)blockIdx.x * 64, i0 = (int64_t)blockIdx.y * 32;
    for (int idx = threadIdx.x; idx < 64 * 32; idx += 128) {
        const int tr = idx >> 5, ic = idx & 31;
        const int64_t t = t0 + tr, i = i0 + ic;
        tile[tr][ic] = (t < N0 && i < m) ? X[t * ldx + i] : 0.f;
    }
    __syncthreads();
    const int ic = threadIdx.x & 31, tg = threadIdx.x >> 5;   // sample, group of 16 directions
    const int64_t i = i0 + ic;
    if (i >= mP) return;
    const int ex = e[i];
    uint32_t packed[S][4];
#pragma unroll
    for (int k = 0; k < S; ++k) packed[k][0] = packed[k][1] = packed[k][2] = packed[k][3] = 0u;
#pragma unroll
    for (int c = 0; c < 16; ++c) {
        long long v = __double2ll_rn(ldexp((double)tile[tg * 16 + c][ic], P_BITS - ex));
#pragma unroll
        for (int k = S - 1; k >= 0; --k) {
            const int dg = (int)((v + 128) & 255) - 128;
            v = (v - dg) >> 8;
            packed[k][c >> 2] |= ((uint32_t)(dg & 0xff)) << (8 * (c & 3));
        }
    }
#pragma unroll
    for (int k = 0; k < S; ++k)
        *reinterpret_cast<uint4 *>(slices + sl_offset(t0 + tg * 16, k, i, mP, S)) =
            make_uint4(packed[k][0], packed[k][1], packed[k][2], packed[k][3]);
}

// ---- host side -------------------------------------------------------------------------------------------------
int sl_make_operand(gpfq_ctx *ctx, SlOperand *op, const int8_t *slices, int64_t rowsP, int64_t kbytes, int n_slices, const int32_t *e,
                    int e_const, bool is_b) {
    using namespace slg;
    if (kbytes % BK || rowsP % TM || ((uintptr_t)slices & 15))
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "slice tensors are padded to whole K blocks and 128-row tiles, 16-byte aligned");
    op->slices = slices;
    op->rowsP = rowsP;
    op->kbytes = kbytes;
    op->n_slices = n_slices;
    op->e = e;
    op->e_const = e_const;
    op->is_b = is_b;
    return GPFQ_OK;
}

// C[M x N] (ldc) = or += sum of the products.  M, N: valid extents; the slice tensors are zero-padded to tile multiples.
int slgemm_i8(gpfq_ctx *ctx, const SlProduct *prod, int nprod, double *C, int64_t ldc, int64_t M, int64_t N, bool accumulate,
              int nbatch, int64_t batch_rows, int64_t batch_c, bool lower_only) {
    SlBatch b;
    b.n = nbatch;
    b.a_rows = b.b_rows = batch_rows;
    b.c = batch_c;
    b.lower_only = lower_only;
    return slgemm_i8_ex(ctx, prod, nprod, C, ldc, M, N, accumulate, b);
}

int slgemm_i8_ex(gpfq_ctx *ctx, const SlProduct *prod, int nprod, double *C, int64_t ldc, int64_t M, int64_t N, bool accumulate,
                 const SlBatch &batch) {
    using namespace slg;
    const int nbatch = batch.n;
    if (nprod < 1 || nprod > 2) return gpfq_fail(ctx, GPFQ_ERR_ARG, "slgemm_i8: 1 or 2 products");
    SlArgs a = {};
    a.nseg = nprod;
    for (int s = 0; s < nprod; ++s) {
        const SlProduct &p = prod[s];
        const int64_t k0b = p.k0b < 0 ? p.k0 : p.k0b;
        if (p.K % BK || p.k0 % BK || k0b % BK || batch.a_k % BK || batch.b_k % BK || p.K / BK > KB_MAX || p.K < BK)
            return gpfq_fail(ctx, GPFQ_ERR_ARG, "slgemm_i8: K = %lld (offset %lld) must be multiples of 64, at most %d",
                             (long long)p.K, (long long)p.k0, KB_MAX * BK);
        if (p.A->is_b || !p.B->is_b || p.A->n_slices > S || p.B->n_slices > S)
            return gpfq_fail(ctx, GPFQ_ERR_ARG, "slgemm_i8: operand roles / slice counts");
        if (p.a_row0 + (nbatch - 1) * batch.a_rows + ceil_div64(M, TM) * TM > p.A->rowsP ||
            p.b_row0 + (nbatch - 1) * batch.b_rows + ceil_div64(N, TN) * TN > p.B->rowsP ||
            p.k0 + (nbatch - 1) * batch.a_k + p.K > p.A->kbytes || k0b + (nbatch - 1) * batch.b_k + p.K > p.B->kbytes)
            return gpfq_fail(ctx, GPFQ_ERR_ARG, "slgemm_i8: operand slices are not padded to the tile grid");
        if (s > 0 && (p.B->e != prod[0].B->e || p.B->e_const != prod[0].B->e_const || p.b_row0 != prod[0].b_row0))
            return gpfq_fail(ctx, GPFQ_ERR_ARG, "slgemm_i8: the products of one call must share the exponents of their B rows");
        SlSeg &g = a.seg[s];
        g.SA = p.A->n_slices;
        g.SB = p.B->n_slices;
        g.D = std::min(std::min(p.D, g.SA + g.SB), MAX_PHASES + 1);
        g.a_row0 = (int)p.a_row0;
        g.b_row0 = (int)p.b_row0;
        g.k0 = (int)p.k0;
        g.k0b = (int)k0b;
        g.kblocks = (int)(p.K / BK);
        g.alpha = p.alpha;
        g.row_mul = p.row_mul;
        g.eA = p.A->e;
        g.eA_const = p.A->e_const;
        g.A = p.A->slices;
        g.B = p.B->slices;
        g.rowsA = p.A->rowsP;
        g.rowsB = p.B->rowsP;
    }
    a.eB = prod[0].B->e;
    a.eB_const = prod[0].B->e_const;
    a.b_row0 = (int)prod[0].b_row0;
    a.tiles_n = (int)ceil_div64(N, TN);
    a.C = C;
    a.ldc = ldc;
    a.M = (int)M;
    a.N = (int)N;
    a.accumulate = accumulate ? 1 : 0;
    a.vec2 = (ldc % 2 == 0) && ((uintptr_t)C % 16 == 0);
    a.batch_rows_a = (int)batch.a_rows;
    a.batch_rows_b = (int)batch.b_rows;
    a.batch_k0a = (int)batch.a_k;
    a.batch_k0b = (int)batch.b_k;
    a.batch_c = batch.c;
    a.lower_only = batch.lower_only ? 1 : 0;
    a.ktri = batch.ktri ? 1 : 0;
    if (nbatch < 1 || nbatch > 65535) return gpfq_fail(ctx, GPFQ_ERR_ARG, "slgemm_i8: 1..65535 batches");
    const bool rowmul = a.seg[0].row_mul || (nprod > 1 && a.seg[1].row_mul);
    auto k = rowmul ? slgemm_i8_kernel<true> : slgemm_i8_kernel<false>;
    CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    const dim3 grid((unsigned)(ceil_div64(M, TM) * a.tiles_n), (unsigned)nbatch);
    k<<<grid, THREADS, SMEM, ctx->stream>>>(a);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

// slices of a row-major fp64 / fp32 matrix (rows x cols, row = output row, K = cols); e: rowsP exponents
template <typename T>
int sl_rowsplit(gpfq_ctx *ctx, const T *X, int64_t ldx, int64_t rows, int64_t cols, int32_t *e, int8_t *slices, int64_t rowsP,
                int64_t colsP, int64_t row0, int64_t grid_rows) {
    const unsigned wgrid = (unsigned)ceil_div64(grid_rows, 8);
    if (colsP <= 32 * 16 * 2)
        sl_rowsplit_warp_kernel<T, 2><<<wgrid, 256, 0, ctx->stream>>>(X, ldx, rows, cols, e, slices, rowsP, colsP, row0, grid_rows);
    else if (colsP <= 32 * 16 * 4)
        sl_rowsplit_warp_kernel<T, 4><<<wgrid, 256, 0, ctx->stream>>>(X, ldx, rows, cols, e, slices, rowsP, colsP, row0, grid_rows);
    else
        sl_rowsplit_kernel<T><<<(unsigned)grid_rows, 256, 0, ctx->stream>>>(X, ldx, rows, cols, e, slices, rowsP, colsP, row0);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}
template int sl_rowsplit<double>(gpfq_ctx *, const double *, int64_t, int64_t, int64_t, int32_t *, int8_t *, int64_t, int64_t, int64_t, int64_t);
template int sl_rowsplit<float>(gpfq_ctx *, const float *, int64_t, int64_t, int64_t, int32_t *, int8_t *, int64_t, int64_t, int64_t, int64_t);

// slices of X^T (and, unless Xq is null, of Xq^T with the SAME per-sample exponents: max over both matrices) for X, Xq
// (N0, m) fp32: (S, mP, N0P) each; scratch: mP ints
int sl_transsplit(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m, int32_t *e, int *scratch,
                  int8_t *slices, int8_t *slices_q, int64_t mP, int64_t N0P) {
    cudaStream_t st = ctx->stream;
    CUDA_TRY(ctx, cudaMemsetAsync(scratch, 0, (size_t)mP * sizeof(int), st));
    const int rows_per_cta = 256;
    dim3 g1((unsigned)ceil_div64(m, 256), (unsigned)ceil_div64(N0, rows_per_cta));
    sl_colmax_kernel<<<g1, 256, 0, st>>>(X, ldx, N0, m, scratch, rows_per_cta);
    KERNEL_CHECK(ctx);
    if (Xq) {
        sl_colmax_kernel<<<g1, 256, 0, st>>>(Xq, ldx, N0, m, scratch, rows_per_cta);
        KERNEL_CHECK(ctx);
    }
    sl_exp_from_max_kernel<<<(unsigned)ceil_div64(mP, 256), 256, 0, st>>>(scratch, m, mP, e);
    KERNEL_CHECK(ctx);
    dim3 g2((unsigned)(N0P / 64), (unsigned)(mP / 32));
    sl_transsplit_kernel<<<g2, 128, 0, st>>>(X, ldx, N0, m, e, slices, mP, N0P);
    KERNEL_CHECK(ctx);
    if (Xq) {
        sl_transsplit_kernel<<<g2, 128, 0, st>>>(Xq, ldx, N0, m, e, slices_q, mP, N0P);
        KERNEL_CHECK(ctx);
    }
    return GPFQ_OK;
}

// ---- diagnostics entry point (include/gpfq.h): C = A B^T through the int8-slice kernel, host arrays ------------------------
extern "C" int gpfq_debug_slgemm(gpfq_ctx *ctx, const double *A, const float *B, int64_t M, int64_t N, int64_t K, int32_t D,
                                 int32_t transposed_b, double *C_out) {
    // A: (M, K) fp64 row-major.  B: (N, K) fp32 row-major, or with transposed_b (K, N) fp32 row-major -- the X^T slicing path.
    using namespace slg;
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (!A || !B || !C_out || M < 1 || N < 1 || K < 1) return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad arguments");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t MP = ceil_div64(M, 128) * 128, NP = ceil_div64(N, 128) * 128, KP = ceil_div64(K, 128) * 128;
    double *dA = nullptr, *dC = nullptr;
    float *dB = nullptr;
    int8_t *sA = nullptr, *sB = nullptr;
    int32_t *e = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_G1, (size_t)M * K * sizeof(double), (void **)&dA));
    GPFQ_TRY(gpfq_ws(ctx, WS_X, (size_t)N * K * sizeof(float), (void **)&dB));
    GPFQ_TRY(gpfq_ws(ctx, WS_G2, (size_t)M * N * sizeof(double), (void **)&dC));
    GPFQ_TRY(gpfq_ws(ctx, WS_I8_SQ, (size_t)S * MP * KP, (void **)&sA));
    GPFQ_TRY(gpfq_ws(ctx, WS_I8_SX, (size_t)S * NP * KP, (void **)&sB));
    GPFQ_TRY(gpfq_ws(ctx, WS_I8_E, (size_t)(MP + 2 * NP + 8) * sizeof(int32_t), (void **)&e));
    CUDA_TRY(ctx, cudaMemcpyAsync(dA, A, (size_t)M * K * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(dB, B, (size_t)N * K * sizeof(float), cudaMemcpyHostToDevice, st));
    GPFQ_TRY(sl_rowsplit<double>(ctx, dA, K, M, K, e, sA, MP, KP, 0, MP));
    if (transposed_b) GPFQ_TRY(sl_transsplit(ctx, dB, nullptr, N, K, N, e + MP, reinterpret_cast<int *>(e + MP + NP), sB, nullptr, NP, KP));
    else GPFQ_TRY(sl_rowsplit<float>(ctx, dB, K, N, K, e + MP, sB, NP, KP, 0, NP));
    SlOperand oa, ob;
    GPFQ_TRY(sl_make_operand(ctx, &oa, sA, MP, KP, S, e, 0, false));
    GPFQ_TRY(sl_make_operand(ctx, &ob, sB, NP, KP, S, e + MP, 0, true));
    int64_t done = 0;
    bool first = true;
    while (done < KP) {     // K chunks of at most KB_MAX blocks: the s32 accumulators cannot overflow
        const int64_t kc = std::min<int64_t>(KP - done, (int64_t)KB_MAX * BK);
        SlProduct p = {&oa, &ob, 0, 0, done, kc, D, 1.0};
        GPFQ_TRY(slgemm_i8(ctx, &p, 1, dC, N, M, N, !first));
        first = false;
        done += kc;
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(C_out, dC, (size_t)M * N * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    return GPFQ_OK;
}
