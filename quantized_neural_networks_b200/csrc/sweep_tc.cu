// sweep_tc.cu -- the range walk of the Dense sweep with one THREAD per neuron and the range's Q terms on the 5th-generation
// tensor cores (symmetric equispaced alphabets; the ternary one of the VGG16 / MNIST configurations has its own specialisation).
//
// What a range of R <= 512 directions [tb, te) has to do for every neuron (quantized_network.py:83-89, :117-119 in Gram form):
//     d_t = P[t] - sum_{tb <= s < t} q_s G2[t][s],   q_t = Q( (d_t + w_t G1[t][t]) / nrm_t^2 )        (guards of :83-87)
// where P already holds everything that does not depend on the range's own decisions (earlier ranges, and the W terms
// sum_{tb <= s < t} w_s G1[t][s] of the range, one batched tcgen05 product before the sweep starts).  The walk is blocked by 32
// directions.  For block b of the range
//     * the Q terms of the EARLIER blocks are an integer matrix product: level indices k'_s = q_s / h (int8, one K-major
//       128-neuron tile in shared memory that grows by 32 bytes per row and block) times the five int8 digit slices of the Gram
//       rows G2[block b, tb : tb + 32 b] -- tcgen05.mma.kind::i8, M = 128 neurons (= TMEM lanes), N = 32 directions, K = 32 per
//       instruction, five s32 accumulators of 32 columns each, exact.  The K steps of blocks <= b - 2 are issued WHILE block b - 1
//       is walked; only the five MMAs of block b - 1's own decisions sit between two walks;
//     * every walker thread then reads ITS neuron's 5 x 32 sums straight out of its TMEM lane (tcgen05.ld 32x32b), combines the
//       digits as one 64-bit integer per direction and scales once: d_t -= h 2^(e_t - 38) I_t;
//     * and walks the 32 directions in registers, fully unrolled: fma, multiply by RN(1 / nrm^2), two compares, select, then one
//       DFMA per remaining direction with the Gram column broadcast from shared memory.  No shuffles, no barriers, no division
//       on the chain (~40 dependent cycles per step; the 4-lanes-per-neuron walk of sweep_pipe_kernel measured ~360).
// Exactness of the short chain: with p = RN(num * rinv) and v = RN(num / den) (what the reference rounds), |p - v| <= 3 ulp, so
// the ternary decision of p (thresholds +- a / 2, ties as _bit_round_parallel breaks them: v = a / 2 -> 0, v = -a / 2 -> -a) is
// the decision of v unless p lies within a few 2^-20 of a threshold (compared as high words, on the integer pipe), is not finite or
// huge, or the perpendicularity guard (:86) fires on a live direction.  Those steps raise a flag; a warp with a flag replays its
// block from the saved residual dots with the literal arithmetic (Markstein-corrected division, the three-level scan).  Random data
// replays one block per neuron (u_0 = 0 at the first step) and about one warp-block in 300 for a near-threshold value.  Alphabets
// with more than three levels round the grid position kr = (p + a) / step with the 1.5 * 2^52 trick; a value within 2^-30 of a step
// of a tie between two levels flags the same way.  The results are level INDICES; the fp64 values of the layer are looked up from
// the stored levels afterwards (stc_q_from_kq_kernel), bit for bit the alphabet's entries.
//
// Kernel anatomy (one CTA per 128 neurons, one CTA per SM, 224 threads):
//   warps 0-3  walkers: thread = neuron = TMEM lane
//   warp 4     TMEM allocator + MMA issuer (one elected lane)
//   warp 5     producer of the Gram digit slices: one 10 KB bulk copy per K block of 64 earlier directions, 3-stage mbarrier ring
//   warp 6     producer of a block's inputs, one block ahead: the P rows and fp32 weights of the CTA's 128 neurons (three TMA boxes,
//              128B swizzle: thread j reads row j conflict-free) and the per-block table (TabA), 2 stages
#include <algorithm>
#include <cfloat>

#include "slgemm_i8.cuh"
#include "sweep_tc.cuh"

namespace stc {
constexpr int NST = 3;
constexpr int THREADS = 224;
constexpr int A_KB = NT * KB;                          // level indices of one K block: 128 rows x 64 B
constexpr int A_BYTES = (MAX_R / KB) * A_KB;
constexpr int TAB_BYTES = (int)sizeof(TabA);
constexpr int D_BYTES = NB * NT * 8, W_BYTES = NB * NT * 4;
constexpr int OFF_B = A_BYTES;
constexpr int OFF_D = OFF_B + NST * B_STAGE;          // 2 sets x 2 TMA boxes (16 directions x 128 neurons, fp64, 128B swizzle)
constexpr int OFF_W = OFF_D + 2 * D_BYTES;            // 2 sets x 1 TMA box (32 directions x 128 neurons, fp32, 128B swizzle)
constexpr int OFF_TAB = OFF_W + 2 * W_BYTES;
constexpr int OFF_Q = OFF_TAB + 2 * TAB_BYTES;
constexpr int OFF_ALPH = OFF_Q + NB * NT;              // the alphabet's levels (replay path of alphabets with more than 3 levels)
constexpr int OFF_BAR = OFF_ALPH + 128 * 8;
constexpr int IN_BYTES = D_BYTES + W_BYTES + TAB_BYTES;   // what one block's inputs add up to (one mbarrier transaction count)
constexpr size_t SMEM = (size_t)OFF_BAR + 256 + 1024 /* alignment slack */;
constexpr int ACC_COLS = S * NB;                       // TMEM columns of one accumulator set
static_assert(TAB_BYTES % 16 == 0 && OFF_TAB % 16 == 0 && OFF_D % 1024 == 0 && OFF_W % 1024 == 0 && OFF_BAR % 8 == 0,
              "bulk copies need 16-byte, swizzled TMA boxes 1024-byte alignment");
static_assert(2 * ACC_COLS <= 512, "two accumulator sets in TMEM");

__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t saddr) {   // K-major, 64-byte rows, SWIZZLE_64B (as slgemm_i8.cu)
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)4 << 61);
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::"r"(
                     i8g::smem_u32(dst)), "l"(map), "r"(i8g::smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
// 16-byte chunk c of row r of a TMA box with 128-byte rows, SWIZZLE_128B: consecutive rows read the same chunk conflict-free
__device__ __forceinline__ int sw128(int r, int c) { return r * 128 + ((c ^ (r & 7)) << 4); }
// 16 columns of each of the five accumulators of this thread's lane, one wait for all of them
__device__ __forceinline__ void tmem_ld_5x16(uint32_t taddr, uint32_t (&v)[S][16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%80];\n"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%81];\n"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47}, [%82];\n"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%83];\n"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%64, %65, %66, %67, %68, %69, %70, %71, %72, %73, %74, %75, %76, %77, %78, %79}, [%84];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        : "=r"(v[0][0]), "=r"(v[0][1]), "=r"(v[0][2]), "=r"(v[0][3]), "=r"(v[0][4]), "=r"(v[0][5]), "=r"(v[0][6]), "=r"(v[0][7]),
          "=r"(v[0][8]), "=r"(v[0][9]), "=r"(v[0][10]), "=r"(v[0][11]), "=r"(v[0][12]), "=r"(v[0][13]), "=r"(v[0][14]), "=r"(v[0][15]),
          "=r"(v[1][0]), "=r"(v[1][1]), "=r"(v[1][2]), "=r"(v[1][3]), "=r"(v[1][4]), "=r"(v[1][5]), "=r"(v[1][6]), "=r"(v[1][7]),
          "=r"(v[1][8]), "=r"(v[1][9]), "=r"(v[1][10]), "=r"(v[1][11]), "=r"(v[1][12]), "=r"(v[1][13]), "=r"(v[1][14]), "=r"(v[1][15]),
          "=r"(v[2][0]), "=r"(v[2][1]), "=r"(v[2][2]), "=r"(v[2][3]), "=r"(v[2][4]), "=r"(v[2][5]), "=r"(v[2][6]), "=r"(v[2][7]),
          "=r"(v[2][8]), "=r"(v[2][9]), "=r"(v[2][10]), "=r"(v[2][11]), "=r"(v[2][12]), "=r"(v[2][13]), "=r"(v[2][14]), "=r"(v[2][15]),
          "=r"(v[3][0]), "=r"(v[3][1]), "=r"(v[3][2]), "=r"(v[3][3]), "=r"(v[3][4]), "=r"(v[3][5]), "=r"(v[3][6]), "=r"(v[3][7]),
          "=r"(v[3][8]), "=r"(v[3][9]), "=r"(v[3][10]), "=r"(v[3][11]), "=r"(v[3][12]), "=r"(v[3][13]), "=r"(v[3][14]), "=r"(v[3][15]),
          "=r"(v[4][0]), "=r"(v[4][1]), "=r"(v[4][2]), "=r"(v[4][3]), "=r"(v[4][4]), "=r"(v[4][5]), "=r"(v[4][6]), "=r"(v[4][7]),
          "=r"(v[4][8]), "=r"(v[4][9]), "=r"(v[4][10]), "=r"(v[4][11]), "=r"(v[4][12]), "=r"(v[4][13]), "=r"(v[4][14]), "=r"(v[4][15])
        : "r"(taddr), "r"(taddr + NB), "r"(taddr + 2 * NB), "r"(taddr + 3 * NB), "r"(taddr + 4 * NB)
        : "memory");
}

// The literal walk of one block from the saved residual dots (own shared-memory column), for a warp that raised a flag:
// gpfq_decide_rcp_inl of dense_gram.cu with the ternary scan.  Rolled loops; decisions go out as level indices.
// SCALED: the neuron's levels are fl(s alph[k]) (per-channel alphabets; a = fl(s alph[K - 1]), `alph` the base alphabet); a neuron
// with s = 0 decides the literal 0 everywhere (its levels are all zero) and never reaches the divisions by a.
// STOCH: stochastic rounding (common.cuh) with the draw of step t0 + t from the neuron's unit key.
// L1: the value of step t is shrunk by its tau (lane t's tau_l: the whole warp replays).
template <bool SCALED, bool STOCH = false, bool L1 = false>
static __device__ __noinline__ void replay_block(unsigned char *dset, const unsigned char *wset, int j, const TabA *tab, double a,
                                                 int8_t *qcol, const double *alph, int K, double s, uint64_t key = 0, int64_t t0 = 0,
                                                 double tau_l = 0.0) {
    // K == 3: the ternary scan with the levels in registers; else the windowed scan of the equispaced levels (common.cuh)
    const bool zero = SCALED && !(a > 0.0);
    const double inv_step = zero ? 0.0 : (SCALED ? gpfq_inv_step_s(alph, K, 1, s) : 0.5 * (double)(K - 1) / a);
    const double inv_h = zero ? 0.0 : (double)(K - 1) / a;
    auto dptr = [&](int t) { return reinterpret_cast<double *>(dset + (t >> 4) * (D_BYTES / 2) + sw128(j, (t & 15) >> 1)) + (t & 1); };
    for (int t = 0; t < NB; ++t) {
        const double d0 = *dptr(t);
        const double wv = (double)reinterpret_cast<const float *>(wset + sw128(j, t >> 2))[t & 3];
        const double nrm = tab->nrm[t];
        const double tau = L1 ? __shfl_sync(0xffffffffu, tau_l, t) : 0.0;
        double q = 0.0;
        if (!(nrm < GPFQ_DEAD_NORM)) {
            double v = wv;
            if (!(fabs(d0) < GPFQ_PERP_DOT)) {
                const double num = fma(wv, tab->g1dd[t], d0), rinv = tab->rinv[t];
                const double q0 = num * rinv;
                const double e = fma(-q0, tab->den[t], num);
                v = fma(e, rinv, q0);
            }
            if (L1) v = gpfq_shrink(v, tau);
            if (zero) q = 0.0;
            else if (STOCH && K == 3) q = gpfq_stoc_round_ternary(v, a, gpfq_draw(key, t0 + t));
            else if (STOCH) q = gpfq_stoc_round_eq<SCALED>(v, alph, K, inv_step, s, gpfq_draw(key, t0 + t));
            else if (K == 3) q = gpfq_bit_round_ternary(v, a);
            else q = SCALED ? gpfq_bit_round_eq_s(v, alph, K, inv_step, s) : gpfq_bit_round_eq(v, alph, K, inv_step);
        }
        qcol[t * NT] = (int8_t)__double2int_rn(q * inv_h);   // level index k' = q / h, h = a / (K - 1); the literal 0 of a dead direction is 0
        for (int u = t + 1; u < NB; ++u) {
            double *du = dptr(u);
            *du = fma(-tab->g2c[t * NB + u], q, *du);
        }
    }
}

// SCALED (per-channel alphabets): neuron jg walks with its own levels fl(scales[jg] levels[k]) -- a = fl(s levels[K - 1]) and the step
// h = a / (K - 1) per walker, from tables prepared with h = 1 (TabA::sc = 2^(e - 38), TabA::ris = rinv / 2); `levels` is the base
// alphabet.  Applying h per walker adds one rounding to the grid position (ris / h: RN(RN(rinv / 2) * RN(1 / h)) against RN(rinv / 2h),
// at most 2 ulp of kr < 2^7), far inside the 2^-30 band that flags a tie; the Q-term scale h 2^(e - 38) stays exact.  The ternary
// thresholds +- a / 2 and their flag window are per walker.
//
// STOCH (stochastic rounding, DESIGN.md 5.6): step t of neuron jg draws r = draw(seed, u0 + jg, t) -- the unit key once per walker, one
// splitmix64 per step, on the integer pipe beside the chain.  Ternary: q = a if p > r a, -a if p <= (r - 1) a, else 0 (on [0, a) the
// literal rule is r < v / a, on (-a, 0) it is r < (v + a) / a); a step is flagged when p lies within 2^-30 a of either threshold.  More
// levels: the grid position kr = (p + a) / step splits into the interval k = floor(kr) and the fraction f = kr - k; the upper level is
// taken when r < f, and a step is flagged when f lies within 2^-30 of 0, 1 or r.  The non-finite / huge and :86 flags are those of
// the nearest walk; a flagged warp replays its block with the literal stoc_round.
//
// L1 (the penalty lambda = *lambdas, DESIGN.md 5.7): lane t of a walker warp forms tau of the block's direction t once per block
// (one division per lane and block), and step t takes it by a shuffle, off the chain.  Ternary: the shrink moves the thresholds
// out by tau -- q = a iff p > r a + tau, -a iff p <= (r - 1) a - tau, with r = 1/2 for nearest rounding -- and a step is flagged
// when p lies within 2^-30 (a + tau) of either.  More levels: the grid position is taken from the shrunk p; the tie / fraction flags
// are those above, and a step whose tau exceeds 2^16 steps is flagged unless |p| < tau (1 - 2^-40), where the shrink gives the
// literal 0 either way (a huge tau would otherwise carry its rounding into the grid position).
template <bool TERN, bool SCALED = false, bool STOCH = false, bool L1 = false>
__global__ void __launch_bounds__(THREADS, 1)
sweep_tc_kernel(const __grid_constant__ CUtensorMap mapP, const __grid_constant__ CUtensorMap mapW, const TabA *__restrict__ tabs,
                const int8_t *__restrict__ g2s, int kbr, int64_t tb, int64_t te, int row0, int64_t nj, int8_t *__restrict__ Kq,
                int64_t krows, int64_t krow0, double a_base, const double *__restrict__ levels, int K,
                const double *__restrict__ scales = nullptr, const uint64_t *__restrict__ seeds = nullptr, int64_t u0 = 0,
                const double *__restrict__ lambdas = nullptr) {
    using namespace i8g;
    extern __shared__ unsigned char stc_smem_raw[];
    // (offset arithmetic on the array itself: the compiler keeps the shared address space, LDS / STS instead of generic accesses)
    unsigned char *smem = stc_smem_raw + ((1024u - (smem_u32(stc_smem_raw) & 1023u)) & 1023u);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
    uint64_t *full = bars, *empty = bars + NST, *in_full = bars + 2 * NST, *in_empty = in_full + 2, *acc_full = in_empty + 2,
             *acc_empty = acc_full + 2, *walk_done = acc_empty + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(walk_done + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nblk = (int)((te - tb + NB - 1) / NB);
    const int64_t blk0 = tb / NB;

    if (tid == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&in_full[s], 1);
            mbar_init(&in_empty[s], NT);
            mbar_init(&acc_full[s], 1);
            mbar_init(&acc_empty[s], NT);
        }
        mbar_init(walk_done, NT);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    double *alph = reinterpret_cast<double *>(smem + OFF_ALPH);
    if (!TERN && tid < K) alph[tid] = levels[tid];
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp < 4) {
        // =============================== walkers: thread j = neuron = TMEM lane ===============================
        const int j = tid;
        const int64_t jg = (int64_t)blockIdx.x * NT + j;
        const bool valid = jg < nj;   // (rows beyond nj exist in P / Wn -- allocation padding -- and hold whatever they hold)
        const double s_u = SCALED ? (valid ? scales[jg] : 0.0) : 1.0;
        const double a = SCALED ? __dmul_rn(s_u, a_base) : a_base;
        const bool zero = SCALED && !(a > 0.0);                     // s = 0: every decision is the literal 0, no replay
        const double h_u = SCALED ? (zero ? 0.0 : a / (double)(K - 1)) : 1.0, inv_hu = SCALED ? (zero ? 0.0 : 1.0 / h_u) : 1.0;
        const double hh = 0.5 * a;
        // flags of the ternary walk, compared as high words: [hi(a / 2) - 1, hi(a / 2) + 1] around the thresholds (a window of ~2^-20
        // relative: one warp-block in ~300 replays), a * 2^40 and above (NaN / Inf included), 1e-10 and below (:86)
        const uint32_t near_lo = (uint32_t)__double2hiint(hh) - 1u, big_hi = (uint32_t)__double2hiint(a * 0x1p40),
                       perp_hi = (uint32_t)__double2hiint(GPFQ_PERP_DOT);
        // more than three levels a_k = -a + k s, s = 2 a / (K - 1): grid position kr = (p + a) / s, nearest level by the 1.5 * 2^52 trick
        const double km1 = (double)(K - 1), step = 2.0 * a / km1, cmid = 0.5 * km1, magic = 6755399441055744.0;
        const uint32_t lane_field = (uint32_t)(warp * 32) << 16;
        const uint64_t key = STOCH ? gpfq_unit_key(seeds[0], u0 + jg) : 0;
        const double lam = L1 ? lambdas[0] : 0.0, inv_st = SCALED ? 0.5 * inv_hu : cmid / a;   // (one step = 2 h)
        for (int b = 0; b < nblk; ++b) {
            const int buf = b & 1;
            const int64_t t0 = tb + (int64_t)b * NB;
            // ---- the block's inputs (TMA, warp 6): this neuron's row of P (two boxes of 16 directions), its weights, the tables
            unsigned char *dset = smem + OFF_D + buf * D_BYTES;
            const unsigned char *wset = smem + OFF_W + buf * W_BYTES;
            const TabA *tab = reinterpret_cast<const TabA *>(smem + OFF_TAB + buf * TAB_BYTES);
            mbar_wait(&in_full[buf], (b >> 1) & 1);
            double d[NB];
#pragma unroll
            for (int c = 0; c < NB / 2; ++c) {
                const double2 v = *reinterpret_cast<const double2 *>(dset + (c >> 3) * (D_BYTES / 2) + sw128(j, c & 7));
                d[2 * c] = v.x;
                d[2 * c + 1] = v.y;
            }
            if (b > 0) {
                // ---- Q terms of the range's earlier blocks: five integer sums per direction out of this thread's TMEM lane
                mbar_wait(&acc_full[buf], ((b - 1) >> 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const uint32_t tacc = tmem_base + lane_field + (uint32_t)(buf * ACC_COLS);
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    uint32_t v[S][16];
                    tmem_ld_5x16(tacc + hf * 16, v);
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        long long I = (long long)(int)v[0][i];
#pragma unroll
                        for (int s = 1; s < S; ++s) I = I * 256 + (long long)(int)v[s][i];
                        const double sc = SCALED ? h_u * tab->sc[hf * 16 + i] : tab->sc[hf * 16 + i];   // exact: sc = 2^(e - 38)
                        d[hf * 16 + i] = fma(-sc, (double)I, d[hf * 16 + i]);
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                mbar_arrive(&acc_empty[buf]);
            }
            // the block's residual dots, kept for a replay (own slots: the P values they came from are spent)
#pragma unroll
            for (int c = 0; c < NB / 2; ++c)
                *reinterpret_cast<double2 *>(dset + (c >> 3) * (D_BYTES / 2) + sw128(j, c & 7)) = make_double2(d[2 * c], d[2 * c + 1]);
            // ---- the walk: 32 steps in registers
            const double2 *g2 = reinterpret_cast<const double2 *>(tab->g2c);
            uint32_t pk[NB / 4];
#pragma unroll
            for (int i = 0; i < NB / 4; ++i) pk[i] = 0u;
            int flag = 0;
            uint32_t m_near = 0xffffffffu, m_big = 0u, m_perp = 0xffffffffu;
            double m_thr = 1e300;   // STOCH ternary: the least |p - threshold| / a of the block
            const double tau_l = L1 ? gpfq_l1_tau(lam, tab->nrm[lane]) : 0.0;   // tau of the block's direction `lane`
#pragma unroll
            for (int t = 0; t < NB; ++t) {
                float4 w4;
                if ((t & 3) == 0) w4 = *reinterpret_cast<const float4 *>(wset + sw128(j, t >> 2));
                const double wv = (double)((t & 3) == 0 ? w4.x : (t & 3) == 1 ? w4.y : (t & 3) == 2 ? w4.z : w4.w);
                const double ri = tab->rinv[t];
                const double num = fma(wv, tab->g1dd[t], d[t]);
                double q;
                if (TERN && L1) {
                    const double p = num * ri;
                    const double tau = __shfl_sync(0xffffffffu, tau_l, t);
                    const double rr = STOCH ? gpfq_draw(key, t0 + t) : 0.5;
                    // the step's thresholds and flag window, off the chain (clamped: tau = inf flags nothing, decides 0)
                    const double up_t = fmin(fma(rr, a, tau), DBL_MAX), dn_t = fmax(fma(rr - 1.0, a, -tau), -DBL_MAX);
                    const double band = 0x1p-30 * fmin(a + tau, DBL_MAX);
                    const bool up = p > up_t, dn = p <= dn_t;
                    q = up ? a : (dn ? -a : 0.0);
                    flag |= (int)!(fmin(fabs(p - up_t), fabs(p - dn_t)) > band);
                    const uint32_t hp = (uint32_t)__double2hiint(p) & 0x7fffffffu;
                    m_big = max(m_big, hp);
                    m_perp = min(m_perp, ((uint32_t)__double2hiint(d[t]) & 0x7fffffffu) | (uint32_t)tab->deadm[t]);
                    pk[t >> 2] |= (up ? 2u : (dn ? 0xfeu : 0u)) << (8 * (t & 3));
                } else if (L1) {
                    const double p = num * ri;
                    const double tau = __shfl_sync(0xffffffffu, tau_l, t);
                    const double ps = fabs(p) <= tau ? 0.0 : p - copysign(tau, p);   // the shrink of p
                    const double kr = fma(ps, inv_st, cmid);
                    double r;
                    int fl;
                    if (STOCH) {
                        const double rr = gpfq_draw(key, t0 + t);
                        const double k0 = fmin(fmax(floor(kr), 0.0), km1 - 1.0);
                        const double f = kr - k0;
                        r = rr < f ? k0 + 1.0 : k0;
                        fl = (int)!(fabs(f) > 0x1p-30) | (int)!(fabs(f - 1.0) > 0x1p-30) | (int)!(fabs(f - rr) > 0x1p-30);
                    } else {
                        const double r0 = (kr + magic) - magic;
                        r = fmin(fmax(r0, 0.0), km1);
                        fl = (int)!(fabs(kr - r0) < 0.5 - 0x1p-30);
                    }
                    const bool live = ri != 0.0;
                    q = live ? fma(r, step, -a) : 0.0;
                    fl |= (int)!(fabs(kr) < 0x1p40) | (int)(fabs(d[t]) < GPFQ_PERP_DOT) |
                          ((int)(tau * inv_st >= 0x1p16) & (int)!(fabs(p) < tau * (1.0 - 0x1p-40)));
                    flag |= fl & (int)live;
                    const int kq = live ? __double2int_rn(fma(r, 2.0, -km1)) : 0;
                    pk[t >> 2] |= ((uint32_t)kq & 0xffu) << (8 * (t & 3));
                } else if (TERN && STOCH) {
                    const double p = num * ri;
                    const double rr = gpfq_draw(key, t0 + t);
                    const double ra = rr * a, rm = (rr - 1.0) * a;       // the thresholds of this step, off the chain
                    const bool up = p > ra, dn = p <= rm;
                    q = up ? a : (dn ? -a : 0.0);
                    m_thr = fmin(m_thr, fmin(fabs(p - ra), fabs(p - rm)));
                    const uint32_t hp = (uint32_t)__double2hiint(p) & 0x7fffffffu;
                    m_big = max(m_big, hp);
                    m_perp = min(m_perp, ((uint32_t)__double2hiint(d[t]) & 0x7fffffffu) | (uint32_t)tab->deadm[t]);
                    pk[t >> 2] |= (up ? 2u : (dn ? 0xfeu : 0u)) << (8 * (t & 3));
                } else if (TERN) {
                    const double p = num * ri;
                    const bool up = p > hh, dn = p <= -hh;
                    q = up ? a : (dn ? -a : 0.0);
                    // the flags on the integer pipe (the fp64 pipe carries the chain): |p| within a few 2^-20 of the threshold,
                    // |p| huge / not finite, and the :86 guard on |d| (dead directions masked out by the table)
                    const uint32_t hp = (uint32_t)__double2hiint(p) & 0x7fffffffu;
                    m_near = min(m_near, hp - near_lo);
                    m_big = max(m_big, hp);
                    m_perp = min(m_perp, ((uint32_t)__double2hiint(d[t]) & 0x7fffffffu) | (uint32_t)tab->deadm[t]);
                    pk[t >> 2] |= (up ? 2u : (dn ? 0xfeu : 0u)) << (8 * (t & 3));   // level index k' = q / h = +-2 (h = a / 2)
                } else if (STOCH) {
                    // grid position kr = (p + a) / step: interval k = floor(kr) (clamped to the K - 1 intervals), fraction f against r
                    const double kr = fma(num, SCALED ? tab->ris[t] * inv_hu : tab->ris[t], cmid);
                    const double rr = gpfq_draw(key, t0 + t);
                    const double k0 = fmin(fmax(floor(kr), 0.0), km1 - 1.0);
                    const double f = kr - k0;
                    const double r = rr < f ? k0 + 1.0 : k0;
                    const bool live = ri != 0.0;
                    q = live ? fma(r, step, -a) : 0.0;
                    flag |= ((int)!(fabs(f) > 0x1p-30) | (int)!(fabs(f - 1.0) > 0x1p-30) | (int)!(fabs(f - rr) > 0x1p-30) |
                             (int)!(fabs(kr) < 0x1p40) | (int)(fabs(d[t]) < GPFQ_PERP_DOT)) & (int)live;
                    const int kq = live ? __double2int_rn(fma(r, 2.0, -km1)) : 0;
                    pk[t >> 2] |= ((uint32_t)kq & 0xffu) << (8 * (t & 3));
                } else {
                    const double kr = fma(num, SCALED ? tab->ris[t] * inv_hu : tab->ris[t], cmid);   // ris = rinv / s
                    const double r0 = (kr + magic) - magic;                  // rint(kr)
                    const double r = fmin(fmax(r0, 0.0), km1);
                    const bool live = ri != 0.0;
                    q = live ? fma(r, step, -a) : 0.0;                       // a dead direction: the literal 0 (:83-84), index 0
                    // a tie between two levels (or anything within 2^-30 of a step of one), a non-finite / huge argument, the :86 guard
                    flag |= ((int)!(fabs(kr - r0) < 0.5 - 0x1p-30) | (int)!(fabs(kr) < 0x1p40) | (int)(fabs(d[t]) < GPFQ_PERP_DOT)) & (int)live;
                    const int kq = live ? __double2int_rn(fma(r, 2.0, -km1)) : 0;   // k' = 2 k - (K - 1)
                    pk[t >> 2] |= ((uint32_t)kq & 0xffu) << (8 * (t & 3));
                }
#pragma unroll
                for (int pp = (t + 1) >> 1; pp < NB / 2; ++pp) {
                    const double2 g = g2[t * (NB / 2) + pp];
                    if (2 * pp > t) d[2 * pp] = fma(-g.x, q, d[2 * pp]);
                    d[2 * pp + 1] = fma(-g.y, q, d[2 * pp + 1]);
                }
                // a branch the compiler cannot remove ends the basic block here: ptxas schedules one step at a time.  (Given the whole
                // walk as ONE block it sinks every update to just before its use -- a serial chain of up to 31 DFMAs in front of the
                // late steps, 2.4 us per block instead of ~1.)
                if (kbr == -1 - t) asm volatile("trap;\n");
            }
            if (TERN && L1) flag |= (int)(m_big >= big_hi) | (int)(m_perp <= perp_hi);
            else if (TERN && STOCH) flag = (int)!(m_thr > 0x1p-30 * a) | (int)(m_big >= big_hi) | (int)(m_perp <= perp_hi);
            else if (TERN) flag = (int)(m_near <= 2u) | (int)(m_big >= big_hi) | (int)(m_perp <= perp_hi);
            if (SCALED && zero) {
                flag = 0;
#pragma unroll
                for (int i = 0; i < NB / 4; ++i) pk[i] = 0u;
            }
            if (__any_sync(0xffffffffu, flag != 0 && valid)) {   // (rows beyond nj hold zeros: they would trip the :86 guard at every step)
                int8_t *qcol = reinterpret_cast<int8_t *>(smem + OFF_Q) + j;
                if (L1) replay_block<SCALED, STOCH, true>(dset, wset, j, tab, a, qcol, alph, K, s_u, key, t0, tau_l);
                else replay_block<SCALED, STOCH>(dset, wset, j, tab, a, qcol, alph, K, s_u, key, t0);
#pragma unroll
                for (int i = 0; i < NB / 4; ++i) {
                    uint32_t w4 = 0u;
#pragma unroll
                    for (int c = 0; c < 4; ++c) w4 |= (uint32_t)(uint8_t)qcol[(4 * i + c) * NT] << (8 * c);
                    pk[i] = w4;
                }
            }
            // ---- hand the decisions over: 32 bytes of this neuron's row of the level-index tile (K block b / 2, 64B swizzle)
            const int sw = (j >> 1) & 3, c16 = 2 * (b & 1);
            if (b + 1 < nblk) {
                unsigned char *arow = smem + (b >> 1) * A_KB + j * KB;
                *reinterpret_cast<uint4 *>(arow + ((c16 ^ sw) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                *reinterpret_cast<uint4 *>(arow + (((c16 + 1) ^ sw) << 4)) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
                asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
                mbar_arrive(walk_done);
            }
            mbar_arrive(&in_empty[buf]);
            // ---- results: the level indices (the residual update of the next range reads them as an int8 operand; the fp64
            // values of the layer are made from them once at the end, stc_q_from_kq_kernel)
            if (valid) {
                int8_t *kq = Kq + sl_offset(t0, 0, krow0 + jg, krows, 1);   // t0 is a multiple of 32: chunk c16 of its K block
                int8_t *kq1 = Kq + sl_offset(t0 + 16, 0, krow0 + jg, krows, 1);
                *reinterpret_cast<uint4 *>(kq) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                *reinterpret_cast<uint4 *>(kq1) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
            }
        }
    } else if (warp == 4) {
        // =============================== MMA issuer ===============================
        // instruction descriptor: D = s32, A = B = signed 8-bit, both K-major, N = 32, M = 128
        const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NB >> 3) << 17) | ((uint32_t)(NT >> 4) << 24);
        const uint32_t a_base = smem_u32(smem), b_base = smem_u32(smem + OFF_B);
        int it = 0;
        for (int b = 1; b < nblk; ++b) {
            const int buf = b & 1, u = (b - 1) >> 1;
            if (u >= 1) mbar_wait(&acc_empty[buf], (u - 1) & 1);   // the walkers have read this set's previous sums
            const uint32_t tacc = tmem_base + (uint32_t)(buf * ACC_COLS);
            for (int kp = 0; kp < b; ++kp) {   // K step kp = the decisions of block kp
                const int kb = kp >> 1, ks = kp & 1, s = it % NST;
                if (ks == 0) mbar_wait(&full[s], (it / NST) & 1);
                if (kp == b - 1) mbar_wait(walk_done, (b - 1) & 1);   // block b - 1 has just been walked
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const bool closes = (ks == 1) || (kp == b - 1);
                if (elect_one()) {
                    const uint64_t da = umma_desc_sw64(a_base + kb * A_KB + ks * 32);
                    const uint64_t db = umma_desc_sw64(b_base + s * B_STAGE + ks * 32);
#pragma unroll
                    for (int sl = 0; sl < S; ++sl)
                        umma_i8(tacc + (uint32_t)(sl * NB), da, db + (uint64_t)((sl * B_SLICE) >> 4), idesc, kp ? 1u : 0u);
                    if (closes) umma_commit(&empty[s]);
                    if (kp == b - 1) umma_commit(&acc_full[buf]);
                }
                __syncwarp();
                if (closes) ++it;
            }
        }
    } else if (warp == 5) {
        // =============================== producer: Gram digit slices ===============================
        if (lane == 0) {
            int it = 0;
            for (int b = 1; b < nblk; ++b) {
                const int8_t *src = g2s + (blk0 + b) * (int64_t)kbr * B_STAGE;
                const int nkb = (b + 1) >> 1;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % NST;
                    if (it >= NST) mbar_wait(&empty[s], ((it / NST) - 1) & 1);
                    mbar_expect_tx(&full[s], B_STAGE);
                    bulk_load(smem + OFF_B + s * B_STAGE, src + (int64_t)kb * B_STAGE, B_STAGE, &full[s]);
                }
            }
        }
    } else if (warp == 6) {
        // =============================== producer: the block's P rows, weights and tables ===============================
        if (lane == 0) {
            const int r0 = row0 + (int)blockIdx.x * NT;
            for (int b = 0; b < nblk; ++b) {
                const int buf = b & 1, u = b >> 1;
                const int c0 = (int)(tb + (int64_t)b * NB);
                if (u >= 1) mbar_wait(&in_empty[buf], (u - 1) & 1);
                mbar_expect_tx(&in_full[buf], IN_BYTES);
                tma_load_2d(smem + OFF_D + buf * D_BYTES, &mapP, &in_full[buf], c0, r0);
                tma_load_2d(smem + OFF_D + buf * D_BYTES + D_BYTES / 2, &mapP, &in_full[buf], c0 + NB / 2, r0);
                tma_load_2d(smem + OFF_W + buf * W_BYTES, &mapW, &in_full[buf], c0, r0);
                bulk_load(smem + OFF_TAB + buf * TAB_BYTES, tabs + blk0 + b, TAB_BYTES, &in_full[buf]);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 4) {
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512));
    }
}

// ---- per-layer tables --------------------------------------------------------------------------------------------
// One CTA per block of 32 directions: digit slices of its Gram rows against the earlier directions of its range (one exponent
// per row: 38 bits below the row maximum, as every other int8-slice operand of this library), and the block's TabA.
__global__ void __launch_bounds__(256)
stc_prepare_kernel(const double *__restrict__ G1, const double *__restrict__ G2, int64_t ldg, int compact, int64_t N0, int64_t R,
                   double h, TabA *__restrict__ tabs, int8_t *__restrict__ g2s) {
    __shared__ int ex_s[NB], bad_s[NB];
    const int64_t blk = blockIdx.x, t0 = blk * NB, tbr = (t0 / R) * R, coff = compact ? tbr : 0;
    const int lo = (int)(t0 - tbr);                     // earlier directions of the range
    const int kbr = (int)(R / KB), nkb = (lo + KB - 1) / KB;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int8_t *out = g2s + blk * (int64_t)kbr * B_STAGE;
    for (int rr = 0; rr < 4; ++rr) {
        const int r = warp * 4 + rr;
        const int64_t t = t0 + r;
        const double *row = G2 + t * ldg + tbr - coff;  // row[c] = G2[t][tbr + c]
        double mx = 0.0;
        int bad = 0;
        if (t < N0)
            for (int c = lane; c < lo; c += 32) {
                const double x = row[c];
                mx = fmax(mx, fabs(x));
                bad |= !isfinite(x);
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            bad |= __shfl_xor_sync(0xffffffffu, bad, o);
        }
        int ex = 0;
        if (mx > 0.0 && !bad) frexp(mx, &ex);
        if (lane == 0) { ex_s[r] = ex; bad_s[r] = bad; }
        const double scale = ldexp(1.0, 8 * S - 2 - ex);
        for (int c0 = lane * 16; c0 < nkb * KB; c0 += 512) {
            uint32_t packed[S][4];
#pragma unroll
            for (int k = 0; k < S; ++k) packed[k][0] = packed[k][1] = packed[k][2] = packed[k][3] = 0u;
            if (t < N0 && c0 < lo && !bad) {
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const double x = (c0 + c < lo) ? row[c0 + c] : 0.0;
                    long long v = __double2ll_rn(x * scale);   // |v| <= 2^38
#pragma unroll
                    for (int k = S - 1; k >= 0; --k) {
                        const int dg = (int)((v + 128) & 255) - 128;   // balanced digit in [-128, 127]
                        v = (v - dg) >> 8;
                        packed[k][c >> 2] |= ((uint32_t)(dg & 0xff)) << (8 * (c & 3));
                    }
                }
            }
            const int kb = c0 >> 6, ch = (c0 >> 4) & 3;
#pragma unroll
            for (int k = 0; k < S; ++k)
                *reinterpret_cast<uint4 *>(out + (int64_t)kb * B_STAGE + k * B_SLICE + r * KB + ((ch ^ ((r >> 1) & 3)) << 4)) =
                    make_uint4(packed[k][0], packed[k][1], packed[k][2], packed[k][3]);
        }
    }
    __syncthreads();
    TabA *tab = tabs + blk;
    for (int e = threadIdx.x; e < NB * NB; e += 256) {
        const int tt = e >> 5, u = e & 31;
        tab->g2c[e] = (u > tt && t0 + u < N0) ? G2[(t0 + u) * ldg + t0 + tt - coff] : 0.0;
    }
    if (threadIdx.x < NB) {
        const int tt = threadIdx.x;
        const int64_t t = t0 + tt;
        const bool live = t < N0;
        const double g2 = live ? G2[t * ldg + t - coff] : 0.0, g1 = live ? G1[t * ldg + t - coff] : 0.0;
        const double nv = (double)(float)sqrt(g2);
        tab->g1dd[tt] = g1;
        tab->nrm[tt] = nv;
        tab->rinv[tt] = nv < GPFQ_DEAD_NORM ? 0.0 : 1.0 / (nv * nv);
        tab->den[tt] = nv * nv;
        tab->deadm[tt] = nv < GPFQ_DEAD_NORM ? 0x7ff00000 : 0;
        tab->ris[tt] = nv < GPFQ_DEAD_NORM ? 0.0 : (1.0 / (nv * nv)) / (2.0 * h);   // h = a / (K - 1): one step is 2 h
        tab->sc[tt] = bad_s[tt] ? __longlong_as_double(0x7ff8000000000000LL) : ldexp(h, ex_s[tt] - (8 * S - 2));
    }
}

// Digit slices of the strictly lower part of every range's G1 tile: one warp per row t, K = the range-local directions c < t - tb.
__global__ void __launch_bounds__(256)
stc_slice_g1_lower_kernel(const double *__restrict__ G1, int64_t ldg, int compact, int64_t N0, int64_t N0P, int64_t R,
                          int32_t *__restrict__ e, int8_t *__restrict__ slices) {
    const int lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (t >= N0P) return;
    const int64_t tbr = (t / R) * R, coff = compact ? tbr : 0;
    const int lo = t < N0 ? (int)(t - tbr) : 0;
    const double *row = G1 + t * ldg + tbr - coff;
    double mx = 0.0;
    for (int c = lane; c < lo; c += 32) mx = fmax(mx, fabs(row[c]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    int ex = 0;
    if (mx > 0.0 && isfinite(mx)) frexp(mx, &ex);
    if (lane == 0) e[t] = ex;
    const double scale = ldexp(1.0, 8 * S - 2 - ex);
    for (int c0 = lane * 16; c0 < (int)R; c0 += 512) {
        uint32_t packed[S][4];
#pragma unroll
        for (int k = 0; k < S; ++k) packed[k][0] = packed[k][1] = packed[k][2] = packed[k][3] = 0u;
        if (c0 < lo) {
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const double x = (c0 + c < lo) ? row[c0 + c] : 0.0;
                long long v = __double2ll_rn(x * scale);
#pragma unroll
                for (int k = S - 1; k >= 0; --k) {
                    const int dg = (int)((v + 128) & 255) - 128;
                    v = (v - dg) >> 8;
                    packed[k][c >> 2] |= ((uint32_t)(dg & 0xff)) << (8 * (c & 3));
                }
            }
        }
#pragma unroll
        for (int k = 0; k < S; ++k)
            *reinterpret_cast<uint4 *>(slices + sl_offset(c0, k, t, N0P, S)) = make_uint4(packed[k][0], packed[k][1], packed[k][2], packed[k][3]);
    }
}

// G1m[t][c] = G1[t][tb(t) + c] for c < t - tb(t), else 0: the strictly lower part of every range's G1 tile, compact (row stride R), fp64
// -- the B operand of the same product on the fp64 pipe (Gram-row form of the sweep, gemm_nt.cuh)
__global__ void stc_mask_g1_lower_kernel(const double *__restrict__ G1, int64_t ldg, int64_t N0, int64_t N0P, int64_t R,
                                         double *__restrict__ G1m) {
    const int64_t t = blockIdx.x;
    const int64_t tbr = (t / R) * R;
    const int lo = t < N0 ? (int)(t - tbr) : 0;
    for (int c = threadIdx.x; c < (int)R; c += blockDim.x) G1m[t * R + c] = c < lo ? G1[t * ldg + tbr + c] : 0.0;
}

// P[j][tb + c] += Do[j][c] (what the earlier ranges contribute, from the Gram-row contraction) for c < n
__global__ void stc_add_outer_kernel(double *__restrict__ P, int64_t ldp, const double *__restrict__ Do, int64_t ldd, int64_t nj, int n) {
    const int64_t j = blockIdx.x;
    if (j >= nj) return;
    for (int c = threadIdx.x; c < n; c += blockDim.x) P[j * ldp + c] += Do[j * ldd + c];
}

// P[j][c] += sum of ns partial results part[k][j][c] (K split of the residual dots over batches), in index order
__global__ void stc_add_partials_kernel(double *__restrict__ P, int64_t ldp, const double *__restrict__ part, int ns, int64_t stride,
                                        int64_t ldd, int64_t nj, int n) {
    const int64_t j = blockIdx.x;
    for (int c = threadIdx.x; c < n; c += blockDim.x) {
        double s = part[j * ldd + c];
        for (int k = 1; k < ns; ++k) s += part[(int64_t)k * stride + j * ldd + c];
        P[j * ldp + c] += s;
    }
}

// Qt[j][t] = the level of index Kq[j][t] for the directions [tb, te): the neuron-major fp64 decisions the Gram-row contraction of the
// later ranges reads
// (scales, per-channel alphabets: neuron j's levels are fl(scales[j] levels[k]))
template <bool SCALED>
__global__ void stc_qt_from_kq_kernel(const int8_t *__restrict__ Kq, int64_t krows, int64_t tb, int64_t te, int64_t nj,
                                      const double *__restrict__ levels, int K, double *__restrict__ Qt, int64_t ldq,
                                      const double *__restrict__ scales) {
    const int64_t j = blockIdx.x;
    const double s = SCALED ? scales[j] : 1.0;
    for (int64_t t = tb + threadIdx.x; t < te; t += blockDim.x) {
        const int k = Kq[sl_offset(t, 0, j, krows, 1)];
        const double lv = SCALED ? __dmul_rn(s, levels[(k + K - 1) >> 1]) : levels[(k + K - 1) >> 1];
        Qt[j * ldq + t] = k == 0 ? 0.0 : lv;
    }
}

// Wn[j][t] = W[t * ldw + wcol0 + j] (fp32, neuron-major, N0P columns, zeros beyond N0): what a walker thread copies per block
__global__ void stc_weights_kernel(const float *__restrict__ W, int64_t ldw, int64_t wcol0, int64_t N0, int64_t N0P, int64_t nj,
                                   float *__restrict__ Wn) {
    __shared__ float tile[32][33];
    const int64_t tb = (int64_t)blockIdx.x * 32, jb = (int64_t)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t t = tb + r, j = jb + threadIdx.x;
        tile[r][threadIdx.x] = (t < N0 && j < nj) ? W[t * ldw + wcol0 + j] : 0.f;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t j = jb + r, t = tb + threadIdx.x;
        if (j < nj && t < N0P) Wn[j * N0P + t] = tile[threadIdx.x][r];
    }
}

// Q[t * ldq + col0 + j] = level of index Kq[j][t] (k' = 2 k - (K - 1); the literal 0 for k' = 0): the layer's quantized weights from
// the level indices of the walk -- the stored levels themselves, bit for bit
template <bool SCALED>
__global__ void stc_q_from_kq_kernel(const int8_t *__restrict__ Kq, int64_t krows, int64_t N0, int64_t nj, const double *__restrict__ levels,
                                     int K, double *__restrict__ Q, int64_t ldq, int64_t col0, const double *__restrict__ scales) {
    __shared__ int8_t tile[32][33];
    const int64_t tb = (int64_t)blockIdx.x * 32, jb = (int64_t)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t j = jb + r, t = tb + threadIdx.x;
        tile[r][threadIdx.x] = (j < nj && t < N0) ? Kq[sl_offset(t, 0, j, krows, 1)] : (int8_t)0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t t = tb + r, j = jb + threadIdx.x;
        if (t < N0 && j < nj) {
            const int k = tile[threadIdx.x][r];
            const double lv = SCALED ? __dmul_rn(scales[j], levels[(k + K - 1) >> 1]) : levels[(k + K - 1) >> 1];
            Q[t * ldq + col0 + j] = k == 0 ? 0.0 : lv;
        }
    }
}
}  // namespace stc

// ---- host side -------------------------------------------------------------------------------------------------
int sweep_tc_prepare(gpfq_ctx *ctx, const double *G1, const double *G2, int64_t ldg, bool compact, int64_t N0, int64_t N0P, int64_t R,
                     double h, TcTables *out) {
    using namespace stc;
    if (R % KB || R > MAX_R || N0P % R || N0P < N0) return gpfq_fail(ctx, GPFQ_ERR_ARG, "sweep_tc: ranges of 64 .. %d directions", MAX_R);
    TabA *tabs = nullptr;
    int8_t *g2s = nullptr;
    const int64_t nblk = N0P / NB;
    GPFQ_TRY(gpfq_ws(ctx, WS_TC_TAB, (size_t)nblk * sizeof(TabA), (void **)&tabs));
    GPFQ_TRY(gpfq_ws(ctx, WS_TC_G2S, (size_t)nblk * (size_t)(R / KB) * B_STAGE, (void **)&g2s));
    stc_prepare_kernel<<<(unsigned)nblk, 256, 0, ctx->stream>>>(G1, G2, ldg, compact ? 1 : 0, N0, R, h, tabs, g2s);
    KERNEL_CHECK(ctx);
    out->tabs = tabs;
    out->g2s = g2s;
    out->R = R;
    return GPFQ_OK;
}

int sweep_tc_slice_g1_lower(gpfq_ctx *ctx, const double *G1, int64_t ldg, bool compact, int64_t N0, int64_t N0P, int64_t R, int32_t *e,
                            int8_t *slices) {
    stc::stc_slice_g1_lower_kernel<<<(unsigned)ceil_div64(N0P, 8), 256, 0, ctx->stream>>>(G1, ldg, compact ? 1 : 0, N0, N0P, R, e, slices);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

int sweep_tc_weights(gpfq_ctx *ctx, const float *W, int64_t ldw, int64_t wcol0, int64_t N0, int64_t N0P, int64_t nj, float *Wn) {
    dim3 grid((unsigned)ceil_div64(N0P, 32), (unsigned)ceil_div64(nj, 32));
    stc::stc_weights_kernel<<<grid, dim3(32, 8), 0, ctx->stream>>>(W, ldw, wcol0, N0, N0P, nj, Wn);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

int sweep_tc_mask_g1_lower(gpfq_ctx *ctx, const double *G1, int64_t ldg, int64_t N0, int64_t N0P, int64_t R, double *G1m) {
    stc::stc_mask_g1_lower_kernel<<<(unsigned)N0P, 128, 0, ctx->stream>>>(G1, ldg, N0, N0P, R, G1m);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

int sweep_tc_add_outer(gpfq_ctx *ctx, double *P, int64_t ldp, const double *Do, int64_t ldd, int64_t nj, int64_t n) {
    stc::stc_add_outer_kernel<<<(unsigned)nj, 128, 0, ctx->stream>>>(P, ldp, Do, ldd, nj, (int)n);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

int sweep_tc_add_partials(gpfq_ctx *ctx, double *P, int64_t ldp, const double *part, int ns, int64_t stride, int64_t ldd, int64_t nj,
                          int64_t n) {
    stc::stc_add_partials_kernel<<<(unsigned)nj, 128, 0, ctx->stream>>>(P, ldp, part, ns, stride, ldd, nj, (int)n);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

int sweep_tc_qt_from_kq(gpfq_ctx *ctx, const int8_t *Kq, int64_t krows, int64_t tb, int64_t te, int64_t nj, const double *levels, int K,
                        double *Qt, int64_t ldq, const double *scales) {
    if (scales) stc::stc_qt_from_kq_kernel<true><<<(unsigned)nj, 128, 0, ctx->stream>>>(Kq, krows, tb, te, nj, levels, K, Qt, ldq, scales);
    else stc::stc_qt_from_kq_kernel<false><<<(unsigned)nj, 128, 0, ctx->stream>>>(Kq, krows, tb, te, nj, levels, K, Qt, ldq, nullptr);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

int sweep_tc_q_from_kq(gpfq_ctx *ctx, const int8_t *Kq, int64_t krows, int64_t N0, int64_t nj, const double *levels, int K, double *Q,
                       int64_t ldq, int64_t col0, const double *scales) {
    dim3 grid((unsigned)ceil_div64(N0, 32), (unsigned)ceil_div64(nj, 32));
    if (scales) stc::stc_q_from_kq_kernel<true><<<grid, dim3(32, 8), 0, ctx->stream>>>(Kq, krows, N0, nj, levels, K, Q, ldq, col0, scales);
    else stc::stc_q_from_kq_kernel<false><<<grid, dim3(32, 8), 0, ctx->stream>>>(Kq, krows, N0, nj, levels, K, Q, ldq, col0, nullptr);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}

// Tensor maps of P (rowsP, ldp) fp64 and Wn (rowsP, ldp) fp32: boxes of 128 neurons x 128 bytes, 128B swizzle
int sweep_tc_bind(gpfq_ctx *ctx, TcTables *tab, const double *P, const float *Wn, int64_t rowsP, int64_t ldp) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return gpfq_fail(ctx, GPFQ_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled is not available from this driver");
    if (rowsP % stc::NT || ldp % stc::NB || ((uintptr_t)P & 15) || ((uintptr_t)Wn & 15))
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "sweep_tc: P / Wn are padded to 128 neurons and whole blocks of directions");
    const cuuint64_t dims[2] = {(cuuint64_t)ldp, (cuuint64_t)rowsP};
    const cuuint32_t estr[2] = {1u, 1u};
    {
        const cuuint64_t strides[1] = {(cuuint64_t)ldp * sizeof(double)};
        const cuuint32_t box[2] = {(cuuint32_t)(stc::NB / 2), (cuuint32_t)stc::NT};
        const CUresult rc = enc(&tab->mapP, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(P), dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (rc != CUDA_SUCCESS) return gpfq_fail(ctx, GPFQ_ERR_CUDA, "cuTensorMapEncodeTiled (P) failed with code %d", (int)rc);
    }
    {
        const cuuint64_t strides[1] = {(cuuint64_t)ldp * sizeof(float)};
        const cuuint32_t box[2] = {(cuuint32_t)stc::NB, (cuuint32_t)stc::NT};
        const CUresult rc = enc(&tab->mapW, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(Wn), dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (rc != CUDA_SUCCESS) return gpfq_fail(ctx, GPFQ_ERR_CUDA, "cuTensorMapEncodeTiled (Wn) failed with code %d", (int)rc);
    }
    tab->rowsP = rowsP;
    return GPFQ_OK;
}

int sweep_tc_range(gpfq_ctx *ctx, const TcTables &tab, int64_t tb, int64_t te, int64_t row0, int64_t nj, int8_t *Kq, int64_t krows,
                   int64_t krow0, double a, const double *levels, int K, const double *scales, int64_t u0) {
    using namespace stc;
    if (tb % tab.R || te - tb > tab.R || te <= tb || row0 % NT || row0 + ceil_div64(nj, NT) * NT > tab.rowsP || !Kq || K < 2 || K > 128)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "sweep_tc: a range starts at a multiple of %lld directions", (long long)tab.R);
    const dim3 grid((unsigned)ceil_div64(nj, NT));
    if (const double *lambdas = ctx->d_l1) {   // L1 penalty: one alphabet on this path, lambdas[0]
        const uint64_t *seeds = ctx->d_seeds;
        auto k = K == 3 ? (scales ? sweep_tc_kernel<true, true, false, true> : sweep_tc_kernel<true, false, false, true>)
                        : (scales ? sweep_tc_kernel<false, true, false, true> : sweep_tc_kernel<false, false, false, true>);
        if (seeds)
            k = K == 3 ? (scales ? sweep_tc_kernel<true, true, true, true> : sweep_tc_kernel<true, false, true, true>)
                       : (scales ? sweep_tc_kernel<false, true, true, true> : sweep_tc_kernel<false, false, true, true>);
        CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        k<<<grid, THREADS, SMEM, ctx->stream>>>(tab.mapP, tab.mapW, tab.tabs, tab.g2s, (int)(tab.R / KB), tb, te, (int)row0, nj, Kq, krows, krow0,
                                                a, levels, K, scales, seeds, u0, lambdas);
    } else if (const uint64_t *seeds = ctx->d_seeds) {   // stochastic rounding: one alphabet on this path, seeds[0]
        auto k = K == 3 ? (scales ? sweep_tc_kernel<true, true, true> : sweep_tc_kernel<true, false, true>)
                        : (scales ? sweep_tc_kernel<false, true, true> : sweep_tc_kernel<false, false, true>);
        CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        k<<<grid, THREADS, SMEM, ctx->stream>>>(tab.mapP, tab.mapW, tab.tabs, tab.g2s, (int)(tab.R / KB), tb, te, (int)row0, nj, Kq, krows, krow0,
                                                a, levels, K, scales, seeds, u0, nullptr);
    } else if (scales) {
        auto k = K == 3 ? sweep_tc_kernel<true, true> : sweep_tc_kernel<false, true>;
        CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        k<<<grid, THREADS, SMEM, ctx->stream>>>(tab.mapP, tab.mapW, tab.tabs, tab.g2s, (int)(tab.R / KB), tb, te, (int)row0, nj, Kq, krows, krow0,
                                                a, levels, K, scales, nullptr, 0, nullptr);
    } else if (K == 3) {
        CUDA_TRY(ctx, cudaFuncSetAttribute(sweep_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        sweep_tc_kernel<true><<<grid, THREADS, SMEM, ctx->stream>>>(tab.mapP, tab.mapW, tab.tabs, tab.g2s, (int)(tab.R / KB), tb, te, (int)row0, nj,
                                                                    Kq, krows, krow0, a, levels, K);
    } else {
        CUDA_TRY(ctx, cudaFuncSetAttribute(sweep_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        sweep_tc_kernel<false><<<grid, THREADS, SMEM, ctx->stream>>>(tab.mapP, tab.mapW, tab.tabs, tab.g2s, (int)(tab.R / KB), tb, te, (int)row0, nj,
                                                                     Kq, krows, krow0, a, levels, K);
    }
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}
