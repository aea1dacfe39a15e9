// conv_corr.cu -- 3x3 / stride 1 / 'SAME' conv layers: per-channel Grams as shifted correlations of the activations.
//
// What the walk of _quantize_filter2D_parallel_jit (quantized_network.py:219-228) consumes per channel are the 9 x 9
// matrices G1[t,s] = <Xq_t, X_s>, G2[t,s] = <Xq_t, Xq_s> (s <= t) of the channel's patch matrix (:789-797, one row per
// tap t = r*3 + c, one column per output pixel p, entry = pixel p + tap - 1 of the zero-padded image).  Substituting
// the pixel s = p + a - 1 that tap a reads:
//
//     G[a, b] = sum over pixels s of  xq[s] * x[s + (b - a)]   restricted to  s - a + 1 inside the image,
//
// i.e. the correlation of the channel image with itself at displacement d = b - a, over all pixels s except ONE border
// row and/or ONE border column (tap row 0 never reads the bottom image row as its own pixel, tap row 2 never the top
// row; columns alike).  For s <= t the displacement is lexicographically <= 0: only 13 displacements exist, so a pixel
// costs 13 exact-product fp64 FMAs per Gram instead of the 81 + 45 of the patch form (126 useful MACs, 168 fp64-pipe
// slots in conv_gram9_nhwc_kernel).  The pixels s are split into nine disjoint regions -- {top row, rows between,
// bottom row} x {left column, columns between, right column} -- whose 13 sums are kept apart and ADDED per (a, b) for
// the regions tap a may sit on.  No subtraction anywhere: a tap direction that only ever reads zeros (a dead channel,
// an image with black margins) gets an exactly zero Gram row, as in the patch form, so the dead-direction guard of
// quantized_network.py:83-84 fires identically.  Sums are exact fp32 x fp32 products accumulated in fp64 in a fixed
// order (tasks per warp in index order, warps in index order): bit-reproducible, and equal to the patch form up to fp64
// re-association (1e-16 relative; the parity budget is 1e-9, SURVEY.md App. C).
//
//   conv_corr9_tma_kernel<RB, BOTH>  lane = channel (NHWC: 32 channels = one 128-byte line per pixel); a warp walks a band
//                                  of RB image rows left to right with a rotating 5-column fp64 register window of xq and
//                                  13 accumulators per lane and Gram.  Operands arrive by TMA (cp.async.bulk.tensor.4d over
//                                  the (N, H, W, C) tensor, zero fill outside the image = the 'SAME' padding) into a
//                                  per-warp mbarrier ring; the warp is its own producer (lane 0 issues the next box before
//                                  multiplying the current one).  X~ == X: G2 = xq x xq from (RB+2)-row windows.  BOTH
//                                  (X~ != X): G1 and G2 in ONE pass.  Substituting t = s + d in G1 makes it
//                                      G1[a, b] = sum over pixels t of  x[t] * xq[t - d],   -d lexicographically >= 0,
//                                  restricted to t - b + 1 inside the image: x centre times the xq window at and BELOW it,
//                                  while G2 is xq centre times the xq window at and ABOVE it.  Both read one (RB+4)-row
//                                  window of xq plus the RB x 5 centre pixels of x: 26 DFMA and (RB+4)/RB + 1 fp32 -> fp64
//                                  conversions per pixel, 8 B per pixel and channel from HBM.  G1's records are split by
//                                  the region of the x pixel t, the assembly adds for G1[a, b] the regions of tap b.  The
//                                  first and the last pixel column of a band go to the left / right region records.  One
//                                  launch covers rows 1 .. H-2 (RB in {8, 6, 4}; {6, 4} with BOTH), one with RB = 1 the top
//                                  and bottom rows.
//   conv_corr9_strip_kernel<SW, RB, CROSS>  the same sums on images 14-64 pixels wide as whole strips of <= 16 columns, in
//                                  two launches (CROSS: xq centre x x window, G1 records split by the xq pixel)
//   conv_corr9_strip1_kernel<SW, RB>  both Grams in one pass on strips, the band kernel's form; picked by width (8 pixels)
//   conv_corr9_assemble_kernel     fixed-order slot sums + the per-tap region sums -> [G1 | G2] per channel in the
//                                  layout conv_sweep_kernel reads
//   corr9_pack_kernel              channel counts a tensor map cannot serve (C < 32, C % 4 != 0) on large images: G images
//                                  side by side as virtual channels of an ordinary tensor; the assembly adds their records
// Images smaller than a box (H < 6 or W < 5) and, by measurement, images below 128 pixels keep the patch form (the
// planner is in gpfq_conv_layer_nhwc, api.cu).
#include <cuda.h>

#include <algorithm>

#include "common.cuh"

namespace corr9 {
constexpr int ND = 13;        // displacements (dy, dx): dy in {-2, -1} x dx in [-2, 2], then dy = 0 x dx in {-2, -1, 0}
constexpr int WARPS = 4;      // warps (tasks in flight) per CTA
constexpr int WC = 5;         // columns per TMA box = phases of the rotating register window
constexpr int REC = 6 * ND;   // doubles per (channel, slot): [pass: cross, auto][pixel column: first, between, last][13]
}  // namespace corr9

struct Corr9Geom {
    int H, W;
    int64_t c_first;   // first channel of this launch
    int n_ch;          // channels of this launch
    int64_t img0, n_img;
    int slots;         // warps per channel group in this launch
    int y_first, y_last;  // pixel rows this launch covers; band b of an image starts at y_first + b * RB
    int two_rows;      // RB = 1 launch over the top and the bottom row: odd slots take y = y_last, even slots y = y_first
};

// ---- TMA-fed variant ---------------------------------------------------------------------------------------------
namespace corr9 {
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n.reg .pred p;\nWAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// box of the (C, W, H, N) tensor at (channel c, column x, row y, image n); coordinates outside the tensor read zeros
__device__ __forceinline__ void tma_load_4d(void *dst, const CUtensorMap *map, uint64_t *bar, int c, int x, int y, int n) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::"r"(
            smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c), "r"(x), "r"(y), "r"(n)
        : "memory");
}
template <int RB, bool BOTH>
struct Ring {
    static constexpr int NS = BOTH ? 2 : 3;                  // boxes in flight per warp
    static constexpr int WR = BOTH ? RB + 4 : RB + 2;        // window rows: two above the band, and two below it for G1
    static constexpr int B_FLOATS = WR * WC * 32;            // xq window: WR rows x 5 columns x 32 channels
    static constexpr int A_FLOATS = BOTH ? RB * WC * 32 : 0;  // x centre pixels, two columns behind
    static constexpr int STAGE_FLOATS = B_FLOATS + A_FLOATS;
    static constexpr size_t WARP_BYTES = (size_t)NS * STAGE_FLOATS * sizeof(float);
    static constexpr size_t SMEM = WARPS * WARP_BYTES + WARPS * NS * sizeof(uint64_t);
};
// One pixel row i of the band into the 13 sums `o`; the window's logical column L (pixel column - 2 + L) sits in physical slot
// (ph + 1 + L) % 5.  G2: xq centre x the xq window at the displacements d (lexicographically <= 0) above it.  G1: x centre x
// the xq window at -d, below it -- the point reflection of the G2 pattern through the centre (row i + 2 + r <-> i + 2 - r,
// column 2 + c <-> 2 - c), so that G1 reads the same window as G2 and lands in the same 13 displacement slots.
template <int WR>
__device__ __forceinline__ void mac_g2(double a, const double (&win)[WR][5], int i, int ph, double (&o)[ND]) {
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 5; ++dx) o[dy * 5 + dx] = fma(a, win[i + dy][(ph + 1 + dx) % 5], o[dy * 5 + dx]);
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) o[10 + dx] = fma(a, win[i + 2][(ph + 1 + dx) % 5], o[10 + dx]);
}
template <int WR>
__device__ __forceinline__ void mac_g1(double a, const double (&win)[WR][5], int i, int ph, double (&o)[ND]) {
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 5; ++dx) o[dy * 5 + dx] = fma(a, win[i + 4 - dy][(ph + 5 - dx) % 5], o[dy * 5 + dx]);
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) o[10 + dx] = fma(a, win[i + 2][(ph + 5 - dx) % 5], o[10 + dx]);
}
}  // namespace corr9

template <int RB, bool BOTH>
__global__ void __launch_bounds__(corr9::WARPS * 32, (RB <= 4 && !BOTH) || RB == 1 ? 3 : 2)
conv_corr9_tma_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapX, Corr9Geom gm,
                      double *__restrict__ partial, int slot_stride, int slot0) {
    using namespace corr9;
    using R = Ring<RB, BOTH>;
    constexpr int NS = R::NS, WR = R::WR;
    extern __shared__ __align__(128) unsigned char corr9_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x * WARPS + warp;
    // a box must start on a 16-byte boundary: channel groups start at c_first rounded down to a multiple of four
    const int c0 = (int)(gm.c_first & ~(int64_t)3) + (int)blockIdx.y * 32;
    const int chl = c0 + lane - (int)gm.c_first;  // channel index inside this launch's range
    const bool chok = chl >= 0 && chl < gm.n_ch;
    float *ring = reinterpret_cast<float *>(corr9_smem + warp * R::WARP_BYTES);
    uint64_t *bars = reinterpret_cast<uint64_t *>(corr9_smem + WARPS * R::WARP_BYTES) + warp * NS;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncwarp();
    const int W = gm.W;
    const int nrows = gm.y_last - gm.y_first + 1;
    const int nbands = gm.two_rows ? 1 : (nrows + RB - 1) / RB;
    // two_rows: this warp's images are slot / 2, slot / 2 + slots / 2, ...; its row is fixed by the slot's parity
    const int64_t ntasks = gm.two_rows ? gm.n_img : gm.n_img * nbands;
    const int64_t t_first = gm.two_rows ? slot / 2 : slot, t_step = gm.two_rows ? gm.slots / 2 : gm.slots;
    const int nstages = (W + 2 + WC - 1) / WC;
    // this lane's record: [pass: G1, G2][first column | between | last column][13]; first / last are read-modify-written in
    // task order by this lane only (the API zeroes the records), `between` is stored once at the end
    double *rec = partial + ((size_t)(chok ? chl : 0) * slot_stride + slot0 + slot) * REC;
    uint32_t it = 0;  // boxes this warp has consumed so far: ring position and mbarrier parity
    double acc[ND], acc1[ND];   // G2, G1 (BOTH)
#pragma unroll
    for (int d = 0; d < ND; ++d) acc[d] = acc1[d] = 0.0;

    // The boxes of this warp's tasks form one stream (task after task, columns left to right); the producer cursor runs
    // NS - 1 boxes ahead of the consumer, across task boundaries, so a new band never starts with an empty ring.
    // (image, band) of a task advance by a fixed step from one task of this warp to its next: no division in the loops
    const int step_img = (int)(gm.two_rows ? t_step : t_step / nbands), step_band = gm.two_rows ? 0 : (int)(t_step % nbands);
    const int img_first = (int)(gm.img0 + (gm.two_rows ? t_first : t_first / nbands));
    const int band_first = gm.two_rows ? 0 : (int)(t_first % nbands);
    const int row_fixed = (slot & 1) ? gm.y_last : gm.y_first;   // two_rows: this warp's row
    int64_t ptask = t_first;
    int pk = 0, pimg = img_first, pband = band_first;
    uint32_t ppos = 0;
    auto produce = [&]() {
        if (ptask < ntasks) {
            if (lane == 0) {
                const int py0 = gm.two_rows ? row_fixed : gm.y_first + pband * RB;
                const int s = (int)(ppos % NS);
                float *dst = ring + s * R::STAGE_FLOATS;
                mbar_expect_tx(&bars[s], (uint32_t)(R::STAGE_FLOATS * sizeof(float)));
                tma_load_4d(dst, &mapQ, &bars[s], c0, pk * WC, py0 - 2, pimg);
                if (BOTH) tma_load_4d(dst + R::B_FLOATS, &mapX, &bars[s], c0, pk * WC - 2, py0, pimg);
            }
            ++ppos;
            if (++pk == nstages) {
                pk = 0;
                ptask += t_step;
                pimg += step_img;
                pband += step_band;
                if (pband >= nbands) { pband -= nbands; ++pimg; }
            }
        }
    };
#pragma unroll
    for (int p = 0; p < NS - 1; ++p) produce();

    int cband = band_first;
    for (int64_t task = t_first; task < ntasks; task += t_step) {
        const int y0 = gm.two_rows ? row_fixed : gm.y_first + cband * RB;
        cband += step_band;
        if (cband >= nbands) cband -= nbands;
        unsigned rowmask = 0;  // bit i: pixel row y0 + i belongs to this launch
#pragma unroll
        for (int i = 0; i < RB; ++i) rowmask |= (y0 + i <= gm.y_last) ? (1u << i) : 0u;
        const bool allrows = rowmask == (1u << RB) - 1u;
        double win[WR][5];
        double ac[RB];
        (void)ac;
#pragma unroll
        for (int r = 0; r < WR; ++r)
#pragma unroll
            for (int c = 0; c < 5; ++c) win[r][c] = 0.0;
        for (int k = 0; k < nstages; ++k) {
            __syncwarp();  // the box consumed in the previous iteration is free again
            produce();
            const uint32_t pos = it + k;
            const int s = (int)(pos % NS);
            mbar_wait(&bars[s], (pos / NS) & 1u);
            const float *tb = ring + s * R::STAGE_FLOATS + lane;
            const float *ta = tb + R::B_FLOATS;
            if (allrows && k >= 1 && k * WC + WC - 1 <= W) {
                // ---- five pixel columns strictly between the first and the last one, every row live: branch-free
#pragma unroll
                for (int ph = 0; ph < WC; ++ph) {
#pragma unroll
                    for (int r = 0; r < WR; ++r) win[r][ph] = (double)tb[(r * WC + ph) * 32];
                    if (BOTH) {
#pragma unroll
                        for (int i = 0; i < RB; ++i) ac[i] = (double)ta[(i * WC + ph) * 32];
                    }
#pragma unroll
                    for (int i = 0; i < RB; ++i) {
                        mac_g2(win[i + 2][(ph + 3) % 5], win, i, ph, acc);
                        if (BOTH) mac_g1(ac[i], win, i, ph, acc1);
                    }
                }
            } else {
                // ---- band ends, ragged last band: one column at a time into `e`, then to the record it belongs to.  The raw
                // fp32 values of a column are read from the box one column ahead (the branches between the columns keep the
                // compiler from hoisting the loads itself, and LDS -> F2F -> DFMA back to back is all latency: ncu, conv10)
                float rawb[WR], rawa[RB];
                (void)rawa;
                auto fetch = [&](int ph) {
#pragma unroll
                    for (int r = 0; r < WR; ++r) rawb[r] = tb[(r * WC + ph) * 32];
                    if (BOTH) {
#pragma unroll
                        for (int i = 0; i < RB; ++i) rawa[i] = ta[(i * WC + ph) * 32];
                    }
                };
                fetch(0);
#pragma unroll
                for (int ph = 0; ph < WC; ++ph) {
                    const int cx = k * WC + ph;  // newest window column (image column cx) lives in physical slot ph
                    if (cx < W + 2) {
#pragma unroll
                        for (int r = 0; r < WR; ++r) win[r][ph] = (double)rawb[r];
                        if (BOTH) {
#pragma unroll
                            for (int i = 0; i < RB; ++i) ac[i] = (double)rawa[i];
                        }
                        if (ph + 1 < WC) fetch(ph + 1);   // inside the box even when that column lies past the image (zeros)
                        if (cx >= 2) {
                            // pixel column cx - 2 = logical window column 2 = physical slot (ph + 3) % 5; the first / last
                            // pixel column have their own records
                            const bool edge = cx == 2 || cx == W + 1;
                            double *o = rec + (cx == 2 ? 0 : 2 * ND);
#pragma unroll
                            for (int pass = BOTH ? 0 : 1; pass < 2; ++pass) {
                                double e[ND];
#pragma unroll
                                for (int d = 0; d < ND; ++d) e[d] = 0.0;
#pragma unroll
                                for (int i = 0; i < RB; ++i) {
                                    const bool live = (rowmask >> i) & 1u;
                                    if (pass == 1) mac_g2(live ? win[i + 2][(ph + 3) % 5] : 0.0, win, i, ph, e);
                                    else mac_g1(live ? ac[i] : 0.0, win, i, ph, e);
                                }
                                if (edge) {
                                    if (chok) {
                                        // fire-and-forget reductions (RED.ADD.F64): nothing waits for the round trip to L2;
                                        // only this lane ever touches the record, and its updates apply in program order
#pragma unroll
                                        for (int d = 0; d < ND; ++d) atomicAdd(o + pass * 3 * ND + d, e[d]);
                                    }
                                } else if (pass == 1) {
#pragma unroll
                                    for (int d = 0; d < ND; ++d) acc[d] += e[d];
                                } else {
#pragma unroll
                                    for (int d = 0; d < ND; ++d) acc1[d] += e[d];
                                }
                            }
                        }
                    }
                }
            }
        }
        it += (uint32_t)nstages;
    }
    if (chok) {
#pragma unroll
        for (int d = 0; d < ND; ++d) {
            rec[3 * ND + ND + d] = acc[d];
            if (BOTH) rec[ND + d] = acc1[d];
        }
    }
}


// ---- strip variant for small images (W in {8, 14, 16, 28, 32, 56, 64}) --------------------------------------------------
// The band walk above pays per band: a window reset, two edge stages of the four to six 5-column stages, reductions to global
// memory for the first / last pixel column -- on 28 x 28 images it runs at 0.27-0.34 of the DFMA rate, on 14 x 14 at 0.17
// (profiles/r1l_conv_corr9_vgg_conv10.md).  Here a task is a band of RB rows x a STRIP of SW <= 16 columns, fetched whole (one
// TMA box of (RB + 2) x (SW + 4) pixels x 32 channels, zero fill outside the image = the padding, plus the RB x SW centre pixels
// of xq for the xq x x pass) and walked as straight-line code: the column index is a compile-time constant, so the rotating
// register window, the column class (first / between / last pixel column) and every shared-memory offset are static, there are
// no edge stages and the three column classes are three register accumulator sets stored once per warp.  G1 and G2 stay two
// launches here: one pass would need the (RB + 4)-row window and 3 x 26 accumulators, past what fits in registers at this occupancy.  W = 28 / 32 are two
// strips (the inner strip boundary is an ordinary "between" column: the halo columns hold real pixels).  Same records as the
// band kernel (conv_corr9_assemble_kernel reads both), same exact products, fixed summation order.
namespace corr9s {
using corr9::ND;
using corr9::REC;
constexpr int WARPS = 4;      // warps per CTA
// boxes per warp: ONE for the bands of four rows -- a strip box is 15-24 KB, and two to three warps per SM sub-partition that take turns
// (one waits for its box while another multiplies) measured faster than one warp that double-buffers; the one-row tasks of the top /
// bottom rows (7-9 KB boxes, 182-208 DFMAs each) keep two in flight
template <int RB> struct Boxes { static constexpr int NS = RB == 1 ? 2 : 1; };
template <int SW, int RB, bool CROSS>
struct Cfg {
    static constexpr int BW = SW + 4;                                  // box columns: the strip and two halo columns either side
    static constexpr int WIN_FLOATS = (RB + 2) * BW * 32;
    static constexpr int CTR_FLOATS = CROSS ? RB * SW * 32 : 0;
    static constexpr int STAGE_FLOATS = WIN_FLOATS + CTR_FLOATS;
    static constexpr int NS = Boxes<RB>::NS;
    static constexpr size_t WARP_BYTES = (size_t)NS * STAGE_FLOATS * sizeof(float);
    static constexpr size_t SMEM = WARPS * WARP_BYTES + WARPS * NS * sizeof(uint64_t);
};
}  // namespace corr9s

template <int SW, int RB, bool CROSS>
__global__ void __launch_bounds__(corr9s::WARPS * 32)
conv_corr9_strip_kernel(const __grid_constant__ CUtensorMap mapWin, const __grid_constant__ CUtensorMap mapCtr, Corr9Geom gm,
                        double *__restrict__ partial, int slot_stride, int slot0) {
    using namespace corr9s;
    using corr9::mbar_expect_tx;
    using corr9::mbar_init;
    using corr9::mbar_wait;
    using corr9::tma_load_4d;
    using C = Cfg<SW, RB, CROSS>;
    constexpr int BW = C::BW, NS = C::NS;
    extern __shared__ __align__(128) unsigned char corr9_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x * WARPS + warp;
    const int c0 = (int)(gm.c_first & ~(int64_t)3) + (int)blockIdx.y * 32;
    const int chl = c0 + lane - (int)gm.c_first;
    const bool chok = chl >= 0 && chl < gm.n_ch;
    float *ring = reinterpret_cast<float *>(corr9_smem + warp * C::WARP_BYTES);
    uint64_t *bars = reinterpret_cast<uint64_t *>(corr9_smem + WARPS * C::WARP_BYTES) + warp * NS;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncwarp();
    const int nstrips = gm.W / SW;
    const int nrows = gm.y_last - gm.y_first + 1;
    const int nbands = gm.two_rows ? 1 : (nrows + RB - 1) / RB;
    const int per_img = nbands * nstrips;                    // tasks of an image: (band, strip) pairs, strip fastest
    const int64_t ntasks = gm.n_img * per_img;               // two_rows: the (image, strip) pairs of this slot's row
    const int64_t t_first = gm.two_rows ? slot / 2 : slot, t_step = gm.two_rows ? gm.slots / 2 : gm.slots;
    const int row_fixed = (slot & 1) ? gm.y_last : gm.y_first;
    // (image, position inside the image) of a task advance by a fixed step from one task of this warp to its next: no division in
    // the loop
    const int step_img = (int)(t_step / per_img), step_in = (int)(t_step % per_img);
    auto fetch = [&](int img, int in, uint32_t pos) {        // lane 0: the box(es) of task (img, in) into ring position pos
        const int band = in / nstrips, strip = in - band * nstrips;   // small 32-bit division
        const int y0 = gm.two_rows ? row_fixed : gm.y_first + band * RB, x0 = strip * SW;
        const int s = (int)(pos % NS);
        float *dst = ring + s * C::STAGE_FLOATS;
        mbar_expect_tx(&bars[s], (uint32_t)(C::STAGE_FLOATS * sizeof(float)));
        tma_load_4d(dst, &mapWin, &bars[s], c0, x0 - 2, y0 - 2, img);
        if (CROSS) tma_load_4d(dst + C::WIN_FLOATS, &mapCtr, &bars[s], c0, x0, y0, img);
    };
    double acc[ND], accF[ND], accL[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) acc[d] = accF[d] = accL[d] = 0.0;
    int img = (int)(gm.img0 + t_first / per_img), in = (int)(t_first % per_img);
    if (t_first < ntasks && lane == 0) fetch(img, in, 0);
    uint32_t pos = 0;
    for (int64_t task = t_first; task < ntasks; task += t_step, ++pos) {
        int nimg = img + step_img, nin = in + step_in;       // this warp's next task
        if (nin >= per_img) { nin -= per_img; ++nimg; }
        if (NS > 1) {
            __syncwarp();      // the box consumed two tasks ago is free again
            if (task + t_step < ntasks && lane == 0) fetch(nimg, nin, pos + 1);
        }
        const int band = in / nstrips, strip = in - band * nstrips;
        const int y0 = gm.two_rows ? row_fixed : gm.y_first + band * RB;
        const bool left_edge = strip == 0, right_edge = strip == nstrips - 1;
        unsigned rowmask = 0;
#pragma unroll
        for (int i = 0; i < RB; ++i) rowmask |= (y0 + i <= gm.y_last) ? (1u << i) : 0u;
        const int s = (int)(pos % NS);
        mbar_wait(&bars[s], (pos / NS) & 1u);
        const float *tb = ring + s * C::STAGE_FLOATS + lane;
        const float *ta = tb + C::WIN_FLOATS;
        // The fp32 -> fp64 conversions run on the XU pipe at a quarter of the DFMA rate (8 cycles per warp instruction) and a warp issues
        // in order: converted right where they are needed they come in bursts that stall the DFMAs behind them (ncu: fp64 pipe 49 %,
        // XU 43 % active, not overlapping).  So the operands of column p + 1 are converted DURING column p, one or two per row of 13
        // DFMAs: a window of SIX physical columns (box column p + 5 goes to slot (p + 5) % 6 while slots p .. p + 4 are in use).
        double win[RB + 2][6];
        double ctr[RB], ctr_n[RB];
        (void)ctr;
        (void)ctr_n;
#pragma unroll
        for (int bc = 0; bc < 5; ++bc)
#pragma unroll
            for (int r = 0; r < RB + 2; ++r) win[r][bc] = (double)tb[(r * BW + bc) * 32];
        if (CROSS) {
#pragma unroll
            for (int i = 0; i < RB; ++i) ctr[i] = (double)ta[(i * SW) * 32];
        }
#pragma unroll
        for (int p = 0; p < SW; ++p) {   // pixel column x0 + p: window = box columns p .. p + 4, physical slots (p + k) % 6
            const bool edge = p == 0 || p == SW - 1;
            double e[ND];
            if (edge) {
#pragma unroll
                for (int d = 0; d < ND; ++d) e[d] = 0.0;
            }
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                double a = CROSS ? ctr[i] : win[i + 2][(p + 2) % 6];
                a = (rowmask >> i) & 1u ? a : 0.0;
                if (edge) {
#pragma unroll
                    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                        for (int dx = 0; dx < 5; ++dx) e[dy * 5 + dx] = fma(a, win[i + dy][(p + dx) % 6], e[dy * 5 + dx]);
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) e[10 + dx] = fma(a, win[i + 2][(p + dx) % 6], e[10 + dx]);
                } else {
#pragma unroll
                    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                        for (int dx = 0; dx < 5; ++dx) acc[dy * 5 + dx] = fma(a, win[i + dy][(p + dx) % 6], acc[dy * 5 + dx]);
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) acc[10 + dx] = fma(a, win[i + 2][(p + dx) % 6], acc[10 + dx]);
                }
                // the next column's operands: window rows i and i + RB (the latter for i < 2), centre pixel of row i
                if (p + 5 < BW) {
                    win[i][(p + 5) % 6] = (double)tb[(i * BW + p + 5) * 32];
                    if (i + RB < RB + 2) win[i + RB][(p + 5) % 6] = (double)tb[((i + RB) * BW + p + 5) * 32];
                    if (RB == 1) win[2][(p + 5) % 6] = (double)tb[(2 * BW + p + 5) * 32];
                }
                if (CROSS && p + 1 < SW) ctr_n[i] = (double)ta[(i * SW + p + 1) * 32];
            }
            if (CROSS) {
#pragma unroll
                for (int i = 0; i < RB; ++i) ctr[i] = ctr_n[i];
            }
            if (edge) {   // the image's first / last pixel column has its own class; a strip boundary inside the image does not
                const bool first = p == 0 && left_edge, last = p == SW - 1 && right_edge;
#pragma unroll
                for (int d = 0; d < ND; ++d) {
                    accF[d] += first ? e[d] : 0.0;
                    accL[d] += last ? e[d] : 0.0;
                    acc[d] += (first || last) ? 0.0 : e[d];
                }
            }
        }
        if (NS == 1) {
            __syncwarp();      // every lane has read the box: fetch the next one into it
            if (task + t_step < ntasks && lane == 0) fetch(nimg, nin, pos + 1);
        }
        img = nimg;
        in = nin;
    }
    if (chok) {
        double *rec = partial + ((size_t)chl * slot_stride + slot0 + slot) * REC + (CROSS ? 0 : 3 * ND);
#pragma unroll
        for (int d = 0; d < ND; ++d) {
            rec[d] = accF[d];
            rec[ND + d] = acc[d];
            rec[2 * ND + d] = accL[d];
        }
    }
}

// One pass for both Grams on strips (X~ != X): a box of RB + 4 rows of xq x (SW + 4) columns plus the RB x SW centre pixels of x
// per task; G2 = xq centre x the window above it, G1 = x centre x the window below it (conv_corr9_tma_kernel's mac_g1).  The
// columns between the first and the last one accumulate in registers (2 x 13 sums); 3 x 26 sums and the (RB + 4)-row window do not
// fit in registers, so the image's first / last pixel column add their sums to lane-private shared-memory records (plain
// read-add-write by the owning lane, in task order) that are stored once per warp like the register sums.
namespace corr9s {
template <int SW, int RB>
struct Cfg1 {
    static constexpr int BW = SW + 4, WR = RB + 4;
    static constexpr int WIN_FLOATS = WR * BW * 32;
    static constexpr int CTR_FLOATS = RB * SW * 32;
    static constexpr int STAGE_FLOATS = WIN_FLOATS + CTR_FLOATS;
    static constexpr int NS = Boxes<RB>::NS;
    static constexpr size_t WARP_BYTES = (size_t)NS * STAGE_FLOATS * sizeof(float);
    static constexpr size_t REC_BYTES = (size_t)2 * 2 * ND * 32 * sizeof(double);   // [first, last][G1, G2][13] x 32 lanes
    static constexpr size_t SMEM = WARPS * (WARP_BYTES + REC_BYTES) + WARPS * NS * sizeof(uint64_t);
};
}  // namespace corr9s

template <int SW, int RB>
__global__ void __launch_bounds__(corr9s::WARPS * 32)
conv_corr9_strip1_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapX, Corr9Geom gm,
                         double *__restrict__ partial, int slot_stride, int slot0) {
    using namespace corr9s;
    using corr9::mbar_expect_tx;
    using corr9::mbar_init;
    using corr9::mbar_wait;
    using corr9::tma_load_4d;
    using C = Cfg1<SW, RB>;
    constexpr int BW = C::BW, WR = C::WR, NS = C::NS;
    extern __shared__ __align__(128) unsigned char corr9_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x * WARPS + warp;
    const int c0 = (int)(gm.c_first & ~(int64_t)3) + (int)blockIdx.y * 32;
    const int chl = c0 + lane - (int)gm.c_first;
    const bool chok = chl >= 0 && chl < gm.n_ch;
    float *ring = reinterpret_cast<float *>(corr9_smem + warp * C::WARP_BYTES);
    double *srec = reinterpret_cast<double *>(corr9_smem + WARPS * C::WARP_BYTES + warp * C::REC_BYTES) + lane;  // [j * 32]
    uint64_t *bars = reinterpret_cast<uint64_t *>(corr9_smem + WARPS * (C::WARP_BYTES + C::REC_BYTES)) + warp * NS;
#pragma unroll
    for (int j = 0; j < 4 * ND; ++j) srec[j * 32] = 0.0;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncwarp();
    const int nstrips = gm.W / SW;
    const int nrows = gm.y_last - gm.y_first + 1;
    const int nbands = gm.two_rows ? 1 : (nrows + RB - 1) / RB;
    const int per_img = nbands * nstrips;
    const int64_t ntasks = gm.n_img * per_img;
    const int64_t t_first = gm.two_rows ? slot / 2 : slot, t_step = gm.two_rows ? gm.slots / 2 : gm.slots;
    const int row_fixed = (slot & 1) ? gm.y_last : gm.y_first;
    const int step_img = (int)(t_step / per_img), step_in = (int)(t_step % per_img);
    auto fetch = [&](int img, int in, uint32_t pos) {
        const int band = in / nstrips, strip = in - band * nstrips;
        const int y0 = gm.two_rows ? row_fixed : gm.y_first + band * RB, x0 = strip * SW;
        const int s = (int)(pos % NS);
        float *dst = ring + s * C::STAGE_FLOATS;
        mbar_expect_tx(&bars[s], (uint32_t)(C::STAGE_FLOATS * sizeof(float)));
        tma_load_4d(dst, &mapQ, &bars[s], c0, x0 - 2, y0 - 2, img);
        tma_load_4d(dst + C::WIN_FLOATS, &mapX, &bars[s], c0, x0, y0, img);
    };
    double acc1[ND], acc2[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) acc1[d] = acc2[d] = 0.0;
    int img = (int)(gm.img0 + t_first / per_img), in = (int)(t_first % per_img);
    if (t_first < ntasks && lane == 0) fetch(img, in, 0);
    uint32_t pos = 0;
    for (int64_t task = t_first; task < ntasks; task += t_step, ++pos) {
        int nimg = img + step_img, nin = in + step_in;
        if (nin >= per_img) { nin -= per_img; ++nimg; }
        if (NS > 1) {
            __syncwarp();
            if (task + t_step < ntasks && lane == 0) fetch(nimg, nin, pos + 1);
        }
        const int band = in / nstrips, strip = in - band * nstrips;
        const int y0 = gm.two_rows ? row_fixed : gm.y_first + band * RB;
        const bool left_edge = strip == 0, right_edge = strip == nstrips - 1;
        unsigned rowmask = 0;
#pragma unroll
        for (int i = 0; i < RB; ++i) rowmask |= (y0 + i <= gm.y_last) ? (1u << i) : 0u;
        const int s = (int)(pos % NS);
        mbar_wait(&bars[s], (pos / NS) & 1u);
        const float *tb = ring + s * C::STAGE_FLOATS + lane;
        const float *ta = tb + C::WIN_FLOATS;
        // window: box columns p .. p + 4 in physical slots (p + k) % 6; box column p + 5 is converted during column p
        double win[WR][6];
        double ctr[RB], ctr_n[RB];
#pragma unroll
        for (int bc = 0; bc < 5; ++bc)
#pragma unroll
            for (int r = 0; r < WR; ++r) win[r][bc] = (double)tb[(r * BW + bc) * 32];
#pragma unroll
        for (int i = 0; i < RB; ++i) ctr[i] = (double)ta[(i * SW) * 32];
#pragma unroll
        for (int p = 0; p < SW; ++p) {
            const bool edge = p == 0 || p == SW - 1;
            double e1[ND], e2[ND];
            if (edge) {
#pragma unroll
                for (int d = 0; d < ND; ++d) e1[d] = e2[d] = 0.0;
            }
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                const bool live = (rowmask >> i) & 1u;
                const double q = live ? win[i + 2][(p + 2) % 6] : 0.0, xc = live ? ctr[i] : 0.0;
                double *o1 = edge ? e1 : acc1, *o2 = edge ? e2 : acc2;
#pragma unroll
                for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                    for (int dx = 0; dx < 5; ++dx) {
                        o2[dy * 5 + dx] = fma(q, win[i + dy][(p + dx) % 6], o2[dy * 5 + dx]);
                        o1[dy * 5 + dx] = fma(xc, win[i + 4 - dy][(p + 4 - dx) % 6], o1[dy * 5 + dx]);
                    }
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    o2[10 + dx] = fma(q, win[i + 2][(p + dx) % 6], o2[10 + dx]);
                    o1[10 + dx] = fma(xc, win[i + 2][(p + 4 - dx) % 6], o1[10 + dx]);
                }
                // the next column's operands, spread over the rows: window rows i, i + RB, ..., centre pixel of row i
                if (p + 5 < BW) {
#pragma unroll
                    for (int r = i; r < WR; r += RB) win[r][(p + 5) % 6] = (double)tb[(r * BW + p + 5) * 32];
                }
                if (p + 1 < SW) ctr_n[i] = (double)ta[(i * SW + p + 1) * 32];
            }
#pragma unroll
            for (int i = 0; i < RB; ++i) ctr[i] = ctr_n[i];
            if (edge) {   // the image's first / last pixel column: the shared-memory records; a strip boundary inside the image: between
                const bool first = p == 0 && left_edge, last = p == SW - 1 && right_edge;
                if (first || last) {
                    double *r = srec + (last ? 2 * ND * 32 : 0);
#pragma unroll
                    for (int d = 0; d < ND; ++d) {
                        r[d * 32] += e1[d];
                        r[(ND + d) * 32] += e2[d];
                    }
                } else {
#pragma unroll
                    for (int d = 0; d < ND; ++d) {
                        acc1[d] += e1[d];
                        acc2[d] += e2[d];
                    }
                }
            }
        }
        if (NS == 1) {
            __syncwarp();
            if (task + t_step < ntasks && lane == 0) fetch(nimg, nin, pos + 1);
        }
        img = nimg;
        in = nin;
    }
    if (chok) {
        double *rec = partial + ((size_t)chl * slot_stride + slot0 + slot) * REC;   // [G1, G2][first, between, last][13]
#pragma unroll
        for (int d = 0; d < ND; ++d) {
            rec[d] = srec[d * 32];
            rec[ND + d] = acc1[d];
            rec[2 * ND + d] = srec[(2 * ND + d) * 32];
            rec[3 * ND + d] = srec[(ND + d) * 32];
            rec[4 * ND + d] = acc2[d];
            rec[5 * ND + d] = srec[(3 * ND + d) * 32];
        }
    }
}

// gram: (n_channels, 2 * 81): [G1 | G2], lower triangle + diagonal valid, zeros above (conv_finalize_kernel's layout).
// partial: records of the launch over rows 1 .. H-2 (left column, interior, right column); rpartial: records of the
// top / bottom row launch (even slots: top-left corner, top row, top-right corner; odd slots: the bottom ones).
__global__ void __launch_bounds__(1024)
conv_corr9_assemble_kernel(const double *__restrict__ partial, int slots, const double *__restrict__ rpartial, int rslots,
                           int same, int g1_by_x, int n_ch, int G, double *__restrict__ gram) {
    using namespace corr9;
    // S[pass][row class: 0 top, 1 between, 2 bottom][column class: 0 first, 1 between, 2 last][13]
    constexpr int NV = 2 * 9 * ND, NP = 4;            // values per channel; slot partitions (one quarter of the CTA each)
    __shared__ double S[2][3][3][ND];
    __shared__ double P[NP][NV];
    const int ch = blockIdx.x, tid = threadIdx.x;
    const int e = tid % 256, part = tid / 256;        // 1024 threads: value e (< 234) x partition `part`
    if (e < NV) {
        const int d = e % ND, cc = (e / ND) % 3, rc = (e / (3 * ND)) % 3, pass = e / (9 * ND);
        const int off = (pass * 3 + cc) * ND + d;
        // The records of a value are summed in a FIXED order whatever the launch geometry: slots in index order dealt
        // round-robin to 16 chains (4 partitions x 4 interleaved sums, independent loads in flight), chains combined in
        // index order; packed layers: the G virtual channels g * n_ch + ch of this channel, g in index order.
        const int n = rc == 1 ? slots : (rslots - (rc == 0 ? 0 : 1) + 1) / 2;
        const size_t stride = rc == 1 ? REC : 2 * REC;
        double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
        for (int g = 0; g < G; ++g) {
            const size_t vch = (size_t)g * n_ch + ch;
            const double *src = rc == 1 ? partial + vch * slots * REC + off
                                        : rpartial + (vch * rslots + (rc == 0 ? 0 : 1)) * REC + off;
            int s = part * 4;
#pragma unroll 2
            for (; s + 4 <= n; s += 4 * NP) {
                t0 += src[(size_t)s * stride];
                t1 += src[(size_t)(s + 1) * stride];
                t2 += src[(size_t)(s + 2) * stride];
                t3 += src[(size_t)(s + 3) * stride];
            }
            if (s < n) {   // the ragged last group of four belongs to exactly one partition
                t0 += src[(size_t)s * stride];
                if (s + 1 < n) t1 += src[(size_t)(s + 1) * stride];
                if (s + 2 < n) t2 += src[(size_t)(s + 2) * stride];
            }
        }
        P[part][e] = (t0 + t1) + (t2 + t3);
    }
    __syncthreads();
    if (tid < NV) {
        const int d = tid % ND, cc = (tid / ND) % 3, rc = (tid / (3 * ND)) % 3, pass = tid / (9 * ND);
        S[pass][rc][cc][d] = (P[0][tid] + P[1][tid]) + (P[2][tid] + P[3][tid]);
    }
    __syncthreads();
    for (int e2 = tid; e2 < 162; e2 += blockDim.x) {
        const int which = e2 / 81, t = (e2 % 81) / 9, s = e2 % 9;
        double v = 0.0;
        if (s <= t) {
            const int ar = t / 3, ac = t % 3, dy = s / 3 - ar, dx = s % 3 - ac;
            const int id = dy < 0 ? (dy + 2) * 5 + dx + 2 : 12 + dx;
            const int pass = (which == 0 && !same) ? 0 : 1;
            // The records are split by the region of the window's centre pixel: the xq pixel tap t reads, or for G1 from the
            // one-pass band kernel (g1_by_x) the x pixel tap s reads (the patch position is the same pixel either way).
            // Tap row 0 never sits on the bottom image row, tap row 2 never on the top row; columns alike.
            const bool by_s = pass == 0 && g1_by_x;
            const int cr = by_s ? s / 3 : ar, ccl = by_s ? s % 3 : ac;
            const int r_lo = cr == 2 ? 1 : 0, r_hi = cr == 0 ? 1 : 2, c_lo = ccl == 2 ? 1 : 0, c_hi = ccl == 0 ? 1 : 2;
            for (int rc = r_lo; rc <= r_hi; ++rc)
                for (int cc = c_lo; cc <= c_hi; ++cc) v += S[pass][rc][cc][id];
        }
        gram[(size_t)ch * 162 + e2] = v;
    }
}

// ---- host side ---------------------------------------------------------------------------------------------------
// Is the geometry eligible, and with how many rows per band?  (0: keep the patch form.)  The channel conditions of the
// tensor map (C >= 32, C % 4 == 0) are the caller's: it can meet them by packing images side by side (corr9_pack_kernel).
int corr9_plan(int kh, int kw, int sh, int sw, int rh, int rw, int padding_same, int H, int W, int force_rb, bool same) {
    if (kh != 3 || kw != 3 || sh != 1 || sw != 1 || rh != 1 || rw != 1 || !padding_same) return 0;
    if (H < 6 || W < corr9::WC) return 0;            // a TMA box (RB + 2 >= 6 rows x 5 columns) must fit in the image
    if ((int64_t)H * W >= ((int64_t)1 << 28)) return 0;
    if ((force_rb == 8 || force_rb == 6 || force_rb == 4) && force_rb + 2 <= H && (same || force_rb != 8)) return force_rb;
    if (!same) {
        // G1 and G2 in one pass: bands of 6 or 4 rows (an 8-row band's 12 x 5 window and 26 sums spill).
        // RB = 6 converts 2.67 values per pixel against RB = 4's 3.0 and moves fewer halo rows: it wins unless it wastes
        // more than 15 % of its band rows.
        const int rows = H - 2;
        const int bands6 = (rows + 5) / 6, bands4 = (rows + 3) / 4;
        return 6 + 2 <= H && ((double)rows >= 0.85 * bands6 * 6 || bands6 * 6 <= bands4 * 4) ? 6 : 4;
    }
    // Rows 1 .. H-2 in bands of RB rows.  Measured (tools/vgg_bench.py --corr-rows, VGG16 and CIFAR10 shapes): RB = 8 wins
    // whenever at least 85 % of its band rows are live (224, 112, 56, 32, 16 rows high), otherwise the band height that
    // wastes fewest rows, with RB = 4 handicapped by 0.1 (more conversions and box traffic per DFMA: on 28 x 28 it wastes
    // least and is still the slowest; RB = 6 is 6 % faster than RB = 8 there; 14 x 14: RB = 6).
    const int rows = H - 2;
    auto live = [&](int rb) { return (double)rows / (double)((rows + rb - 1) / rb * rb); };
    if (8 + 2 <= H && live(8) >= 0.85) return 8;
    int best = 0;
    double best_live = -1.0;
    const int cand[3] = {8, 6, 4};
    for (int i = 0; i < 3; ++i) {
        const int rb = cand[i];
        if (rb + 2 > H) continue;
        const double score = live(rb) - (rb == 4 ? 0.1 : 0.0);
        if (score > best_live + 1e-9) { best_live = score; best = rb; }
    }
    return best;
}

// ---- image packing ---------------------------------------------------------------------------------------------------
// lane = channel needs 32 channels per warp and a 16-byte channel pitch.  Layers with few channels (the first conv layer:
// C = 3; a rank of a multi-GPU job that owns 8 of 64 channels) are repacked so that G = 32 / gcd(n_ch, 32) images sit side
// by side as "virtual channels": out[(ng, y, x, g * n_ch + c)] = act[(ng * G + g, y, x, c_first + c)], zeros past the last
// image.  Every virtual channel is an ordinary channel of an ordinary (n / G, H, W, G n_ch) tensor for the correlation
// kernels; conv_corr9_assemble_kernel adds the G records of a real channel (g in index order).
__global__ void __launch_bounds__(256)
corr9_pack_kernel(const float *__restrict__ act, int64_t n_valid, int hw, int64_t C, int64_t c_first, int n_ch, int G,
                  int64_t img0, int pix_per_warp, float *__restrict__ out) {
    // blockIdx.y: group of G images; every warp copies a run of pixels, 32 virtual channels (one 128-byte line) at a time
    const int lane = threadIdx.x & 31, VC = G * n_ch;
    const int64_t ng = blockIdx.y;
    const int p0 = (int)((blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * pix_per_warp);
    const int p1 = min(hw, p0 + pix_per_warp);
    if (p0 >= p1) return;
    for (int vb = 0; vb < VC; vb += 32) {
        const int v = vb + lane;
        if (v >= VC) continue;
        const int g = v / n_ch, c = v - g * n_ch;
        const int64_t n = img0 + ng * G + g;
        float *dst = out + (ng * hw + p0) * VC + v;
        if (n < n_valid) {
            const float *src = act + (n * hw + p0) * C + c_first + c;
            int p = p0;
            for (; p + 8 <= p1; p += 8) {
                float t[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) t[u] = __ldg(src + (int64_t)u * C);
#pragma unroll
                for (int u = 0; u < 8; ++u) dst[(int64_t)u * VC] = t[u];
                src += 8 * C;
                dst += (int64_t)8 * VC;
            }
            for (; p < p1; ++p) {
                *dst = __ldg(src);
                src += C;
                dst += VC;
            }
        } else {
            for (int p = p0; p < p1; ++p) {
                *dst = 0.f;
                dst += VC;
            }
        }
    }
}

// Packs images [img0, img0 + imgs) (img0 a multiple of G) of channels [c_first, c_first + n_ch) into `out`, which holds
// the packed tensor of ALL images: groups [img0 / G, ceil((img0 + imgs) / G)) are written.
int corr9_pack_stage(gpfq_ctx *ctx, const float *act, int64_t n_img, int H, int Wd, int64_t C, int64_t c_first, int n_ch, int G,
                     int64_t img0, int64_t imgs, float *out) {
    const int hw = H * Wd;
    const int64_t VC = (int64_t)G * n_ch, ngrp = ceil_div64(imgs, G);
    // enough warps for ~8 CTAs per SM over the whole launch, at least 32 pixels per warp
    int64_t ppw = ceil_div64((int64_t)hw * ngrp, (int64_t)ctx->sm_count * 64);
    ppw = std::max<int64_t>(32, std::min<int64_t>(ppw, hw));
    const int64_t warps = ceil_div64(hw, ppw);
    for (int64_t g0 = 0; g0 < ngrp; g0 += 65535) {   // gridDim.y limit
        const int64_t gn = std::min<int64_t>(65535, ngrp - g0);
        dim3 grid((unsigned)ceil_div64(warps, 8), (unsigned)gn);
        corr9_pack_kernel<<<grid, 256, 0, ctx->stream>>>(act, std::min<int64_t>(n_img, img0 + imgs), hw, C, c_first, n_ch, G,
                                                         img0 + g0 * G, (int)ppw, out + (img0 / G + g0) * hw * VC);
        KERNEL_CHECK(ctx);
    }
    return GPFQ_OK;
}

template <int RB, bool BOTH>
static int corr9_resident_ctas() {
    using namespace corr9;
    // a failed query only costs launch geometry (the caller plans for one CTA per SM): its error is consumed HERE, where it
    // arose, so that it can neither leak into the next launch check nor swallow an unrelated pending error
    int a = 0;
    if (cudaFuncSetAttribute(conv_corr9_tma_kernel<RB, BOTH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Ring<RB, BOTH>::SMEM) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, conv_corr9_tma_kernel<RB, BOTH>, WARPS * 32, Ring<RB, BOTH>::SMEM) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return a;
}

// X~ != X on strips: both Grams in one pass (conv_corr9_strip1_kernel) or the two-pass pair, by strip width.  Measured per layer
// (B200, VGG16 and CIFAR10 benches, profiles/r3_corr9_onepass.md): one pass wins on 8-pixel images (0.305 -> 0.219 ms, 0.342 ->
// 0.331 ms) and loses on 14- to 64-wide ones (VGG16 56 x 56 x 256: 3.66 -> 5.39 ms), where its shared-memory records and
// (RB + 4)-row boxes leave one CTA of four warps per SM against the pair's eight warps.
static constexpr bool corr9_strip_onepass_sw(int sw) { return sw == 8; }
static int corr9_strip_width(int Wd);
static bool corr9_strip_onepass(int Wd);
template <int SW, int RB>
static int corr9_strip_resident_ctas(bool same) {
    using namespace corr9s;
    int a = 0, b = 0;
    if constexpr (corr9_strip_onepass_sw(SW)) {
        if (!same) {
            if (cudaFuncSetAttribute(conv_corr9_strip1_kernel<SW, RB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg1<SW, RB>::SMEM) != cudaSuccess ||
                cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, conv_corr9_strip1_kernel<SW, RB>, WARPS * 32, Cfg1<SW, RB>::SMEM) != cudaSuccess) {
                cudaGetLastError();
                return 0;
            }
            return a;
        }
    }
    if (cudaFuncSetAttribute(conv_corr9_strip_kernel<SW, RB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg<SW, RB, false>::SMEM) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, conv_corr9_strip_kernel<SW, RB, false>, WARPS * 32, Cfg<SW, RB, false>::SMEM) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    if constexpr (!corr9_strip_onepass_sw(SW)) {
        if (same) return a;
        if (cudaFuncSetAttribute(conv_corr9_strip_kernel<SW, RB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg<SW, RB, true>::SMEM) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, conv_corr9_strip_kernel<SW, RB, true>, WARPS * 32, Cfg<SW, RB, true>::SMEM) != cudaSuccess) {
            cudaGetLastError();
            return 0;
        }
        return a < b ? a : b;
    }
    return a;
}

// Slots (warps per channel group) that fill every SM with as many CTAs of four warps as stay resident.  Wd: the image width (the
// strip kernel of small images has its own occupancy; there the slot count is rounded DOWN to whole CTAs so that the launch is one
// wave -- every warp gets the same number of tasks, and 1.5 waves cost two: measured on VGG16's 28 x 28 layers).
int corr9_pick_slots(gpfq_ctx *ctx, int RB, bool same, int64_t c_first, int n_ch, int64_t ntasks, int Wd) {
    using namespace corr9;
    if (RB < 1 || RB > 8) return WARPS;
    if (const int sw = ctx->corr_strip == 2 ? 0 : corr9_strip_width(Wd)) {
        const int rb = RB == 1 ? 1 : 4, wi = sw == 8 ? 0 : sw == 14 ? 1 : 2;
        int &socc = ctx->corr_strip_occ[same ? 1 : 0][rb == 1 ? 0 : 1][wi];
        if (!socc) {
            socc = rb == 1 ? (sw == 8 ? corr9_strip_resident_ctas<8, 1>(same) : sw == 14 ? corr9_strip_resident_ctas<14, 1>(same) : corr9_strip_resident_ctas<16, 1>(same))
                           : (sw == 8 ? corr9_strip_resident_ctas<8, 4>(same) : sw == 14 ? corr9_strip_resident_ctas<14, 4>(same) : corr9_strip_resident_ctas<16, 4>(same));
            if (socc < 1) socc = 1;
        }
        const int64_t groups = ceil_div64(n_ch + (c_first & 3), 32);
        int64_t ctas = std::max<int64_t>(1, (int64_t)ctx->sm_count * socc / groups);    // CTAs per channel group: one wave, rounded down
        ctas = std::min<int64_t>(ctas, std::max<int64_t>(1, ceil_div64(ntasks, corr9s::WARPS)));
        return (int)(ctas * corr9s::WARPS);
    }
    int &occ = ctx->corr_occ[same ? 1 : 0][RB];      // per context (= per device): no state shared between engines / threads
    if (!occ) {
        occ = same ? (RB == 8 ? corr9_resident_ctas<8, false>() : RB == 6 ? corr9_resident_ctas<6, false>()
                      : RB == 4 ? corr9_resident_ctas<4, false>() : corr9_resident_ctas<1, false>())
                   : (RB == 6 ? corr9_resident_ctas<6, true>() : RB == 4 ? corr9_resident_ctas<4, true>() : corr9_resident_ctas<1, true>());
        if (occ < 1) occ = 1;                        // the occupancy query failed: plan for one CTA per SM
    }
    const int64_t groups = ceil_div64(n_ch + (c_first & 3), 32);
    int64_t per = ceil_div64((int64_t)ctx->sm_count * occ * WARPS, groups);
    per = std::min<int64_t>(per, std::max<int64_t>(1, ntasks));
    return (int)(ceil_div64(per, WARPS) * WARPS);
}

typedef CUresult (*Corr9EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static Corr9EncodeFn corr9_encode_fn() {
    static Corr9EncodeFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<Corr9EncodeFn>(p);
    }
    return fn;
}

// Can the activation tensor be read through a tensor map at all (driver entry point, alignment)?
int corr9_tensor_ok(const float *act, const float *actq) {
    return corr9_encode_fn() != nullptr && ((uintptr_t)act & 15) == 0 && ((uintptr_t)actq & 15) == 0;
}

// (C, W, H, N) fp32 tensor map with a 32-channel x `cols`-column x `rows`-row box
static bool corr9_make_map(CUtensorMap *map, const float *act, int64_t n_img_total, int H, int W, int64_t C, int rows,
                           int cols = corr9::WC) {
    Corr9EncodeFn enc = corr9_encode_fn();
    if (!enc) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n_img_total};
    const cuuint64_t strides[3] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4, (cuuint64_t)H * W * C * 4};  // bytes, dims 1..3
    const cuuint32_t box[4] = {32u, (cuuint32_t)cols, (cuuint32_t)rows, 1u};
    const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float *>(act), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// X~ == X: G2 only; otherwise G1 and G2 in one pass (an (RB + 4)-row window of xq and the RB x 5 centre pixels of x per box)
template <int RB, bool BOTH>
static int launch_corr9(gpfq_ctx *ctx, const float *actq, const float *actx, const Corr9Geom &gm, int64_t C, int64_t n_img_total,
                        double *partial, int slot_stride, int slot0) {
    using namespace corr9;
    using R = Ring<RB, BOTH>;
    dim3 grid((unsigned)(gm.slots / WARPS), (unsigned)ceil_div64(gm.n_ch + (gm.c_first & 3), 32));
    CUtensorMap mq_win, mx_ctr;
    bool ok = corr9_make_map(&mq_win, actq, n_img_total, gm.H, gm.W, C, R::WR);
    if (ok && BOTH) ok = corr9_make_map(&mx_ctr, actx, n_img_total, gm.H, gm.W, C, RB);
    if (!ok) return gpfq_fail(ctx, GPFQ_ERR_CUDA, "cuTensorMapEncodeTiled failed for the (%lld, %d, %d, %lld) activations",
                              (long long)n_img_total, gm.H, gm.W, (long long)C);
    CUDA_TRY(ctx, cudaFuncSetAttribute(conv_corr9_tma_kernel<RB, BOTH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R::SMEM));
    conv_corr9_tma_kernel<RB, BOTH><<<grid, WARPS * 32, R::SMEM, ctx->stream>>>(mq_win, BOTH ? mx_ctr : mq_win, gm, partial, slot_stride, slot0);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}


template <int SW, int RB>
static int launch_corr9_strip(gpfq_ctx *ctx, const float *actq, const float *actx, bool same, const Corr9Geom &gm, int64_t C,
                              int64_t n_img_total, double *partial, int slot_stride, int slot0) {
    using namespace corr9s;
    cudaStream_t st = ctx->stream;
    dim3 grid((unsigned)(gm.slots / WARPS), (unsigned)ceil_div64(gm.n_ch + (gm.c_first & 3), 32));
    CUtensorMap mq_win, mq_ctr, mx_win;
    if constexpr (corr9_strip_onepass_sw(SW)) {
        if (!same) {   // both Grams in one launch
        using C1 = Cfg1<SW, RB>;
        if (!corr9_make_map(&mq_win, actq, n_img_total, gm.H, gm.W, C, C1::WR, SW + 4) ||
            !corr9_make_map(&mq_ctr, actx, n_img_total, gm.H, gm.W, C, RB, SW))
            return gpfq_fail(ctx, GPFQ_ERR_CUDA, "cuTensorMapEncodeTiled failed for the (%lld, %d, %d, %lld) activations",
                             (long long)n_img_total, gm.H, gm.W, (long long)C);
        CUDA_TRY(ctx, cudaFuncSetAttribute(conv_corr9_strip1_kernel<SW, RB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C1::SMEM));
        conv_corr9_strip1_kernel<SW, RB><<<grid, WARPS * 32, C1::SMEM, st>>>(mq_win, mq_ctr, gm, partial, slot_stride, slot0);
        KERNEL_CHECK(ctx);
        return GPFQ_OK;
        }
    }
    bool ok = corr9_make_map(&mq_win, actq, n_img_total, gm.H, gm.W, C, RB + 2, SW + 4);
    if (ok && !same)
        ok = corr9_make_map(&mq_ctr, actq, n_img_total, gm.H, gm.W, C, RB, SW) &&
             corr9_make_map(&mx_win, actx, n_img_total, gm.H, gm.W, C, RB + 2, SW + 4);
    if (!ok) return gpfq_fail(ctx, GPFQ_ERR_CUDA, "cuTensorMapEncodeTiled failed for the (%lld, %d, %d, %lld) activations",
                              (long long)n_img_total, gm.H, gm.W, (long long)C);
    CUDA_TRY(ctx, cudaFuncSetAttribute(conv_corr9_strip_kernel<SW, RB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)Cfg<SW, RB, false>::SMEM));
    conv_corr9_strip_kernel<SW, RB, false><<<grid, WARPS * 32, Cfg<SW, RB, false>::SMEM, st>>>(mq_win, mq_win, gm, partial, slot_stride, slot0);
    KERNEL_CHECK(ctx);
    if constexpr (!corr9_strip_onepass_sw(SW)) {
        if (!same) {
            CUDA_TRY(ctx, cudaFuncSetAttribute(conv_corr9_strip_kernel<SW, RB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)Cfg<SW, RB, true>::SMEM));
            conv_corr9_strip_kernel<SW, RB, true><<<grid, WARPS * 32, Cfg<SW, RB, true>::SMEM, st>>>(mx_win, mq_ctr, gm, partial, slot_stride, slot0);
            KERNEL_CHECK(ctx);
        }
    }
    return GPFQ_OK;
}

// strip width of the small-image variant for an image width (0: none)
// (measured on VGG16: 56-wide layers 4.00 -> 3.66 ms as four strips, 112-wide ones 3.50 -> 3.65 ms: those keep the band kernel)
static int corr9_strip_width(int Wd) { return Wd == 8 ? 8 : (Wd == 14 || Wd == 28 || Wd == 56) ? 14 : (Wd == 16 || Wd == 32 || Wd == 64) ? 16 : 0; }
static bool corr9_strip_onepass(int Wd) { return corr9_strip_onepass_sw(corr9_strip_width(Wd)); }

template <int SW>
static int corr9_strip_stage(gpfq_ctx *ctx, const float *actq, const float *act, bool same, Corr9Geom gm, int64_t C, int64_t n_img_total,
                             double *partial, int slot_stride, int slot0, int slots, double *rpartial, int rslot_stride, int rslot0,
                             int rslots) {
    if (gm.H > 2) {
        gm.slots = slots; gm.y_first = 1; gm.y_last = gm.H - 2; gm.two_rows = 0;
        GPFQ_TRY((launch_corr9_strip<SW, 4>(ctx, actq, act, same, gm, C, n_img_total, partial, slot_stride, slot0)));
    }
    gm.slots = rslots; gm.y_first = 0; gm.y_last = gm.H - 1; gm.two_rows = 1;
    GPFQ_TRY((launch_corr9_strip<SW, 1>(ctx, actq, act, same, gm, C, n_img_total, rpartial, rslot_stride, rslot0)));
    return GPFQ_OK;
}

// does the correlation form of images of this width use the strip kernel
int corr9_uses_strips(gpfq_ctx *ctx, int Wd) { return ctx->corr_strip != 2 && corr9_strip_width(Wd) != 0; }

// Correlation sums of channels [c_first, c_first + n_ch) over images [img0, img0 + n_img) of a tensor of n_img_total
// images: fills slots [slot0, slot0 + slots) of `partial` (rows 1 .. H-2) and [rslot0, rslot0 + rslots) of `rpartial`
// (top / bottom row) of every channel.  Both record arrays must be zeroed by the caller.
int conv_corr9_stage(gpfq_ctx *ctx, const float *act, const float *actq, bool same, int64_t img0, int64_t n_img,
                     int64_t n_img_total, int H, int Wd, int64_t C, int64_t c_first, int n_ch, int RB, double *partial,
                     int slot_stride, int slot0, int slots, double *rpartial, int rslot_stride, int rslot0, int rslots) {
    using namespace corr9;
    if (slots % WARPS || rslots % WARPS || rslots < 2)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "corr9: slot counts must be multiples of %d", WARPS);
    if (n_img_total >= ((int64_t)1 << 31)) return gpfq_fail(ctx, GPFQ_ERR_ARG, "corr9: too many images");
    Corr9Geom gm;
    gm.H = H; gm.W = Wd; gm.c_first = c_first; gm.n_ch = n_ch; gm.img0 = img0; gm.n_img = n_img;
    if (const int sw = ctx->corr_strip == 2 ? 0 : corr9_strip_width(Wd)) {   // small images: whole strips as straight-line code
        gm.slots = 0; gm.y_first = gm.y_last = gm.two_rows = 0;
        if (sw == 8) return corr9_strip_stage<8>(ctx, actq, act, same, gm, C, n_img_total, partial, slot_stride, slot0, slots, rpartial, rslot_stride, rslot0, rslots);
        if (sw == 14) return corr9_strip_stage<14>(ctx, actq, act, same, gm, C, n_img_total, partial, slot_stride, slot0, slots, rpartial, rslot_stride, rslot0, rslots);
        return corr9_strip_stage<16>(ctx, actq, act, same, gm, C, n_img_total, partial, slot_stride, slot0, slots, rpartial, rslot_stride, rslot0, rslots);
    }
    if (H > 2) {
        gm.slots = slots; gm.y_first = 1; gm.y_last = H - 2; gm.two_rows = 0;
        const int rc = same ? RB : -RB;
        switch (rc) {
            case 8: GPFQ_TRY((launch_corr9<8, false>(ctx, actq, act, gm, C, n_img_total, partial, slot_stride, slot0))); break;
            case 6: GPFQ_TRY((launch_corr9<6, false>(ctx, actq, act, gm, C, n_img_total, partial, slot_stride, slot0))); break;
            case 4: GPFQ_TRY((launch_corr9<4, false>(ctx, actq, act, gm, C, n_img_total, partial, slot_stride, slot0))); break;
            case -6: GPFQ_TRY((launch_corr9<6, true>(ctx, actq, act, gm, C, n_img_total, partial, slot_stride, slot0))); break;
            case -4: GPFQ_TRY((launch_corr9<4, true>(ctx, actq, act, gm, C, n_img_total, partial, slot_stride, slot0))); break;
            default: return gpfq_fail(ctx, GPFQ_ERR_ARG, "corr9: no kernel for %d rows per band (X~ %s X)", RB, same ? "==" : "!=");
        }
    }
    gm.slots = rslots; gm.y_first = 0; gm.y_last = H - 1; gm.two_rows = 1;
    if (same) GPFQ_TRY((launch_corr9<1, false>(ctx, actq, act, gm, C, n_img_total, rpartial, rslot_stride, rslot0)));
    else GPFQ_TRY((launch_corr9<1, true>(ctx, actq, act, gm, C, n_img_total, rpartial, rslot_stride, rslot0)));
    return GPFQ_OK;
}

// n_ch real channels; G > 1: the records belong to G * n_ch virtual channels of a packed tensor
// gram[ch] = sum over the G virtual channels g * n_ch + ch of gv[.], g in index order (packed layers)
__global__ void conv_corr9_sum_groups_kernel(const double *__restrict__ gv, int n_ch, int G, double *__restrict__ gram) {
    const int ch = blockIdx.x;
    for (int e = threadIdx.x; e < 162; e += blockDim.x) {
        double v = 0.0;
        for (int g = 0; g < G; ++g) v += gv[((size_t)g * n_ch + ch) * 162 + e];
        gram[(size_t)ch * 162 + e] = v;
    }
}

int conv_corr9_assemble_stage(gpfq_ctx *ctx, const double *partial, int slots, const double *rpartial, int rslots,
                              bool same, int Wd, int n_ch, int G, double *gram) {
    const int g1_by_x = corr9_uses_strips(ctx, Wd) && !corr9_strip_onepass(Wd) ? 0 : 1;   // which kernel wrote the G1 records (conv_corr9_stage)
    if (G > 1) {
        // Packed layers (VGG16's first layer: 3 real channels, G = 32): one CTA per REAL channel would walk G x slots records
        // alone (measured: 1.05 ms of that layer's 1.95).  Assemble every virtual channel on its own CTA, then add the G
        // matrices of a channel in index order -- the Gram entries are sums of the records either way, the order stays fixed.
        double *gv = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_MISC, (size_t)G * n_ch * 162 * sizeof(double), (void **)&gv));
        conv_corr9_assemble_kernel<<<(unsigned)(G * n_ch), 1024, 0, ctx->stream>>>(partial, slots, rpartial, rslots, same ? 1 : 0,
                                                                                    g1_by_x, G * n_ch, 1, gv);
        KERNEL_CHECK(ctx);
        conv_corr9_sum_groups_kernel<<<(unsigned)n_ch, 192, 0, ctx->stream>>>(gv, n_ch, G, gram);
        KERNEL_CHECK(ctx);
        return GPFQ_OK;
    }
    conv_corr9_assemble_kernel<<<(unsigned)n_ch, 1024, 0, ctx->stream>>>(partial, slots, rpartial, rslots, same ? 1 : 0, g1_by_x, n_ch, G, gram);
    KERNEL_CHECK(ctx);
    return GPFQ_OK;
}
