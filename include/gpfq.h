/* gpfq.h -- C ABI of libgpfq: the GPFQ greedy path-following quantizer on NVIDIA B200 (sm_100a).
 *
 * Drop-in boundary for the hot path of elybrand/quantized_neural_networks
 * (scripts/quantized_network.py).  The reference has no FFI; its boundary is method level, with
 * HDF5 files as the hand-off.  Each entry point below names the reference code it replaces.
 * All pointers are BORROWED for the duration of a call; the library never frees caller memory
 * and every output buffer is caller-allocated.  Plain C: no C++ or torch types in signatures.
 *
 * Data contract (identical to what the reference's workers read):
 *   X, Xq  float32, one ROW per data direction t, contiguous along the m samples
 *          ((N0, m) `wX`/`qX` datasets written with transpose=True, quantized_network.py:469-492;
 *           (kh*kw, n_patches) `wX_channel{c}`/`qX_channel{c}` datasets, :789-797)
 *   W      float32 Keras kernel, (N0, N1) row-major for Dense -- a neuron is a COLUMN (:553);
 *          (kh, kw, C, F) for Conv2D -- the "neuron" is W[:, :, c, f] flattened C-order (:215)
 *   alphabet  float64, K levels, as produced by `rad * linspace(-1, 1, K)` (:396, :544-545).  Any levels are accepted and
 *          rounded to literally; the fast kernels are chosen from the levels themselves (ascending within 1 % of a step of a
 *          grid: windowed rounding; on the symmetric grid, see "sweep_walk": the tensor-core walk and the int8 residual form)
 *   Q      float64, same shape/strides convention as W (`Q = zeros(W.shape)`, :535, :833)
 */
#ifndef GPFQ_H_
#define GPFQ_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPFQ_VERSION 100

typedef struct gpfq_ctx gpfq_ctx;

/* return codes (0 = success).  The reference logs and re-raises worker exceptions
 * (quantized_network.py:563-565, :719-721); the Python wrapper turns non-zero codes into the same. */
enum {
    GPFQ_OK = 0,
    GPFQ_ERR_ARG = 1,         /* bad shape / NULL pointer / unsupported K */
    GPFQ_ERR_CUDA = 2,        /* a CUDA runtime call or kernel failed (message has the detail) */
    GPFQ_ERR_OOM = 3,         /* device or pinned-host allocation failed */
    GPFQ_ERR_UNSUPPORTED = 4  /* valid request this build cannot serve (e.g. no sm_100 device) */
};

/* flags */
#define GPFQ_X_DEVICE (1u << 0)   /* X / Xq (and patch pointers) are device pointers */
#define GPFQ_W_DEVICE (1u << 1)   /* W is a device pointer */
#define GPFQ_Q_DEVICE (1u << 2)   /* Q_out is a device pointer */
#define GPFQ_ALL_DEVICE (GPFQ_X_DEVICE | GPFQ_W_DEVICE | GPFQ_Q_DEVICE)
#define GPFQ_METHOD_AUTO (0u << 4)    /* pick streaming vs Gram+sweep by the measured cost table */
#define GPFQ_METHOD_STREAM (1u << 4)  /* literal residual walk (the reference's dtype ladder: fp32-rounded w*X), u on chip */
#define GPFQ_METHOD_GRAM (2u << 4)    /* Gram stage + blocked triangular sweep */
#define GPFQ_METHOD_STREAM_FAST (3u << 4) /* residual walk on exact fp32 x fp32 products (the Gram form's numerics) */
#define GPFQ_METHOD_MASK (3u << 4)
#define GPFQ_NO_SYNC (1u << 8)        /* all-device calls only: return after enqueueing */

#define GPFQ_MAX_K 64                 /* alphabet levels per alphabet */

/* per-call report (optional, may be NULL).  Times are CUDA-event milliseconds on the library's
 * stream; they are 0 when GPFQ_NO_SYNC is set. */
typedef struct gpfq_stats {
    int32_t method;          /* GPFQ_METHOD_STREAM, _GRAM or _STREAM_FAST actually used (>>4) */
    int32_t kernel_launches; /* kernels launched by this call */
    float ms_total;          /* whole call, including copies for host pointers */
    float ms_h2d, ms_d2h;    /* copies (host-pointer calls) */
    float ms_gram;           /* Gram stage (dense) or patch-Gram stage (conv) */
    float ms_sweep;          /* triangular sweep */
    float ms_stream;         /* streaming walk */
    int64_t weights;         /* quantized weights produced (per alphabet x n_alphabets) */
    int64_t bytes_algorithmic; /* algorithmic HBM bytes of the dominant kernel (DESIGN.md) */
    int64_t flops_algorithmic; /* algorithmic fp64 flops of the dominant kernel */
    int32_t gram_kernel;     /* Dense Gram stage ran as: 0 none, 1 fp64 DMMA (mma.sync), 2 int8 slices on tcgen05,
                                3 block-diagonal tiles only (residual form of the sweep's outer level);
                                conv NHWC entry point: 4 = correlation form (13 displacement sums per Gram),
                                5 = correlation form on images packed side by side as virtual channels */
    int32_t reserved;        /* bit 0: contractions of the residual-form sweep ran on tcgen05 (int8 slices); bit 1: the sweep's ranges were
                                walked by the tensor-core walk (sweep_tc_kernel) */
} gpfq_stats;

/* ---- lifetime ------------------------------------------------------------------------------
 * One context per GPU per process (the reference: one ProcessPoolExecutor per layer, :549, :706). */
int gpfq_create(int device, gpfq_ctx **out);
void gpfq_destroy(gpfq_ctx *ctx);
const char *gpfq_last_error(const gpfq_ctx *ctx); /* never NULL; valid until the next call */
int gpfq_version(void);
/* Launch on the caller's stream (a cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream);
 * NULL restores the library's own stream; for the default stream pass cudaStreamLegacy ((void*)0x1)
 * or cudaStreamPerThread ((void*)0x2), not 0. */
int gpfq_set_stream(gpfq_ctx *ctx, void *cuda_stream);
/* Tuning / A-B switches (profiling and tests; the defaults pick by shape):
 *   "gram_kernel"  0 auto, 1 fp64 DMMA contraction, 2 int8 slices on tcgen05 (Dense Gram stage)
 *   "i8_pairs_d"   0 default, else keep int8 slice pairs with k + l <= value (2..10; 10 = every pair)
 *   "conv_kernel"  0 TMA-staged patch Grams / correlation form from NHWC activations, 1 direct LDG, 2 generic,
 *                  3 as 0 but the NHWC entry point uses the shared-memory planes kernel (patch form: 126 MACs per column)
 *   "corr_pack"    correlation form, images packed side by side as virtual channels: 0 when the channel count cannot be
 *                  mapped (C < 32 or C % 4 != 0) and the images are large, 1 always, 2 never
 *   "corr_small"   1: correlation form also on images below 128 pixels (default: the planes kernel is faster there)
 *   "corr_rows"    correlation form: image rows per band (0 auto by image height, or 4 / 6 / 8; 8 only when X~ == X,
 *                  the one-pass G1 + G2 kernel of X~ != X has bands of 4 or 6 rows and plans its own height otherwise)
 *   "corr_strip"   correlation form on small images (widths 8, 14, 16, 28, 32, 56, 64): 0 the strip kernel (whole strips of <= 16 columns as
 *                  straight-line code), 2 the band kernel
 *   "sweep_walk"   range walk of the Gram-row sweep for one alphabet on the symmetric grid (every level within 2^-40 a of
 *                  -a + k 2a / (K - 1), a = the top level; for odd K the middle level exactly 0, three levels exactly {-a, 0, a}):
 *                  0 auto (the tensor-core walk sweep_tc_kernel from 2048 directions, below that sweep_pipe / sweep_tile),
 *                  1 always the tensor-core walk, 2 always sweep_pipe / sweep_tile; other alphabets always walk with
 *                  sweep_pipe / sweep_tile.  The residual form walks with sweep_tc_kernel when its contractions run on
 *                  tcgen05, with sweep_pipe / sweep_tile when they run on the fp64 pipe ("sweep_i8")
 *   "sweep_i8"     contractions of the residual-form sweep: 0 auto (int8 slices on tcgen05 unless the direction norms spread
 *                  beyond what one exponent per sample keeps: then fp64 DMMA; one 4-byte read-back decides), 1 always int8
 *                  slices on tcgen05, 2 fp64 DMMA
 *   "sweep_outer"  0 auto, 1 Gram rows of all earlier directions, 2 carried residuals (3 m N0 N1 MACs: wins when m << N0),
 *                  3 carried residuals as one chain (default: two halves of the neurons on two streams, so that one half's
 *                  contractions fill the other half's latency-bound walk) */
int gpfq_set_option(gpfq_ctx *ctx, const char *key, int64_t value);
/* Stage times of an earlier call: calls_back = 0 is the most recent API call, 1 the one before, ...
 * (a ring of 128).  For GPFQ_NO_SYNC calls, synchronise the stream first; unfinished events read 0. */
int gpfq_query_stats(gpfq_ctx *ctx, int32_t calls_back, gpfq_stats *out);
/* Release cached device/pinned workspaces (they are otherwise kept between calls). */
int gpfq_trim(gpfq_ctx *ctx);
/* Bytes of partial Gram workspace the last conv call (gpfq_conv_channels, gpfq_conv_layer_nhwc, gpfq_conv_gram_nhwc) asked
 * for: 0 for kernels above 128 taps.  For the kernel sizes without a specialised kernel it stays within 1 GiB unless a single
 * partial slot of every channel is larger. */
int64_t gpfq_conv_partial_bytes(gpfq_ctx *ctx);

/* ---- Dense layer ---------------------------------------------------------------------------
 * Replaces QuantizedNeuralNetwork._quantize_layer_parallel after data collection
 * (quantized_network.py:543-567): the pool fan-out of _quantize_neuron_parallel (:91-121) over
 * neurons j0 <= j < j1 (a shard; pass 0, N1 for the whole layer).
 *   X, Xq : (N0, m) float32, row stride ldx elements.  Xq == X (same pointer) or Xq == NULL
 *           selects the first-layer path (one Gram).
 *   W     : (N0, N1) float32, row stride ldw.
 *   alphabets : n_alphabets alphabets stored back to back, the a-th has K[a] float64 levels.
 *           n_alphabets > 1 batches several (bits, alphabet_scalar) grid points over the same
 *           X, Xq, W (quantize_pretrained_cnn.py:32-48 walks that grid one process pool at a time).
 *   Q_out : n_alphabets matrices (N0, N1) float64, row stride ldq, the a-th at Q_out + a*N0*ldq.
 *           Only columns j0..j1-1 are written.
 */
int gpfq_dense_layer(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0,
                     int64_t m, const float *W, int64_t ldw, int64_t N1, int64_t j0, int64_t j1,
                     const double *alphabets, const int32_t *K, int32_t n_alphabets,
                     double *Q_out, int64_t ldq, uint32_t flags, gpfq_stats *stats);

/* ---- Dense layer, sweep stage from Gram matrices already on the device ------------------------------
 * Multi-GPU sample split of the Gram stage (BASELINE north_star; SURVEY 8e item 4): the two m-length contractions of
 * every greedy step (quantized_network.py:83-89) only enter through G2 = Xq Xq^T and G1 = Xq X^T, which are SUMS over
 * samples.  Each rank of a job contracts its own m / world samples with gpfq_gram_matrices (device outputs), the
 * (N0, N0) fp64 partial matrices are summed with ONE all-reduce (NCCL over NVLink), and every rank then walks its own
 * neurons j0..j1-1 from the summed matrices with this call -- X / Xq are never replicated.
 *   G1, G2 : (N0, N0) float64 DEVICE pointers (GPFQ_X_DEVICE must be set), contiguous rows, lower triangle +
 *            diagonal valid; G1 == G2 or G1 == NULL: first layer (X == Xq).
 *   W, alphabets, K, Q_out, ldq, j0, j1: as gpfq_dense_layer (GPFQ_W_DEVICE / GPFQ_Q_DEVICE say where W / Q_out live).
 */
int gpfq_dense_layer_from_gram(gpfq_ctx *ctx, const double *G1, const double *G2, int64_t N0, const float *W,
                               int64_t ldw, int64_t N1, int64_t j0, int64_t j1, const double *alphabets,
                               const int32_t *K, int32_t n_alphabets, double *Q_out, int64_t ldq, uint32_t flags,
                               gpfq_stats *stats);

/* ---- Conv2D / DepthwiseConv2D channels -------------------------------------------------------
 * Replaces the channel loop of QuantizedCNN._quantize_conv2D_layer_parallel_jit (:844-860) and
 * the pool part of _quantize_channel_parallel_jit (:699-721), i.e. _quantize_filter2D_parallel_jit
 * (:185-233) for every filter f of channels c0 <= c < c0 + n_channels in ONE call.
 *   Xp[i], Xqp[i] : patch matrices of channel c0+i, (kk, n_patches) float32 contiguous
 *                   (kk = kh*kw, row r*kw+col, quantized_network.py:175-179, :789-797).
 *                   Xqp == NULL or Xqp[i] == Xp[i]: first conv layer (X == Xq).
 *   W     : pointer to W[0, 0, 0, 0] of the (kh, kw, C, F) float32 kernel; tap t = r*kw+col of
 *           channel c, filter f is W[t*C*F + c*F + f].
 *   Q_out : float64, same indexing; only channels c0..c0+n_channels-1 are written; the a-th
 *           alphabet's tensor starts at Q_out + a*kk*C*F.
 */
int gpfq_conv_channels(gpfq_ctx *ctx, const float *const *Xp, const float *const *Xqp,
                       int64_t n_patches, int32_t kk, const float *W, int64_t C, int64_t F,
                       int64_t c0, int64_t n_channels, const double *alphabets, const int32_t *K,
                       int32_t n_alphabets, double *Q_out, uint32_t flags, gpfq_stats *stats);

/* ---- Conv2D layer straight from the NHWC activations ------------------------------------------
 * Coarser override point: replaces _build_patch_array (:729-809, tf.image.extract_patches per
 * channel) + the channel loop above.  act/actq: (n_img, H, Wd, C) float32 as stored by
 * _get_layer_data_generator (:468, :494-495); the patch matrices are never materialised on the
 * host.  padding_same: 1 = 'SAME', 0 = 'VALID' (:856).  actq == act or NULL: first layer.
 */
int gpfq_conv_layer_nhwc(gpfq_ctx *ctx, const float *act, const float *actq, int64_t n_img,
                         int64_t H, int64_t Wd, int64_t C, int32_t kh, int32_t kw, int32_t stride_h,
                         int32_t stride_w, int32_t rate_h, int32_t rate_w, int32_t padding_same,
                         const float *W, int64_t F, int64_t c0, int64_t n_channels,
                         const double *alphabets, const int32_t *K, int32_t n_alphabets,
                         double *Q_out, uint32_t flags, gpfq_stats *stats);

/* ---- Conv2D layer split over IMAGES (multi-GPU) -------------------------------------------------------------------
 * The 9-step walk of a channel (quantized_network.py:219-228) sees its patch matrices only through the kk x kk matrices
 * G1 = Xq X^T, G2 = Xq Xq^T, which are sums over patches, i.e. over images.  A multi-GPU job therefore gives each rank
 * n_img / world images of EVERY channel (1 / world of the activations over its own PCIe link, no replication):
 *   gpfq_conv_gram_nhwc        per-channel [G1 | G2] (2 kk^2 float64 per channel, lower triangles + diagonals valid, G1 == G2
 *                              when actq == act / NULL) of channels c0 .. c0+n_ch-1 over the given images.  gram_out lives
 *                              on the device when GPFQ_Q_DEVICE is set, else on the host.  With device activations AND a
 *                              device gram_out, GPFQ_NO_SYNC returns after enqueueing (the all-reduce that follows is
 *                              ordered on the same stream).
 *   (one all-reduce of the n_ch x 2 kk^2 doubles, e.g. NCCL over NVLink: 83 KB for 64 channels)
 *   gpfq_conv_layer_from_gram  the walks of every filter of channels c0 .. c0+n_ch-1 from such matrices (device pointer,
 *                              GPFQ_X_DEVICE; channel i of the range at gram + i * 2 kk^2).  W / Q_out as in
 *                              gpfq_conv_channels (GPFQ_W_DEVICE / GPFQ_Q_DEVICE say where they live).
 * Both serve every kernel up to 128 taps, kh * kw <= 128 (11 x 11 included); a larger kernel returns GPFQ_ERR_UNSUPPORTED
 * (gpfq_conv_layer_nhwc and gpfq_conv_channels still take it, one Dense problem per channel).
 */
int gpfq_conv_gram_nhwc(gpfq_ctx *ctx, const float *act, const float *actq, int64_t n_img, int64_t H, int64_t Wd,
                        int64_t C, int32_t kh, int32_t kw, int32_t stride_h, int32_t stride_w, int32_t rate_h,
                        int32_t rate_w, int32_t padding_same, int64_t c0, int64_t n_channels, double *gram_out,
                        uint32_t flags);
int gpfq_conv_layer_from_gram(gpfq_ctx *ctx, const double *gram, int32_t kk, const float *W, int64_t C, int64_t F,
                              int64_t c0, int64_t n_channels, const double *alphabets, const int32_t *K,
                              int32_t n_alphabets, double *Q_out, uint32_t flags, gpfq_stats *stats);

/* ---- grouped Conv2D (groups > 1: ResNeXt, RegNet, ConvNeXt's Conv2D(groups=C), ShuffleNet) ---------------------------------
 * The counterparts of gpfq_conv_layer_nhwc and gpfq_conv_layer_from_gram for a Conv2D with `groups` groups, in one call.  C is the
 * number of INPUT channels (of the activations / Grams); W and Q_out are the (kh, kw, Cg, F) kernel of the layer, Cg = C / groups:
 * tap t of input channel c and filter f < Fg = F / groups of c's group g = c / Cg is W[t*Cg*F + (c % Cg)*F + g*Fg + f], and input
 * channel c is walked against those Fg filters only (the filters of other groups never see it).  c0 / n_channels index input
 * channels as in the Gram stage (gpfq_conv_gram_nhwc is shared: Grams do not depend on groups), so a channel range may start or
 * end inside a group; only its channels' entries of Q_out are written.  The a-th alphabet's tensor starts at
 * Q_out + a*kk*Cg*F.  groups must be >= 1 and divide both C and F (GPFQ_ERR_ARG otherwise); groups = 1 is the ungrouped call.
 * stats.weights counts kk * n_channels * Fg * n_alphabets.  A depthwise layer (groups = C) is a DepthwiseConv2D with
 * depth_multiplier Fg whose kernel is stored (kh, kw, 1, C*Fg).
 */
int gpfq_conv_layer_nhwc_grouped(gpfq_ctx *ctx, const float *act, const float *actq, int64_t n_img, int64_t H, int64_t Wd,
                                 int64_t C, int32_t kh, int32_t kw, int32_t stride_h, int32_t stride_w, int32_t rate_h,
                                 int32_t rate_w, int32_t padding_same, const float *W, int64_t F, int64_t c0,
                                 int64_t n_channels, const double *alphabets, const int32_t *K, int32_t n_alphabets,
                                 double *Q_out, uint32_t flags, gpfq_stats *stats, int32_t groups);
int gpfq_conv_layer_from_gram_grouped(gpfq_ctx *ctx, const double *gram, int32_t kk, const float *W, int64_t C, int64_t F,
                                      int64_t c0, int64_t n_channels, const double *alphabets, const int32_t *K,
                                      int32_t n_alphabets, double *Q_out, uint32_t flags, gpfq_stats *stats, int32_t groups);

/* ---- per-channel alphabets --------------------------------------------------------------------------------------------------
 * The counterparts of the entry points above with one scale per unit: unit u (a Dense neuron, or the kernel slice W[:, :, ci, f] of
 * a conv layer, ci < Cw = C / groups) walks with the levels fl64(s_u * alphabet[k]) -- one correctly rounded product per level,
 * what NumPy's `rad_u * alphabet` gives for a scalar rad_u -- instead of the alphabet itself.  Every decision and guard is the
 * reference's, taken with the unit's own levels; the outputs are those levels, or the literal 0 of a dead direction.  s_u = 0 gives
 * the unit an all-zero Q.  `scales` is HOST memory, like the alphabets: every scale a call reads must be finite and >= 0
 * (GPFQ_ERR_ARG otherwise, before any work); GPFQ_NO_SYNC all-device calls stay asynchronous.
 *   Dense:  scales[a * N1 + j] for the global neuron j (a shard j0..j1 reads its own slice).
 *   Conv:   scales[a * Cw * F + ci * F + f]; groups as in the _grouped entry points (1 = ungrouped; gpfq_conv_channels: C = Cw).
 *   MSQ:    element i of W rounds with scales[i % n_units] (n_units >= 1: the last axis of a Dense or conv kernel, or its (Cw, F)).
 * A scaled call runs the kernels its per-layer counterpart runs (the tensor-core walk and the int8 residual form apply each neuron's
 * own level step; stats.reserved reports them as for per-layer calls).
 */
int gpfq_dense_layer_scaled(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m, const float *W,
                            int64_t ldw, int64_t N1, int64_t j0, int64_t j1, const double *alphabets, const int32_t *K,
                            int32_t n_alphabets, double *Q_out, int64_t ldq, uint32_t flags, gpfq_stats *stats,
                            const double *scales);
int gpfq_dense_layer_from_gram_scaled(gpfq_ctx *ctx, const double *G1, const double *G2, int64_t N0, const float *W, int64_t ldw,
                                      int64_t N1, int64_t j0, int64_t j1, const double *alphabets, const int32_t *K,
                                      int32_t n_alphabets, double *Q_out, int64_t ldq, uint32_t flags, gpfq_stats *stats,
                                      const double *scales);
int gpfq_conv_channels_scaled(gpfq_ctx *ctx, const float *const *Xp, const float *const *Xqp, int64_t n_patches, int32_t kk,
                              const float *W, int64_t C, int64_t F, int64_t c0, int64_t n_channels, const double *alphabets,
                              const int32_t *K, int32_t n_alphabets, double *Q_out, uint32_t flags, gpfq_stats *stats,
                              const double *scales);
int gpfq_conv_layer_nhwc_scaled(gpfq_ctx *ctx, const float *act, const float *actq, int64_t n_img, int64_t H, int64_t Wd,
                                int64_t C, int32_t kh, int32_t kw, int32_t stride_h, int32_t stride_w, int32_t rate_h,
                                int32_t rate_w, int32_t padding_same, const float *W, int64_t F, int64_t c0, int64_t n_channels,
                                const double *alphabets, const int32_t *K, int32_t n_alphabets, double *Q_out, uint32_t flags,
                                gpfq_stats *stats, int32_t groups, const double *scales);
int gpfq_conv_layer_from_gram_scaled(gpfq_ctx *ctx, const double *gram, int32_t kk, const float *W, int64_t C, int64_t F,
                                     int64_t c0, int64_t n_channels, const double *alphabets, const int32_t *K,
                                     int32_t n_alphabets, double *Q_out, uint32_t flags, gpfq_stats *stats, int32_t groups,
                                     const double *scales);
int gpfq_msq_scaled(gpfq_ctx *ctx, const float *W, int64_t n, const double *alphabet, int32_t K, const double *scales,
                    int64_t n_units, double *Q_out, uint32_t flags);

/* ---- stochastic rounding (SPFQ) --------------------------------------------------------------------------------------------
 * Context state, like gpfq_set_stream: every later call that quantizes (the Dense, conv, _grouped, _scaled, MSQ and bit_round
 * entry points) rounds with this mode; Gram-only calls ignore it.  GPFQ_ROUND_NEAREST (the default) is the reference's nearest-
 * level rounding, bit for bit.  GPFQ_ROUND_STOCHASTIC runs the same path-following walk with the nearest quantizer replaced by
 * unbiased stochastic rounding between the two bracketing levels (Zhang & Saab, SPFQ, 2023):
 *   splitmix64(x)    = the SplitMix64 finaliser of x + 0x9E3779B97F4A7C15 (mod 2^64)
 *   draw(seed, u, t) = (splitmix64(splitmix64(seed ^ splitmix64(u)) ^ t) >> 11) * 2^-53               exact fp64 in [0, 1)
 *   stoc_round(v, A, r) = A[0] unless v > A[0] (NaN included); A[K-1] if v >= A[K-1]; else, with k = max{i : A[i] <= v} and
 *                         p = (v - A[k]) / (A[k+1] - A[k]) in fp64, A[k+1] if r < p else A[k]
 * A greedy step keeps the reference's guards: the literal 0 for a dead direction, stoc_round(w_t) when |d| < 1e-10, else
 * stoc_round(num / nrm^2), with A the alphabet or the unit's levels fl(s_u * A[k]) and r = draw(seeds[a], u, t) for alphabet a.
 * Unit and step ids are global, so results do not depend on shards, channel ranges, conv paths or the Gram split:
 *   Dense: u = neuron (column) j, t = direction;   Conv: u = ci * F + f (ci < C / groups, f the filter), t = tap r * kw + col;
 *   MSQ / bit_round: u = flat element index, t = 0.
 * `seeds` (n_seeds >= 1, host) are copied into the context; a call with more alphabets than seeds, or with an alphabet that is
 * not non-decreasing and finite, returns GPFQ_ERR_ARG before any work.  A stochastic call runs the kernels of its nearest
 * counterpart (the tensor-core walk and the int8 residual form included), with equal stats.method, gram_kernel, reserved and launch
 * count; every option applies as for nearest rounding. */
#define GPFQ_ROUND_NEAREST 0
#define GPFQ_ROUND_STOCHASTIC 1
int gpfq_set_rounding(gpfq_ctx *ctx, int32_t mode, const uint64_t *seeds, int32_t n_seeds);

/* ---- sparse GPFQ: an L1 penalty on every greedy step -----------------------------------------------------------------------
 * Context state, like gpfq_set_rounding: every later Dense, conv, _grouped and _scaled call walks with the penalty lambdas[a] for
 * alphabet a (n_lambdas = 0 turns it off, the default); Gram-only calls, gpfq_msq* and gpfq_bit_round ignore it.  One greedy step
 * of unit u at step t (unit and step as for stochastic rounding), in fp64 with correct rounding:
 *   q = 0                                                    if nrm < 1e-16 (dead direction)
 *   den = fl(nrm * nrm);  v = w_t if |d| < 1e-10 else fl(num / den)           (the reference's value)
 *   tau = fl(lambda / den)
 *   v' = 0 if |v| <= tau, else fl(v - copysign(tau, v))                       (NaN: the comparison is false, v' = NaN)
 *   q = Q(v')   with the call's quantizer: nearest (first level on ties) or stoc_round, levels A[k] or fl(s_u * A[k])
 * In the main branch v' = s_lambda(num) / den with s_lambda(x) = sign(x) max(|x| - lambda, 0): the exact minimiser over real p of
 * 1/2 |u_{t-1} + w_t X_t - p Xq_t|^2 + lambda |p|, then quantized; the shrink in value space also covers the :86 branch.
 * lambda = 0 reproduces the call without the penalty bit for bit (tau = +0; only the sign of a zero v changes, which neither
 * quantizer sees).  Zeros come from an alphabet with a 0 level (odd K of the symmetric alphabets).  Each lambda must be finite
 * and >= 0 (else GPFQ_ERR_ARG from this call, the state unchanged); a quantizing call with more alphabets than lambdas returns
 * GPFQ_ERR_ARG before any work.  The lambdas are staged like the seeds: GPFQ_NO_SYNC calls stay asynchronous.  A call with the
 * penalty runs the kernels of its counterpart without it, with equal stats.method, gram_kernel, reserved and launch count. */
int gpfq_set_l1_penalty(gpfq_ctx *ctx, const double *lambdas, int32_t n_lambdas);

/* ---- MSQ baseline ---------------------------------------------------------------------------
 * Plain nearest-level rounding of every weight (_bit_round_parallel :40-57 applied elementwise,
 * as in quantize_pretrained_mlp.py:97-117).  n elements, contiguous. */
int gpfq_msq(gpfq_ctx *ctx, const float *W, int64_t n, const double *alphabet, int32_t K,
             double *Q_out, uint32_t flags);

/* The scalar quantizer itself on fp64 inputs: out[i] = alphabet[argmin_k |alphabet[k] - t[i]|], first
 * minimal index on ties (_bit_round_parallel, quantized_network.py:40-57). */
int gpfq_bit_round(gpfq_ctx *ctx, const double *t, int64_t n, const double *alphabet, int32_t K,
                   double *out, uint32_t flags);

/* ---- diagnostics ------------------------------------------------------------------------------
 * The Gram stage alone: G2 = Xq Xq^T and (if G1_out != NULL) G1 = Xq X^T over the m samples, fp64,
 * (N0, N0) row-major, LOWER triangle + diagonal valid.  These replace the m-length dot/norm calls
 * of quantized_network.py:83-89; tests check them against an fp64 NumPy Gram.
 * GPFQ_X_DEVICE / GPFQ_Q_DEVICE say where X/Xq and the outputs live.  With GPFQ_Q_DEVICE the matrices are contracted
 * in place into the caller's buffers (zeroed first: entries above the diagonal are finite, so partial matrices of a
 * sample split can be all-reduced whole) and GPFQ_NO_SYNC returns after enqueueing. */
int gpfq_gram_matrices(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0,
                       int64_t m, double *G1_out, double *G2_out, uint32_t flags);

/* The int8-slice tcgen05 contraction the residual-form sweep uses for U += W_r X_r - Q_r Xq_r and D_r = U Xq_r^T
 * (whole ranges of the updates / dots of quantized_network.py:119, :86-89), exposed for tests: C = A B^T with
 * A (M, K) float64 and B (N, K) float32 host arrays -- or, with transposed_b, B given as (K, N) (the X^T slicing path) --
 * keeping digit-slice pairs with s_a + s_b <= D (2..10).  C_out: (M, N) float64 host array. */
int gpfq_debug_slgemm(gpfq_ctx *ctx, const double *A, const float *B, int64_t M, int64_t N, int64_t K, int32_t D,
                      int32_t transposed_b, double *C_out);

#ifdef __cplusplus
}
#endif
#endif /* GPFQ_H_ */
