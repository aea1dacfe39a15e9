// api.cu -- C ABI of libgpfq (include/gpfq.h): context, workspaces, host<->device staging, method choice.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>

#include <algorithm>
#include <cmath>

#include "common.cuh"

// kernels / stages implemented in the other translation units
int dense_gram_path(gpfq_ctx *, const float *, const float *, int64_t, int64_t, int64_t, const float *, int64_t,
                    int64_t, int64_t, const double *, const int *, const int *, int, double *, int64_t, int64_t,
                    gpfq_stats *, const double *G1_pre = nullptr, const double *G2_pre = nullptr, const double *d_scales = nullptr,
                    int64_t u0 = 0);
int dense_stream_path(gpfq_ctx *, const float *, const float *, int64_t, int64_t, int64_t, const float *, int64_t,
                      int64_t, int64_t, const double *, const int *, const int *, int, double *, int64_t, int64_t,
                      gpfq_stats *, const double *d_scales, int64_t u0);
int dense_gram_only(gpfq_ctx *, const float *, const float *, int64_t, int64_t, int64_t, double *, double *);
bool dense_gram_uses_i8(gpfq_ctx *, int64_t, int64_t, bool);
int conv_supported_kk(int kk);
int conv_pick_chunks(gpfq_ctx *, int64_t, int, int64_t *, int, bool, int64_t part_rows = 0);
bool conv_specialised_kk(int kk);
int conv_gram_stage(gpfq_ctx *, int, ConvPtrs, bool, int64_t, int, int, int64_t, double *, bool, int);
int conv_finalize_stage(gpfq_ctx *, const double *, int, int, int, bool, double *);
int conv_sweep_stage(gpfq_ctx *, int, const double *, const float *, double *, int64_t, int64_t, int64_t, int,
                     const double *, const int *, const int *, int, int64_t, const double *);
int im2col_stage(gpfq_ctx *, const float *, int64_t, int, int, int64_t, int64_t, int, int, int, int, int, int, int,
                 int, int, int, int, float *, int64_t);
int msq_stage(gpfq_ctx *, const void *, int, int64_t, const double *, int, int, double *, const double *, int64_t);  // ctx->d_seeds
int nhwc9_plan(int, int, int, int, int, int, int, int, int *, int *);
int corr9_plan(int, int, int, int, int, int, int, int, int, int, bool);
int corr9_pack_stage(gpfq_ctx *, const float *, int64_t, int, int, int64_t, int64_t, int, int, int64_t, int64_t, float *);
int corr9_pick_slots(gpfq_ctx *, int, bool, int64_t, int, int64_t, int);
int corr9_uses_strips(gpfq_ctx *, int);
int corr9_tensor_ok(const float *, const float *);
int conv_corr9_stage(gpfq_ctx *, const float *, const float *, bool, int64_t, int64_t, int64_t, int, int, int64_t, int64_t, int,
                     int, double *, int, int, int, double *, int, int, int);
int conv_corr9_assemble_stage(gpfq_ctx *, const double *, int, const double *, int, bool, int, int, int, double *);
int conv_gram9_nhwc_stage(gpfq_ctx *, const float *, const float *, bool, int64_t, int64_t, int, int, int64_t, int64_t, int,
                          int, int, int, int, int, int, int, double *, int);

// ---------------------------------------------------------------------------------------------
int gpfq_fail(gpfq_ctx *ctx, int code, const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}

int gpfq_ws(gpfq_ctx *ctx, int slot, size_t bytes, void **out) {
    DevBuf &b = ctx->ws[slot];
    if (bytes == 0) bytes = 16;
    if (b.cap < bytes) {
        if (b.p) {
            // pending kernels may still read the old buffer
            CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
            for (auto &s : ctx->aux_stream) if (s) CUDA_TRY(ctx, cudaStreamSynchronize(s));
            CUDA_TRY(ctx, cudaFree(b.p));
            b.p = nullptr;
            b.cap = 0;
        }
        size_t cap = (bytes + ((size_t)1 << 20) - 1) & ~(((size_t)1 << 20) - 1);
        cudaError_t e = cudaMalloc(&b.p, cap);
        if (e != cudaSuccess) {
            b.p = nullptr;
            cudaGetLastError();
            return gpfq_fail(ctx, GPFQ_ERR_OOM, "cudaMalloc of %zu bytes (workspace %d) failed: %s", cap, slot,
                             cudaGetErrorString(e));
        }
        b.cap = cap;
    }
    *out = b.p;
    return GPFQ_OK;
}

int gpfq_pinned(gpfq_ctx *ctx, int slot, size_t bytes, void **out) {
    DevBuf &b = ctx->pinned[slot];
    if (bytes == 0) bytes = 16;
    if (b.cap < bytes) {
        if (b.p) {
            CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            CUDA_TRY(ctx, cudaFreeHost(b.p));
            b.p = nullptr;
            b.cap = 0;
        }
        cudaError_t e = cudaMallocHost(&b.p, bytes);
        if (e != cudaSuccess) {
            b.p = nullptr;
            cudaGetLastError();
            return gpfq_fail(ctx, GPFQ_ERR_OOM, "cudaMallocHost of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        }
        b.cap = bytes;
    }
    *out = b.p;
    return GPFQ_OK;
}

extern "C" int gpfq_version(void) { return GPFQ_VERSION; }

extern "C" int gpfq_create(int device, gpfq_ctx **out) {
    if (!out) return GPFQ_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        return GPFQ_ERR_UNSUPPORTED;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return GPFQ_ERR_CUDA;
    if (prop.major != 10) return GPFQ_ERR_UNSUPPORTED;  // built for sm_100a only
    if (cudaSetDevice(device) != cudaSuccess) return GPFQ_ERR_CUDA;
    gpfq_ctx *ctx = new gpfq_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    bool ok = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    ctx->ring.resize(GPFQ_RING);
    for (auto &r : ctx->ring)
        for (int i = 0; ok && i < 8; ++i) ok = cudaEventCreate(&r.e[i]) == cudaSuccess;
    ctx->cur = &ctx->ring[0];
    for (int i = 0; ok && i < 4; ++i) ok = cudaEventCreateWithFlags(&ctx->ev_copy[i], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok && i < 12; ++i) ok = cudaEventCreateWithFlags(&ctx->ev_chain[i], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok && i < 8; ++i) ok = cudaStreamCreateWithFlags(&ctx->aux_stream[i], cudaStreamNonBlocking) == cudaSuccess;
    if (!ok) {
        delete ctx;
        return GPFQ_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    *out = ctx;
    return GPFQ_OK;
}

extern "C" int64_t gpfq_conv_partial_bytes(gpfq_ctx *ctx) { return ctx ? ctx->conv_part_bytes : 0; }

extern "C" int gpfq_trim(gpfq_ctx *ctx) {
    if (!ctx) return GPFQ_ERR_ARG;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->copy_stream);
    for (auto &s : ctx->aux_stream) if (s) cudaStreamSynchronize(s);
    for (auto &b : ctx->ws) {
        if (b.p) cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    for (auto &b : ctx->pinned) {
        if (b.p) cudaFreeHost(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    ctx->alph_cache.clear();
    ctx->alph_used = 0;
    ctx->i8_oom_bytes = 0;
    return GPFQ_OK;
}

extern "C" void gpfq_destroy(gpfq_ctx *ctx) {
    if (!ctx) return;
    gpfq_trim(ctx);
    for (auto &r : ctx->ring)
        for (auto &e : r.e) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->ev_copy) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->ev_chain) if (e) cudaEventDestroy(e);
    for (auto &s : ctx->aux_stream) if (s) cudaStreamDestroy(s);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;
}

extern "C" const char *gpfq_last_error(const gpfq_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

extern "C" int gpfq_set_option(gpfq_ctx *ctx, const char *key, int64_t value) {
    if (!ctx || !key) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (!strcmp(key, "gram_kernel")) {          // 0 auto, 1 fp64 DMMA, 2 int8 slices on tcgen05
        if (value < 0 || value > 2) return gpfq_fail(ctx, GPFQ_ERR_ARG, "gram_kernel must be 0, 1 or 2");
        ctx->gram_variant = (int)value;
    } else if (!strcmp(key, "i8_pairs_d")) {    // 0 default; else keep slice pairs with k + l <= value
        if (value != 0 && (value < 2 || value > 10)) return gpfq_fail(ctx, GPFQ_ERR_ARG, "i8_pairs_d must be 0 or 2..10");
        ctx->i8_pairs_d = (int)value;
    } else if (!strcmp(key, "corr_pack")) {   // correlation form, image packing: 0 auto, 1 always (tests), 2 never
        if (value < 0 || value > 2) return gpfq_fail(ctx, GPFQ_ERR_ARG, "corr_pack must be 0, 1 or 2");
        ctx->corr_pack = (int)value;
    } else if (!strcmp(key, "corr_small")) {   // correlation form also on images below 128 pixels (tests)
        ctx->corr_direct_small = value != 0;
    } else if (!strcmp(key, "corr_rows")) {   // correlation form: rows per band (0 auto, 4, 6 or 8)
        if (value != 0 && value != 4 && value != 6 && value != 8) return gpfq_fail(ctx, GPFQ_ERR_ARG, "corr_rows must be 0, 4, 6 or 8");
        ctx->corr_rb = (int)value;
    } else if (!strcmp(key, "corr_strip")) {    // correlation form on small images: 0 strip kernel (W in {8, 14, 16, 28, 32, 56, 64}), 2 band kernel
        if (value != 0 && value != 2) return gpfq_fail(ctx, GPFQ_ERR_ARG, "corr_strip must be 0 or 2");
        ctx->corr_strip = (int)value;
    } else if (!strcmp(key, "conv_kernel")) {   // 0 TMA-staged / correlation form, 1 direct LDG, 2 generic, 3 NHWC planes kernel
        if (value < 0 || value > 3) return gpfq_fail(ctx, GPFQ_ERR_ARG, "conv_kernel must be 0, 1, 2 or 3");
        ctx->conv_variant = (int)value;
    } else if (!strcmp(key, "sweep_outer")) {   // 0 auto, 1 Gram rows, 2 carried residuals (low-rank form, m << N0),
        // 3 carried residuals as ONE chain (no two-stream split of the neurons)
        if (value < 0 || value > 3) return gpfq_fail(ctx, GPFQ_ERR_ARG, "sweep_outer must be 0, 1, 2 or 3");
        ctx->lowrank_variant = (int)value;
    } else if (!strcmp(key, "sweep_walk")) {    // range walk of the Gram-row sweep (one symmetric equispaced alphabet): 0 auto,
                                                 // 1 tensor-core walk (sweep_tc.cu), 2 sweep_pipe / sweep_tile kernels
        if (value < 0 || value > 2) return gpfq_fail(ctx, GPFQ_ERR_ARG, "sweep_walk must be 0, 1 or 2");
        ctx->sweep_walk = (int)value;
    } else if (!strcmp(key, "sweep_i8")) {      // residual-form sweep contractions: 0 auto, 1 int8 slices on tcgen05, 2 fp64 DMMA
        if (value < 0 || value > 2) return gpfq_fail(ctx, GPFQ_ERR_ARG, "sweep_i8 must be 0, 1 or 2");
        ctx->sweep_i8 = (int)value;
    } else {
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "unknown option '%s'", key);
    }
    return GPFQ_OK;
}

extern "C" int gpfq_set_rounding(gpfq_ctx *ctx, int32_t mode, const uint64_t *seeds, int32_t n_seeds) {
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (mode == GPFQ_ROUND_NEAREST) {
        ctx->rounding = mode;
        ctx->seeds.clear();
        return GPFQ_OK;
    }
    if (mode != GPFQ_ROUND_STOCHASTIC) return gpfq_fail(ctx, GPFQ_ERR_ARG, "unknown rounding mode %d", mode);
    if (!seeds || n_seeds < 1) return gpfq_fail(ctx, GPFQ_ERR_ARG, "stochastic rounding needs n_seeds >= 1 seeds");
    ctx->rounding = mode;
    ctx->seeds.assign(seeds, seeds + n_seeds);
    return GPFQ_OK;
}

extern "C" int gpfq_set_l1_penalty(gpfq_ctx *ctx, const double *lambdas, int32_t n_lambdas) {
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (n_lambdas < 0 || (n_lambdas > 0 && !lambdas)) return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad n_lambdas=%d", n_lambdas);
    for (int i = 0; i < n_lambdas; ++i)
        if (!std::isfinite(lambdas[i]) || !(lambdas[i] >= 0.0))
            return gpfq_fail(ctx, GPFQ_ERR_ARG, "L1 penalty %d must be finite and >= 0", i);
    ctx->l1.assign(lambdas, lambdas + n_lambdas);
    return GPFQ_OK;
}

extern "C" int gpfq_set_stream(gpfq_ctx *ctx, void *cuda_stream) {
    if (!ctx) return GPFQ_ERR_ARG;
    cudaStream_t next = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    if (next != ctx->stream) {
        // workspaces are shared between calls: work queued on the old stream must finish before the new
        // stream may reuse them
        cudaSetDevice(ctx->device);
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) cudaGetLastError();
        ctx->stream = next;
    }
    return GPFQ_OK;
}

// ---------------------------------------------------------------------------------------------
// alphabets: validate, flatten to device (levels + prefix offsets)
// ---------------------------------------------------------------------------------------------
struct Alphabets {
    const double *d_levels = nullptr;
    const int *d_koff = nullptr;
    const int *d_flags = nullptr;  // per alphabet: 1 = ascending and equispaced (fast rounding window)
    std::vector<int> h_koff, h_flags;
};

static int alphabet_is_equispaced(const double *a, int K) {
    if (K < 2) return 0;
    const double step = (a[K - 1] - a[0]) / (K - 1);
    if (!(step > 0.0) || !std::isfinite(step)) return 0;
    for (int k = 0; k < K; ++k)
        if (!(fabs(a[k] - (a[0] + k * step)) <= 0.01 * step)) return 0;
    return 1;
}

static int upload_alphabets(gpfq_ctx *ctx, const double *alphabets, const int32_t *K, int n_alph, Alphabets *out) {
    if (!alphabets || !K || n_alph < 1 || n_alph > 1024) return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad alphabet arguments");
    out->h_koff.assign(n_alph + 1, 0);
    for (int a = 0; a < n_alph; ++a) {
        if (K[a] < 1 || K[a] > GPFQ_MAX_K)
            return gpfq_fail(ctx, GPFQ_ERR_ARG, "alphabet %d has %d levels (supported: 1..%d)", a, K[a], GPFQ_MAX_K);
        out->h_koff[a + 1] = out->h_koff[a] + K[a];
    }
    const size_t nlev = out->h_koff[n_alph];
    const size_t lev_bytes = nlev * sizeof(double);
    out->h_flags.assign(n_alph, 0);
    for (int a = 0; a < n_alph; ++a) out->h_flags[a] = alphabet_is_equispaced(alphabets + out->h_koff[a], K[a]);
    const size_t koff_bytes = (n_alph + 1) * sizeof(int);
    const size_t bytes = (lev_bytes + koff_bytes + n_alph * sizeof(int) + 15) & ~(size_t)15;
    std::vector<char> blob(bytes, 0);
    memcpy(blob.data(), alphabets, lev_bytes);
    memcpy(blob.data() + lev_bytes, out->h_koff.data(), koff_bytes);
    memcpy(blob.data() + lev_bytes + koff_bytes, out->h_flags.data(), n_alph * sizeof(int));
    const size_t cap = (size_t)1 << 20;
    char *d = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_ALPH, cap, (void **)&d));
    const AlphEntry *hit = nullptr;
    for (const auto &e : ctx->alph_cache)
        if (e.blob.size() == bytes && memcmp(e.blob.data(), blob.data(), bytes) == 0) { hit = &e; break; }
    if (!hit) {
        if (bytes > cap) return gpfq_fail(ctx, GPFQ_ERR_ARG, "alphabet table too large");
        if (ctx->alph_used + bytes > cap || ctx->alph_cache.size() >= 256) {
            CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));  // kernels may still read the old entries
            ctx->alph_cache.clear();
            ctx->alph_used = 0;
        }
        ctx->alph_cache.emplace_back();
        AlphEntry &e = ctx->alph_cache.back();
        e.blob.swap(blob);
        e.off = ctx->alph_used;
        ctx->alph_used += bytes;
        CUDA_TRY(ctx, cudaMemcpyAsync(d + e.off, e.blob.data(), bytes, cudaMemcpyHostToDevice, ctx->stream));
        hit = &e;
    }
    ctx->h_alph = alphabets;   // host view for the duration of the call (the int8 sweep contractions need the level spacing)
    ctx->h_koff = out->h_koff.data();
    ctx->h_flags = out->h_flags.data();
    out->d_levels = reinterpret_cast<const double *>(d + hit->off);
    out->d_koff = reinterpret_cast<const int *>(d + hit->off + lev_bytes);
    out->d_flags = reinterpret_cast<const int *>(d + hit->off + lev_bytes + koff_bytes);
    return GPFQ_OK;
}

// Per-unit scales (per-channel alphabets): n_alph rows of n scales, row a read from scales + a * lds, each finite and >= 0.
static int check_scales(gpfq_ctx *ctx, const double *scales, int n_alph, int64_t n, int64_t lds) {
    if (!scales) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL scales");
    for (int a = 0; a < n_alph; ++a)
        for (int64_t j = 0; j < n; ++j) {
            const double v = scales[a * lds + j];
            if (!(v >= 0.0) || !std::isfinite(v))
                return gpfq_fail(ctx, GPFQ_ERR_ARG, "scale %lld of alphabet %d is %g (scales must be finite and >= 0)", (long long)j, a, v);
        }
    return GPFQ_OK;
}

// ... staged on the device as (n_alph, n) on the call's stream, like the alphabets (pageable source: staged before the call
// returns, so GPFQ_NO_SYNC calls stay asynchronous).  The kernels of the call read them in stream order.
static int upload_scales(gpfq_ctx *ctx, const double *scales, int n_alph, int64_t n, int64_t lds, const double **out) {
    double *d = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_SCALES, (size_t)n_alph * n * sizeof(double), (void **)&d));
    CUDA_TRY(ctx, cudaMemcpy2DAsync(d, n * sizeof(double), scales, lds * sizeof(double), n * sizeof(double), n_alph,
                                    cudaMemcpyHostToDevice, ctx->stream));
    *out = d;
    return GPFQ_OK;
}

// Stochastic rounding: a seed for every alphabet of the call, and levels the bracketing search can rely on (non-decreasing and
// finite).  Nothing to check for nearest rounding.
static int check_rounding(gpfq_ctx *ctx, const double *alphabets, const int32_t *K, int n_alph) {
    if (ctx->rounding != GPFQ_ROUND_STOCHASTIC || !alphabets || !K) return GPFQ_OK;
    if ((size_t)n_alph > ctx->seeds.size())
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "%d alphabets but %zu stochastic-rounding seeds", n_alph, ctx->seeds.size());
    int64_t off = 0;
    for (int a = 0; a < n_alph; ++a) {
        if (K[a] < 1 || K[a] > GPFQ_MAX_K) return GPFQ_OK;   // upload_alphabets reports it
        for (int k = 0; k < K[a]; ++k) {
            const double v = alphabets[off + k];
            if (!std::isfinite(v) || (k > 0 && !(alphabets[off + k - 1] <= v)))
                return gpfq_fail(ctx, GPFQ_ERR_ARG, "stochastic rounding: alphabet %d must be non-decreasing and finite", a);
        }
        off += K[a];
    }
    return GPFQ_OK;
}

// The seeds of this call on the device (one per alphabet, read by the walks in stream order; pageable source: staged before the
// call returns, so GPFQ_NO_SYNC calls stay asynchronous), or nullptr for nearest rounding and for Gram-only calls.
static int stage_seeds(gpfq_ctx *ctx, int n_alph) {
    ctx->d_seeds = nullptr;
    if (ctx->rounding != GPFQ_ROUND_STOCHASTIC || ctx->gram_only_out) return GPFQ_OK;
    uint64_t *d = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_SEEDS, (size_t)n_alph * sizeof(uint64_t), (void **)&d));
    CUDA_TRY(ctx, cudaMemcpyAsync(d, ctx->seeds.data(), (size_t)n_alph * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    ctx->d_seeds = d;
    return GPFQ_OK;
}

// L1 penalty: one lambda for every alphabet of the call.  Nothing to check when it is off.
static int check_l1(gpfq_ctx *ctx, int n_alph) {
    if (ctx->l1.empty() || (size_t)n_alph <= ctx->l1.size()) return GPFQ_OK;
    return gpfq_fail(ctx, GPFQ_ERR_ARG, "%d alphabets but %zu L1 penalties", n_alph, ctx->l1.size());
}

// The lambdas of this call on the device (one per alphabet, read by the walks in stream order; staged like the seeds, so
// GPFQ_NO_SYNC calls stay asynchronous), or nullptr when the penalty is off and for Gram-only calls.
static int stage_l1(gpfq_ctx *ctx, int n_alph) {
    ctx->d_l1 = nullptr;
    if (ctx->l1.empty() || ctx->gram_only_out) return GPFQ_OK;
    double *d = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_L1_LAMBDA, (size_t)n_alph * sizeof(double), (void **)&d));
    CUDA_TRY(ctx, cudaMemcpyAsync(d, ctx->l1.data(), (size_t)n_alph * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    ctx->d_l1 = d;
    return GPFQ_OK;
}

cudaError_t gpfq_record(gpfq_ctx *ctx, int which, cudaStream_t s) {
    ctx->cur->rec[which] = true;
    return cudaEventRecord(ctx->cur->e[which], s);
}

static void begin_call(gpfq_ctx *ctx, int kind) {
    ctx->cur = &ctx->ring[ctx->calls % GPFQ_RING];
    ctx->calls++;
    for (bool &r : ctx->cur->rec) r = false;
    ctx->cur->kind = kind;
    ctx->cur->st = gpfq_stats{};
    ctx->launches = 0;
}

static float ev_ms(const CallRecord &r, int a, int b) {
    float ms = 0.f;
    if (!r.rec[a] || !r.rec[b]) return 0.f;
    if (cudaEventElapsedTime(&ms, r.e[a], r.e[b]) != cudaSuccess) { cudaGetLastError(); return 0.f; }
    return ms;
}

// events: 0 call start, 5 inputs resident, 2 main stage start, 3 main stage end, 4 sweep end, 6 before D2H, 1 call end
static void fill_times(CallRecord &r) {
    gpfq_stats &st = r.st;
    st.ms_total = ev_ms(r, 0, 1);
    st.ms_h2d = ev_ms(r, 0, 5);
    if (r.kind == 1) {
        st.ms_stream = ev_ms(r, 2, 3);
        st.ms_d2h = ev_ms(r, 6, 1);
    } else {
        st.ms_gram = ev_ms(r, 2, 3);
        st.ms_sweep = ev_ms(r, 3, 4);
        st.ms_d2h = r.kind == 0 ? ev_ms(r, 6, 1) : ev_ms(r, 4, 1);
    }
}

static void end_call(gpfq_ctx *ctx, gpfq_stats *stats, bool synced) {
    CallRecord &r = *ctx->cur;
    if (stats) r.st = *stats;  // static fields filled by the stage code
    r.st.kernel_launches = ctx->launches;
    if (synced) fill_times(r);
    if (stats) *stats = r.st;
}

extern "C" int gpfq_query_stats(gpfq_ctx *ctx, int32_t calls_back, gpfq_stats *out) {
    if (!ctx || !out || calls_back < 0 || calls_back >= GPFQ_RING || calls_back >= ctx->calls) return GPFQ_ERR_ARG;
    CallRecord &r = ctx->ring[(ctx->calls - 1 - calls_back) % GPFQ_RING];
    fill_times(r);
    *out = r.st;
    return GPFQ_OK;
}

// ---------------------------------------------------------------------------------------------
// Dense
// ---------------------------------------------------------------------------------------------
static int choose_dense_method(gpfq_ctx *ctx, uint32_t flags, int64_t N0, int64_t m, int64_t nj, bool same, int n_alph) {
    const uint32_t want = flags & GPFQ_METHOD_MASK;
    if (want != GPFQ_METHOD_AUTO) return (int)want;
    // Cost table (DESIGN.md "method choice"), calibrated on B200 (tools/dense_bench.py), fp64-pipe slots at the measured
    // 18.5 T slots/s:
    //   streaming : 3 slots per (sample, direction, neuron), per alphabet; a step (row ingest + CTA-wide reduction +
    //               decision) takes 0.6 us + 0.37 us per 2048 samples; long sample axes (residual not in registers) ~4x
    //   Gram+sweep: Gram stage (DMMA: m N0^2 / 2 slots per Gram; int8 tcgen05: see below) once, then per alphabet
    //               N0^2 nj slots of contractions and a serial walk of ~0.6 us per direction and round of CTAs
    const double slots_per_s = 18.5e12 * 0.6;
    const bool u_in_regs = m <= 512 * 16;
    const double waves = ceil((double)nj / (double)ctx->sm_count);
    const double epv = ceil((double)m / 2048.0);
    double t_stream = n_alph * (3.0 * (double)m * N0 * nj / slots_per_s * (u_in_regs ? 1.0 : 4.0));
    const double t_steps = n_alph * waves * (double)N0 * (0.6e-6 + 0.37e-6 * (u_in_regs ? epv : 4.0 * epv));
    if (t_stream < t_steps) t_stream = t_steps;
    double t_gram_stage = (same ? 0.5 : 1.0) * (double)m * N0 * N0 / slots_per_s;
    if (dense_gram_uses_i8(ctx, N0, m, same)) {
        // int8 slices on tcgen05: 15 slice pairs, lower-triangular 128 x 256 tiles, ~2e15 int8 op/s sustained (the
        // single-CTA tile is bound by the L2 -> shared-memory operand stream), plus the slicing pass and launches
        const double tile_area = (double)N0 * N0 * 0.5 + 192.0 * N0;
        t_gram_stage = (same ? 1.0 : 2.0) * (15.0 * 2.0 * tile_area * (double)m / 2.0e15 + 24.0 * N0 * (double)m / 5e12) + 4e-5;
    }
    const double sweep_rounds = ceil((double)ceil_div64(nj, 32) * n_alph / (2.0 * ctx->sm_count));
    double t_gram = t_gram_stage + n_alph * ((double)N0 * N0 * nj / slots_per_s) + sweep_rounds * (double)N0 * 0.6e-6;
    const double gram_bytes = (same ? 1.0 : 2.0) * 8.0 * N0 * N0;
    if (gram_bytes > 48e9) return GPFQ_METHOD_STREAM_FAST;
    return t_gram < t_stream ? GPFQ_METHOD_GRAM : GPFQ_METHOD_STREAM_FAST;
}

// scales (nullable, host): per-neuron scales, neuron j of alphabet a at scales[a * lds + j].
static int dense_layer(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m, const float *W,
                       int64_t ldw, int64_t N1, int64_t j0, int64_t j1, const double *alphabets, const int32_t *K, int32_t n_alph,
                       double *Q_out, int64_t ldq, uint32_t flags, gpfq_stats *stats, const double *scales, int64_t lds,
                       int64_t ubase = 0) {
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (stats) memset(stats, 0, sizeof(*stats));
    if (!X || !W || !Q_out) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL X, W or Q_out");
    if (N0 < 1 || m < 1 || N1 < 1 || ldx < m || ldw < N1 || ldq < N1 || j0 < 0 || j1 > N1 || j0 > j1)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad shape: N0=%lld m=%lld N1=%lld ldx=%lld ldw=%lld ldq=%lld j0=%lld j1=%lld",
                         (long long)N0, (long long)m, (long long)N1, (long long)ldx, (long long)ldw, (long long)ldq,
                         (long long)j0, (long long)j1);
    if (N0 > 2000000 || m > ((int64_t)1 << 40)) return gpfq_fail(ctx, GPFQ_ERR_ARG, "shape too large");
    if ((flags & GPFQ_NO_SYNC) && (flags & GPFQ_ALL_DEVICE) != GPFQ_ALL_DEVICE)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "GPFQ_NO_SYNC needs all-device pointers");
    const int64_t nj = j1 - j0;
    if (scales && n_alph >= 1) GPFQ_TRY(check_scales(ctx, scales + j0, n_alph, nj, lds));
    GPFQ_TRY(check_rounding(ctx, alphabets, K, n_alph));
    GPFQ_TRY(check_l1(ctx, n_alph));
    if (nj == 0) return GPFQ_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const bool same = (Xq == nullptr || Xq == X);
    cudaStream_t s = ctx->stream;
    const int method = choose_dense_method(ctx, flags, N0, m, nj, same, n_alph);
    begin_call(ctx, method == GPFQ_METHOD_GRAM ? 0 : 1);
    CUDA_TRY(ctx, gpfq_record(ctx, 0, s));

    Alphabets al;
    GPFQ_TRY(upload_alphabets(ctx, alphabets, K, n_alph, &al));
    GPFQ_TRY(stage_seeds(ctx, n_alph));
    GPFQ_TRY(stage_l1(ctx, n_alph));
    const double *d_scales = nullptr;
    if (scales) GPFQ_TRY(upload_scales(ctx, scales + j0, n_alph, nj, lds, &d_scales));

    const float *dX = X, *dXq = same ? X : Xq, *dW = W;
    int64_t dldx = ldx, dldw = ldw, dj0 = j0;
    if (!(flags & GPFQ_X_DEVICE)) {
        float *bx = nullptr, *bq = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_X, (size_t)N0 * m * sizeof(float), (void **)&bx));
        CUDA_TRY(ctx, cudaMemcpy2DAsync(bx, m * sizeof(float), X, ldx * sizeof(float), m * sizeof(float), N0,
                                        cudaMemcpyHostToDevice, s));
        dX = dXq = bx;
        if (!same) {
            GPFQ_TRY(gpfq_ws(ctx, WS_XQ, (size_t)N0 * m * sizeof(float), (void **)&bq));
            CUDA_TRY(ctx, cudaMemcpy2DAsync(bq, m * sizeof(float), Xq, ldx * sizeof(float), m * sizeof(float), N0,
                                            cudaMemcpyHostToDevice, s));
            dXq = bq;
        }
        dldx = m;
    }
    if (!(flags & GPFQ_W_DEVICE)) {
        float *bw = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_W, (size_t)N0 * nj * sizeof(float), (void **)&bw));
        CUDA_TRY(ctx, cudaMemcpy2DAsync(bw, nj * sizeof(float), W + j0, ldw * sizeof(float), nj * sizeof(float), N0,
                                        cudaMemcpyHostToDevice, s));
        dW = bw;
        dldw = nj;
        dj0 = 0;
    }
    double *dQ = Q_out;
    int64_t dldq = ldq, col0 = j0;
    if (!(flags & GPFQ_Q_DEVICE)) {
        GPFQ_TRY(gpfq_ws(ctx, WS_Q, (size_t)n_alph * N0 * nj * sizeof(double), (void **)&dQ));
        dldq = nj;
        col0 = 0;
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 5, s));

    if (method == GPFQ_METHOD_GRAM)
        GPFQ_TRY(dense_gram_path(ctx, dX, dXq, dldx, N0, m, dW, dldw, dj0, nj, al.d_levels, al.d_koff, al.d_flags, n_alph, dQ,
                                 dldq, col0, stats, nullptr, nullptr, d_scales, ubase + j0));
    else {
        ctx->stream_literal = (method == GPFQ_METHOD_STREAM);
        GPFQ_TRY(dense_stream_path(ctx, dX, dXq, dldx, N0, m, dW, dldw, dj0, nj, al.d_levels, al.h_koff.data(),
                                   al.h_flags.data(), n_alph, dQ, dldq, col0, stats, d_scales, ubase + j0));
        if (stats) stats->method = method >> 4;
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 6, s));
    if (!(flags & GPFQ_Q_DEVICE)) {
        for (int a = 0; a < n_alph; ++a)
            CUDA_TRY(ctx, cudaMemcpy2DAsync(Q_out + (int64_t)a * N0 * ldq + j0, ldq * sizeof(double),
                                            dQ + (int64_t)a * N0 * nj, nj * sizeof(double), nj * sizeof(double), N0,
                                            cudaMemcpyDeviceToHost, s));
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 1, s));
    if (stats) stats->weights = N0 * nj * n_alph;
    const bool synced = !(flags & GPFQ_NO_SYNC);
    if (synced) CUDA_TRY(ctx, cudaStreamSynchronize(s));
    end_call(ctx, stats, synced);
    return GPFQ_OK;
}

extern "C" int gpfq_dense_layer(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m,
                                const float *W, int64_t ldw, int64_t N1, int64_t j0, int64_t j1,
                                const double *alphabets, const int32_t *K, int32_t n_alph, double *Q_out,
                                int64_t ldq, uint32_t flags, gpfq_stats *stats) {
    return dense_layer(ctx, X, Xq, ldx, N0, m, W, ldw, N1, j0, j1, alphabets, K, n_alph, Q_out, ldq, flags, stats, nullptr, 0);
}

extern "C" int gpfq_dense_layer_scaled(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m,
                                       const float *W, int64_t ldw, int64_t N1, int64_t j0, int64_t j1,
                                       const double *alphabets, const int32_t *K, int32_t n_alph, double *Q_out,
                                       int64_t ldq, uint32_t flags, gpfq_stats *stats, const double *scales) {
    if (ctx && !scales) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL scales");
    return dense_layer(ctx, X, Xq, ldx, N0, m, W, ldw, N1, j0, j1, alphabets, K, n_alph, Q_out, ldq, flags, stats, scales, N1);
}

// Sweep stage alone, from Gram matrices the caller already holds on the device (sample-split Gram stage of a multi-GPU
// job: every rank contracts its m / world samples with gpfq_gram_matrices, the (N0, N0) partial Grams are summed with
// one NCCL all-reduce, then each rank sweeps its own neurons from the summed matrices).
static int dense_layer_from_gram(gpfq_ctx *ctx, const double *G1, const double *G2, int64_t N0, const float *W, int64_t ldw,
                                 int64_t N1, int64_t j0, int64_t j1, const double *alphabets, const int32_t *K, int32_t n_alph,
                                 double *Q_out, int64_t ldq, uint32_t flags, gpfq_stats *stats, const double *scales) {
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (stats) memset(stats, 0, sizeof(*stats));
    if (!G2 || !W || !Q_out) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL G2, W or Q_out");
    if (N0 < 1 || N1 < 1 || ldw < N1 || ldq < N1 || j0 < 0 || j1 > N1 || j0 > j1)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad shape: N0=%lld N1=%lld ldw=%lld ldq=%lld j0=%lld j1=%lld", (long long)N0,
                         (long long)N1, (long long)ldw, (long long)ldq, (long long)j0, (long long)j1);
    if (!(flags & GPFQ_X_DEVICE)) return gpfq_fail(ctx, GPFQ_ERR_ARG, "G1 / G2 must be device pointers (GPFQ_X_DEVICE)");
    if ((flags & GPFQ_NO_SYNC) && (flags & GPFQ_ALL_DEVICE) != GPFQ_ALL_DEVICE)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "GPFQ_NO_SYNC needs all-device pointers");
    const int64_t nj = j1 - j0;
    if (scales && n_alph >= 1) GPFQ_TRY(check_scales(ctx, scales + j0, n_alph, nj, N1));
    GPFQ_TRY(check_rounding(ctx, alphabets, K, n_alph));
    GPFQ_TRY(check_l1(ctx, n_alph));
    if (nj == 0) return GPFQ_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    begin_call(ctx, 0);
    CUDA_TRY(ctx, gpfq_record(ctx, 0, s));
    Alphabets al;
    GPFQ_TRY(upload_alphabets(ctx, alphabets, K, n_alph, &al));
    GPFQ_TRY(stage_seeds(ctx, n_alph));
    GPFQ_TRY(stage_l1(ctx, n_alph));
    const double *d_scales = nullptr;
    if (scales) GPFQ_TRY(upload_scales(ctx, scales + j0, n_alph, nj, N1, &d_scales));
    const float *dW = W;
    int64_t dldw = ldw, dj0 = j0;
    if (!(flags & GPFQ_W_DEVICE)) {
        float *bw = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_W, (size_t)N0 * nj * sizeof(float), (void **)&bw));
        CUDA_TRY(ctx, cudaMemcpy2DAsync(bw, nj * sizeof(float), W + j0, ldw * sizeof(float), nj * sizeof(float), N0,
                                        cudaMemcpyHostToDevice, s));
        dW = bw;
        dldw = nj;
        dj0 = 0;
    }
    double *dQ = Q_out;
    int64_t dldq = ldq, col0 = j0;
    if (!(flags & GPFQ_Q_DEVICE)) {
        GPFQ_TRY(gpfq_ws(ctx, WS_Q, (size_t)n_alph * N0 * nj * sizeof(double), (void **)&dQ));
        dldq = nj;
        col0 = 0;
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 5, s));
    GPFQ_TRY(dense_gram_path(ctx, nullptr, nullptr, 0, N0, 0, dW, dldw, dj0, nj, al.d_levels, al.d_koff, al.d_flags, n_alph,
                             dQ, dldq, col0, stats, (G1 == nullptr || G1 == G2) ? nullptr : G1, G2, d_scales, j0));
    CUDA_TRY(ctx, gpfq_record(ctx, 6, s));
    if (!(flags & GPFQ_Q_DEVICE)) {
        for (int a = 0; a < n_alph; ++a)
            CUDA_TRY(ctx, cudaMemcpy2DAsync(Q_out + (int64_t)a * N0 * ldq + j0, ldq * sizeof(double),
                                            dQ + (int64_t)a * N0 * nj, nj * sizeof(double), nj * sizeof(double), N0,
                                            cudaMemcpyDeviceToHost, s));
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 1, s));
    if (stats) stats->weights = N0 * nj * n_alph;
    const bool synced = !(flags & GPFQ_NO_SYNC);
    if (synced) CUDA_TRY(ctx, cudaStreamSynchronize(s));
    end_call(ctx, stats, synced);
    return GPFQ_OK;
}

extern "C" int gpfq_dense_layer_from_gram(gpfq_ctx *ctx, const double *G1, const double *G2, int64_t N0, const float *W,
                                          int64_t ldw, int64_t N1, int64_t j0, int64_t j1, const double *alphabets,
                                          const int32_t *K, int32_t n_alph, double *Q_out, int64_t ldq, uint32_t flags,
                                          gpfq_stats *stats) {
    return dense_layer_from_gram(ctx, G1, G2, N0, W, ldw, N1, j0, j1, alphabets, K, n_alph, Q_out, ldq, flags, stats, nullptr);
}

extern "C" int gpfq_dense_layer_from_gram_scaled(gpfq_ctx *ctx, const double *G1, const double *G2, int64_t N0, const float *W,
                                                 int64_t ldw, int64_t N1, int64_t j0, int64_t j1, const double *alphabets,
                                                 const int32_t *K, int32_t n_alph, double *Q_out, int64_t ldq, uint32_t flags,
                                                 gpfq_stats *stats, const double *scales) {
    if (ctx && !scales) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL scales");
    return dense_layer_from_gram(ctx, G1, G2, N0, W, ldw, N1, j0, j1, alphabets, K, n_alph, Q_out, ldq, flags, stats, scales);
}

// Diagnostics: the Gram stage alone (tests check it against an fp64 NumPy Gram).
// G1_out/G2_out: (N0, N0) fp64, lower triangle + diagonal valid; G1_out may be NULL.
extern "C" int gpfq_gram_matrices(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m,
                                  double *G1_out, double *G2_out, uint32_t flags) {
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (!X || !G2_out || N0 < 1 || m < 1 || ldx < m) return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad arguments");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const bool same = (Xq == nullptr || Xq == X);
    cudaStream_t s = ctx->stream;
    const float *dX = X, *dXq = same ? X : Xq;
    int64_t dld = ldx;
    if (!(flags & GPFQ_X_DEVICE)) {
        float *bx = nullptr, *bq = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_X, (size_t)N0 * m * sizeof(float), (void **)&bx));
        CUDA_TRY(ctx, cudaMemcpy2DAsync(bx, m * sizeof(float), X, ldx * sizeof(float), m * sizeof(float), N0,
                                        cudaMemcpyHostToDevice, s));
        dX = dXq = bx;
        if (!same) {
            GPFQ_TRY(gpfq_ws(ctx, WS_XQ, (size_t)N0 * m * sizeof(float), (void **)&bq));
            CUDA_TRY(ctx, cudaMemcpy2DAsync(bq, m * sizeof(float), Xq, ldx * sizeof(float), m * sizeof(float), N0,
                                            cudaMemcpyHostToDevice, s));
            dXq = bq;
        }
        dld = m;
    }
    double *g1 = nullptr, *g2 = nullptr;
    if (flags & GPFQ_Q_DEVICE) {
        // device outputs (the sample-split Gram stage of a multi-GPU job): contract straight into the caller's
        // matrices, zeroed first so that what an all-reduce sums above the diagonal is finite
        if (!same && !G1_out) return gpfq_fail(ctx, GPFQ_ERR_ARG, "G1_out is NULL but Xq != X");
        g2 = G2_out;
        g1 = same ? g2 : G1_out;
        CUDA_TRY(ctx, cudaMemsetAsync(g2, 0, (size_t)N0 * N0 * sizeof(double), s));
        if (!same) CUDA_TRY(ctx, cudaMemsetAsync(g1, 0, (size_t)N0 * N0 * sizeof(double), s));
        GPFQ_TRY(dense_gram_only(ctx, dX, dXq, dld, N0, m, g1, g2));
        if (same && G1_out && G1_out != G2_out)
            CUDA_TRY(ctx, cudaMemcpyAsync(G1_out, g2, (size_t)N0 * N0 * sizeof(double), cudaMemcpyDeviceToDevice, s));
        if (!(flags & GPFQ_NO_SYNC)) CUDA_TRY(ctx, cudaStreamSynchronize(s));
        return GPFQ_OK;
    }
    GPFQ_TRY(gpfq_ws(ctx, WS_G2, (size_t)N0 * N0 * sizeof(double), (void **)&g2));
    g1 = g2;
    if (!same) GPFQ_TRY(gpfq_ws(ctx, WS_G1, (size_t)N0 * N0 * sizeof(double), (void **)&g1));
    GPFQ_TRY(dense_gram_only(ctx, dX, dXq, dld, N0, m, g1, g2));
    CUDA_TRY(ctx, cudaMemcpyAsync(G2_out, g2, (size_t)N0 * N0 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (G1_out) CUDA_TRY(ctx, cudaMemcpyAsync(G1_out, g1, (size_t)N0 * N0 * sizeof(double), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    return GPFQ_OK;
}

// ---------------------------------------------------------------------------------------------
// Conv
// ---------------------------------------------------------------------------------------------
// Host Q of a grouped layer, (kk, Cg, F) per alphabet: channel c's entries are row c % Cg of its group's Fg columns in every
// tap.  Channels c0 .. c0+n_ch-1 cover a partial first group, whole groups and a partial last group; whole groups are one
// pitched copy over all taps, a partial group one per tap.
static int conv_copy_q_grouped(gpfq_ctx *ctx, double *Q_out, const double *dQ, int kk, int64_t Cg, int64_t F, int64_t Fg,
                               int64_t c0, int64_t n_ch, int n_alph, size_t wcount) {
    cudaStream_t s = ctx->stream;
    const size_t pitch = (size_t)F * sizeof(double);
    auto box = [&](int64_t r0, int64_t r1, int64_t g0, int64_t g1) -> int {  // rows [r0, r1) of groups [g0, g1)
        if (r1 <= r0 || g1 <= g0) return GPFQ_OK;
        const size_t width = (size_t)(g1 - g0) * Fg * sizeof(double);
        for (int a = 0; a < n_alph; ++a) {
            const size_t off = (size_t)a * wcount + (size_t)r0 * F + (size_t)g0 * Fg;
            if (r0 == 0 && r1 == Cg) {
                CUDA_TRY(ctx, cudaMemcpy2DAsync(Q_out + off, pitch, dQ + off, pitch, width, (size_t)kk * Cg, cudaMemcpyDeviceToHost, s));
                continue;
            }
            for (int t = 0; t < kk; ++t) {
                const size_t o = off + (size_t)t * Cg * F;
                CUDA_TRY(ctx, cudaMemcpy2DAsync(Q_out + o, pitch, dQ + o, pitch, width, (size_t)(r1 - r0), cudaMemcpyDeviceToHost, s));
            }
        }
        return GPFQ_OK;
    };
    const int64_t c1 = c0 + n_ch, w0 = ceil_div64(c0, Cg), w1 = c1 / Cg;  // whole groups [w0, w1)
    if (w0 > w1) return box(c0 % Cg, c1 % Cg, c0 / Cg, c0 / Cg + 1);    // inside one group
    GPFQ_TRY(box(c0 % Cg, Cg, c0 / Cg, w0));
    GPFQ_TRY(box(0, Cg, w0, w1));
    return box(0, c1 % Cg, w1, w1 + 1);
}

// W / Q_out: (kk, C / groups, F); channel c walks the F / groups filters of its group c / (C / groups).
// d_scales (nullable): (n_alph, C / groups, F) per-unit scales on the device.
static int conv_finish(gpfq_ctx *ctx, int kk, const double *partial, int n_ch, int n_chunks, bool same,
                       const float *W, int64_t C, int64_t F, int64_t c0, const Alphabets &al, int n_alph,
                       double *Q_out, uint32_t flags, double *gram_ready = nullptr, int64_t groups = 1,
                       const double *d_scales = nullptr) {
    cudaStream_t s = ctx->stream;
    double *gram = gram_ready;  // per-channel [G1 | G2] already assembled (correlation form): no partials to sum
    if (!gram) {
        GPFQ_TRY(gpfq_ws(ctx, WS_CG, (size_t)n_ch * 2 * kk * kk * sizeof(double), (void **)&gram));
        GPFQ_TRY(conv_finalize_stage(ctx, partial, n_ch, n_chunks, kk, same, gram));
    }
    if (ctx->gram_only_out) {
        // gpfq_conv_gram_nhwc: the caller wants the per-channel [G1 | G2] of these images, not the walk (image split of a
        // multi-GPU job: the matrices of all ranks are summed first)
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->gram_only_out, gram, (size_t)n_ch * 2 * kk * kk * sizeof(double),
                                      (flags & GPFQ_Q_DEVICE) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
        CUDA_TRY(ctx, gpfq_record(ctx, 4, s));
        return GPFQ_OK;
    }
    const float *dW = W;
    const int64_t Cg = C / groups;
    const size_t wcount = (size_t)kk * Cg * F;
    if (!(flags & GPFQ_W_DEVICE)) {
        float *bw = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_W, wcount * sizeof(float), (void **)&bw));
        CUDA_TRY(ctx, cudaMemcpyAsync(bw, W, wcount * sizeof(float), cudaMemcpyHostToDevice, s));
        dW = bw;
    }
    double *dQ = Q_out;
    if (!(flags & GPFQ_Q_DEVICE)) GPFQ_TRY(gpfq_ws(ctx, WS_Q, (size_t)n_alph * wcount * sizeof(double), (void **)&dQ));
    GPFQ_TRY(conv_sweep_stage(ctx, kk, gram, dW, dQ, C, F, c0, n_ch, al.d_levels, al.d_koff, al.d_flags, n_alph, groups, d_scales));
    CUDA_TRY(ctx, gpfq_record(ctx, 4, s));
    if (!(flags & GPFQ_Q_DEVICE) && groups > 1)
        return conv_copy_q_grouped(ctx, Q_out, dQ, kk, Cg, F, F / groups, c0, n_ch, n_alph, wcount);
    if (!(flags & GPFQ_Q_DEVICE)) {
        for (int a = 0; a < n_alph; ++a) {
            const size_t off = (size_t)a * wcount + (size_t)c0 * F;
            CUDA_TRY(ctx, cudaMemcpy2DAsync(Q_out + off, C * F * sizeof(double), dQ + off, C * F * sizeof(double),
                                            (size_t)n_ch * F * sizeof(double), kk, cudaMemcpyDeviceToHost, s));
        }
    }
    return GPFQ_OK;
}

static void conv_stats(gpfq_ctx *ctx, gpfq_stats *st, int kk, int64_t n, int64_t n_ch, int64_t F, bool same, int n_alph) {
    if (!st) return;
    st->weights = (int64_t)kk * n_ch * F * n_alph;
    st->method = GPFQ_METHOD_GRAM >> 4;
    st->bytes_algorithmic = (same ? 1 : 2) * 4LL * kk * n * n_ch;
    st->flops_algorithmic = (same ? 0 : 2LL * kk * kk * n * n_ch) + (int64_t)kk * (kk + 1) * n * n_ch;
    // conv_gramx_kernel forms the lower triangles + diagonals of both Grams (of G2 alone in the first-layer form):
    // kk (kk + 1) / 2 MACs = kk (kk + 1) flops per column, channel and Gram
    if (!conv_specialised_kk(kk)) st->flops_algorithmic = (same ? 1 : 2) * (int64_t)kk * (kk + 1) * n * n_ch;
}

// scales (nullable, host): (n_alph, C, F) per-unit scales.
static int conv_channels(gpfq_ctx *ctx, const float *const *Xp, const float *const *Xqp, int64_t n, int32_t kk, const float *W,
                         int64_t C, int64_t F, int64_t c0, int64_t n_ch, const double *alphabets, const int32_t *K,
                         int32_t n_alph, double *Q_out, uint32_t flags, gpfq_stats *stats, const double *scales) {
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (stats) memset(stats, 0, sizeof(*stats));
    if (!Xp || !W || !Q_out) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL Xp, W or Q_out");
    if (n < 1 || kk < 1 || C < 1 || F < 1 || c0 < 0 || n_ch < 0 || c0 + n_ch > C || n_ch > 65535)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad shape: n=%lld kk=%d C=%lld F=%lld c0=%lld n_ch=%lld", (long long)n, kk,
                         (long long)C, (long long)F, (long long)c0, (long long)n_ch);
    if ((flags & GPFQ_NO_SYNC) && (flags & GPFQ_ALL_DEVICE) != GPFQ_ALL_DEVICE)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "GPFQ_NO_SYNC needs all-device pointers");
    if (scales && n_alph >= 1) GPFQ_TRY(check_scales(ctx, scales, n_alph, C * F, C * F));
    GPFQ_TRY(check_rounding(ctx, alphabets, K, n_alph));
    GPFQ_TRY(check_l1(ctx, n_alph));
    ctx->conv_part_bytes = 0;
    if (n_ch == 0) return GPFQ_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    bool same = (Xqp == nullptr);
    if (!same) {
        same = true;
        for (int64_t i = 0; i < n_ch; ++i) same = same && (Xqp[i] == Xp[i] || Xqp[i] == nullptr);
    }
    for (int64_t i = 0; i < n_ch; ++i)
        if (!Xp[i] || (!same && !Xqp[i])) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL patch pointer for channel %lld", (long long)i);

    if (!conv_supported_kk(kk)) {
        // kernels above 128 taps: each channel is a (kk, F) Dense problem over n_patches samples
        int64_t launches = 0;
        for (int64_t i = 0; i < n_ch; ++i) {
            const int64_t c = c0 + i;
            // per-alphabet outputs are kk*C*F apart, which is exactly N0*ldq for N0=kk, ldq=C*F
            GPFQ_TRY(dense_layer(ctx, Xp[i], same ? Xp[i] : Xqp[i], n, kk, n, W + c * F, C * F, F, 0, F, alphabets, K, n_alph,
                                 Q_out + c * F, C * F, (flags & ~GPFQ_NO_SYNC) | GPFQ_METHOD_GRAM, stats,
                                 scales ? scales + c * F : nullptr, C * F, c * F));   // unit ids c * F + f
            launches += stats ? stats->kernel_launches : 0;
        }
        if (stats) { stats->kernel_launches = (int)launches; stats->weights = (int64_t)kk * n_ch * F * n_alph; }
        return GPFQ_OK;
    }

    cudaStream_t s = ctx->stream;
    begin_call(ctx, 2);
    CUDA_TRY(ctx, gpfq_record(ctx, 0, s));
    Alphabets al;
    GPFQ_TRY(upload_alphabets(ctx, alphabets, K, n_alph, &al));
    GPFQ_TRY(stage_seeds(ctx, n_alph));
    GPFQ_TRY(stage_l1(ctx, n_alph));
    const double *d_scales = nullptr;
    if (scales) GPFQ_TRY(upload_scales(ctx, scales, n_alph, C * F, C * F, &d_scales));

    bool vec_ok = n % 4 == 0;  // float4 / bulk-copy paths: every row of every patch matrix 16-byte aligned
    if (flags & GPFQ_X_DEVICE)
        for (int64_t i = 0; i < n_ch; ++i)
            vec_ok = vec_ok && ((uintptr_t)Xp[i] % 16 == 0) && (same || (uintptr_t)Xqp[i] % 16 == 0);
    int64_t chunk_cols = 0;
    const int n_chunks = conv_pick_chunks(ctx, n, (int)n_ch, &chunk_cols, kk, vec_ok);
    double *partial = nullptr;
    ctx->conv_part_bytes = (int64_t)n_ch * n_chunks * 2 * kk * kk * (int64_t)sizeof(double);
    GPFQ_TRY(gpfq_ws(ctx, WS_CPART, (size_t)ctx->conv_part_bytes, (void **)&partial));
    const float **d_ptrs = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_PTRS, (size_t)2 * n_ch * sizeof(float *), (void **)&d_ptrs));
    std::vector<const float *> h_ptrs(2 * n_ch);
    const size_t ch_bytes = (size_t)kk * n * sizeof(float);

    CUDA_TRY(ctx, gpfq_record(ctx, 2, s));
    if (flags & GPFQ_X_DEVICE) {
        for (int64_t i = 0; i < n_ch; ++i) {
            h_ptrs[i] = Xp[i];
            h_ptrs[n_ch + i] = same ? Xp[i] : Xqp[i];
        }
        CUDA_TRY(ctx, cudaMemcpyAsync(d_ptrs, h_ptrs.data(), h_ptrs.size() * sizeof(float *), cudaMemcpyHostToDevice, s));
        ConvPtrs p{d_ptrs, d_ptrs + n_ch};
        GPFQ_TRY(conv_gram_stage(ctx, kk, p, same, n, (int)n_ch, n_chunks, chunk_cols, partial, vec_ok, n_chunks));
    } else {
        // host patches: double-buffered channel batches, copies on the copy stream overlap the Gram kernel
        const size_t per_ch = ch_bytes * (same ? 1 : 2);
        const size_t budget = (size_t)6 << 30;
        int64_t bch = (int64_t)std::max<size_t>(1, budget / per_ch);
        bch = std::min<int64_t>(bch, n_ch);
        if (bch * 2 > n_ch && n_ch >= 2) bch = (n_ch + 1) / 2;  // at least two batches so copy and compute overlap
        float *buf[2] = {nullptr, nullptr};
        GPFQ_TRY(gpfq_ws(ctx, WS_PATCH_A, (size_t)bch * per_ch, (void **)&buf[0]));
        GPFQ_TRY(gpfq_ws(ctx, WS_PATCH_B, (size_t)bch * per_ch, (void **)&buf[1]));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[2], s));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[2], 0));
        int bi = 0;
        for (int64_t b0 = 0; b0 < n_ch; b0 += bch, ++bi) {
            const int64_t nb = std::min<int64_t>(bch, n_ch - b0);
            float *dst = buf[bi & 1];
            // the compute that last read this buffer must be done before we overwrite it
            if (bi >= 2) CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[bi & 1], 0));
            for (int64_t i = 0; i < nb; ++i) {
                float *dx = dst + (size_t)i * (per_ch / sizeof(float));
                CUDA_TRY(ctx, cudaMemcpyAsync(dx, Xp[b0 + i], ch_bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
                h_ptrs[b0 + i] = dx;
                h_ptrs[n_ch + b0 + i] = dx;
                if (!same) {
                    float *dq = dx + (size_t)kk * n;
                    CUDA_TRY(ctx, cudaMemcpyAsync(dq, Xqp[b0 + i], ch_bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
                    h_ptrs[n_ch + b0 + i] = dq;
                }
            }
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[3], ctx->copy_stream));
            CUDA_TRY(ctx, cudaStreamWaitEvent(s, ctx->ev_copy[3], 0));
            // pointer tables for this batch (pageable source: the copy is staged before the call returns)
            CUDA_TRY(ctx, cudaMemcpyAsync(d_ptrs + b0, h_ptrs.data() + b0, nb * sizeof(float *), cudaMemcpyHostToDevice, s));
            CUDA_TRY(ctx, cudaMemcpyAsync(d_ptrs + n_ch + b0, h_ptrs.data() + n_ch + b0, nb * sizeof(float *),
                                          cudaMemcpyHostToDevice, s));
            ConvPtrs p{d_ptrs + b0, d_ptrs + n_ch + b0};
            GPFQ_TRY(conv_gram_stage(ctx, kk, p, same, n, (int)nb, n_chunks, chunk_cols,
                                     partial + (size_t)b0 * n_chunks * 2 * kk * kk, vec_ok, n_chunks));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[bi & 1], s));
        }
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 3, s));
    GPFQ_TRY(conv_finish(ctx, kk, partial, (int)n_ch, n_chunks, same, W, C, F, c0, al, n_alph, Q_out, flags, nullptr, 1, d_scales));
    CUDA_TRY(ctx, gpfq_record(ctx, 1, s));
    gpfq_stats local = {};
    conv_stats(ctx, stats ? stats : &local, kk, n, n_ch, F, same, n_alph);
    const bool synced = !(flags & GPFQ_NO_SYNC);
    if (synced) CUDA_TRY(ctx, cudaStreamSynchronize(s));
    end_call(ctx, stats ? stats : &local, synced);
    return GPFQ_OK;
}

extern "C" int gpfq_conv_channels(gpfq_ctx *ctx, const float *const *Xp, const float *const *Xqp, int64_t n,
                                  int32_t kk, const float *W, int64_t C, int64_t F, int64_t c0, int64_t n_ch,
                                  const double *alphabets, const int32_t *K, int32_t n_alph, double *Q_out,
                                  uint32_t flags, gpfq_stats *stats) {
    return conv_channels(ctx, Xp, Xqp, n, kk, W, C, F, c0, n_ch, alphabets, K, n_alph, Q_out, flags, stats, nullptr);
}

extern "C" int gpfq_conv_channels_scaled(gpfq_ctx *ctx, const float *const *Xp, const float *const *Xqp, int64_t n,
                                         int32_t kk, const float *W, int64_t C, int64_t F, int64_t c0, int64_t n_ch,
                                         const double *alphabets, const int32_t *K, int32_t n_alph, double *Q_out,
                                         uint32_t flags, gpfq_stats *stats, const double *scales) {
    if (ctx && !scales) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL scales");
    return conv_channels(ctx, Xp, Xqp, n, kk, W, C, F, c0, n_ch, alphabets, K, n_alph, Q_out, flags, stats, scales);
}

// gpfq_conv_layer_nhwc(_grouped): W / Q_out (kh, kw, C / groups, F).
static int conv_layer_nhwc(gpfq_ctx *ctx, const float *act, const float *actq, int64_t n_img, int64_t H, int64_t Wd, int64_t C,
                           int32_t kh, int32_t kw, int32_t sh, int32_t sw, int32_t rh, int32_t rw, int32_t padding_same,
                           const float *W, int64_t F, int64_t c0, int64_t n_ch, const double *alphabets, const int32_t *K,
                           int32_t n_alph, double *Q_out, uint32_t flags, gpfq_stats *stats, int64_t groups,
                           const double *scales) {
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (stats) memset(stats, 0, sizeof(*stats));
    if (!act || !W || !Q_out) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL act, W or Q_out");
    if (n_img < 1 || H < 1 || Wd < 1 || C < 1 || F < 1 || kh < 1 || kw < 1 || sh < 1 || sw < 1 || rh < 1 || rw < 1 ||
        c0 < 0 || n_ch < 0 || c0 + n_ch > C || H > 65535 || Wd > 65535)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad conv geometry");
    if (groups < 1 || C % groups || F % groups)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad groups=%lld for C=%lld, F=%lld", (long long)groups, (long long)C, (long long)F);
    const int64_t Cg = C / groups, Fg = F / groups;
    const int kk = kh * kw;
    if (scales && n_alph >= 1) GPFQ_TRY(check_scales(ctx, scales, n_alph, Cg * F, Cg * F));
    if (!ctx->gram_only_out) GPFQ_TRY(check_rounding(ctx, alphabets, K, n_alph));
    if (!ctx->gram_only_out) GPFQ_TRY(check_l1(ctx, n_alph));
    ctx->conv_part_bytes = 0;
    if (n_ch == 0) return GPFQ_OK;
    // TensorFlow extract_patches geometry (quantized_network.py:158-172)
    const int keh = (kh - 1) * rh + 1, kew = (kw - 1) * rw + 1;
    int Ho, Wo, pt = 0, pl = 0;
    if (padding_same) {
        Ho = (int)((H + sh - 1) / sh);
        Wo = (int)((Wd + sw - 1) / sw);
        const int64_t ph = std::max<int64_t>((int64_t)(Ho - 1) * sh + keh - H, 0);
        const int64_t pw = std::max<int64_t>((int64_t)(Wo - 1) * sw + kew - Wd, 0);
        pt = (int)(ph / 2);
        pl = (int)(pw / 2);
    } else {
        if (H < keh || Wd < kew) return gpfq_fail(ctx, GPFQ_ERR_ARG, "VALID padding: input smaller than the kernel");
        Ho = (int)((H - keh) / sh + 1);
        Wo = (int)((Wd - kew) / sw + 1);
    }
    const int64_t n = n_img * Ho * Wo;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const bool same = (actq == nullptr || actq == act);
    if (!conv_supported_kk(kk)) {
        // Kernels above 128 taps (13 x 11, 12 x 12, ...; the reference takes any size, quantized_network.py:686-727) have no
        // batched Gram / walk kernel: patches of one channel at a time on the device (im2col), then that channel is a
        // (kk, F) Dense problem over n patches -- what gpfq_conv_channels does for such sizes from host patch matrices.
        if (ctx->gram_only_out) return gpfq_fail(ctx, GPFQ_ERR_UNSUPPORTED, "kernel %dx%d has no Gram-only (image split) path", kh, kw);
        const size_t abytes_g = (size_t)n_img * H * Wd * C * sizeof(float);
        const float *gA = act, *gAq = same ? act : actq;
        if (!(flags & GPFQ_X_DEVICE)) {
            float *ba = nullptr, *bq = nullptr;
            GPFQ_TRY(gpfq_ws(ctx, WS_ACT_A, abytes_g, (void **)&ba));
            CUDA_TRY(ctx, cudaMemcpyAsync(ba, act, abytes_g, cudaMemcpyHostToDevice, s));
            gA = gAq = ba;
            if (!same) {
                GPFQ_TRY(gpfq_ws(ctx, WS_ACT_B, abytes_g, (void **)&bq));
                CUDA_TRY(ctx, cudaMemcpyAsync(bq, actq, abytes_g, cudaMemcpyHostToDevice, s));
                gAq = bq;
            }
        }
        float *pa = nullptr, *pq = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_PATCH_A, (size_t)kk * n * sizeof(float), (void **)&pa));
        pq = pa;
        if (!same) GPFQ_TRY(gpfq_ws(ctx, WS_PATCH_B, (size_t)kk * n * sizeof(float), (void **)&pq));
        int64_t launches = 0;
        for (int64_t i = 0; i < n_ch; ++i) {
            const int64_t c = c0 + i;
            GPFQ_TRY(im2col_stage(ctx, gA, n_img, (int)H, (int)Wd, C, c, 1, kh, kw, sh, sw, rh, rw, pt, pl, Ho, Wo, pa, (int64_t)kk * n));
            if (!same)
                GPFQ_TRY(im2col_stage(ctx, gAq, n_img, (int)H, (int)Wd, C, c, 1, kh, kw, sh, sw, rh, rw, pt, pl, Ho, Wo, pq, (int64_t)kk * n));
            // channel c against the Fg filters of its group (all F when ungrouped); per-alphabet outputs are kk*Cg*F apart, which is
            // exactly N0*ldq for N0 = kk, ldq = Cg*F
            const int64_t off = (c % Cg) * F + (c / Cg) * Fg;
            GPFQ_TRY(dense_layer(ctx, pa, same ? pa : pq, n, kk, n, W + off, Cg * F, Fg, 0, Fg, alphabets, K, n_alph, Q_out + off,
                                 Cg * F, ((flags & ~GPFQ_NO_SYNC) | GPFQ_X_DEVICE | GPFQ_METHOD_GRAM), stats,
                                 scales ? scales + off : nullptr, Cg * F, off));   // unit ids (c % Cg) * F + g * Fg + f
            launches += (stats ? stats->kernel_launches : 0) + (same ? 1 : 2);
        }
        if (stats) { stats->kernel_launches = (int)launches; stats->weights = (int64_t)kk * n_ch * Fg * n_alph; }
        return GPFQ_OK;
    }
    begin_call(ctx, 2);
    CUDA_TRY(ctx, gpfq_record(ctx, 0, s));
    Alphabets al;
    GPFQ_TRY(upload_alphabets(ctx, alphabets, K, n_alph, &al));
    GPFQ_TRY(stage_seeds(ctx, n_alph));
    GPFQ_TRY(stage_l1(ctx, n_alph));
    const double *d_scales = nullptr;
    if (scales) GPFQ_TRY(upload_scales(ctx, scales, n_alph, Cg * F, Cg * F, &d_scales));
    const float *dA = act, *dAq = same ? act : actq;
    const size_t img_elems = (size_t)H * Wd * C;
    const size_t abytes = (size_t)n_img * img_elems * sizeof(float);
    const bool host_act = !(flags & GPFQ_X_DEVICE);
    // Host activations: the images go over in chunks on the copy stream while the compute stream turns the chunks
    // that have landed into patches and partial Grams (the Gram is a sum over patches, so image chunks are just
    // more partial slots, summed in index order by the finalize kernel).
    int64_t ipc = n_img;  // images per chunk
    if (host_act) {
        const size_t target = (size_t)96 << 20;
        ipc = (int64_t)std::max<size_t>(1, target / (img_elems * sizeof(float)));
        ipc = std::max<int64_t>(ipc, ceil_div64(n_img, 32));  // at most 32 chunks
        ipc = std::min<int64_t>(ceil_div64(ipc, 4) * 4, n_img);
    }
    int n_ic = (int)ceil_div64(n_img, ipc);
    if (host_act && !conv_specialised_kk(kk)) {
        // every image chunk adds partial slots: keep the partial workspace of conv_gramx_kernel within CONV_PART_LIMIT
        // (conv_pick_chunks trims the column chunks), with fewer, larger image chunks when many channels meet a large kernel
        const int64_t max_ic = std::max<int64_t>(1, CONV_PART_LIMIT / (n_ch * 2 * kk * kk * (int64_t)sizeof(double)));
        if (n_ic > max_ic) {
            ipc = std::min<int64_t>(ceil_div64(ceil_div64(n_img, max_ic), 4) * 4, n_img);
            n_ic = (int)ceil_div64(n_img, ipc);
        }
    }
    if (host_act) {
        float *ba = nullptr, *bq = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_ACT_A, abytes, (void **)&ba));
        dA = dAq = ba;
        if (!same) {
            GPFQ_TRY(gpfq_ws(ctx, WS_ACT_B, abytes, (void **)&bq));
            dAq = bq;
        }
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 5, s));
    const int corr_rb = ctx->conv_variant == 0 ? corr9_plan(kh, kw, sh, sw, rh, rw, padding_same, (int)H, (int)Wd, ctx->corr_rb, same) : 0;
    // what a tensor map of the activations needs: 32-channel boxes on a 16-byte channel pitch; and lane = channel wants a
    // full warp of channels.  Otherwise G images are packed side by side as virtual channels first (conv_corr.cu).
    // Measured (tools/vgg_bench.py --net cifar / --conv-kernel 3): on 8 x 8 images the per-band start-up outweighs the 6.5x
    // fewer MACs and the shared-memory planes kernel wins; packing pays for itself only on large images whose channel
    // count cannot be mapped directly (VGG's first layer: 7.0 -> 3.6 ms; with the strip kernel also on images from 1024 pixels:
    // CIFAR10's 32 x 32 x 3 first layer 0.50 -> 0.23 ms); channel shards of 8-16 channels run faster unpacked with idle lanes.
    const bool corr_direct = C >= 32 && C % 4 == 0 && n_ch >= 8 && (H * Wd >= 128 || (H * Wd >= 64 && corr9_uses_strips(ctx, (int)Wd)));
    int corr_G = 1;
    if (corr_rb && !(C >= 32 && C % 4 == 0) && (H * Wd >= 4096 || (H * Wd >= 1024 && corr9_uses_strips(ctx, (int)Wd))) && ctx->corr_pack != 2) {
        int g = 32, a = (int)(n_ch % 32);
        while (a) { const int t = g % a; g = a; a = t; }   // g = gcd(n_ch, 32)
        corr_G = 32 / g;
        const double packed = (double)ceil_div64(n_img, corr_G) * corr_G * H * Wd * n_ch * sizeof(float) * (same ? 1 : 2);
        if (corr_G * n_ch > 4096 || packed > 32e9) corr_G = 1;   // keep the patch form
    }
    if (ctx->corr_pack == 1 && corr_rb) {   // tests: pack whatever the shape
        int g = 32, a = (int)(n_ch % 32);
        while (a) { const int t = g % a; g = a; a = t; }
        corr_G = 32 / g;
        if (corr_G == 1 || corr_G * n_ch > 4096) corr_G = (corr_G * n_ch > 4096) ? 1 : 2;
    }
    if (corr_rb && (corr_G > 1 || (corr_direct && ctx->corr_pack != 1) || (ctx->corr_direct_small && C >= 32 && C % 4 == 0 && n_ch >= 8)) &&
        corr9_tensor_ok(dA, dAq)) {
        // ---- correlation form: 13 displacement sums per Gram straight from the activations (conv_corr.cu)
        const bool pack = corr_G > 1;
        const int64_t VC = pack ? (int64_t)corr_G * n_ch : C;            // channels of the tensor the kernels see
        const int vch = pack ? (int)VC : (int)n_ch;                       // channels (records) of this call
        const int64_t vc0 = pack ? 0 : c0;
        int64_t cipc = ipc;                                               // images per host chunk: whole groups when packing
        if (pack) cipc = std::min<int64_t>(ceil_div64(cipc, corr_G) * corr_G, ceil_div64(n_img, corr_G) * corr_G);
        const int cn_ic = (int)ceil_div64(n_img, cipc);
        const int64_t units_per_chunk = pack ? cipc / corr_G : cipc;      // tensor "images" per chunk
        const int64_t units_total = pack ? ceil_div64(n_img, corr_G) : n_img;
        const int nbands = (int)ceil_div64(H - 2, corr_rb);                        // rows 1 .. H-2 in bands
        const int per_ic = corr9_pick_slots(ctx, corr_rb, same, vc0, vch, units_per_chunk * nbands, (int)Wd);
        const int bper_ic = corr9_pick_slots(ctx, 1, same, vc0, vch, 2 * units_per_chunk, (int)Wd);   // top and bottom row of every image
        const int slots = cn_ic * per_ic, bslots = cn_ic * bper_ic;
        double *partial = nullptr, *bpartial = nullptr, *gram = nullptr;
        float *pkA = nullptr, *pkQ = nullptr;
        const size_t part_bytes = (size_t)vch * slots * 78 * sizeof(double);      // 2 passes x 3 column classes x 13 sums
        const size_t bpart_bytes = (size_t)vch * bslots * 78 * sizeof(double);
        ctx->conv_part_bytes = (int64_t)part_bytes;
        GPFQ_TRY(gpfq_ws(ctx, WS_CPART, part_bytes, (void **)&partial));
        GPFQ_TRY(gpfq_ws(ctx, WS_CORR_B, bpart_bytes, (void **)&bpartial));
        GPFQ_TRY(gpfq_ws(ctx, WS_CG, (size_t)n_ch * 2 * kk * kk * sizeof(double), (void **)&gram));
        if (pack) {
            const size_t pk_bytes = (size_t)units_total * H * Wd * VC * sizeof(float);
            GPFQ_TRY(gpfq_ws(ctx, WS_PATCH_A, pk_bytes, (void **)&pkA));
            pkQ = pkA;
            if (!same) GPFQ_TRY(gpfq_ws(ctx, WS_PATCH_B, pk_bytes, (void **)&pkQ));
        }
        CUDA_TRY(ctx, cudaMemsetAsync(partial, 0, part_bytes, s));
        CUDA_TRY(ctx, cudaMemsetAsync(bpartial, 0, bpart_bytes, s));
        CUDA_TRY(ctx, gpfq_record(ctx, 2, s));
        if (host_act) {
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[2], s));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[2], 0));
        }
        for (int ic = 0; ic < cn_ic; ++ic) {
            const int64_t img0 = (int64_t)ic * cipc;
            const int64_t imgs = std::min<int64_t>(cipc, n_img - img0);
            if (host_act) {
                const size_t off = (size_t)img0 * img_elems, bytes = (size_t)imgs * img_elems * sizeof(float);
                CUDA_TRY(ctx, cudaMemcpyAsync(const_cast<float *>(dA) + off, act + off, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
                if (!same)
                    CUDA_TRY(ctx, cudaMemcpyAsync(const_cast<float *>(dAq) + off, actq + off, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
                CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[ic & 1], ctx->copy_stream));
                CUDA_TRY(ctx, cudaStreamWaitEvent(s, ctx->ev_copy[ic & 1], 0));
            }
            if (pack) {
                GPFQ_TRY(corr9_pack_stage(ctx, dA, n_img, (int)H, (int)Wd, C, c0, (int)n_ch, corr_G, img0, imgs, pkA));
                if (!same) GPFQ_TRY(corr9_pack_stage(ctx, dAq, n_img, (int)H, (int)Wd, C, c0, (int)n_ch, corr_G, img0, imgs, pkQ));
                GPFQ_TRY(conv_corr9_stage(ctx, pkA, pkQ, same, img0 / corr_G, ceil_div64(imgs, corr_G), units_total, (int)H, (int)Wd, VC,
                                          0, vch, corr_rb, partial, slots, ic * per_ic, per_ic, bpartial, bslots, ic * bper_ic, bper_ic));
            } else {
                GPFQ_TRY(conv_corr9_stage(ctx, dA, dAq, same, img0, imgs, n_img, (int)H, (int)Wd, C, c0, (int)n_ch, corr_rb, partial, slots,
                                          ic * per_ic, per_ic, bpartial, bslots, ic * bper_ic, bper_ic));
            }
        }
        GPFQ_TRY(conv_corr9_assemble_stage(ctx, partial, slots, bpartial, bslots, same, (int)Wd, (int)n_ch, pack ? corr_G : 1, gram));
        CUDA_TRY(ctx, gpfq_record(ctx, 3, s));
        GPFQ_TRY(conv_finish(ctx, kk, nullptr, (int)n_ch, 0, same, W, C, F, c0, al, n_alph, Q_out, flags, gram, groups, d_scales));
        CUDA_TRY(ctx, gpfq_record(ctx, 1, s));
        gpfq_stats local = {};
        gpfq_stats *st = stats ? stats : &local;
        conv_stats(ctx, st, kk, n, n_ch, Fg, same, n_alph);
        st->bytes_algorithmic = (same ? 1 : 2) * 4LL * n_img * H * Wd * n_ch;  // the activations, once
        st->flops_algorithmic = (same ? 1 : 2) * 26LL * n_img * H * Wd * n_ch;  // 13 MACs per pixel, channel and Gram
        st->gram_kernel = pack ? 5 : 4;
        const bool synced = !(flags & GPFQ_NO_SYNC);
        if (synced) CUDA_TRY(ctx, cudaStreamSynchronize(s));
        end_call(ctx, st, synced);
        return GPFQ_OK;
    }
    int planeP = 0, bandR = 0;
    if ((ctx->conv_variant == 0 || ctx->conv_variant == 3) && nhwc9_plan(kh, kw, sh, sw, rh, rw, Ho, Wo, &planeP, &bandR)) {
        // ---- fused path: Grams straight from the activations, no patch matrices
        const int64_t ctas = ceil_div64(n_ch, 8);                            // CTAs of 8 channels per image slot
        int64_t per_ic = ceil_div64(4LL * 2 * ctx->sm_count, ctas * n_ic);  // ~4 waves of two CTAs per SM overall
        per_ic = std::max<int64_t>(1, std::min<int64_t>(per_ic, ipc));
        const int slots = (int)(n_ic * per_ic);
        double *partial = nullptr;
        const size_t part_bytes = (size_t)ctas * 8 * slots * 2 * kk * kk * sizeof(double);
        ctx->conv_part_bytes = (int64_t)part_bytes;
        GPFQ_TRY(gpfq_ws(ctx, WS_CPART, part_bytes, (void **)&partial));
        CUDA_TRY(ctx, cudaMemsetAsync(partial, 0, part_bytes, s));  // short chunks leave slots unused
        CUDA_TRY(ctx, gpfq_record(ctx, 2, s));
        if (host_act) {
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[2], s));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[2], 0));
        }
        for (int ic = 0; ic < n_ic; ++ic) {
            const int64_t img0 = (int64_t)ic * ipc;
            const int64_t imgs = std::min<int64_t>(ipc, n_img - img0);
            if (host_act) {
                const size_t off = (size_t)img0 * img_elems, bytes = (size_t)imgs * img_elems * sizeof(float);
                CUDA_TRY(ctx, cudaMemcpyAsync(const_cast<float *>(dA) + off, act + off, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
                if (!same)
                    CUDA_TRY(ctx, cudaMemcpyAsync(const_cast<float *>(dAq) + off, actq + off, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
                CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[ic & 1], ctx->copy_stream));
                CUDA_TRY(ctx, cudaStreamWaitEvent(s, ctx->ev_copy[ic & 1], 0));
            }
            GPFQ_TRY(conv_gram9_nhwc_stage(ctx, dA, dAq, same, img0, imgs, (int)H, (int)Wd, C, c0, (int)n_ch, Ho, Wo, pt, pl,
                                           planeP, bandR, (int)per_ic, partial + (size_t)ic * per_ic * 2 * kk * kk, slots));
        }
        CUDA_TRY(ctx, gpfq_record(ctx, 3, s));
        GPFQ_TRY(conv_finish(ctx, kk, partial, (int)n_ch, slots, same, W, C, F, c0, al, n_alph, Q_out, flags, nullptr, groups, d_scales));
        CUDA_TRY(ctx, gpfq_record(ctx, 1, s));
        gpfq_stats local = {};
        gpfq_stats *st = stats ? stats : &local;
        conv_stats(ctx, st, kk, n, n_ch, Fg, same, n_alph);
        st->bytes_algorithmic = (same ? 1 : 2) * 4LL * n_img * H * Wd * n_ch;  // the activations, once
        const bool synced = !(flags & GPFQ_NO_SYNC);
        if (synced) CUDA_TRY(ctx, cudaStreamSynchronize(s));
        end_call(ctx, st, synced);
        return GPFQ_OK;
    }
    const int64_t hw_out = (int64_t)Ho * Wo;
    const int64_t n_c = ipc * hw_out;  // patch columns of a full image chunk
    bool vec_ok = n_c % 4 == 0 && ((n_img - (int64_t)(n_ic - 1) * ipc) * hw_out) % 4 == 0;
    int64_t chunk_cols = 0;
    const int n_chunks = conv_pick_chunks(ctx, n_c, (int)std::min<int64_t>(n_ch, 64), &chunk_cols, kk, vec_ok, n_ch * n_ic);
    const int slots = n_ic * n_chunks;
    double *partial = nullptr;
    const size_t part_bytes = (size_t)n_ch * slots * 2 * kk * kk * sizeof(double);
    ctx->conv_part_bytes = (int64_t)part_bytes;
        GPFQ_TRY(gpfq_ws(ctx, WS_CPART, part_bytes, (void **)&partial));
    if (n_ic > 1) CUDA_TRY(ctx, cudaMemsetAsync(partial, 0, part_bytes, s));  // a short last chunk leaves slots unused
    const size_t ch_elems = (size_t)kk * n_c;
    const size_t per_ch = ch_elems * sizeof(float);
    const size_t budget = (size_t)8 << 30;
    int64_t bch = (int64_t)std::max<size_t>(1, budget / (per_ch * (same ? 1 : 2)));
    bch = std::min<int64_t>(bch, n_ch);
    float *pa = nullptr, *pq = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_PATCH_A, (size_t)bch * per_ch, (void **)&pa));
    if (!same) GPFQ_TRY(gpfq_ws(ctx, WS_PATCH_B, (size_t)bch * per_ch, (void **)&pq));
    const float **d_ptrs = nullptr;
    GPFQ_TRY(gpfq_ws(ctx, WS_PTRS, (size_t)2 * bch * n_ic * sizeof(float *), (void **)&d_ptrs));
    CUDA_TRY(ctx, gpfq_record(ctx, 2, s));
    if (host_act) {  // the copy stream may not overwrite the staging buffers before earlier work on s is done
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[2], s));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[2], 0));
    }
    std::vector<const float *> h_ptrs((size_t)2 * bch * n_ic);
    for (int ic = 0; ic < n_ic; ++ic) {
        const int64_t img0 = (int64_t)ic * ipc;
        const int64_t imgs = std::min<int64_t>(ipc, n_img - img0);
        const int64_t n_this = imgs * hw_out;
        if (host_act) {
            const size_t off = (size_t)img0 * img_elems, bytes = (size_t)imgs * img_elems * sizeof(float);
            CUDA_TRY(ctx, cudaMemcpyAsync(const_cast<float *>(dA) + off, act + off, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
            if (!same)
                CUDA_TRY(ctx, cudaMemcpyAsync(const_cast<float *>(dAq) + off, actq + off, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_copy[ic & 1], ctx->copy_stream));
            CUDA_TRY(ctx, cudaStreamWaitEvent(s, ctx->ev_copy[ic & 1], 0));
        }
        // patch pointers of this chunk: channel i at pa + i * kk * n_this (rows stay 16-byte aligned when vec_ok)
        const float **hp = h_ptrs.data() + (size_t)2 * bch * ic;
        for (int64_t i = 0; i < bch; ++i) {
            hp[i] = pa + (size_t)i * kk * n_this;
            hp[bch + i] = same ? hp[i] : pq + (size_t)i * kk * n_this;
        }
        const float **dp = d_ptrs + (size_t)2 * bch * ic;
        CUDA_TRY(ctx, cudaMemcpyAsync(dp, hp, (size_t)2 * bch * sizeof(float *), cudaMemcpyHostToDevice, s));
        const int chunks_this = (int)ceil_div64(n_this, chunk_cols);
        for (int64_t b0 = 0; b0 < n_ch; b0 += bch) {
            const int64_t nb = std::min<int64_t>(bch, n_ch - b0);
            GPFQ_TRY(im2col_stage(ctx, dA + (size_t)img0 * img_elems, imgs, (int)H, (int)Wd, C, c0 + b0, (int)nb, kh, kw, sh, sw,
                                  rh, rw, pt, pl, Ho, Wo, pa, (int64_t)kk * n_this));
            if (!same)
                GPFQ_TRY(im2col_stage(ctx, dAq + (size_t)img0 * img_elems, imgs, (int)H, (int)Wd, C, c0 + b0, (int)nb, kh, kw,
                                      sh, sw, rh, rw, pt, pl, Ho, Wo, pq, (int64_t)kk * n_this));
            ConvPtrs p{dp, dp + bch};
            GPFQ_TRY(conv_gram_stage(ctx, kk, p, same, n_this, (int)nb, chunks_this, chunk_cols,
                                     partial + ((size_t)b0 * slots + (size_t)ic * n_chunks) * 2 * kk * kk, vec_ok, slots));
        }
    }
    CUDA_TRY(ctx, gpfq_record(ctx, 3, s));
    GPFQ_TRY(conv_finish(ctx, kk, partial, (int)n_ch, slots, same, W, C, F, c0, al, n_alph, Q_out, flags, nullptr, groups, d_scales));
    CUDA_TRY(ctx, gpfq_record(ctx, 1, s));
    gpfq_stats local = {};
    conv_stats(ctx, stats ? stats : &local, kk, n, n_ch, Fg, same, n_alph);
    const bool synced = !(flags & GPFQ_NO_SYNC);
    if (synced) CUDA_TRY(ctx, cudaStreamSynchronize(s));
    end_call(ctx, stats ? stats : &local, synced);
    return GPFQ_OK;
}

extern "C" int gpfq_conv_layer_nhwc(gpfq_ctx *ctx, const float *act, const float *actq, int64_t n_img, int64_t H,
                                    int64_t Wd, int64_t C, int32_t kh, int32_t kw, int32_t sh, int32_t sw, int32_t rh,
                                    int32_t rw, int32_t padding_same, const float *W, int64_t F, int64_t c0,
                                    int64_t n_ch, const double *alphabets, const int32_t *K, int32_t n_alph,
                                    double *Q_out, uint32_t flags, gpfq_stats *stats) {
    return conv_layer_nhwc(ctx, act, actq, n_img, H, Wd, C, kh, kw, sh, sw, rh, rw, padding_same, W, F, c0, n_ch, alphabets, K,
                           n_alph, Q_out, flags, stats, 1, nullptr);
}

extern "C" int gpfq_conv_layer_nhwc_grouped(gpfq_ctx *ctx, const float *act, const float *actq, int64_t n_img, int64_t H,
                                            int64_t Wd, int64_t C, int32_t kh, int32_t kw, int32_t sh, int32_t sw, int32_t rh,
                                            int32_t rw, int32_t padding_same, const float *W, int64_t F, int64_t c0,
                                            int64_t n_ch, const double *alphabets, const int32_t *K, int32_t n_alph,
                                            double *Q_out, uint32_t flags, gpfq_stats *stats, int32_t groups) {
    return conv_layer_nhwc(ctx, act, actq, n_img, H, Wd, C, kh, kw, sh, sw, rh, rw, padding_same, W, F, c0, n_ch, alphabets, K,
                           n_alph, Q_out, flags, stats, groups, nullptr);
}

extern "C" int gpfq_conv_layer_nhwc_scaled(gpfq_ctx *ctx, const float *act, const float *actq, int64_t n_img, int64_t H,
                                           int64_t Wd, int64_t C, int32_t kh, int32_t kw, int32_t sh, int32_t sw, int32_t rh,
                                           int32_t rw, int32_t padding_same, const float *W, int64_t F, int64_t c0,
                                           int64_t n_ch, const double *alphabets, const int32_t *K, int32_t n_alph,
                                           double *Q_out, uint32_t flags, gpfq_stats *stats, int32_t groups,
                                           const double *scales) {
    if (ctx && !scales) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL scales");
    return conv_layer_nhwc(ctx, act, actq, n_img, H, Wd, C, kh, kw, sh, sw, rh, rw, padding_same, W, F, c0, n_ch, alphabets, K,
                           n_alph, Q_out, flags, stats, groups, scales);
}

// Gram stage of a conv layer alone (see include/gpfq.h): the same planner and kernels as gpfq_conv_layer_nhwc, stopped
// before the walk.
extern "C" int gpfq_conv_gram_nhwc(gpfq_ctx *ctx, const float *act, const float *actq, int64_t n_img, int64_t H, int64_t Wd,
                                   int64_t C, int32_t kh, int32_t kw, int32_t sh, int32_t sw, int32_t rh, int32_t rw,
                                   int32_t padding_same, int64_t c0, int64_t n_ch, double *gram_out, uint32_t flags) {
    if (!ctx) return GPFQ_ERR_ARG;
    if (!gram_out) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL gram_out");
    static const double unit[2] = {-1.0, 1.0};   // the walk never runs: any alphabet / kernel pointer will do
    static const int32_t two = 2;
    static const float w_dummy = 0.f;
    ctx->gram_only_out = gram_out;
    // W_DEVICE keeps the (unused) kernel from being copied; Q_DEVICE in `flags` says where gram_out lives; GPFQ_NO_SYNC
    // (device inputs and outputs only) returns after enqueueing: the copy into gram_out is ordered on the stream
    uint32_t f = flags | GPFQ_W_DEVICE;
    if ((f & GPFQ_ALL_DEVICE) != GPFQ_ALL_DEVICE) f &= ~GPFQ_NO_SYNC;
    const int rc = gpfq_conv_layer_nhwc(ctx, act, actq, n_img, H, Wd, C, kh, kw, sh, sw, rh, rw, padding_same, &w_dummy, 1, c0, n_ch,
                                        unit, &two, 1, gram_out, f, nullptr);
    ctx->gram_only_out = nullptr;
    return rc;
}

// Walk stage of a conv layer from per-channel Gram matrices on the device (see include/gpfq.h); W / Q_out (kk, C / groups, F).
static int conv_layer_from_gram(gpfq_ctx *ctx, const double *gram, int32_t kk, const float *W, int64_t C, int64_t F, int64_t c0,
                                int64_t n_ch, const double *alphabets, const int32_t *K, int32_t n_alph, double *Q_out,
                                uint32_t flags, gpfq_stats *stats, int64_t groups, const double *scales) {
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (stats) memset(stats, 0, sizeof(*stats));
    if (!gram || !W || !Q_out) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL gram, W or Q_out");
    if (!(flags & GPFQ_X_DEVICE)) return gpfq_fail(ctx, GPFQ_ERR_ARG, "gram must be a device pointer (GPFQ_X_DEVICE)");
    if (C < 1 || F < 1 || c0 < 0 || n_ch < 0 || c0 + n_ch > C) return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad channel range");
    if (groups < 1 || C % groups || F % groups)
        return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad groups=%lld for C=%lld, F=%lld", (long long)groups, (long long)C, (long long)F);
    if (!conv_supported_kk(kk)) return gpfq_fail(ctx, GPFQ_ERR_UNSUPPORTED, "kernel size kk=%d has no walk kernel", kk);
    if (scales && n_alph >= 1) GPFQ_TRY(check_scales(ctx, scales, n_alph, C / groups * F, C / groups * F));
    GPFQ_TRY(check_rounding(ctx, alphabets, K, n_alph));
    GPFQ_TRY(check_l1(ctx, n_alph));
    if (n_ch == 0) return GPFQ_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    begin_call(ctx, 2);
    CUDA_TRY(ctx, gpfq_record(ctx, 0, s));
    Alphabets al;
    GPFQ_TRY(upload_alphabets(ctx, alphabets, K, n_alph, &al));
    GPFQ_TRY(stage_seeds(ctx, n_alph));
    GPFQ_TRY(stage_l1(ctx, n_alph));
    const double *d_scales = nullptr;
    if (scales) GPFQ_TRY(upload_scales(ctx, scales, n_alph, C / groups * F, C / groups * F, &d_scales));
    CUDA_TRY(ctx, gpfq_record(ctx, 5, s));
    CUDA_TRY(ctx, gpfq_record(ctx, 2, s));
    CUDA_TRY(ctx, gpfq_record(ctx, 3, s));
    GPFQ_TRY(conv_finish(ctx, kk, nullptr, (int)n_ch, 0, false, W, C, F, c0, al, n_alph, Q_out, flags, const_cast<double *>(gram),
                         groups, d_scales));
    CUDA_TRY(ctx, gpfq_record(ctx, 1, s));
    gpfq_stats local = {};
    gpfq_stats *st = stats ? stats : &local;
    st->weights = (int64_t)kk * n_ch * (F / groups) * n_alph;
    st->method = GPFQ_METHOD_GRAM >> 4;
    const bool synced = !(flags & GPFQ_NO_SYNC);
    if (synced) CUDA_TRY(ctx, cudaStreamSynchronize(s));
    end_call(ctx, st, synced);
    return GPFQ_OK;
}

extern "C" int gpfq_conv_layer_from_gram(gpfq_ctx *ctx, const double *gram, int32_t kk, const float *W, int64_t C, int64_t F,
                                         int64_t c0, int64_t n_ch, const double *alphabets, const int32_t *K, int32_t n_alph,
                                         double *Q_out, uint32_t flags, gpfq_stats *stats) {
    return conv_layer_from_gram(ctx, gram, kk, W, C, F, c0, n_ch, alphabets, K, n_alph, Q_out, flags, stats, 1, nullptr);
}

extern "C" int gpfq_conv_layer_from_gram_grouped(gpfq_ctx *ctx, const double *gram, int32_t kk, const float *W, int64_t C,
                                                 int64_t F, int64_t c0, int64_t n_ch, const double *alphabets, const int32_t *K,
                                                 int32_t n_alph, double *Q_out, uint32_t flags, gpfq_stats *stats,
                                                 int32_t groups) {
    return conv_layer_from_gram(ctx, gram, kk, W, C, F, c0, n_ch, alphabets, K, n_alph, Q_out, flags, stats, groups, nullptr);
}

extern "C" int gpfq_conv_layer_from_gram_scaled(gpfq_ctx *ctx, const double *gram, int32_t kk, const float *W, int64_t C,
                                                int64_t F, int64_t c0, int64_t n_ch, const double *alphabets, const int32_t *K,
                                                int32_t n_alph, double *Q_out, uint32_t flags, gpfq_stats *stats,
                                                int32_t groups, const double *scales) {
    if (ctx && !scales) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL scales");
    return conv_layer_from_gram(ctx, gram, kk, W, C, F, c0, n_ch, alphabets, K, n_alph, Q_out, flags, stats, groups, scales);
}

// scales (nullable, float32 W): element i rounds to the levels scales[i % n_units] * alphabet.
static int round_elements(gpfq_ctx *ctx, const void *W, int is_f64, int64_t n, const double *alphabet, int32_t K,
                          double *Q_out, uint32_t flags, const double *scales = nullptr, int64_t n_units = 0) {
    if (!ctx) return GPFQ_ERR_ARG;
    ctx->err.clear();
    if (!W || !Q_out || n < 0) return gpfq_fail(ctx, GPFQ_ERR_ARG, "bad arguments");
    if (scales) {
        if (n_units < 1) return gpfq_fail(ctx, GPFQ_ERR_ARG, "n_units must be >= 1");
        GPFQ_TRY(check_scales(ctx, scales, 1, n_units, n_units));
    }
    GPFQ_TRY(check_rounding(ctx, alphabet, &K, 1));
    if (n == 0) return GPFQ_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    begin_call(ctx, 2);
    cudaStream_t s = ctx->stream;
    Alphabets al;
    GPFQ_TRY(upload_alphabets(ctx, alphabet, &K, 1, &al));
    GPFQ_TRY(stage_seeds(ctx, 1));
    ctx->d_l1 = nullptr;   // MSQ and bit_round have no greedy step: the penalty does not apply
    const double *d_scales = nullptr;
    if (scales) GPFQ_TRY(upload_scales(ctx, scales, 1, n_units, n_units, &d_scales));
    const size_t esz = is_f64 ? sizeof(double) : sizeof(float);
    const void *dW = W;
    if (!(flags & GPFQ_W_DEVICE)) {
        void *bw = nullptr;
        GPFQ_TRY(gpfq_ws(ctx, WS_W, (size_t)n * esz, &bw));
        CUDA_TRY(ctx, cudaMemcpyAsync(bw, W, (size_t)n * esz, cudaMemcpyHostToDevice, s));
        dW = bw;
    }
    double *dQ = Q_out;
    if (!(flags & GPFQ_Q_DEVICE)) GPFQ_TRY(gpfq_ws(ctx, WS_Q, (size_t)n * sizeof(double), (void **)&dQ));
    GPFQ_TRY(msq_stage(ctx, dW, is_f64, n, al.d_levels, K, al.h_flags[0], dQ, d_scales, n_units));
    if (!(flags & GPFQ_Q_DEVICE))
        CUDA_TRY(ctx, cudaMemcpyAsync(Q_out, dQ, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (!(flags & GPFQ_NO_SYNC) || !(flags & GPFQ_Q_DEVICE)) CUDA_TRY(ctx, cudaStreamSynchronize(s));
    return GPFQ_OK;
}

extern "C" int gpfq_msq(gpfq_ctx *ctx, const float *W, int64_t n, const double *alphabet, int32_t K, double *Q_out,
                        uint32_t flags) {
    return round_elements(ctx, W, 0, n, alphabet, K, Q_out, flags);
}

extern "C" int gpfq_msq_scaled(gpfq_ctx *ctx, const float *W, int64_t n, const double *alphabet, int32_t K, const double *scales,
                               int64_t n_units, double *Q_out, uint32_t flags) {
    if (ctx && !scales) return gpfq_fail(ctx, GPFQ_ERR_ARG, "NULL scales");
    return round_elements(ctx, W, 0, n, alphabet, K, Q_out, flags, scales, n_units);
}

extern "C" int gpfq_bit_round(gpfq_ctx *ctx, const double *t, int64_t n, const double *alphabet, int32_t K,
                              double *out, uint32_t flags) {
    return round_elements(ctx, t, 1, n, alphabet, K, out, flags);
}
