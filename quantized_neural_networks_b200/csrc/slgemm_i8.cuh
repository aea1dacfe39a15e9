// slgemm_i8.cuh -- host interface of the int8-slice tcgen05 contraction (slgemm_i8.cu).
#pragma once
#include "i8_common.cuh"

// Layout of a sliced operand in HBM: the SHARED-MEMORY IMAGE of its tiles.  K-block tiled -- everything one pipeline stage
// fetches is a handful of contiguous 4-8 KB runs -- and already 64B-swizzled (16-byte chunk c of row r sits at chunk
// c ^ ((r >> 1) & 3), the pattern UMMA's SWIZZLE_64B descriptors expect), so a stage is filled by plain 1-D bulk copies
// (cp.async.bulk: one request per 4-8 KB; the same boxes through a tensor map cost one 64-byte request per row and capped an
// SM at ~40 GB/s):
//   byte (slice s, row r, K position c)  at  ((c / 64 * n_slices + s) * rowsP + r) * 64 + ((c / 16 % 4) ^ (r / 2 % 4)) * 16 + c % 16
__host__ __device__ __forceinline__ int64_t sl_offset(int64_t c, int s, int64_t r, int64_t rowsP, int n_slices) {
    return (((c >> 6) * n_slices + s) * rowsP + r) * 64 + ((((c >> 4) & 3) ^ ((r >> 1) & 3)) << 4) + (c & 15);
}

struct SlOperand {          // a sliced matrix on the device: n_slices x rowsP x kbytes int8 (K-block tiled, sl_offset) + row exponents
    const int8_t *slices = nullptr;
    int64_t rowsP = 0, kbytes = 0;
    int n_slices = 0;
    const int32_t *e = nullptr;   // nullptr: e_const for every row
    int e_const = 0;
    bool is_b = false;            // used as the B operand (output columns: 64-row tiles) or as the A operand (128-row tiles)
};

struct SlProduct {          // one segment: alpha * A[a_row0 : a_row0 + M, k0 : k0 + K] B[b_row0 : b_row0 + N, k0 : k0 + K]^T
    const SlOperand *A, *B;
    int64_t a_row0, b_row0, k0, K;
    int D;
    double alpha;
    int64_t k0b = -1;       // first K byte of the B operand when it differs from A's (-1: k0)
    const double *row_mul = nullptr;   // optional fp64 multiplier per A row (indexed like the A rows): alpha * row_mul[row]
};

struct SlBatch {            // blockIdx.y batches: per batch the A rows advance by a_rows, the B rows (and the exponents of both) by
    int n = 1;              // b_rows, A's first K byte by a_k and C by c elements
    int64_t a_rows = 0, b_rows = 0, a_k = 0, c = 0;
    int64_t b_k = 0;           // ... and B's first K byte by b_k (K split over batches: a_k = b_k = the chunk, c = one partial result)
    bool lower_only = false;   // skip tiles entirely above the diagonal (block-diagonal Gram tiles)
    bool ktri = false;         // B is strictly lower triangular in (row, K): column tile tj only needs the K blocks 0 .. tj
};

int sl_make_operand(gpfq_ctx *ctx, SlOperand *op, const int8_t *slices, int64_t rowsP, int64_t kbytes, int n_slices, const int32_t *e,
                    int e_const, bool is_b);
// C[M x N] (ldc) = or += sum of the products (at most two, sharing the exponents of their B rows).  M, N: valid extents; the
// slice tensors are zero-padded to the 128-row / 64-column / 64-byte tile grid.
// nbatch > 1: blockIdx.y batches whose A and B rows advance by batch_rows and whose C advances by batch_c elements (the
// block-diagonal Gram tiles of the residual-form sweep); lower_only skips tiles entirely above the diagonal.
int slgemm_i8(gpfq_ctx *ctx, const SlProduct *prod, int nprod, double *C, int64_t ldc, int64_t M, int64_t N, bool accumulate,
              int nbatch = 1, int64_t batch_rows = 0, int64_t batch_c = 0, bool lower_only = false);
int slgemm_i8_ex(gpfq_ctx *ctx, const SlProduct *prod, int nprod, double *C, int64_t ldc, int64_t M, int64_t N, bool accumulate,
                 const SlBatch &batch);
// 5 digit slices + row exponents of `grid_rows` rows (rows >= `rows` and columns >= cols are zeros) of a row-major matrix,
// written as rows row0 .. row0 + grid_rows - 1 of a 5 x rowsP x colsP slice tensor (e: exponent of row row0 + r at e[row0 + r])
template <typename T>
int sl_rowsplit(gpfq_ctx *ctx, const T *X, int64_t ldx, int64_t rows, int64_t cols, int32_t *e, int8_t *slices, int64_t rowsP,
                int64_t colsP, int64_t row0, int64_t grid_rows);
int sl_transsplit(gpfq_ctx *ctx, const float *X, const float *Xq, int64_t ldx, int64_t N0, int64_t m, int32_t *e, int *scratch,
                  int8_t *slices, int8_t *slices_q, int64_t mP, int64_t N0P);
