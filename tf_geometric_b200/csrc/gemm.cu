// K4 (SIMT path): C = act(op(A) @ op(B) + bias + beta*C) in exact fp32 (FFMA), 128x128x8 tiles, 8x8 micro-tiles.
// This is the general fallback (any transpose, any shape, split-K for tall-skinny weight-gradient reductions).
// The forward projections x@W of the hot path go through the tcgen05 kernel in gemm_tc.cu when it applies.
#include "common.cuh"
#include <algorithm>

namespace tfgk {

constexpr int BM = 128, BN = 128, BK = 8;
constexpr int kGemmThreads = 256;
constexpr int PAD = 4;

struct GemmParams {
    const float *A; int64_t lda;
    const float *B; int64_t ldb;
    const float *bias; int act; float beta;
    int M, N, K;
    float *C; int64_t ldc;
    float *partial;     // split-K scratch [S][M][N] or nullptr
    int k_chunk;        // K range per z-slice (multiple of BK)
};

template <bool TA, bool TB>
__global__ void __launch_bounds__(kGemmThreads) sgemm_kernel(const GemmParams p) {
    __shared__ __align__(16) float As[BK][BM + PAD];
    __shared__ __align__(16) float Bs[BK][BN + PAD];
    const int t = threadIdx.x;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const int k_begin = blockIdx.z * p.k_chunk;
    const int k_end = min(p.K, k_begin + p.k_chunk);
    const int ty = t / 16, tx = t % 16;

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

    float ra[4], rb[4];
    auto load_tiles = [&](int k0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int m, k;
            if (TA) { m = t % BM; k = t / BM + 2 * i; } else { k = t % BK; m = t / BK + 32 * i; }
            const int gm = m0 + m, gk = k0 + k;
            ra[i] = (gm < p.M && gk < k_end) ? __ldg(TA ? p.A + (int64_t)gk * p.lda + gm : p.A + (int64_t)gm * p.lda + gk) : 0.0f;
            int n, kb;
            if (TB) { kb = t % BK; n = t / BK + 32 * i; } else { n = t % BN; kb = t / BN + 2 * i; }
            const int gn = n0 + n, gkb = k0 + kb;
            rb[i] = (gn < p.N && gkb < k_end) ? __ldg(TB ? p.B + (int64_t)gn * p.ldb + gkb : p.B + (int64_t)gkb * p.ldb + gn) : 0.0f;
        }
    };
    auto store_tiles = [&]() {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int m, k;
            if (TA) { m = t % BM; k = t / BM + 2 * i; } else { k = t % BK; m = t / BK + 32 * i; }
            As[k][m] = ra[i];
            int n, kb;
            if (TB) { kb = t % BK; n = t / BK + 32 * i; } else { n = t % BN; kb = t / BN + 2 * i; }
            Bs[kb][n] = rb[i];
        }
    };

    if (k_begin < k_end) load_tiles(k_begin);
    for (int k0 = k_begin; k0 < k_end; k0 += BK) {
        store_tiles();
        __syncthreads();
        if (k0 + BK < k_end) load_tiles(k0 + BK);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&As[k][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&Bs[k][64 + tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }

#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int gm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (gm >= p.M) continue;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int gn = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
            if (gn >= p.N) continue;
            if (p.partial) {
                p.partial[((int64_t)blockIdx.z * p.M + gm) * p.N + gn] = acc[i][j];
            } else {
                float v = acc[i][j];
                float *c = p.C + (int64_t)gm * p.ldc + gn;
                if (p.beta != 0.0f) v += p.beta * (*c);
                if (p.bias) v += p.bias[gn];
                *c = apply_act(v, p.act);
            }
        }
    }
}

__global__ void splitk_reduce_kernel(const GemmParams p, int S) {
    const int64_t total = (int64_t)p.M * p.N;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        float v = 0.0f;
        for (int z = 0; z < S; ++z) v += p.partial[(int64_t)z * total + i];   // fixed order: deterministic
        const int m = (int)(i / p.N), n = (int)(i % p.N);
        float *c = p.C + (int64_t)m * p.ldc + n;
        if (p.beta != 0.0f) v += p.beta * (*c);
        if (p.bias) v += p.bias[n];
        *c = apply_act(v, p.act);
    }
}

static int choose_splits(int M, int N, int K) {
    const int64_t tiles = ceil_div64(M, BM) * ceil_div64(N, BN);
    if (tiles >= 148 || K < 4096) return 1;
    int64_t s = (148 * 2) / tiles;
    const int64_t by_k = ceil_div64(K, 1024);
    if (s > by_k) s = by_k;
    return (int)(s < 1 ? 1 : s);
}

__global__ void __launch_bounds__(256) l2_normalize_kernel(const float *__restrict__ x, int64_t ldx, int32_t N, int32_t D,
                                                           float *__restrict__ out, int64_t ldo) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= N) return;
    float ss = 0.0f;
    for (int c = lane; c < D; c += 32) { const float v = x[r * ldx + c]; ss += v * v; }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    const float inv = rsqrtf(fmaxf(ss, 1e-12f));
    for (int c = lane; c < D; c += 32) out[r * ldo + c] = x[r * ldx + c] * inv;
}

// Column sums of a tall matrix: out[c] = sum_r x[r, c] (the bias gradients db = 1^T dY of every layer's backward pass).
// Two deterministic stages: each block sums a contiguous slab of rows per column (threads own columns, so a warp reads a
// contiguous row segment), partials are then added in block order.
constexpr int kColsumThreads = 256;

__global__ void __launch_bounds__(kColsumThreads) colsum_partial_kernel(const float *__restrict__ x, int64_t ldx, int64_t n_rows,
                                                                       int32_t D, int64_t rows_per_block, float *__restrict__ partial) {
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
    const int64_t r1 = r0 + rows_per_block < n_rows ? r0 + rows_per_block : n_rows;
    // a block covers the columns in passes of blockDim.x; inside a pass thread t owns column c0 + t
    for (int c = threadIdx.x; c < D; c += kColsumThreads) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        int64_t r = r0;
        for (; r + 4 <= r1; r += 4) {
            a0 += x[r * ldx + c];
            a1 += x[(r + 1) * ldx + c];
            a2 += x[(r + 2) * ldx + c];
            a3 += x[(r + 3) * ldx + c];
        }
        for (; r < r1; ++r) a0 += x[r * ldx + c];
        partial[(int64_t)blockIdx.x * D + c] = (a0 + a1) + (a2 + a3);
    }
}

__global__ void __launch_bounds__(kColsumThreads) colsum_final_kernel(const float *__restrict__ partial, int32_t n_blocks, int32_t D,
                                                                     float *__restrict__ out) {
    const int c = blockIdx.x * kColsumThreads + threadIdx.x;
    if (c >= D) return;
    float acc = 0.f;
    for (int b = 0; b < n_blocks; ++b) acc += partial[(int64_t)b * D + c];
    out[c] = acc;
}

}  // namespace tfgk

using namespace tfgk;

static int colsum_blocks(int64_t n_rows) {
    int64_t b = ceil_div64(n_rows, 512);
    if (b > 148 * 8) b = 148 * 8;
    return (int)(b < 1 ? 1 : b);
}

extern "C" int tfgk_colsum_workspace_bytes(int64_t n_rows, int32_t D, size_t *out_bytes) {
    TFGK_CHECK_ARG(out_bytes != nullptr && n_rows >= 0 && D >= 0, "colsum_workspace_bytes: bad argument");
    *out_bytes = (size_t)colsum_blocks(n_rows) * (size_t)(D > 0 ? D : 1) * sizeof(float);
    return TFGK_OK;
}

extern "C" int tfgk_colsum_f32(const float *x, int64_t ldx, int64_t n_rows, int32_t D, float *out, void *workspace,
                               size_t workspace_bytes, void *stream) {
    TFGK_CHECK_ARG(n_rows >= 0 && D >= 0, "colsum: negative size");
    if (D == 0) return TFGK_OK;
    TFGK_CHECK_ARG(out != nullptr && (n_rows == 0 || (x != nullptr && ldx >= D)), "colsum: bad argument");
    const int nb = colsum_blocks(n_rows);
    TFGK_CHECK_ARG(workspace != nullptr && workspace_bytes >= (size_t)nb * D * sizeof(float), "colsum: workspace too small");
    cudaStream_t st = as_stream(stream);
    const int64_t rows_per_block = ceil_div64(n_rows > 0 ? n_rows : 1, nb);
    colsum_partial_kernel<<<nb, kColsumThreads, 0, st>>>(x, ldx, n_rows, D, rows_per_block, static_cast<float *>(workspace));
    TFGK_LAUNCH_CHECK();
    colsum_final_kernel<<<(unsigned)ceil_div64(D, kColsumThreads), kColsumThreads, 0, st>>>(static_cast<float *>(workspace), nb, D, out);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

namespace tfgk {
}  // namespace tfgk

using namespace tfgk;

extern "C" int tfgk_gemm_workspace_bytes(int32_t M, int32_t N, int32_t K, size_t *out_bytes) {
    TFGK_CHECK_ARG(out_bytes != nullptr, "gemm_workspace_bytes: null output");
    TFGK_CHECK_ARG(M >= 0 && N >= 0 && K >= 0, "gemm_workspace_bytes: negative size");
    const int s = (M == 0 || N == 0) ? 1 : choose_splits(M, N, K);
    *out_bytes = s > 1 ? (size_t)s * M * N * sizeof(float) : 0;
    return TFGK_OK;
}

// tensor-core path (gemm_tc.cu); returns TFGK_ERR_UNSUPPORTED when the shape/layout does not qualify
extern "C" int tfgk_gemm_tc_f32(const float *A, int64_t lda, const float *B, int64_t ldb, const float *bias, int act,
                                int32_t M, int32_t N, int32_t K, float *C, int64_t ldc, void *stream);

extern "C" int tfgk_gemm_f32(const float *A, int64_t lda, int transA, const float *B, int64_t ldb, int transB,
                             const float *bias, int act, float beta, int32_t M, int32_t N, int32_t K,
                             float *C, int64_t ldc, void *workspace, size_t workspace_bytes, void *stream) {
    TFGK_CHECK_ARG(M >= 0 && N >= 0 && K >= 0, "gemm: negative size");
    TFGK_CHECK_ARG(act == TFGK_ACT_NONE || act == TFGK_ACT_RELU, "gemm: unknown activation %d", act);
    if (M == 0 || N == 0) return TFGK_OK;
    TFGK_CHECK_ARG(C != nullptr && ldc >= N, "gemm: bad C");
    TFGK_CHECK_ARG(K == 0 || (A && B), "gemm: null operand");
    TFGK_CHECK_ARG(K == 0 || (lda >= (transA ? M : K) && ldb >= (transB ? K : N)), "gemm: leading dimension too small");
    cudaStream_t st = as_stream(stream);

    if (!transA && beta == 0.0f && K > 0) {
        // tall projections (and dX = dY W^T with transB): the multi-block tcgen05 kernel (gemm_proj.cu), N cut into blocks
        // of <= 128 columns
        if (N <= 512 && (int64_t)M * K >= (1 << 14)) {
            tfgk_proj_block blocks[4];
            int nb = 0;
            for (int c0 = 0; c0 < N; c0 += 128, ++nb) {
                const int w = N - c0 < 128 ? N - c0 : 128;
                blocks[nb].B = transB ? B + (int64_t)c0 * ldb : B + c0; blocks[nb].ldb = ldb; blocks[nb].ncols = w;
                blocks[nb].transB = transB ? 1 : 0;
                blocks[nb].bias = bias ? bias + c0 : nullptr; blocks[nb].act = act;
                blocks[nb].C = C + c0; blocks[nb].ldc = ldc;
            }
            const float *parts[1] = {A};
            const int rcp = tfgk_gemm_proj_f32(parts, 1, 0, lda, M, K, blocks, nb, 0, 0, stream);
            if (rcp != TFGK_ERR_UNSUPPORTED) return rcp;
        }
        if (!transB) {
            const int rc = tfgk_gemm_tc_f32(A, lda, B, ldb, bias, act, M, N, K, C, ldc, stream);
            if (rc != TFGK_ERR_UNSUPPORTED) return rc;
        }
    }

    GemmParams p;
    p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.bias = bias; p.act = act; p.beta = beta;
    p.M = M; p.N = N; p.K = K; p.C = C; p.ldc = ldc; p.partial = nullptr;
    int S = choose_splits(M, N, K);
    if (S > 1 && (workspace == nullptr || workspace_bytes < (size_t)S * M * N * sizeof(float))) S = 1;
    p.k_chunk = (int)(ceil_div64(ceil_div64(K > 0 ? K : 1, S), BK) * BK);
    if (S > 1) p.partial = static_cast<float *>(workspace);
    dim3 grid((unsigned)ceil_div64(M, BM), (unsigned)ceil_div64(N, BN), (unsigned)S);
    TFGK_CHECK_ARG(grid.y <= 65535, "gemm: N too large for the SIMT path (N=%d)", N);
    if (transA && transB) sgemm_kernel<true, true><<<grid, kGemmThreads, 0, st>>>(p);
    else if (transA)      sgemm_kernel<true, false><<<grid, kGemmThreads, 0, st>>>(p);
    else if (transB)      sgemm_kernel<false, true><<<grid, kGemmThreads, 0, st>>>(p);
    else                  sgemm_kernel<false, false><<<grid, kGemmThreads, 0, st>>>(p);
    TFGK_LAUNCH_CHECK();
    if (S > 1) {
        splitk_reduce_kernel<<<(unsigned)std::min<int64_t>(ceil_div64((int64_t)M * N, 256), 148 * 8), 256, 0, st>>>(p, S);
        TFGK_LAUNCH_CHECK();
    }
    return TFGK_OK;
}

extern "C" int tfgk_l2_normalize_f32(const float *x, int64_t ldx, int32_t N, int32_t D, float *out, int64_t ldo,
                                     void *stream) {
    TFGK_CHECK_ARG(N >= 0 && D >= 0, "l2_normalize: negative size");
    if (N == 0 || D == 0) return TFGK_OK;
    TFGK_CHECK_ARG(x && out && ldx >= D && ldo >= D, "l2_normalize: bad argument");
    l2_normalize_kernel<<<(unsigned)ceil_div64(N, 8), 256, 0, as_stream(stream)>>>(x, ldx, N, D, out, ldo);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}
