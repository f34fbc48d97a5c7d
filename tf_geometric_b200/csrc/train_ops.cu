// Training-mode kernels (SURVEY.md 8(f)4): dropout masks, per-head weighted aggregation and the GAT softmax backward.
// The reference obtains all of these from TensorFlow autodiff / tf.nn.dropout (gat.py:73-114, gcn.py:262,
// nn/sampling/drop_edge.py); here they are explicit kernels that reuse the destination-sorted CSR of the forward
// pass (and its transpose for the scatter-shaped gradients), deterministic, no atomics.
#include "common.cuh"
#include "rng.cuh"

namespace tfgk {
namespace {

constexpr int kTrainThreads = 256;
constexpr int kTrainWarps = kTrainThreads / 32;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// dropout weight of element idx: 1/(1-rate) when kept, 0 when dropped (tf.nn.dropout: keep iff u >= rate)
__device__ __forceinline__ float keep_scale(float rate, float scale, uint64_t seed, uint32_t stream, uint64_t idx) {
    if (rate <= 0.0f) return 1.0f;
    return random_uniform(seed, stream, idx) >= rate ? scale : 0.0f;
}

__global__ void dropout_kernel(const float *__restrict__ x, int64_t n, float rate, float scale, uint64_t seed,
                               uint32_t stream, float *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = x ? x[i] : 1.0f;
    const float k = keep_scale(rate, scale, seed, stream, (uint64_t)i);
    out[i] = k == 0.0f ? 0.0f : __fmul_rn(v, k);
}

// ---- per-head weighted aggregation -----------------------------------------------------------------------------
struct HeadsParams {
    const int64_t *rowptr;
    const int32_t *col;
    const int32_t *emap;     // position of edge e in the weight table (NULL: e itself)
    const float *w;          // [*, H]
    const float *src;
    int64_t lds;
    int32_t N, H, dh, mode;
    float rate, scale;
    uint64_t seed;
    uint32_t stream;
    float alpha;
    const float *bias;
    int act;
    float *out;
    int64_t ldo;
};

template <bool DROP = true>
__device__ __forceinline__ float head_weight(const HeadsParams &p, int64_t e, int h) {
    const int64_t pos = p.emap ? (int64_t)p.emap[e] : e;
    const float w = p.w[pos * p.H + h];
    if (!DROP) return w;                             // compiled without the generator: fewer registers, more warps
    const float k = keep_scale(p.rate, p.scale, p.seed, p.stream, (uint64_t)(pos * p.H + h));
    return k == 0.0f ? 0.0f : (p.rate > 0.0f ? __fmul_rn(w, k) : w);
}

// generic shape: one warp per destination row, lanes over output columns
__global__ void __launch_bounds__(kTrainThreads) spmm_heads_kernel(const HeadsParams p) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r = (int64_t)blockIdx.x * kTrainWarps + warp;
    if (r >= p.N) return;
    const int64_t e0 = p.rowptr[r], e1 = p.rowptr[r + 1];
    const int H = p.H, dh = p.dh;
    if (p.mode == TFGK_HEADS_REDUCE) {
        for (int u = lane; u < dh; u += 32) {
            float tot = 0.0f;
            for (int h = 0; h < H; ++h) {
                float acc = 0.0f;
                for (int64_t e = e0; e < e1; ++e)
                    acc = __fadd_rn(acc, __fmul_rn(p.src[(int64_t)p.col[e] * p.lds + (int64_t)h * dh + u], head_weight(p, e, h)));
                tot = h == 0 ? acc : __fadd_rn(tot, acc);
            }
            float v = __fmul_rn(tot, p.alpha);
            if (p.bias) v += p.bias[u];
            p.out[r * p.ldo + u] = apply_act(v, p.act);
        }
        return;
    }
    const int D = H * dh;
    for (int c = lane; c < D; c += 32) {
        const int h = c / dh;
        const int sc = p.mode == TFGK_HEADS_BROADCAST ? c - h * dh : c;
        float acc = 0.0f;
        for (int64_t e = e0; e < e1; ++e)
            acc = __fadd_rn(acc, __fmul_rn(p.src[(int64_t)p.col[e] * p.lds + sc], head_weight(p, e, h)));
        float v = __fmul_rn(acc, p.alpha);
        if (p.bias) v += p.bias[c];
        p.out[r * p.ldo + c] = apply_act(v, p.act);
    }
}

// H*dh == 128, split layout, 16-byte aligned rows: every lane owns one float4 of the output row and the head it
// belongs to; U edges in flight per iteration
template <int U, bool DROP>
__global__ void __launch_bounds__(kTrainThreads) spmm_heads128_kernel(const HeadsParams p) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r = (int64_t)blockIdx.x * kTrainWarps + warp;
    if (r >= p.N) return;
    const int64_t e0 = p.rowptr[r], e1 = p.rowptr[r + 1];
    const int h = (lane * 4) / p.dh;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int64_t e = e0;
    for (; e + U <= e1; e += U) {
        float4 v[U];
        float w[U];
#pragma unroll
        for (int i = 0; i < U; ++i) {
            v[i] = *reinterpret_cast<const float4 *>(p.src + (int64_t)p.col[e + i] * p.lds + lane * 4);
            w[i] = head_weight<DROP>(p, e + i, h);
        }
#pragma unroll
        for (int i = 0; i < U; ++i) {
            acc.x = __fadd_rn(acc.x, __fmul_rn(v[i].x, w[i]));
            acc.y = __fadd_rn(acc.y, __fmul_rn(v[i].y, w[i]));
            acc.z = __fadd_rn(acc.z, __fmul_rn(v[i].z, w[i]));
            acc.w = __fadd_rn(acc.w, __fmul_rn(v[i].w, w[i]));
        }
    }
    for (; e < e1; ++e) {
        const float4 v = *reinterpret_cast<const float4 *>(p.src + (int64_t)p.col[e] * p.lds + lane * 4);
        const float w = head_weight<DROP>(p, e, h);
        acc.x = __fadd_rn(acc.x, __fmul_rn(v.x, w));
        acc.y = __fadd_rn(acc.y, __fmul_rn(v.y, w));
        acc.z = __fadd_rn(acc.z, __fmul_rn(v.z, w));
        acc.w = __fadd_rn(acc.w, __fmul_rn(v.w, w));
    }
    float4 o;
    o.x = __fmul_rn(acc.x, p.alpha); o.y = __fmul_rn(acc.y, p.alpha);
    o.z = __fmul_rn(acc.z, p.alpha); o.w = __fmul_rn(acc.w, p.alpha);
    if (p.bias) {
        const float4 b = *reinterpret_cast<const float4 *>(p.bias + lane * 4);
        o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
    }
    o.x = apply_act(o.x, p.act); o.y = apply_act(o.y, p.act); o.z = apply_act(o.z, p.act); o.w = apply_act(o.w, p.act);
    *reinterpret_cast<float4 *>(p.out + r * p.ldo + lane * 4) = o;
}

// ---- GAT softmax backward ---------------------------------------------------------------------------------------
struct GatBwdParams {
    const int64_t *rowptr;
    const int32_t *col;
    const float *att;        // [E, H] softmax coefficients BEFORE dropout, CSR order
    const float *G;          // gradient w.r.t. the aggregated rows (before bias / activation)
    int64_t ldg;
    const float *V;
    int64_t ldv;
    int32_t N, H, dv, split;
    float rate, scale;
    uint64_t seed;
    uint32_t stream;
    float *ds;               // [E, H] out: gradient w.r.t. the raw (already scaled) scores
};

// one warp per destination row; sweep 1: da = <G_r, V_col> per edge and head, delta = sum a*da; sweep 2: ds = a (da - delta)
__global__ void __launch_bounds__(kTrainThreads) gat_softmax_bwd_kernel(const GatBwdParams p) {
    extern __shared__ float smem[];   // [warps][H]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r = (int64_t)blockIdx.x * kTrainWarps + warp;
    if (r >= p.N) return;
    const int H = p.H, dv = p.dv;
    float *delta = smem + (size_t)warp * H;
    const int64_t start = p.rowptr[r];
    const int deg = (int)(p.rowptr[r + 1] - start);
    const float *att = p.att + start * H;
    float *ds = p.ds + start * H;
    const int32_t *col = p.col + start;
    const float *grow = p.G + r * p.ldg;
    const float inv_h = 1.0f / (float)H;

    for (int h = lane; h < H; h += 32) delta[h] = 0.0f;
    __syncwarp();
    for (int e = 0; e < deg; ++e) {
        const float *vrow = p.V + (int64_t)col[e] * p.ldv;
        for (int h = 0; h < H; ++h) {
            float d = 0.0f;
            if (p.split) {
                for (int u = lane; u < dv; u += 32) d += grow[h * dv + u] * vrow[h * dv + u];
            } else {
                for (int u = lane; u < dv; u += 32) d += grow[u] * vrow[h * dv + u];
            }
            d = warp_sum(d);
            if (lane == 0) {
                if (!p.split) d *= inv_h;
                const int64_t idx = (int64_t)e * H + h;
                d *= keep_scale(p.rate, p.scale, p.seed, p.stream, (uint64_t)((start + e) * H + h));
                ds[idx] = d;
                delta[h] += att[idx] * d;
            }
        }
    }
    __syncwarp();
    for (int idx = lane; idx < deg * H; idx += 32) ds[idx] = att[idx] * (ds[idx] - delta[idx % H]);
}

// split layout with H*dv == 128 (dv a multiple of 4 dividing 128): lane owns one float4; the dot products of all heads
// are reduced at once inside groups of dv/4 lanes
template <int U, int MINB, bool DROP>
__global__ void __launch_bounds__(kTrainThreads, MINB) gat_softmax_bwd128_kernel(const GatBwdParams p) {
    extern __shared__ float smem[];   // [warps][H]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r = (int64_t)blockIdx.x * kTrainWarps + warp;
    if (r >= p.N) return;
    const int H = p.H;
    const int group = p.dv >> 2;                // lanes per head (power of two)
    const int h = lane / group;
    const bool leader = (lane % group) == 0;
    float *delta = smem + (size_t)warp * H;
    const int64_t start = p.rowptr[r];
    const int deg = (int)(p.rowptr[r + 1] - start);
    const float *att = p.att + start * H;
    float *ds = p.ds + start * H;
    const int32_t *col = p.col + start;
    const float4 g = *reinterpret_cast<const float4 *>(p.G + r * p.ldg + lane * 4);
    float dacc = 0.0f;
    auto finish = [&](float d, int e) {
        for (int off = group >> 1; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
        if (leader) {
            const int64_t idx = (int64_t)e * H + h;
            if (DROP) d *= keep_scale(p.rate, p.scale, p.seed, p.stream, (uint64_t)((start + e) * H + h));
            ds[idx] = d;
            dacc += att[idx] * d;
        }
    };
    int e = 0;
    for (; e + U <= deg; e += U) {                  // U gathered value rows in flight
        float4 v[U];
#pragma unroll
        for (int i = 0; i < U; ++i) v[i] = *reinterpret_cast<const float4 *>(p.V + (int64_t)col[e + i] * p.ldv + lane * 4);
#pragma unroll
        for (int i = 0; i < U; ++i) finish(g.x * v[i].x + g.y * v[i].y + g.z * v[i].z + g.w * v[i].w, e + i);
    }
    for (; e < deg; ++e) {
        const float4 v = *reinterpret_cast<const float4 *>(p.V + (int64_t)col[e] * p.ldv + lane * 4);
        finish(g.x * v.x + g.y * v.y + g.z * v.z + g.w * v.w, e);
    }
    if (leader) delta[h] = dacc;
    __syncwarp();
    for (int idx = lane; idx < deg * H; idx += 32) ds[idx] = att[idx] * (ds[idx] - delta[idx % H]);
}

inline bool pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }

}  // namespace
}  // namespace tfgk

using namespace tfgk;

extern "C" {

int tfgk_dropout_f32(const float *x, int64_t n, float rate, uint64_t seed, uint32_t rng_stream, float *out, void *stream) {
    TFGK_CHECK_ARG(n >= 0, "dropout: negative size");
    TFGK_CHECK_ARG(rate >= 0.0f && rate < 1.0f, "dropout: rate %g outside [0, 1)", (double)rate);
    if (n == 0) return TFGK_OK;
    TFGK_CHECK_ARG(out != nullptr, "dropout: null output");
    const float scale = 1.0f / (1.0f - rate);
    dropout_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, as_stream(stream)>>>(x, n, rate, scale, seed, rng_stream, out);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

int tfgk_spmm_heads_f32(const int64_t *rowptr, const int32_t *col, const int32_t *emap, const float *w,
                        const float *src, int64_t lds, int32_t n_dst, int32_t H, int32_t dh, int mode,
                        float drop_rate, uint64_t seed, uint32_t rng_stream, float alpha,
                        const float *bias, int act, float *out, int64_t ldo, void *stream) {
    TFGK_CHECK_ARG(n_dst >= 0 && H >= 1 && dh >= 1, "spmm_heads: bad size (n_dst=%d H=%d dh=%d)", n_dst, H, dh);
    TFGK_CHECK_ARG(mode == TFGK_HEADS_SPLIT || mode == TFGK_HEADS_BROADCAST || mode == TFGK_HEADS_REDUCE,
                   "spmm_heads: unknown mode %d", mode);
    TFGK_CHECK_ARG(act == TFGK_ACT_NONE || act == TFGK_ACT_RELU, "spmm_heads: unknown activation %d", act);
    TFGK_CHECK_ARG(drop_rate >= 0.0f && drop_rate < 1.0f, "spmm_heads: drop rate %g outside [0, 1)", (double)drop_rate);
    if (n_dst == 0) return TFGK_OK;
    TFGK_CHECK_ARG(rowptr && out, "spmm_heads: null pointer");
    const int64_t out_cols = mode == TFGK_HEADS_REDUCE ? dh : (int64_t)H * dh;
    const int64_t src_cols = mode == TFGK_HEADS_BROADCAST ? dh : (int64_t)H * dh;
    TFGK_CHECK_ARG(ldo >= out_cols && lds >= src_cols, "spmm_heads: leading dimension too small");
    HeadsParams p;
    p.rowptr = rowptr; p.col = col; p.emap = emap; p.w = w; p.src = src; p.lds = lds;
    p.N = n_dst; p.H = H; p.dh = dh; p.mode = mode;
    p.rate = drop_rate; p.scale = 1.0f / (1.0f - drop_rate); p.seed = seed; p.stream = rng_stream;
    p.alpha = alpha; p.bias = bias; p.act = act; p.out = out; p.ldo = ldo;
    const unsigned blocks = (unsigned)ceil_div64(n_dst, kTrainWarps);
    const bool fast = mode == TFGK_HEADS_SPLIT && (int64_t)H * dh == 128 && dh % 4 == 0 && aligned16(src) && aligned16(out) &&
                      lds % 4 == 0 && ldo % 4 == 0 && (!bias || aligned16(bias));
    if (fast) {
        if (drop_rate > 0.0f) spmm_heads128_kernel<4, true><<<blocks, kTrainThreads, 0, as_stream(stream)>>>(p);
        else spmm_heads128_kernel<4, false><<<blocks, kTrainThreads, 0, as_stream(stream)>>>(p);
    } else
        spmm_heads_kernel<<<blocks, kTrainThreads, 0, as_stream(stream)>>>(p);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

int tfgk_gat_softmax_bwd_f32(const int64_t *rowptr, const int32_t *col, const float *att,
                             const float *G, int64_t ldg, const float *V, int64_t ldv,
                             int32_t n_dst, int32_t H, int32_t dv, int split_value_heads,
                             float drop_rate, uint64_t seed, uint32_t rng_stream, float *ds, void *stream) {
    TFGK_CHECK_ARG(n_dst >= 0 && H >= 1 && dv >= 1, "gat_softmax_bwd: bad size (n_dst=%d H=%d dv=%d)", n_dst, H, dv);
    TFGK_CHECK_ARG(drop_rate >= 0.0f && drop_rate < 1.0f, "gat_softmax_bwd: drop rate %g outside [0, 1)", (double)drop_rate);
    if (n_dst == 0) return TFGK_OK;
    TFGK_CHECK_ARG(rowptr && G && V, "gat_softmax_bwd: null pointer");
    const int64_t g_cols = split_value_heads ? (int64_t)H * dv : dv;
    TFGK_CHECK_ARG(ldg >= g_cols && ldv >= (int64_t)H * dv, "gat_softmax_bwd: leading dimension too small");
    GatBwdParams p;
    p.rowptr = rowptr; p.col = col; p.att = att; p.G = G; p.ldg = ldg; p.V = V; p.ldv = ldv;
    p.N = n_dst; p.H = H; p.dv = dv; p.split = split_value_heads ? 1 : 0;
    p.rate = drop_rate; p.scale = 1.0f / (1.0f - drop_rate); p.seed = seed; p.stream = rng_stream; p.ds = ds;
    const unsigned blocks = (unsigned)ceil_div64(n_dst, kTrainWarps);
    const size_t smem = (size_t)kTrainWarps * H * sizeof(float);
    TFGK_CHECK_ARG(smem <= 48 * 1024, "gat_softmax_bwd: too many heads (%d)", H);
    const bool fast = p.split && (int64_t)H * dv == 128 && dv % 4 == 0 && pow2(dv >> 2) && aligned16(G) && aligned16(V) &&
                      ldg % 4 == 0 && ldv % 4 == 0;
    if (fast) {
        if (drop_rate > 0.0f) gat_softmax_bwd128_kernel<4, 4, true><<<blocks, kTrainThreads, smem, as_stream(stream)>>>(p);
        else gat_softmax_bwd128_kernel<4, 4, false><<<blocks, kTrainThreads, smem, as_stream(stream)>>>(p);
    } else
        gat_softmax_bwd_kernel<<<blocks, kTrainThreads, smem, as_stream(stream)>>>(p);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

}  // extern "C"
