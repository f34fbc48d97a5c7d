// K3: edge softmax (tfgk_segment_softmax_f32) and the fused GAT aggregation (tfgk_gat_fused_f32).
//
// One warp owns one destination row r of the self-looped CSR and runs three phases without leaving the SM:
//   A   stream the K rows of the neighbours (one coalesced 4*A-byte request per edge), dot them with Q[r] per head,
//       write the raw scores s[e,h] to the [E,H] attention buffer and keep the exact per-head maximum;
//   B1  walk the row's H*deg scores flat and coalesced: p = exp(s - max), accumulate the per-head denominators;
//   B2  stream the V rows of the neighbours and accumulate  a_e * V[col_e]  in CSR (= reference) order, with
//       a_e = p_e / (sum + 1e-8)  exactly as nn/kernel/segment.py:26-33 computes it.
// K and V are each read once per edge, Q and the output once per node: 4*(A+U)+4 bytes per edge - the HBM
// roofline of the reference's 5-pass segment_softmax + two [E,A] gathers + SpMM pipeline (SURVEY.md 8d).
// No tensor cores: the per-edge dot products are 16-wide and the kernel is bound by the gathers.
#include "common.cuh"

namespace tfgk {

constexpr int kGatThreads = 256;
constexpr int kGatWarps = kGatThreads / 32;
constexpr int kMaxHeadsFast = 32;

__device__ __forceinline__ float4 ldg4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }

struct GatParams {
    const int64_t *rowptr;
    const int32_t *col;
    const float *Q; int64_t ldq;
    const float *K; int64_t ldk;
    const float *V; int64_t ldv;
    int32_t N, H, dqk, dv;
    float scale;
    int split;
    const float *bias;
    int act;
    float *att;          // NOT restrict/const: written and re-read by the same warp
    int write_att;
    float *out; int64_t ldo;
    // optional work plan (tfgk_plan)
    int32_t n_tasks;
    const int32_t *task_row, *task_nrows;
    const int64_t *task_e0, *task_e1;
    const int32_t *task_slot;
    int32_t n_hubs;
    const int32_t *hub_row, *hub_slot0, *hub_nslots;
    float *scratch;      // per slot: [A] partial sums | [32] running max per lane | [32] denominators per lane
    float *stats;        // optional [N, 2H]: per (row, head) softmax maximum and denominator (+1e-8), kept for the backward pass
};

// ---- fast path: float4 lanes, H | 32, dqk/4 a power of two, heads concatenated ---------------------------------
template <int NCK, int NCV, int U>
__global__ void __launch_bounds__(kGatThreads) gat_fast_kernel(const GatParams p) {
    __shared__ float s_max[kGatWarps][kMaxHeadsFast];
    __shared__ float s_den[kGatWarps][kMaxHeadsFast];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r = (int64_t)blockIdx.x * kGatWarps + warp;
    if (r >= p.N) return;   // warp-uniform
    const int H = p.H;
    const int A = H * p.dqk, VW = H * p.dv;
    const int lanes_per_head = p.dqk >> 2;
    const int64_t start = p.rowptr[r];
    const int deg = (int)(p.rowptr[r + 1] - start);
    float *att = p.att + start * H;

    // ---------------- phase A: scores ----------------
    int kcol[NCK];
    bool kok[NCK];
    float4 q[NCK];
    float mx[NCK];
#pragma unroll
    for (int k = 0; k < NCK; ++k) {
        kcol[k] = (lane + 32 * k) * 4;
        kok[k] = kcol[k] < A;
        q[k] = kok[k] ? ldg4(p.Q + r * p.ldq + kcol[k]) : make_float4(0.f, 0.f, 0.f, 0.f);
        mx[k] = -FLT_MAX;
    }
    for (int t = 0; t < deg; t += 32) {
        const int e = t + lane;
        const int my_c = e < deg ? ld_stream_i32(p.col + start + e) : 0;
        const int nb = min(32, deg - t);
        for (int j = 0; j < nb; j += U) {
            float4 kk[U][NCK];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int c = __shfl_sync(0xffffffffu, my_c, j + u);
                const float *rowp = p.K + (int64_t)c * p.ldk;
#pragma unroll
                for (int k = 0; k < NCK; ++k)
                    if (j + u < nb && kok[k]) kk[u][k] = ldg4(rowp + kcol[k]);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const bool ok = j + u < nb;   // warp-uniform
#pragma unroll
                for (int k = 0; k < NCK; ++k) {
                    float d = 0.0f;
                    if (ok && kok[k])
                        d = q[k].x * kk[u][k].x + q[k].y * kk[u][k].y + q[k].z * kk[u][k].z + q[k].w * kk[u][k].w;
                    for (int off = 1; off < lanes_per_head; off <<= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
                    if (ok && kok[k]) {
                        const float s = __fdiv_rn(d, p.scale);
                        mx[k] = fmaxf(mx[k], s);
                        if ((lane & (lanes_per_head - 1)) == 0) att[(int64_t)(t + j + u) * H + kcol[k] / p.dqk] = s;
                    }
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < NCK; ++k)
        if (kok[k] && (lane & (lanes_per_head - 1)) == 0) s_max[warp][kcol[k] / p.dqk] = mx[k];
    __syncwarp();

    // ---------------- phase B1: exp and denominators (flat, coalesced; head of a lane = lane % H) -------------
    {
        const float m = s_max[warp][lane & (H - 1)];
        float part = 0.0f;
        const int total = deg * H;
        for (int f = 0; f < total; f += 32) {
            const int idx = f + lane;
            if (idx < total) {
                const float pexp = expf(att[idx] - m);
                att[idx] = pexp;
                part += pexp;
            }
        }
        for (int off = 16; off >= H; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
        s_den[warp][lane & (H - 1)] = part + 1e-8f;
    }
    __syncwarp();

    // ---------------- phase B2: weighted aggregation of V ----------------
    int vcol[NCV], vhead[NCV];
    bool vok[NCV];
    float den[NCV];
    float acc[NCV][4];
#pragma unroll
    for (int k = 0; k < NCV; ++k) {
        vcol[k] = (lane + 32 * k) * 4;
        vok[k] = vcol[k] < VW;
        vhead[k] = vok[k] ? vcol[k] / p.dv : 0;
        den[k] = s_den[warp][vhead[k]];
        acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.0f;
    }
    for (int t = 0; t < deg; t += 32) {
        const int e = t + lane;
        const int my_c = e < deg ? __ldg(p.col + start + e) : 0;
        const int nb = min(32, deg - t);
        for (int j = 0; j < nb; j += U) {
            float4 vv[U][NCV];
            float pe[U][NCV];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int c = __shfl_sync(0xffffffffu, my_c, j + u);
                const float *rowp = p.V + (int64_t)c * p.ldv;
#pragma unroll
                for (int k = 0; k < NCV; ++k)
                    if (j + u < nb && vok[k]) {
                        vv[u][k] = ldg4(rowp + vcol[k]);
                        pe[u][k] = att[(int64_t)(t + j + u) * H + vhead[k]];
                    }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (j + u < nb) {
#pragma unroll
                    for (int k = 0; k < NCV; ++k) {
                        if (vok[k]) {
                            const float a = __fdiv_rn(pe[u][k], den[k]);
                            acc[k][0] = __fadd_rn(acc[k][0], __fmul_rn(vv[u][k].x, a));
                            acc[k][1] = __fadd_rn(acc[k][1], __fmul_rn(vv[u][k].y, a));
                            acc[k][2] = __fadd_rn(acc[k][2], __fmul_rn(vv[u][k].z, a));
                            acc[k][3] = __fadd_rn(acc[k][3], __fmul_rn(vv[u][k].w, a));
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < NCV; ++k) {
        if (!vok[k]) continue;
        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) b = ldg4(p.bias + vcol[k]);
        float4 o;
        o.x = apply_act(acc[k][0] + b.x, p.act);
        o.y = apply_act(acc[k][1] + b.y, p.act);
        o.z = apply_act(acc[k][2] + b.z, p.act);
        o.w = apply_act(acc[k][3] + b.w, p.act);
        *reinterpret_cast<float4 *>(p.out + r * p.ldo + vcol[k]) = o;
    }
    if (p.write_att) {
        __syncwarp();
        const float dn = s_den[warp][lane & (H - 1)];
        const int total = deg * H;
        for (int f = 0; f < total; f += 32) {
            const int idx = f + lane;
            if (idx < total) att[idx] = __fdiv_rn(att[idx], dn);
        }
    }
}

// ---- single-pass path (dqk == dv): one walk over the edges with an online softmax ----------------------------------
// Per edge the K row gives the per-head score, and the V row is consumed in the same iteration:
//     m' = max(m, s);  acc = acc * exp(m - m') + exp(s - m') * V[col];  l = l * exp(m - m') + exp(s - m')
// (U edges share one rescale).  K and V are each read once, together - when the caller projects them into one
// [N, A+U] buffer (V == K + A, same leading dimension) the two 16-byte loads of a lane hit the same 1 KB DRAM
// burst.  No score scratch is touched unless the attention coefficients are requested.  The result differs from the
// reference's max -> exp -> sum -> divide order only by the rounding of the rescales (<= 1e-6 relative).
template <int NC, int U>
__global__ void __launch_bounds__(kGatThreads) gat_online_kernel(const GatParams p) {
    __shared__ float s_max[kGatWarps][kMaxHeadsFast];
    __shared__ float s_den[kGatWarps][kMaxHeadsFast];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r = (int64_t)blockIdx.x * kGatWarps + warp;
    if (r >= p.N) return;
    const int H = p.H;
    const int A = H * p.dqk;
    const int lanes_per_head = p.dqk >> 2;
    const bool head_leader = (lane & (lanes_per_head - 1)) == 0;
    const int64_t start = p.rowptr[r];
    const int deg = (int)(p.rowptr[r + 1] - start);
    float *att = p.att ? p.att + start * H : nullptr;
    const bool want_att = p.write_att != 0;

    int ccol[NC];
    bool cok[NC];
    float4 q[NC];
    float mx[NC], den[NC];
    float acc[NC][4];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        ccol[k] = (lane + 32 * k) * 4;
        cok[k] = ccol[k] < A;
        q[k] = cok[k] ? ldg4(p.Q + r * p.ldq + ccol[k]) : make_float4(0.f, 0.f, 0.f, 0.f);
        mx[k] = -FLT_MAX;
        den[k] = 0.0f;
        acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.0f;
    }
    for (int t = 0; t < deg; t += 32) {
        const int e = t + lane;
        const int my_c = e < deg ? ld_stream_i32(p.col + start + e) : 0;
        const int nb = min(32, deg - t);
        for (int j = 0; j < nb; j += U) {
            float4 kk[U][NC], vv[U][NC];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int c = __shfl_sync(0xffffffffu, my_c, j + u);
                const float *krow = p.K + (int64_t)c * p.ldk;
                const float *vrow = p.V + (int64_t)c * p.ldv;
#pragma unroll
                for (int k = 0; k < NC; ++k)
                    if (j + u < nb && cok[k]) {
                        kk[u][k] = ldg4(krow + ccol[k]);
                        vv[u][k] = ldg4(vrow + ccol[k]);
                    }
            }
            float sc[U][NC];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const bool ok = j + u < nb;       // warp-uniform
#pragma unroll
                for (int k = 0; k < NC; ++k) {
                    float d = 0.0f;
                    if (ok && cok[k])
                        d = q[k].x * kk[u][k].x + q[k].y * kk[u][k].y + q[k].z * kk[u][k].z + q[k].w * kk[u][k].w;
                    for (int off = 1; off < lanes_per_head; off <<= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
                    sc[u][k] = ok ? __fdiv_rn(d, p.scale) : -FLT_MAX;
                    if (want_att && ok && cok[k] && head_leader) att[(int64_t)(t + j + u) * H + ccol[k] / p.dqk] = sc[u][k];
                }
            }
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                float m_new = mx[k];
#pragma unroll
                for (int u = 0; u < U; ++u) m_new = fmaxf(m_new, sc[u][k]);
                const float corr = expf(mx[k] - m_new);        // exp(-huge) = 0 on the first group
                mx[k] = m_new;
                den[k] *= corr;
                acc[k][0] *= corr; acc[k][1] *= corr; acc[k][2] *= corr; acc[k][3] *= corr;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (j + u < nb && cok[k]) {
                        const float pe = expf(sc[u][k] - m_new);
                        den[k] += pe;
                        acc[k][0] = fmaf(pe, vv[u][k].x, acc[k][0]);
                        acc[k][1] = fmaf(pe, vv[u][k].y, acc[k][1]);
                        acc[k][2] = fmaf(pe, vv[u][k].z, acc[k][2]);
                        acc[k][3] = fmaf(pe, vv[u][k].w, acc[k][3]);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        if (!cok[k]) continue;
        const float inv = 1.0f / (den[k] + 1e-8f);
        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) b = ldg4(p.bias + ccol[k]);
        float4 o;
        o.x = apply_act(acc[k][0] * inv + b.x, p.act);
        o.y = apply_act(acc[k][1] * inv + b.y, p.act);
        o.z = apply_act(acc[k][2] * inv + b.z, p.act);
        o.w = apply_act(acc[k][3] * inv + b.w, p.act);
        *reinterpret_cast<float4 *>(p.out + r * p.ldo + ccol[k]) = o;
        if (want_att && head_leader) {
            s_max[warp][ccol[k] / p.dqk] = mx[k];
            s_den[warp][ccol[k] / p.dqk] = den[k] + 1e-8f;
        }
    }
    if (want_att) {      // raw scores -> coefficients, flat and coalesced (head of a lane = lane % H)
        __syncwarp();
        const float m = s_max[warp][lane & (H - 1)], dn = s_den[warp][lane & (H - 1)];
        const int total = deg * H;
        for (int f = 0; f < total; f += 32) {
            const int idx = f + lane;
            if (idx < total) att[idx] = __fdiv_rn(expf(att[idx] - m), dn);
        }
    }
}

// ---- single-pass path on a cp.async ring (A == H*dv <= 128) ----------------------------------------------------------
// Same arithmetic as gat_online_kernel, same memory pipeline as spmm_async_kernel (see spmm.cu): a warp owns
// kGatAsyncRows consecutive destination rows = one contiguous CSR range and streams it in rounds of U edges; every
// round is 2*U LDGSTS per lane (the K and the V slice of each neighbour) into a per-warp ring of S stages tracked by
// commit groups, so (S-1)*U neighbour pairs are always in flight per warp at 64 registers.  The online softmax is
// updated per edge (one expf), which lets a round straddle row boundaries.
constexpr int kGatAsyncRows = 32;
constexpr int kGatAsyncWarps = 4;

__device__ __forceinline__ void gat_cp_async16(uint32_t dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}

template <int U, int S>
__global__ void __launch_bounds__(kGatAsyncWarps * 32) gat_async_kernel(const GatParams p) {
    static_assert(32 % U == 0, "a round must not straddle an index chunk");
    constexpr int RPC = 32 / U;
    static_assert(S <= RPC, "index chunk refill assumes the prologue stays inside chunk 0");
    extern __shared__ __align__(16) uint8_t gat_ring[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t task = (int64_t)blockIdx.x * kGatAsyncWarps + warp;
    int64_t r0, r1, e_begin, e_stop;
    int slot = -1;
    if (p.task_row != nullptr) {
        if (task >= p.n_tasks) return;
        r0 = p.task_row[task];
        r1 = r0 + p.task_nrows[task];
        e_begin = p.task_e0[task];
        e_stop = p.task_e1[task];
        slot = p.task_slot[task];
    } else {
        r0 = task * kGatAsyncRows;
        if (r0 >= p.N) return;
        r1 = min((int64_t)p.N, r0 + kGatAsyncRows);
        e_begin = p.rowptr[r0];
        e_stop = p.rowptr[r1];
    }
    const int64_t rp_hi = p.rowptr[min(r0 + lane + 1, r1)];
    const int n_edges = (int)(e_stop - e_begin);
    const int n_rounds = (n_edges + U - 1) / U;
    const int A = p.H * p.dqk;
    const int lanes_per_head = p.dqk >> 2;
    const int ccol = lane * 4;
    const bool cok = ccol < A;
    const uint32_t row_bytes = (uint32_t)A * 4u;
    const uint32_t stage_bytes = 2u * U * row_bytes;          // [U][K slice row | V slice row]
    uint8_t *my_ring = gat_ring + (size_t)warp * S * stage_bytes;
    const uint32_t ring_addr = (uint32_t)__cvta_generic_to_shared(my_ring);

    int64_t r = r0;
    int row_end = slot >= 0 ? 0x7fffffff : (int)(__shfl_sync(0xffffffffu, rp_hi, 0) - e_begin);   // hub slices never close
    float4 q = cok ? ldg4(p.Q + r * p.ldq + ccol) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 q_next = (cok && r + 1 < r1) ? ldg4(p.Q + (r + 1) * p.ldq + ccol) : make_float4(0.f, 0.f, 0.f, 0.f);
    float mx = -FLT_MAX, den = 0.0f, a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.bias && cok) bias = ldg4(p.bias + ccol);

    auto finalize_row = [&]() {
        if (cok) {
            const float inv = 1.0f / (den + 1e-8f);
            float4 o;
            o.x = apply_act(a0 * inv + bias.x, p.act);
            o.y = apply_act(a1 * inv + bias.y, p.act);
            o.z = apply_act(a2 * inv + bias.z, p.act);
            o.w = apply_act(a3 * inv + bias.w, p.act);
            *reinterpret_cast<float4 *>(p.out + r * p.ldo + ccol) = o;
            if (p.stats != nullptr && (lane % lanes_per_head) == 0) {      // training: (max, denominator) instead of [E, H] coefficients
                p.stats[r * 2 * p.H + lane / lanes_per_head] = mx;
                p.stats[r * 2 * p.H + p.H + lane / lanes_per_head] = den + 1e-8f;
            }
        }
        mx = -FLT_MAX; den = 0.0f; a0 = a1 = a2 = a3 = 0.0f;
        ++r;
        q = q_next;
        if (r < r1) {
            row_end = (int)(__shfl_sync(0xffffffffu, rp_hi, (int)(r - r0)) - e_begin);
            if (cok && r + 1 < r1) q_next = ldg4(p.Q + (r + 1) * p.ldq + ccol);
        }
    };
    auto load_chunk = [&](int c) {
        const int e = c * 32 + lane;
        return e < n_edges ? ld_stream_i32(p.col + e_begin + e) : 0;
    };
    auto issue = [&](int g, int ci) {
        if (g < n_rounds) {
            const int base = (g % RPC) * U;
            const uint32_t dst0 = ring_addr + (uint32_t)(g % S) * stage_bytes;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int c = __shfl_sync(0xffffffffu, ci, base + u);
                if (g * U + u < n_edges && cok) {
                    gat_cp_async16(dst0 + (2 * u) * row_bytes + ccol * 4, p.K + (int64_t)c * p.ldk + ccol);
                    gat_cp_async16(dst0 + (2 * u + 1) * row_bytes + ccol * 4, p.V + (int64_t)c * p.ldv + ccol);
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    int ca = load_chunk(0), cb = load_chunk(1);
#pragma unroll
    for (int g = 0; g < S - 1; ++g) issue(g, ca);

    for (int g = 0; g < n_rounds; ++g) {
        {
            const int gn = g + S - 1;
            issue(gn, ((gn / RPC) & 1) ? cb : ca);
        }
        asm volatile("cp.async.wait_group %0;" ::"n"(S - 1) : "memory");
        const uint8_t *sbuf = my_ring + (size_t)(g % S) * stage_bytes;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = g * U + u;
            if (e < n_edges) {
                while (e == row_end) finalize_row();
                float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
                if (cok) {
                    kk = *reinterpret_cast<const float4 *>(sbuf + (size_t)(2 * u) * row_bytes + ccol * 4);
                    vv = *reinterpret_cast<const float4 *>(sbuf + (size_t)(2 * u + 1) * row_bytes + ccol * 4);
                }
                float d = q.x * kk.x + q.y * kk.y + q.z * kk.z + q.w * kk.w;
                for (int off = 1; off < lanes_per_head; off <<= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
                const float s = __fdiv_rn(d, p.scale);
                // one exponential per edge: the new maximum is either s (rescale the running sums) or mx (scale the term)
                const bool up = s > mx;
                const float t = expf(up ? mx - s : s - mx);
                const float corr = up ? t : 1.0f, pe = up ? 1.0f : t;
                mx = up ? s : mx;
                den = fmaf(den, corr, pe);
                a0 = fmaf(a0, corr, pe * vv.x);
                a1 = fmaf(a1, corr, pe * vv.y);
                a2 = fmaf(a2, corr, pe * vv.z);
                a3 = fmaf(a3, corr, pe * vv.w);
            }
        }
        if ((g + S) % RPC == 0) {                 // the last round of chunk `dead` has been issued: refill its register
            const int dead = (g + S) / RPC - 1;
            if (dead & 1) cb = load_chunk(dead + 2); else ca = load_chunk(dead + 2);
        }
    }
    if (slot >= 0) {                      // hub slice: partial (sums, max, denominator), merged by gat_hub_fixup_kernel
        float *dst = p.scratch + (int64_t)slot * (A + 64);
        if (cok) *reinterpret_cast<float4 *>(dst + ccol) = make_float4(a0, a1, a2, a3);
        dst[A + lane] = mx;
        dst[A + 32 + lane] = den;
        return;
    }
    while (r < r1) finalize_row();
}

// ---- the same kernel with the neighbour rows fetched by TMA tile::gather4 (north_star: "staged through TMA") ------------------
// K and V are projected into ONE [N, 2A] buffer (nn/conv/gat.py), so a tensor map over that buffer with a box of 2A columns x 1
// row lets ONE cp.async.bulk.tensor...tile::gather4 fetch the key AND the value rows of four neighbours (4 x 2A x 4 bytes = 4 KB
// at A = 128) into the warp's ring stage, completing its mbarrier with the transaction bytes.  Arithmetic, edge order and the
// online softmax are those of gat_async_kernel: same bits.  Requires V == K + A columns in the same buffer (ldk == ldv).
__device__ __forceinline__ void gat_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (spin > (1u << 28)) __trap();
    }
}

template <int S>
__global__ void __launch_bounds__(kGatAsyncWarps * 32) gat_gather4_kernel(const GatParams p, const __grid_constant__ TensorMap tmap) {
    constexpr int U = 4, RPC = 32 / U;
    static_assert(S <= RPC, "index chunk refill assumes the prologue stays inside chunk 0");
    extern __shared__ __align__(128) uint8_t gat_g4_ring[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int A = p.H * p.dqk;
    const uint32_t edge_bytes = 2u * (uint32_t)A * 4u;            // [K row | V row] of one neighbour, contiguous in the KV buffer
    const uint32_t tx_bytes = U * edge_bytes;
    const uint32_t stage_bytes = (tx_bytes + 127u) & ~127u;
    uint8_t *my_ring = gat_g4_ring + (size_t)warp * S * stage_bytes;
    const uint32_t ring_addr = (uint32_t)__cvta_generic_to_shared(my_ring);
    uint64_t *bars = reinterpret_cast<uint64_t *>(gat_g4_ring + (size_t)kGatAsyncWarps * S * stage_bytes) + warp * S;
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(bars);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < S; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8 * i));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const int64_t task = (int64_t)blockIdx.x * kGatAsyncWarps + warp;
    int64_t r0, r1, e_begin, e_stop;
    int slot = -1;
    if (p.task_row != nullptr) {
        if (task >= p.n_tasks) return;
        r0 = p.task_row[task];
        r1 = r0 + p.task_nrows[task];
        e_begin = p.task_e0[task];
        e_stop = p.task_e1[task];
        slot = p.task_slot[task];
    } else {
        r0 = task * kGatAsyncRows;
        if (r0 >= p.N) return;
        r1 = min((int64_t)p.N, r0 + kGatAsyncRows);
        e_begin = p.rowptr[r0];
        e_stop = p.rowptr[r1];
    }
    const int64_t rp_hi = p.rowptr[min(r0 + lane + 1, r1)];
    const int n_edges = (int)(e_stop - e_begin);
    const int n_rounds = (n_edges + U - 1) / U;
    const int lanes_per_head = p.dqk >> 2;
    const int ccol = lane * 4;
    const bool cok = ccol < A;
    const uint32_t row_bytes = (uint32_t)A * 4u;

    int64_t r = r0;
    int row_end = slot >= 0 ? 0x7fffffff : (int)(__shfl_sync(0xffffffffu, rp_hi, 0) - e_begin);
    float4 q = cok ? ldg4(p.Q + r * p.ldq + ccol) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 q_next = (cok && r + 1 < r1) ? ldg4(p.Q + (r + 1) * p.ldq + ccol) : make_float4(0.f, 0.f, 0.f, 0.f);
    float mx = -FLT_MAX, den = 0.0f, a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.bias && cok) bias = ldg4(p.bias + ccol);

    auto finalize_row = [&]() {
        if (cok) {
            const float inv = 1.0f / (den + 1e-8f);
            float4 o;
            o.x = apply_act(a0 * inv + bias.x, p.act);
            o.y = apply_act(a1 * inv + bias.y, p.act);
            o.z = apply_act(a2 * inv + bias.z, p.act);
            o.w = apply_act(a3 * inv + bias.w, p.act);
            *reinterpret_cast<float4 *>(p.out + r * p.ldo + ccol) = o;
            if (p.stats != nullptr && (lane % lanes_per_head) == 0) {
                p.stats[r * 2 * p.H + lane / lanes_per_head] = mx;
                p.stats[r * 2 * p.H + p.H + lane / lanes_per_head] = den + 1e-8f;
            }
        }
        mx = -FLT_MAX; den = 0.0f; a0 = a1 = a2 = a3 = 0.0f;
        ++r;
        q = q_next;
        if (r < r1) {
            row_end = (int)(__shfl_sync(0xffffffffu, rp_hi, (int)(r - r0)) - e_begin);
            if (cok && r + 1 < r1) q_next = ldg4(p.Q + (r + 1) * p.ldq + ccol);
        }
    };
    auto load_chunk = [&](int c) {
        const int e = c * 32 + lane;
        return e < n_edges ? ld_stream_i32(p.col + e_begin + e) : 0;
    };
    auto issue = [&](int g, int ci) {
        if (g < n_rounds) {
            const int base = (g % RPC) * U;
            const int valid = min(U, n_edges - g * U);
            const int c0 = __shfl_sync(0xffffffffu, ci, base);
            int c1 = __shfl_sync(0xffffffffu, ci, base + 1), c2 = __shfl_sync(0xffffffffu, ci, base + 2);
            int c3 = __shfl_sync(0xffffffffu, ci, base + 3);
            if (valid < 2) c1 = c0;
            if (valid < 3) c2 = c0;
            if (valid < 4) c3 = c0;
            if (lane == 0) {
                const uint32_t bar = bar0 + 8 * (uint32_t)(g % S);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(tx_bytes) : "memory");
                asm volatile(
                    "cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
                    ::"r"(ring_addr + (uint32_t)(g % S) * stage_bytes), "l"(&tmap), "r"(0), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
                    : "memory");
            }
        }
    };

    int ca = load_chunk(0), cb = load_chunk(1);
#pragma unroll
    for (int g = 0; g < S - 1; ++g) issue(g, ca);

    for (int g = 0; g < n_rounds; ++g) {
        __syncwarp();                               // every lane has finished reading the stage that is re-armed now
        {
            const int gn = g + S - 1;
            issue(gn, ((gn / RPC) & 1) ? cb : ca);
        }
        gat_mbar_wait(bar0 + 8 * (uint32_t)(g % S), (uint32_t)(g / S) & 1u);
        const uint8_t *sbuf = my_ring + (size_t)(g % S) * stage_bytes;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = g * U + u;
            if (e < n_edges) {
                while (e == row_end) finalize_row();
                float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
                if (cok) {
                    kk = *reinterpret_cast<const float4 *>(sbuf + (size_t)u * edge_bytes + ccol * 4);
                    vv = *reinterpret_cast<const float4 *>(sbuf + (size_t)u * edge_bytes + row_bytes + ccol * 4);
                }
                float d = q.x * kk.x + q.y * kk.y + q.z * kk.z + q.w * kk.w;
                for (int off = 1; off < lanes_per_head; off <<= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
                const float s = __fdiv_rn(d, p.scale);
                const bool up = s > mx;
                const float t = expf(up ? mx - s : s - mx);
                const float corr = up ? t : 1.0f, pe = up ? 1.0f : t;
                mx = up ? s : mx;
                den = fmaf(den, corr, pe);
                a0 = fmaf(a0, corr, pe * vv.x);
                a1 = fmaf(a1, corr, pe * vv.y);
                a2 = fmaf(a2, corr, pe * vv.z);
                a3 = fmaf(a3, corr, pe * vv.w);
            }
        }
        if ((g + S) % RPC == 0) {
            const int dead = (g + S) / RPC - 1;
            if (dead & 1) cb = load_chunk(dead + 2); else ca = load_chunk(dead + 2);
        }
    }
    if (slot >= 0) {
        float *dst = p.scratch + (int64_t)slot * (A + 64);
        if (cok) *reinterpret_cast<float4 *>(dst + ccol) = make_float4(a0, a1, a2, a3);
        dst[A + lane] = mx;
        dst[A + 32 + lane] = den;
        return;
    }
    while (r < r1) finalize_row();
}

// merges the (sums, max, denominator) partials of every hub row with the log-sum-exp rule, in slice order
__global__ void __launch_bounds__(256) gat_hub_fixup_kernel(const GatParams p) {
    const int lane = threadIdx.x & 31;
    const int h = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (h >= p.n_hubs) return;
    const int64_t r = p.hub_row[h];
    const int s0 = p.hub_slot0[h], ns = p.hub_nslots[h];
    const int A = p.H * p.dqk;
    const int ccol = lane * 4;
    const bool cok = ccol < A;
    const int64_t stride = A + 64;
    float m = -FLT_MAX;
    for (int s = 0; s < ns; ++s) m = fmaxf(m, p.scratch[(int64_t)(s0 + s) * stride + A + lane]);
    float den = 0.0f, a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int s = 0; s < ns; ++s) {
        const float *src = p.scratch + (int64_t)(s0 + s) * stride;
        const float sc = expf(src[A + lane] - m);
        den = fmaf(src[A + 32 + lane], sc, den);
        if (cok) {
            const float4 v = *reinterpret_cast<const float4 *>(src + ccol);
            a0 = fmaf(v.x, sc, a0); a1 = fmaf(v.y, sc, a1); a2 = fmaf(v.z, sc, a2); a3 = fmaf(v.w, sc, a3);
        }
    }
    if (cok && p.stats != nullptr && (lane % (p.dqk >> 2)) == 0) {
        p.stats[r * 2 * p.H + lane / (p.dqk >> 2)] = m;
        p.stats[r * 2 * p.H + p.H + lane / (p.dqk >> 2)] = den + 1e-8f;
    }
    if (cok) {
        const float inv = 1.0f / (den + 1e-8f);
        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) b = ldg4(p.bias + ccol);
        float4 o;
        o.x = apply_act(a0 * inv + b.x, p.act);
        o.y = apply_act(a1 * inv + b.y, p.act);
        o.z = apply_act(a2 * inv + b.z, p.act);
        o.w = apply_act(a3 * inv + b.w, p.act);
        *reinterpret_cast<float4 *>(p.out + r * p.ldo + ccol) = o;
    }
}

template <int U, int S>
static int launch_gat_async(const GatParams &p, cudaStream_t st) {
    const size_t smem = (size_t)kGatAsyncWarps * S * 2 * U * (size_t)(p.H * p.dqk) * 4;
    TFGK_CUDA(ensure_dynamic_smem(gat_async_kernel<U, S>, smem));
    const int64_t n_tasks = p.task_row ? p.n_tasks : ceil_div64(p.N, kGatAsyncRows);
    const unsigned blocks = (unsigned)ceil_div64(n_tasks, kGatAsyncWarps);
    gat_async_kernel<U, S><<<blocks, kGatAsyncWarps * 32, smem, st>>>(p);
    TFGK_LAUNCH_CHECK();
    if (p.task_row && p.n_hubs > 0) {
        gat_hub_fixup_kernel<<<(unsigned)ceil_div64(p.n_hubs, 8), 256, 0, st>>>(p);
        TFGK_LAUNCH_CHECK();
    }
    return TFGK_OK;
}

template <int S>
static int launch_gat_gather4(const GatParams &p, cudaStream_t st) {
    const int A = p.H * p.dqk;
    if (p.V != p.K + A || p.ldk != p.ldv || 2 * A > 256 || (p.ldk % 4) != 0) return TFGK_ERR_UNSUPPORTED;
    TensorMap tmap;
    const int rc = make_row_tensor_map(&tmap, p.K, p.ldk, (int64_t)1 << 31, 2 * A);      // rows bounded by the int32 column ids
    if (rc != TFGK_OK) return rc;
    const size_t stage_pitch = ((size_t)4 * 2 * A * 4 + 127) & ~(size_t)127;
    const size_t smem = (size_t)kGatAsyncWarps * S * stage_pitch + (size_t)kGatAsyncWarps * S * 8;
    TFGK_CUDA(ensure_dynamic_smem(gat_gather4_kernel<S>, smem));
    const int64_t n_tasks = p.task_row ? p.n_tasks : ceil_div64(p.N, kGatAsyncRows);
    const unsigned blocks = (unsigned)ceil_div64(n_tasks, kGatAsyncWarps);
    gat_gather4_kernel<S><<<blocks, kGatAsyncWarps * 32, smem, st>>>(p, tmap);
    TFGK_LAUNCH_CHECK();
    if (p.task_row && p.n_hubs > 0) {
        gat_hub_fixup_kernel<<<(unsigned)ceil_div64(p.n_hubs, 8), 256, 0, st>>>(p);
        TFGK_LAUNCH_CHECK();
    }
    return TFGK_OK;
}

static int dispatch_gat_async(const GatParams &p, cudaStream_t st) {
    // TMA tile::gather4 ring with two stages whenever K and V sit side by side in one buffer (the layers project them that
    // way): 18.74 ms against 19.97 ms for the cp.async ring at the products shape on a B200, three / four stages lose resident
    // warps (22.1 / 26.3 ms; profiles/r2_kernel_variants_final.json).  Separate K and V buffers, or a tensor map the driver
    // cannot encode, take the cp.async ring.
    const int rc = launch_gat_gather4<2>(p, st);
    if (rc != TFGK_ERR_UNSUPPORTED) return rc;
    return launch_gat_async<2, 3>(p, st);
}

// ---- generic path: any H / dqk / dv, split or averaged heads (correctness first) --------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}

__global__ void __launch_bounds__(kGatThreads) gat_generic_kernel(const GatParams p) {
    extern __shared__ float smem[];   // [warps][2][H]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r = (int64_t)blockIdx.x * kGatWarps + warp;
    if (r >= p.N) return;
    const int H = p.H;
    float *s_max = smem + (size_t)warp * 2 * H;
    float *s_den = s_max + H;
    const int64_t start = p.rowptr[r];
    const int deg = (int)(p.rowptr[r + 1] - start);
    float *att = p.att + start * H;
    const int32_t *col = p.col + start;

    for (int h = lane; h < H; h += 32) s_max[h] = -FLT_MAX;
    __syncwarp();
    for (int e = 0; e < deg; ++e) {
        const float *krow = p.K + (int64_t)col[e] * p.ldk;
        const float *qrow = p.Q + r * p.ldq;
        for (int h = 0; h < H; ++h) {
            float d = 0.0f;
            for (int j = lane; j < p.dqk; j += 32) d += qrow[h * p.dqk + j] * krow[h * p.dqk + j];
            d = warp_sum(d);
            if (lane == 0) {
                const float s = __fdiv_rn(d, p.scale);
                att[(int64_t)e * H + h] = s;
                s_max[h] = fmaxf(s_max[h], s);
            }
        }
    }
    __syncwarp();
    for (int h = 0; h < H; ++h) {
        const float m = s_max[h];
        float part = 0.0f;
        for (int e = lane; e < deg; e += 32) {
            const float pexp = expf(att[(int64_t)e * H + h] - m);
            att[(int64_t)e * H + h] = pexp;
            part += pexp;
        }
        part = warp_sum(part);
        if (lane == 0) s_den[h] = part + 1e-8f;
    }
    __syncwarp();
    if (p.split) {
        for (int c = lane; c < H * p.dv; c += 32) {
            const int hv = c / p.dv;
            const float dn = s_den[hv];
            float acc = 0.0f;
            for (int e = 0; e < deg; ++e) {
                const float a = __fdiv_rn(att[(int64_t)e * H + hv], dn);
                acc = __fadd_rn(acc, __fmul_rn(p.V[(int64_t)col[e] * p.ldv + c], a));
            }
            if (p.bias) acc += p.bias[c];
            p.out[r * p.ldo + c] = apply_act(acc, p.act);
        }
    } else {
        for (int u = lane; u < p.dv; u += 32) {
            float tot = 0.0f;
            for (int h = 0; h < H; ++h) {
                const float dn = s_den[h];
                float acc = 0.0f;
                for (int e = 0; e < deg; ++e) {
                    const float a = __fdiv_rn(att[(int64_t)e * H + h], dn);
                    acc = __fadd_rn(acc, __fmul_rn(p.V[(int64_t)col[e] * p.ldv + h * p.dv + u], a));
                }
                tot = h == 0 ? acc : __fadd_rn(tot, acc);     // tf.add_n over heads
            }
            tot = __fdiv_rn(tot, (float)H);
            if (p.bias) tot += p.bias[u];
            p.out[r * p.ldo + u] = apply_act(tot, p.act);
        }
    }
    if (p.write_att) {
        __syncwarp();
        for (int idx = lane; idx < deg * H; idx += 32) att[idx] = __fdiv_rn(att[idx], s_den[idx % H]);
    }
}

// ---- stand-alone segment softmax over CSR segments ------------------------------------------------------------
__global__ void __launch_bounds__(kGatThreads) segment_softmax_kernel(const int64_t *__restrict__ rowptr,
                                                                      const float *__restrict__ score, int32_t n_seg,
                                                                      int32_t H, float *__restrict__ out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r = (int64_t)blockIdx.x * kGatWarps + warp;
    if (r >= n_seg) return;
    const int64_t start = rowptr[r];
    const int deg = (int)(rowptr[r + 1] - start);
    const float *s = score + start * H;
    float *o = out + start * H;
    for (int h = 0; h < H; ++h) {
        float m = -FLT_MAX;
        for (int e = lane; e < deg; e += 32) m = fmaxf(m, s[(int64_t)e * H + h]);
        m = warp_max(m);
        float part = 0.0f;
        for (int e = lane; e < deg; e += 32) {
            const float pexp = expf(s[(int64_t)e * H + h] - m);
            o[(int64_t)e * H + h] = pexp;
            part += pexp;
        }
        const float den = warp_sum(part) + 1e-8f;
        for (int e = lane; e < deg; e += 32) o[(int64_t)e * H + h] = __fdiv_rn(o[(int64_t)e * H + h], den);
    }
}

static inline bool is_pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }

template <int NC>
static int launch_gat_online(const GatParams &p, cudaStream_t st) {
    constexpr int U = NC == 1 ? 4 : 2;
    const unsigned blocks = (unsigned)ceil_div64(p.N, kGatWarps);
    gat_online_kernel<NC, U><<<blocks, kGatThreads, 0, st>>>(p);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

template <int NCK, int NCV>
static int launch_gat_fast(const GatParams &p, cudaStream_t st) {
    constexpr int U = (NCK + NCV <= 2) ? 4 : 2;
    const unsigned blocks = (unsigned)ceil_div64(p.N, kGatWarps);
    gat_fast_kernel<NCK, NCV, U><<<blocks, kGatThreads, 0, st>>>(p);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

template <int NCK>
static int dispatch_gat_v(const GatParams &p, int ncv, cudaStream_t st) {
    switch (ncv) {
        case 1: return launch_gat_fast<NCK, 1>(p, st);
        case 2: return launch_gat_fast<NCK, 2>(p, st);
        case 3: return launch_gat_fast<NCK, 3>(p, st);
        default: return launch_gat_fast<NCK, 4>(p, st);
    }
}

}  // namespace tfgk

using namespace tfgk;

extern "C" int tfgk_segment_softmax_f32(const int64_t *rowptr, const float *score, int32_t n_seg, int32_t H,
                                        float *out, void *stream) {
    TFGK_CHECK_ARG(n_seg >= 0 && H >= 1, "segment_softmax: bad size (n_seg=%d, H=%d)", n_seg, H);
    if (n_seg == 0) return TFGK_OK;
    TFGK_CHECK_ARG(rowptr && out, "segment_softmax: null pointer");
    segment_softmax_kernel<<<(unsigned)ceil_div64(n_seg, kGatWarps), kGatThreads, 0, as_stream(stream)>>>(
        rowptr, score, n_seg, H, out);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

static int gat_fused_impl(const int64_t *rowptr, const int32_t *col,
                          const float *Q, int64_t ldq, const float *K, int64_t ldk, const float *V, int64_t ldv,
                          int32_t N, int32_t H, int32_t dqk, int32_t dv, float scale, int split_value_heads,
                          const float *bias, int act, float *att, int write_att, float *out, int64_t ldo,
                          const tfgk_plan *plan, float *stats, void *stream) {
    TFGK_CHECK_ARG(N >= 0 && H >= 1 && dqk >= 1 && dv >= 1, "gat: bad size (N=%d H=%d dqk=%d dv=%d)", N, H, dqk, dv);
    TFGK_CHECK_ARG(act == TFGK_ACT_NONE || act == TFGK_ACT_RELU, "gat: unknown activation %d", act);
    TFGK_CHECK_ARG(scale > 0.0f, "gat: scale must be positive");
    if (N == 0) return TFGK_OK;
    TFGK_CHECK_ARG(rowptr && col && Q && K && V && out, "gat: null pointer");
    TFGK_CHECK_ARG(att != nullptr || (!write_att), "gat: write_att needs an attention buffer");
    const int A = H * dqk, VW = H * dv;
    const int out_w = split_value_heads ? VW : dv;
    TFGK_CHECK_ARG(ldq >= A && ldk >= A && ldv >= VW && ldo >= out_w, "gat: leading dimension too small");

    GatParams p;
    p.rowptr = rowptr; p.col = col;
    p.Q = Q; p.ldq = ldq; p.K = K; p.ldk = ldk; p.V = V; p.ldv = ldv;
    p.N = N; p.H = H; p.dqk = dqk; p.dv = dv; p.scale = scale; p.split = split_value_heads;
    p.bias = bias; p.act = act; p.att = att; p.write_att = write_att; p.out = out; p.ldo = ldo;
    p.n_tasks = 0; p.task_row = nullptr; p.task_nrows = nullptr; p.task_e0 = nullptr; p.task_e1 = nullptr;
    p.task_slot = nullptr; p.n_hubs = 0; p.hub_row = nullptr; p.hub_slot0 = nullptr; p.hub_nslots = nullptr; p.scratch = nullptr;
    p.stats = stats;
    if (plan != nullptr && plan->n_tasks > 0) {
        if (plan->n_hubs > 0)
            TFGK_CHECK_ARG(plan->scratch != nullptr && plan->scratch_bytes >= (size_t)plan->n_slots * (H * dv + 64) * sizeof(float),
                           "gat: plan scratch too small (need %zu bytes)", (size_t)plan->n_slots * (H * dv + 64) * sizeof(float));
        p.n_tasks = plan->n_tasks; p.task_row = plan->task_row; p.task_nrows = plan->task_nrows;
        p.task_e0 = plan->task_e0; p.task_e1 = plan->task_e1; p.task_slot = plan->task_slot;
        p.n_hubs = plan->n_hubs; p.hub_row = plan->hub_row; p.hub_slot0 = plan->hub_slot0;
        p.hub_nslots = plan->hub_nslots; p.scratch = plan->scratch;
    }
    cudaStream_t st = as_stream(stream);

    const bool fast = split_value_heads && is_pow2(H) && H <= kMaxHeadsFast && dqk % 4 == 0 && is_pow2(dqk / 4) &&
                      dqk <= 128 && dv % 4 == 0 && A <= 512 && VW <= 512 && ldq % 4 == 0 && ldk % 4 == 0 &&
                      ldv % 4 == 0 && ldo % 4 == 0 && aligned16(Q) && aligned16(K) && aligned16(V) && aligned16(out) &&
                      (!bias || aligned16(bias));
    if (fast && dqk == dv && A <= 128 && !write_att) return dispatch_gat_async(p, st);
    if (stats != nullptr) return TFGK_ERR_UNSUPPORTED;      // only the streaming kernel keeps (max, denominator)
    if (fast && dqk == dv) {
        switch ((A + 127) / 128) {
            case 1: return launch_gat_online<1>(p, st);
            case 2: return launch_gat_online<2>(p, st);
            case 3: return launch_gat_online<3>(p, st);
            default: return launch_gat_online<4>(p, st);
        }
    }
    if (att == nullptr) return set_error(TFGK_ERR_WORKSPACE, "gat: this shape needs the [E,H] attention scratch buffer");
    if (fast) {
        const int nck = (A + 127) / 128, ncv = (VW + 127) / 128;
        switch (nck) {
            case 1: return dispatch_gat_v<1>(p, ncv, st);
            case 2: return dispatch_gat_v<2>(p, ncv, st);
            case 3: return dispatch_gat_v<3>(p, ncv, st);
            default: return dispatch_gat_v<4>(p, ncv, st);
        }
    }
    const size_t smem = (size_t)kGatWarps * 2 * H * sizeof(float);
    TFGK_CHECK_ARG(smem <= 48 * 1024, "gat: too many heads for the generic path (H=%d)", H);
    gat_generic_kernel<<<(unsigned)ceil_div64(N, kGatWarps), kGatThreads, smem, st>>>(p);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

extern "C" int tfgk_gat_fused_f32(const int64_t *rowptr, const int32_t *col,
                                  const float *Q, int64_t ldq, const float *K, int64_t ldk, const float *V, int64_t ldv,
                                  int32_t N, int32_t H, int32_t dqk, int32_t dv, float scale, int split_value_heads,
                                  const float *bias, int act, float *att, int write_att, float *out, int64_t ldo,
                                  const tfgk_plan *plan, void *stream) {
    return gat_fused_impl(rowptr, col, Q, ldq, K, ldk, V, ldv, N, H, dqk, dv, scale, split_value_heads, bias, act, att, write_att,
                          out, ldo, plan, nullptr, stream);
}

extern "C" int tfgk_gat_fused_stats_f32(const int64_t *rowptr, const int32_t *col,
                                        const float *Q, int64_t ldq, const float *K, int64_t ldk, const float *V, int64_t ldv,
                                        int32_t N, int32_t H, int32_t dqk, int32_t dv, float scale,
                                        const float *bias, int act, float *out, int64_t ldo, float *stats,
                                        const tfgk_plan *plan, void *stream) {
    TFGK_CHECK_ARG(stats != nullptr, "gat_fused_stats: stats buffer is required");
    return gat_fused_impl(rowptr, col, Q, ldq, K, ldk, V, ldv, N, H, dqk, dv, scale, 1, bias, act, nullptr, 0, out, ldo, plan,
                          stats, stream);
}
