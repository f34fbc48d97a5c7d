// K1: gather - edge-apply - segment-reduce over a destination-sorted CSR  (tfgk_spmm_f32).
//
//   out[r,:] = epilogue( REDUCE_{e in [rowptr[r], rowptr[r+1])} w[e] * h[col[e], :] )
//
// HBM-bound (0.25-0.5 flop/byte): no tensor cores.  Mapping: a group of G lanes owns one destination row and
// each lane owns NC vectors of VEC consecutive feature columns, so one gathered source row is one coalesced
// G*VEC*4-byte request (512 B for D=128).  Edge ids/weights are read once, coalesced, G at a time and broadcast
// with shuffles; U gathered rows are kept in flight per group before any of them is consumed.  Accumulation is
// fp32, strictly in CSR (= input) order with separate multiply and add roundings, which makes SUM/MEAN
// bit-identical to tf.math.unsorted_segment_sum's sequential CPU loop (no atomics anywhere => deterministic).
//
// Algorithmic bytes per launch (DESIGN.md): E*(4*D + 4 [+4 weighted]) + N*(4*D + 8).
#include "common.cuh"

namespace tfgk {

template <int VEC> struct Vec;
template <> struct Vec<4> { using T = float4; };
template <> struct Vec<1> { using T = float; };

template <int VEC>
__device__ __forceinline__ void load_vec(const float *p, float (&v)[VEC]) {
    if constexpr (VEC == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4 *>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
        v[0] = __ldg(p);
    }
}

template <int VEC>
__device__ __forceinline__ void store_vec(float *p, const float (&v)[VEC]) {
    if constexpr (VEC == 4) {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
        p[0] = v[0];
    }
}

struct SpmmParams {
    const int64_t *rowptr;
    const int32_t *col;
    const float *w;
    const float *h;
    int64_t ldh;
    int32_t n_dst;
    int32_t D;
    int reduce;
    float alpha;
    const float *addend;
    int64_t ld_addend;
    float beta;
    const float *bias;
    int act;
    float *out;
    int64_t ldo;
    // optional work plan (tfgk_plan): tasks + hub slices; task_row == nullptr -> implicit blocks of consecutive rows
    int32_t n_tasks;
    const int32_t *task_row, *task_nrows;
    const int64_t *task_e0, *task_e1;
    const int32_t *task_slot;
    int32_t n_hubs;
    const int32_t *hub_row, *hub_slot0, *hub_nslots;
    float *scratch;
};

constexpr int kSpmmThreads = 256;

// G: lanes per row (power of two), NC: vectors per lane, IS_MAX: max-reduce instead of sum/mean, U: rows in flight
template <int VEC, int G, int NC, bool IS_MAX, int U>
__global__ void __launch_bounds__(kSpmmThreads) spmm_kernel(const SpmmParams p) {
    constexpr int RPW = 32 / G;   // rows per warp
    const int lane = threadIdx.x & 31;
    const int gl = lane & (G - 1);
    const int grp = lane / G;
    const int64_t warp_global = (int64_t)blockIdx.x * (kSpmmThreads / 32) + (threadIdx.x >> 5);
    const int64_t r = warp_global * RPW + grp;
    const bool row_ok = r < p.n_dst;

    int64_t start = 0;
    int deg = 0;
    if (row_ok) {
        start = p.rowptr[r];
        deg = (int)(p.rowptr[r + 1] - start);
    }
    int deg_max = deg;
    if constexpr (RPW > 1) {
#pragma unroll
        for (int off = 16; off >= G; off >>= 1) deg_max = max(deg_max, __shfl_xor_sync(0xffffffffu, deg_max, off));
    }

    int coff[NC];
    bool cok[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        coff[k] = (gl + k * G) * VEC;
        cok[k] = coff[k] < p.D;
    }

    float acc[NC][VEC];
#pragma unroll
    for (int k = 0; k < NC; ++k)
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[k][v] = IS_MAX ? -FLT_MAX : 0.0f;

    const bool weighted = p.w != nullptr;
    const float *__restrict__ h = p.h;

    for (int t = 0; t < deg_max; t += G) {
        // coalesced read of up to G (col, w) pairs of this row
        const int e = t + gl;
        int my_c = 0;
        float my_w = 1.0f;
        if (e < deg) {
            my_c = ld_stream_i32(p.col + start + e);
            if (weighted) my_w = ld_stream_f32(p.w + start + e);
        }
        const int nb = min(G, deg - t);           // edges of this row in the batch (may be <= 0)
        const int nb_max = min(G, deg_max - t);   // warp-uniform trip count
        for (int j = 0; j < nb_max; j += U) {
            float v[U][NC][VEC];
            float ww[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int src = j + u;
                const int c = __shfl_sync(0xffffffffu, my_c, src, G);
                ww[u] = __shfl_sync(0xffffffffu, my_w, src, G);
                const bool ok = src < nb;
                const float *rowp = h + (int64_t)c * p.ldh;
#pragma unroll
                for (int k = 0; k < NC; ++k) {
                    if (ok && cok[k]) load_vec<VEC>(rowp + coff[k], v[u][k]);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (j + u < nb) {
#pragma unroll
                    for (int k = 0; k < NC; ++k) {
                        if (cok[k]) {
#pragma unroll
                            for (int x = 0; x < VEC; ++x) {
                                const float m = __fmul_rn(v[u][k][x], ww[u]);   // gcn_mapper rounding
                                acc[k][x] = IS_MAX ? fmaxf(acc[k][x], m) : __fadd_rn(acc[k][x], m);
                            }
                        }
                    }
                }
            }
        }
    }

    if (!row_ok) return;
    const bool is_mean = p.reduce == TFGK_REDUCE_MEAN;
    const float cnt = (float)max(deg, 1);
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        if (!cok[k]) continue;
        float o[VEC];
        float ad[VEC];
        float bs[VEC];
        if (p.addend) load_vec<VEC>(p.addend + r * p.ld_addend + coff[k], ad);
        if (p.bias) load_vec<VEC>(p.bias + coff[k], bs);
#pragma unroll
        for (int x = 0; x < VEC; ++x) {
            float a = acc[k][x];
            if (is_mean) a = __fdiv_rn(a, cnt);
            if (p.addend) a = __fadd_rn(__fmul_rn(a, p.alpha), __fmul_rn(ad[x], p.beta));
            else if (p.alpha != 1.0f) a = __fmul_rn(a, p.alpha);
            if (p.bias) a = __fadd_rn(a, bs[x]);
            o[x] = apply_act(a, p.act);
        }
        store_vec<VEC>(p.out + r * p.ldo + coff[k], o);
    }
}

// ------------------------------------------------------------------------------------------------------------
// cp.async ring.  Register double-buffering cannot overlap two gather rounds: a warp has six counting scoreboard
// slots, ptxas puts the loads of both rounds on the same slots, and the first use of round g then also waits for
// round g+1 (decoded from SASS, profiles/r1_notes.md).  LDGSTS copies are tracked by commit groups instead, so a
// per-warp shared-memory ring of S stages x U rows keeps (S-1)*U rows in flight per warp with no register cost.
// Each lane copies - and later reads back - only its own 16-byte slices: shared memory is used as an asynchronous
// extension of the register file, no cross-lane traffic, no barriers.  Edge streaming: a warp owns kAsyncRows consecutive
// rows = a contiguous CSR range, walked in rounds of U edges across row boundaries.  Same rounding and order => same bits.
// ------------------------------------------------------------------------------------------------------------
constexpr int kAsyncRows = 32;
constexpr int kAsyncWarps = 4;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int NC, bool IS_MAX, int U, int S>
__global__ void __launch_bounds__(kAsyncWarps * 32) spmm_async_kernel(const SpmmParams p, uint32_t row_bytes) {
    static_assert(32 % U == 0, "a round must not straddle an index chunk");
    constexpr int RPC = 32 / U;
    extern __shared__ __align__(16) uint8_t ring_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t task = (int64_t)blockIdx.x * kAsyncWarps + warp;
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
        r0 = task * kAsyncRows;
        if (r0 >= p.n_dst) return;
        r1 = min((int64_t)p.n_dst, r0 + kAsyncRows);
        e_begin = p.rowptr[r0];
        e_stop = p.rowptr[r1];
    }
    const int64_t rp_lo = p.rowptr[min(r0 + lane, r1)];
    const int64_t rp_hi = p.rowptr[min(r0 + lane + 1, r1)];
    const int n_edges = (int)(e_stop - e_begin);
    const int n_rounds = (n_edges + U - 1) / U;
    const bool weighted = p.w != nullptr;
    const uint32_t stage_bytes = U * row_bytes;
    uint8_t *my_ring = ring_raw + (size_t)warp * S * stage_bytes;
    const uint32_t ring_addr = (uint32_t)__cvta_generic_to_shared(my_ring);

    int coff[NC];
    bool cok[NC];
    float acc[NC][4];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        coff[k] = (lane + 32 * k) * 4;
        cok[k] = coff[k] < p.D;
#pragma unroll
        for (int x = 0; x < 4; ++x) acc[k][x] = IS_MAX ? -FLT_MAX : 0.0f;
    }
    int64_t r = r0;
    // a hub slice (slot >= 0) never closes its row: the partial sum goes to the scratch slot instead
    int row_end = slot >= 0 ? 0x7fffffff : (int)(__shfl_sync(0xffffffffu, rp_hi, 0) - e_begin);
    const bool is_mean = p.reduce == TFGK_REDUCE_MEAN;

    auto finalize_row = [&]() {
        const int64_t row_start = __shfl_sync(0xffffffffu, rp_lo, (int)(r - r0));
        const int deg = (int)(row_end + e_begin - row_start);
        const float cnt = (float)max(deg, 1);
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            if (cok[k]) {
                float ad[4], bs[4], o[4];
                if (p.addend) load_vec<4>(p.addend + r * p.ld_addend + coff[k], ad);
                if (p.bias) load_vec<4>(p.bias + coff[k], bs);
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    float a = acc[k][x];
                    if (is_mean) a = __fdiv_rn(a, cnt);
                    if (p.addend) a = __fadd_rn(__fmul_rn(a, p.alpha), __fmul_rn(ad[x], p.beta));
                    else if (p.alpha != 1.0f) a = __fmul_rn(a, p.alpha);
                    if (p.bias) a = __fadd_rn(a, bs[x]);
                    o[x] = apply_act(a, p.act);
                    acc[k][x] = IS_MAX ? -FLT_MAX : 0.0f;
                }
                store_vec<4>(p.out + r * p.ldo + coff[k], o);
            }
        }
        ++r;
        if (r < r1) row_end = (int)(__shfl_sync(0xffffffffu, rp_hi, (int)(r - r0)) - e_begin);
    };
    auto load_chunk = [&](int c, int &ci, float &wi) {
        const int e = c * 32 + lane;
        ci = 0;
        wi = 1.0f;
        if (e < n_edges) {
            ci = ld_stream_i32(p.col + e_begin + e);
            if (weighted) wi = ld_stream_f32(p.w + e_begin + e);
        }
    };
    // copy round g (edges [g*U, g*U+U)) into ring stage g % S; always commits one group (possibly empty)
    auto issue = [&](int g, int ci) {
        if (g < n_rounds) {
            const int base = (g % RPC) * U;
            const uint32_t dst0 = ring_addr + (uint32_t)(g % S) * stage_bytes;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int c = __shfl_sync(0xffffffffu, ci, base + u);
                if (g * U + u < n_edges) {
                    const float *rowp = p.h + (int64_t)c * p.ldh;
#pragma unroll
                    for (int k = 0; k < NC; ++k)
                        if (cok[k]) cp_async16(dst0 + u * row_bytes + coff[k] * 4, rowp + coff[k]);
                }
            }
        }
        cp_async_commit();
    };

    // Index registers (ca: even chunks, cb: odd chunks) are dead once the chunk's last round has been ISSUED; its
    // weights are needed until that round is CONSUMED, S-1 iterations later: wa/wb serve the consumer, wna/wnb hold the
    // weights fetched ahead together with the indices (requires S <= 2*RPC, asserted below).
    static_assert(S <= 2 * RPC, "weight look-ahead registers would be overwritten before they are consumed");
    int ca, cb;
    float wa, wb, wna = 1.0f, wnb = 1.0f;
    load_chunk(0, ca, wa);
    load_chunk(1, cb, wb);
    // prologue: S-1 rounds in flight (they all live in chunk 0 / 1 as long as (S-1)*U <= 64)
#pragma unroll
    for (int g = 0; g < S - 1; ++g) issue(g, ((g / RPC) & 1) ? cb : ca);
    if (S - 1 >= RPC) load_chunk(2, ca, wna);       // chunk 0 was issued completely by the prologue

    for (int g = 0; g < n_rounds; ++g) {
        // keep the pipe full: round g+S-1 goes into the stage consumed in the previous iteration
        {
            const int gn = g + S - 1;
            issue(gn, ((gn / RPC) & 1) ? cb : ca);
        }
        cp_async_wait<S - 1>();                     // round g has landed (groups retire in order)
        const int cc = g / RPC;
        const float wi = (cc & 1) ? wb : wa;
        const int base = (g % RPC) * U;
        const uint8_t *sbuf = my_ring + (size_t)(g % S) * stage_bytes;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = g * U + u;
            const float we = __shfl_sync(0xffffffffu, wi, base + u);
            if (e < n_edges) {
                while (e == row_end) finalize_row();
#pragma unroll
                for (int k = 0; k < NC; ++k) {
                    if (cok[k]) {
                        const float4 v = *reinterpret_cast<const float4 *>(sbuf + (size_t)u * row_bytes + coff[k] * 4);
                        const float m0 = __fmul_rn(v.x, we), m1 = __fmul_rn(v.y, we), m2 = __fmul_rn(v.z, we), m3 = __fmul_rn(v.w, we);
                        acc[k][0] = IS_MAX ? fmaxf(acc[k][0], m0) : __fadd_rn(acc[k][0], m0);
                        acc[k][1] = IS_MAX ? fmaxf(acc[k][1], m1) : __fadd_rn(acc[k][1], m1);
                        acc[k][2] = IS_MAX ? fmaxf(acc[k][2], m2) : __fadd_rn(acc[k][2], m2);
                        acc[k][3] = IS_MAX ? fmaxf(acc[k][3], m3) : __fadd_rn(acc[k][3], m3);
                    }
                }
            }
        }
        // the index chunk that the LAST issued round (g+S-1) no longer needs can be refilled: chunk j is dead once
        // round (j+1)*RPC - 1 has been issued, i.e. when g + S - 1 == (j+1)*RPC - 1
        if ((g + 1) % RPC == 0) {                   // chunk cc fully consumed: promote the look-ahead weights
            if (cc & 1) wb = wnb; else wa = wna;
        }
        if ((g + S) % RPC == 0) {
            const int dead = (g + S) / RPC - 1;
            if (dead & 1) load_chunk(dead + 2, cb, wnb); else load_chunk(dead + 2, ca, wna);
        }
    }
    if (slot >= 0) {                                  // hub slice: raw partial, merged by spmm_hub_fixup_kernel
#pragma unroll
        for (int k = 0; k < NC; ++k)
            if (cok[k]) store_vec<4>(p.scratch + (int64_t)slot * p.D + coff[k], acc[k]);
        return;
    }
    while (r < r1) finalize_row();
}

// ------------------------------------------------------------------------------------------------------------
// TMA tile::gather4 variant (north_star: "staged through TMA into shared memory").  Same edge streaming, ring and
// arithmetic as spmm_async_kernel, but a round of U = 4 edges is ONE instruction
//     cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4 [ring stage], [tensor map of h, {0, c0, c1, c2, c3}], [mbarrier]
// issued by one lane: the TMA unit fetches the four neighbour rows (box = D columns x 1 row each) and completes the
// stage's mbarrier with 4 * row_bytes transaction bytes.  That is a quarter of the TMA issues of a 1-D cp.async.bulk
// copy per row, and frees the 4 LDGSTS issue slots per lane and round of the cp.async ring.  Each warp owns S mbarriers;
// a stage is re-armed only after every lane has read it (__syncwarp before the elected lane issues).  Rows beyond the edge range repeat a valid row id (the bytes still count
// towards the stage's transaction total) and are ignored by the consumer.  Same rounding and order => same bits.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_wait_parity(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (spin > (1u << 28)) __trap();     // a lost transaction becomes a launch failure, never a hang
    }
}

__device__ __forceinline__ void tma_gather4(uint32_t dst, const TensorMap *map, int c0, int c1, int c2, int c3, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
        ::"r"(dst), "l"(map), "r"(0), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar) : "memory");
}

template <bool IS_MAX, int S>
__global__ void __launch_bounds__(kAsyncWarps * 32) spmm_gather4_kernel(const SpmmParams p, uint32_t row_bytes,
                                                                          const __grid_constant__ TensorMap tmap) {
    constexpr int U = 4, RPC = 32 / U;
    static_assert(S <= 2 * RPC, "weight look-ahead registers would be overwritten before they are consumed");
    extern __shared__ __align__(128) uint8_t g4_ring[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t tx_bytes = U * row_bytes;
    const uint32_t stage_bytes = (tx_bytes + 127u) & ~127u;      // TMA destinations are 128-byte aligned
    uint8_t *my_ring = g4_ring + (size_t)warp * S * stage_bytes;
    const uint32_t ring_addr = (uint32_t)__cvta_generic_to_shared(my_ring);
    uint64_t *bars = reinterpret_cast<uint64_t *>(g4_ring + (size_t)kAsyncWarps * S * stage_bytes) + warp * S;
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(bars);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < S; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8 * i));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const int64_t task = (int64_t)blockIdx.x * kAsyncWarps + warp;
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
        r0 = task * kAsyncRows;
        if (r0 >= p.n_dst) return;
        r1 = min((int64_t)p.n_dst, r0 + kAsyncRows);
        e_begin = p.rowptr[r0];
        e_stop = p.rowptr[r1];
    }
    const int64_t rp_lo = p.rowptr[min(r0 + lane, r1)];
    const int64_t rp_hi = p.rowptr[min(r0 + lane + 1, r1)];
    const int n_edges = (int)(e_stop - e_begin);
    const int n_rounds = (n_edges + U - 1) / U;
    const bool weighted = p.w != nullptr;
    constexpr int NCX = 2;                         // up to 256 columns: two float4 slices per lane
    int coff[NCX];
    bool cok[NCX];
    float acc[NCX][4];
#pragma unroll
    for (int k = 0; k < NCX; ++k) {
        coff[k] = (lane + 32 * k) * 4;
        cok[k] = coff[k] < p.D;
#pragma unroll
        for (int x = 0; x < 4; ++x) acc[k][x] = IS_MAX ? -FLT_MAX : 0.0f;
    }
    int64_t r = r0;
    int row_end = slot >= 0 ? 0x7fffffff : (int)(__shfl_sync(0xffffffffu, rp_hi, 0) - e_begin);
    const bool is_mean = p.reduce == TFGK_REDUCE_MEAN;

    auto finalize_row = [&]() {
        const int64_t row_start = __shfl_sync(0xffffffffu, rp_lo, (int)(r - r0));
        const int deg = (int)(row_end + e_begin - row_start);
        const float cnt = (float)max(deg, 1);
#pragma unroll
        for (int k = 0; k < NCX; ++k) {
            if (cok[k]) {
                float ad[4], bs[4], o[4];
                if (p.addend) load_vec<4>(p.addend + r * p.ld_addend + coff[k], ad);
                if (p.bias) load_vec<4>(p.bias + coff[k], bs);
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    float a = acc[k][x];
                    if (is_mean) a = __fdiv_rn(a, cnt);
                    if (p.addend) a = __fadd_rn(__fmul_rn(a, p.alpha), __fmul_rn(ad[x], p.beta));
                    else if (p.alpha != 1.0f) a = __fmul_rn(a, p.alpha);
                    if (p.bias) a = __fadd_rn(a, bs[x]);
                    o[x] = apply_act(a, p.act);
                    acc[k][x] = IS_MAX ? -FLT_MAX : 0.0f;
                }
                store_vec<4>(p.out + r * p.ldo + coff[k], o);
            }
        }
        ++r;
        if (r < r1) row_end = (int)(__shfl_sync(0xffffffffu, rp_hi, (int)(r - r0)) - e_begin);
    };
    auto load_chunk = [&](int c, int &ci, float &wi) {
        const int e = c * 32 + lane;
        ci = 0;
        wi = 1.0f;
        if (e < n_edges) {
            ci = ld_stream_i32(p.col + e_begin + e);
            if (weighted) wi = ld_stream_f32(p.w + e_begin + e);
        }
    };
    // round g (edges [4g, 4g+4)) -> ring stage g % S: one gather4, armed and issued by lane 0
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
                tma_gather4(ring_addr + (uint32_t)(g % S) * stage_bytes, &tmap, c0, c1, c2, c3, bar);
            }
        }
    };

    int ca, cb;
    float wa, wb, wna = 1.0f, wnb = 1.0f;
    load_chunk(0, ca, wa);
    load_chunk(1, cb, wb);
#pragma unroll
    for (int g = 0; g < S - 1; ++g) issue(g, ((g / RPC) & 1) ? cb : ca);
    if (S - 1 >= RPC) load_chunk(2, ca, wna);

    for (int g = 0; g < n_rounds; ++g) {
        __syncwarp();                               // every lane has finished reading stage (g-1) % S, which is re-armed now
        {
            const int gn = g + S - 1;
            issue(gn, ((gn / RPC) & 1) ? cb : ca);
        }
        mbar_wait_parity(bar0 + 8 * (uint32_t)(g % S), (uint32_t)(g / S) & 1u);
        const int cc = g / RPC;
        const float wi = (cc & 1) ? wb : wa;
        const int base = (g % RPC) * U;
        const uint8_t *sbuf = my_ring + (size_t)(g % S) * stage_bytes;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = g * U + u;
            const float we = __shfl_sync(0xffffffffu, wi, base + u);
            if (e < n_edges) {
                while (e == row_end) finalize_row();
#pragma unroll
                for (int k = 0; k < NCX; ++k) {
                    if (cok[k]) {
                        const float4 v = *reinterpret_cast<const float4 *>(sbuf + (size_t)u * row_bytes + coff[k] * 4);
                        const float m0 = __fmul_rn(v.x, we), m1 = __fmul_rn(v.y, we), m2 = __fmul_rn(v.z, we), m3 = __fmul_rn(v.w, we);
                        acc[k][0] = IS_MAX ? fmaxf(acc[k][0], m0) : __fadd_rn(acc[k][0], m0);
                        acc[k][1] = IS_MAX ? fmaxf(acc[k][1], m1) : __fadd_rn(acc[k][1], m1);
                        acc[k][2] = IS_MAX ? fmaxf(acc[k][2], m2) : __fadd_rn(acc[k][2], m2);
                        acc[k][3] = IS_MAX ? fmaxf(acc[k][3], m3) : __fadd_rn(acc[k][3], m3);
                    }
                }
            }
        }
        if ((g + 1) % RPC == 0) {
            if (cc & 1) wb = wnb; else wa = wna;
        }
        if ((g + S) % RPC == 0) {
            const int dead = (g + S) / RPC - 1;
            if (dead & 1) load_chunk(dead + 2, cb, wnb); else load_chunk(dead + 2, ca, wna);
        }
    }
    if (slot >= 0) {
#pragma unroll
        for (int k = 0; k < NCX; ++k)
            if (cok[k]) store_vec<4>(p.scratch + (int64_t)slot * p.D + coff[k], acc[k]);
        return;
    }
    while (r < r1) finalize_row();
}

// merges the slices of every hub row in slice order (deterministic) and applies the epilogue; one warp per hub row
template <bool IS_MAX>
__global__ void __launch_bounds__(256) spmm_hub_fixup_kernel(const SpmmParams p) {
    const int lane = threadIdx.x & 31;
    const int h = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (h >= p.n_hubs) return;
    const int64_t r = p.hub_row[h];
    const int s0 = p.hub_slot0[h], ns = p.hub_nslots[h];
    const float cnt = (float)max((int)(p.rowptr[r + 1] - p.rowptr[r]), 1);
    for (int c = lane * 4; c < p.D; c += 128) {
        float acc[4] = {IS_MAX ? -FLT_MAX : 0.f, IS_MAX ? -FLT_MAX : 0.f, IS_MAX ? -FLT_MAX : 0.f, IS_MAX ? -FLT_MAX : 0.f};
        for (int s = 0; s < ns; ++s) {
            float v[4];
            load_vec<4>(p.scratch + (int64_t)(s0 + s) * p.D + c, v);
#pragma unroll
            for (int x = 0; x < 4; ++x) acc[x] = IS_MAX ? fmaxf(acc[x], v[x]) : __fadd_rn(acc[x], v[x]);
        }
        float ad[4], bs[4], o[4];
        if (p.addend) load_vec<4>(p.addend + r * p.ld_addend + c, ad);
        if (p.bias) load_vec<4>(p.bias + c, bs);
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            float a = acc[x];
            if (p.reduce == TFGK_REDUCE_MEAN) a = __fdiv_rn(a, cnt);
            if (p.addend) a = __fadd_rn(__fmul_rn(a, p.alpha), __fmul_rn(ad[x], p.beta));
            else if (p.alpha != 1.0f) a = __fmul_rn(a, p.alpha);
            if (p.bias) a = __fadd_rn(a, bs[x]);
            o[x] = apply_act(a, p.act);
        }
        store_vec<4>(p.out + r * p.ldo + c, o);
    }
}

template <int NC, int U, int S>
static int launch_spmm_async(const SpmmParams &p, cudaStream_t st) {
    const uint32_t row_bytes = (uint32_t)p.D * 4u;
    const size_t smem = (size_t)kAsyncWarps * S * U * row_bytes;
    if (smem > 200 * 1024) return TFGK_ERR_UNSUPPORTED;
    const int64_t n_tasks = p.task_row ? p.n_tasks : ceil_div64(p.n_dst, kAsyncRows);
    const unsigned blocks = (unsigned)ceil_div64(n_tasks, kAsyncWarps);
    if (p.reduce == TFGK_REDUCE_MAX) {
        TFGK_CUDA(ensure_dynamic_smem(spmm_async_kernel<NC, true, U, S>, smem));
        spmm_async_kernel<NC, true, U, S><<<blocks, kAsyncWarps * 32, smem, st>>>(p, row_bytes);
    } else {
        TFGK_CUDA(ensure_dynamic_smem(spmm_async_kernel<NC, false, U, S>, smem));
        spmm_async_kernel<NC, false, U, S><<<blocks, kAsyncWarps * 32, smem, st>>>(p, row_bytes);
    }
    TFGK_LAUNCH_CHECK();
    if (p.task_row && p.n_hubs > 0) {
        const unsigned fb = (unsigned)ceil_div64(p.n_hubs, 8);
        if (p.reduce == TFGK_REDUCE_MAX) spmm_hub_fixup_kernel<true><<<fb, 256, 0, st>>>(p);
        else spmm_hub_fixup_kernel<false><<<fb, 256, 0, st>>>(p);
        TFGK_LAUNCH_CHECK();
    }
    return TFGK_OK;
}

template <int S>
static int launch_spmm_gather4(const SpmmParams &p, int64_t h_rows, cudaStream_t st) {
    if (p.D > 256 || p.D % 4 != 0 || p.ldh % 4 != 0) return TFGK_ERR_UNSUPPORTED;
    const uint32_t row_bytes = (uint32_t)p.D * 4u;
    const size_t stage_pitch = ((size_t)4 * row_bytes + 127) & ~(size_t)127;
    const size_t smem = (size_t)kAsyncWarps * S * stage_pitch + (size_t)kAsyncWarps * S * 8;
    if (smem > 200 * 1024) return TFGK_ERR_UNSUPPORTED;
    TensorMap tmap;
    const int rc = make_row_tensor_map(&tmap, p.h, p.ldh, h_rows, p.D);
    if (rc != TFGK_OK) return rc;
    const int64_t n_tasks = p.task_row ? p.n_tasks : ceil_div64(p.n_dst, kAsyncRows);
    const unsigned blocks = (unsigned)ceil_div64(n_tasks, kAsyncWarps);
    if (p.reduce == TFGK_REDUCE_MAX) {
        TFGK_CUDA(ensure_dynamic_smem(spmm_gather4_kernel<true, S>, smem));
        spmm_gather4_kernel<true, S><<<blocks, kAsyncWarps * 32, smem, st>>>(p, row_bytes, tmap);
    } else {
        TFGK_CUDA(ensure_dynamic_smem(spmm_gather4_kernel<false, S>, smem));
        spmm_gather4_kernel<false, S><<<blocks, kAsyncWarps * 32, smem, st>>>(p, row_bytes, tmap);
    }
    TFGK_LAUNCH_CHECK();
    if (p.task_row && p.n_hubs > 0) {
        const unsigned fb = (unsigned)ceil_div64(p.n_hubs, 8);
        if (p.reduce == TFGK_REDUCE_MAX) spmm_hub_fixup_kernel<true><<<fb, 256, 0, st>>>(p);
        else spmm_hub_fixup_kernel<false><<<fb, 256, 0, st>>>(p);
        TFGK_LAUNCH_CHECK();
    }
    return TFGK_OK;
}

// float4 rows of 257..512 columns (gather4 takes up to 256)
static int dispatch_spmm_async(const SpmmParams &p, cudaStream_t st) {
    const int lanes = (p.D + 3) / 4;
    if (lanes <= 96) return launch_spmm_async<3, 4, 3>(p, st);
    return launch_spmm_async<4, 2, 4>(p, st);
}

template <int VEC, int G, int NC, int U>
static int launch_spmm(const SpmmParams &p, cudaStream_t st) {
    constexpr int rows_per_block = (kSpmmThreads / 32) * (32 / G);
    const int64_t blocks = ceil_div64(p.n_dst, rows_per_block);
    if (p.reduce == TFGK_REDUCE_MAX)
        spmm_kernel<VEC, G, NC, true, U><<<(unsigned)blocks, kSpmmThreads, 0, st>>>(p);
    else
        spmm_kernel<VEC, G, NC, false, U><<<(unsigned)blocks, kSpmmThreads, 0, st>>>(p);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

template <int VEC>
static int dispatch_spmm(const SpmmParams &p, int lanes, cudaStream_t st) {
    // lanes = number of VEC-wide vectors in a row (<= 128)
    if (lanes <= 1) return launch_spmm<VEC, 1, 1, 8>(p, st);
    if (lanes <= 2) return launch_spmm<VEC, 2, 1, 8>(p, st);
    if (lanes <= 4) return launch_spmm<VEC, 4, 1, 8>(p, st);
    if (lanes <= 8) return launch_spmm<VEC, 8, 1, 8>(p, st);
    if (lanes <= 16) return launch_spmm<VEC, 16, 1, 8>(p, st);
    if (lanes <= 32) return launch_spmm<VEC, 32, 1, 8>(p, st);
    if (lanes <= 64) return launch_spmm<VEC, 32, 2, 4>(p, st);
    if (lanes <= 96) return launch_spmm<VEC, 32, 3, 2>(p, st);
    return launch_spmm<VEC, 32, 4, 2>(p, st);
}

}  // namespace tfgk

using namespace tfgk;

extern "C" int tfgk_spmm_f32(const int64_t *rowptr, const int32_t *col, const float *w,
                             const float *h, int64_t ldh, int32_t n_dst, int32_t D, int reduce,
                             float alpha, const float *addend, int64_t ld_addend, float beta,
                             const float *bias, int act,
                             float *out, int64_t ldo, const tfgk_plan *plan, void *stream) {
    TFGK_CHECK_ARG(n_dst >= 0 && D >= 0, "spmm: negative size (n_dst=%d, D=%d)", n_dst, D);
    if (plan != nullptr && plan->n_hubs > 0)
        TFGK_CHECK_ARG(plan->scratch != nullptr && plan->scratch_bytes >= (size_t)plan->n_slots * D * sizeof(float),
                       "spmm: plan scratch too small (need %zu bytes)", (size_t)plan->n_slots * D * sizeof(float));
    TFGK_CHECK_ARG(reduce >= TFGK_REDUCE_SUM && reduce <= TFGK_REDUCE_MAX, "spmm: unknown reduce %d", reduce);
    TFGK_CHECK_ARG(act == TFGK_ACT_NONE || act == TFGK_ACT_RELU, "spmm: unknown activation %d", act);
    if (n_dst == 0 || D == 0) return TFGK_OK;
    TFGK_CHECK_ARG(rowptr && out && h, "spmm: null pointer");
    TFGK_CHECK_ARG(ldh >= D && ldo >= D && (!addend || ld_addend >= D), "spmm: leading dimension < D");

    const bool vec4 = (D % 4 == 0) && (ldh % 4 == 0) && (ldo % 4 == 0) && aligned16(h) && aligned16(out) &&
                      (!addend || ((ld_addend % 4 == 0) && aligned16(addend))) && (!bias || aligned16(bias));
    const int vec = vec4 ? 4 : 1;
    const int cols_per_launch = 128 * vec;   // 32 lanes x NC<=4 vectors
    for (int c0 = 0; c0 < D; c0 += cols_per_launch) {
        SpmmParams p;
        p.rowptr = rowptr; p.col = col; p.w = w;
        p.h = h + c0; p.ldh = ldh; p.n_dst = n_dst;
        p.D = (D - c0 < cols_per_launch) ? D - c0 : cols_per_launch;
        p.reduce = reduce; p.alpha = alpha;
        p.addend = addend ? addend + c0 : nullptr; p.ld_addend = ld_addend; p.beta = beta;
        p.bias = bias ? bias + c0 : nullptr; p.act = act;
        p.out = out + c0; p.ldo = ldo;
        p.n_tasks = 0; p.task_row = nullptr; p.task_nrows = nullptr; p.task_e0 = nullptr; p.task_e1 = nullptr;
        p.task_slot = nullptr; p.n_hubs = 0; p.hub_row = nullptr; p.hub_slot0 = nullptr; p.hub_nslots = nullptr;
        p.scratch = nullptr;
        // the plan applies when the whole width runs in one launch of the streaming kernel (scratch rows are D wide)
        const bool use_plan = plan != nullptr && plan->n_tasks > 0 && vec4 && D >= 32 && D <= cols_per_launch;
        if (use_plan) {
            p.n_tasks = plan->n_tasks; p.task_row = plan->task_row; p.task_nrows = plan->task_nrows;
            p.task_e0 = plan->task_e0; p.task_e1 = plan->task_e1; p.task_slot = plan->task_slot;
            p.n_hubs = plan->n_hubs; p.hub_row = plan->hub_row; p.hub_slot0 = plan->hub_slot0;
            p.hub_nslots = plan->hub_nslots; p.scratch = plan->scratch;
        }
        const int lanes = (p.D + vec - 1) / vec;
        // Float4 rows of 32..256 columns: the TMA tile::gather4 ring with three stages (profiles/r2_kernel_variants_final.json,
        // B200: D = 128 9.55 ms against 9.87 ms for the cp.async ring, D = 100 9.51 against 10.24; three stages beat four, six
        // and eight, which cost resident warps).  Wider float4 rows: the cp.async ring.  Everything else, and any row when no
        // tensor map can be encoded: the per-row LDG kernel.
        if (vec4 && p.D >= 32 && p.D <= 256) {
            // the ABI does not carry the number of source rows: the tensor map is bounded by the index type instead
            // (column ids were validated against n_cols when the CSR was built)
            const int rcg = launch_spmm_gather4<3>(p, (int64_t)1 << 31, as_stream(stream));
            if (rcg != TFGK_ERR_UNSUPPORTED) { if (rcg != TFGK_OK) return rcg; continue; }
        } else if (vec4 && p.D > 256) {
            const int rca = dispatch_spmm_async(p, as_stream(stream));
            if (rca != TFGK_ERR_UNSUPPORTED) { if (rca != TFGK_OK) return rca; continue; }
        }
        const int rc = vec4 ? dispatch_spmm<4>(p, lanes, as_stream(stream)) : dispatch_spmm<1>(p, lanes, as_stream(stream));
        if (rc != TFGK_OK) return rc;
    }
    return TFGK_OK;
}
