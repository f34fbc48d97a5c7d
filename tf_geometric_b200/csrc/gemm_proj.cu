// K4 (round 2): the dense projections of the hot path as ONE launch over several column blocks, optionally with the A
// operand gathered tile by tile from other GPUs' memory (fused all-gather -> GEMM over NVLink peer mappings, K5).
//
//   C_b[M, n_b] = act_b(A[M, K] @ W_b[K, n_b] + bias_b)     for b in 0..nb-1  (n_b <= 128, nb <= 4)
//
// replaces x@W at nn/conv/gcn.py:272 and the three projections x@Wq, x@Wk, x@W of nn/conv/gat.py:52,61,70, which the
// round-1 path ran as three launches that each re-read x.  Differences from gemm_tc.cu (same 3xTF32 arithmetic, same bits):
//   * column blocks: CTA b handles block b % nb for the row tiles of its group b / nb; the nb CTAs of a group walk the
//     same tiles in the same order, so x is read from HBM once and from L2 nb-1 times (A traffic is 4(MK), not 4 nb MK);
//   * W_b (hi | lo) resident in shared memory for K rounded up to 8 (not 32), the MMA issuer skips the UMMA_K steps
//     beyond K and the producers skip the 16-byte chunks beyond it: K = 100 costs 13 k-steps instead of 16;
//   * epilogue through shared memory: tcgen05.ld 32 columns per round trip -> +bias -> act -> per-warp staging tile ->
//     full 128-byte row segments per store instruction (the round-1 epilogue wrote 16 bytes per row per instruction);
//   * A may be split into `n_parts` row blocks living at different base pointers (the other ranks' copies of x, mapped
//     through CUDA IPC): the producers' cp.async then read straight over NVLink, tile by tile, while the tensor core
//     works on the previous tiles - no halo buffer for x, no separate exchange step.  Tiles are walked starting at part
//     `first_part` so that every rank pulls from a different peer at any moment.
#include "common.cuh"
#include "tfgk_tc.cuh"

namespace tfgk {
namespace proj {

using namespace tc;

constexpr int kMaxBlocks = 4;
constexpr int kMaxParts = 8;
// warp roles: 0-3 converters (lo = a - trunc(a) on landed k-blocks), 4-11 epilogue (TMEM lane quarter = warp % 4, two
// warps per quarter split the columns), 12 MMA issuer, 13-14 loaders (cp.async into the ring as soon as a stage is free)
constexpr int kProducerWarps = 4, kEpilogueWarps = 8, kLoaderWarps = 2;
constexpr int kLoaderWarp0 = kProducerWarps + kEpilogueWarps + 1;
constexpr int kThreadsProj = (kProducerWarps + kEpilogueWarps + 1 + kLoaderWarps) * 32;      // 480
constexpr int kBarrierBytes = 192;
constexpr int kUN = 128;                 // accumulator columns per buffer
constexpr int kTmemColsProj = 256;       // 2 accumulator buffers
constexpr int kPassCols = 16;             // accumulator columns per TMEM round trip of an epilogue warp
constexpr int kStageRowBytes = 80;       // 16 floats + 16 B pad: conflict-free row-wise STS.128, segment-wise LDS.128
constexpr int kStageBytes = 32 * kStageRowBytes;

struct Params {
    const float *A[kMaxParts];
    int64_t lda, part_rows;
    int n_parts, first_tile, local_part;
    int M, K, nb, tiles_m, n_groups;
    const float *B[kMaxBlocks]; int64_t ldb[kMaxBlocks];
    const float *bias[kMaxBlocks]; int act[kMaxBlocks]; int ncols[kMaxBlocks]; int transb[kMaxBlocks];
    float *C[kMaxBlocks]; int64_t ldc[kMaxBlocks];
};

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// ---- epilogue: TMEM -> registers -> per-warp staging tile -> full row segments per store ------------------------------------
__device__ __forceinline__ int tile_index(const Params &p, int group, int it) {
    int tl = group + it * p.n_groups + p.first_tile;
    return tl >= p.tiles_m ? tl - p.tiles_m : tl;
}

__device__ __forceinline__ void epilogue_loop(const Params &p, int cb, int group, int un, int ncols, uint32_t tmem_base,
                                              uint8_t *stage_base, const float *s_bias, uint64_t *acc_full, uint64_t *acc_empty,
                                              int my_tiles, int warp, int lane) {
    auto tile_of = [&](int it) { return tile_index(p, group, it); };
        const int ew = warp - kProducerWarps;                 // 0..7
        const int q = warp & 3, half = ew >> 2;               // TMEM lane quarter (= warp % 4) and column half of this warp
        uint8_t *stg = stage_base + ew * kStageBytes;
        const uint32_t stg_addr = smem_u32(stg);
        float *__restrict__ Cb = p.C[cb];
        const int64_t ldc = p.ldc[cb];
        const int act = p.act[cb];
        const bool vec_ok = (ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(Cb) & 15) == 0);
        const int seg_row = lane >> 2, seg_chunk = lane & 3;  // store phase: 8 rows x 64 bytes per instruction
        const int n_pass = un / kPassCols;
        const int pass0 = half == 0 ? 0 : (n_pass + 1) / 2, pass1 = half == 0 ? (n_pass + 1) / 2 : n_pass;
        for (int it = 0; it < my_tiles; ++it) {
            const int buf = it & 1;
            const int tile = tile_of(it);
            mbar_wait(&acc_full[buf], (uint32_t)((it >> 1) & 1));
            tc_fence_after();
            const int64_t row0 = (int64_t)tile * BM + q * 32;
            if (pass0 >= pass1) {                             // nothing to read (a single pass belongs to the other half)
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[buf]);
            }
            for (int ps = pass0; ps < pass1; ++ps) {
                const int c0 = ps * kPassCols;
                uint32_t r[16];
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * kUN + c0);
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                    "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (ps + 1 == pass1) {                        // this warp's share is drained: one arrive per warp frees the buffer
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[buf]);
                }
#pragma unroll
                for (int j = 0; j < 16; j += 4) {
                    const float v0 = apply_act(__uint_as_float(r[j]) + s_bias[c0 + j], act);
                    const float v1 = apply_act(__uint_as_float(r[j + 1]) + s_bias[c0 + j + 1], act);
                    const float v2 = apply_act(__uint_as_float(r[j + 2]) + s_bias[c0 + j + 2], act);
                    const float v3 = apply_act(__uint_as_float(r[j + 3]) + s_bias[c0 + j + 3], act);
                    st_shared_v4(stg_addr + (uint32_t)lane * kStageRowBytes + (uint32_t)j * 4u, v0, v1, v2, v3);
                }
                __syncwarp();
                const int col = c0 + seg_chunk * 4;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int rl = j * 8 + seg_row;
                    const int64_t row = row0 + rl;
                    const float4 v = *reinterpret_cast<const float4 *>(stg + rl * kStageRowBytes + seg_chunk * 16);
                    if (row < p.M) {
                        float *dst = Cb + row * ldc + col;
                        if (vec_ok && col + 4 <= ncols) {
                            *reinterpret_cast<float4 *>(dst) = v;
                        } else {
                            if (col < ncols) dst[0] = v.x;
                            if (col + 1 < ncols) dst[1] = v.y;
                            if (col + 2 < ncols) dst[2] = v.z;
                            if (col + 3 < ncols) dst[3] = v.w;
                        }
                    }
                }
                __syncwarp();
            }
        }
}

// ---- the kernel: A operands in tensor memory ("TS" form of tcgen05.mma) ----------------------------------------------------
// Why tensor memory (profiles/r2_notes.md): with the split A operands in shared memory, a ring stage makes one trip
// free -> load -> convert -> MMA -> commit -> free in ~3000 cycles whatever its size, and next to the resident W the ring
// holds raw + lo tiles for only 96 K-columns - less than one 128 x 104 row tile - so a row tile costs about one full trip
// (4.3 us) where its 39 MMAs need 1.3 us.  Here the ring in shared memory holds RAW k-blocks only (16 KB per 32 columns,
// up to six stages) and the split operands live in TENSOR MEMORY: the converter warps read their own row of a landed
// k-block, compute hi = trunc_tf32(a) and lo = a - hi in registers and store both with tcgen05.st into a 4-slot ring
// (2 x 32 columns per slot) next to the two accumulators: 256 + 256 = all 512 TMEM columns.  The MMAs then take A from
// tensor memory and only W from shared memory, which also halves their shared-memory traffic.  Twice the K-columns in
// flight in shared memory plus four k-blocks in tensor memory cover the trip latency.
constexpr int kTsSlots = 4;
constexpr int kTsTmemCols = 512;
constexpr int kTsBarrierBytes = 256;
constexpr int kTsAcol0 = 2 * kUN;                 // first TMEM column of the A ring

struct PlanTS {
    uint32_t kpad8, b_bytes, raw_bytes, stages, total;
    __host__ __device__ explicit PlanTS(int K) {
        kpad8 = (uint32_t)((K + 7) / 8) * 8;
        b_bytes = (uint32_t)kUN * kpad8 * 4u;
        raw_bytes = BM * BK * 4u;
        const uint32_t fixed = 2u * b_bytes + kEpilogueWarps * kStageBytes + kTsBarrierBytes + kUN * 4u;
        const uint32_t budget = 227u * 1024u;
        stages = 0;
        for (uint32_t st = 6; st >= 2; --st)
            if (fixed + st * raw_bytes <= budget) { stages = st; break; }
        total = fixed + stages * raw_bytes;
    }
};

__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

#define TFGK_ST32(taddr, v)                                                                                                    \
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "                                                              \
                 "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"                                                   \
                 "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"                                          \
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),         \
                   "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),               \
                   "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),             \
                   "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31]) : "memory")

template <int STAGES>
__global__ void __launch_bounds__(kThreadsProj, 1) gemm_proj_ts_kernel(const Params p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const PlanTS L(p.K);
    uint8_t *b_hi_ptr = smem, *b_lo_ptr = smem + L.b_bytes;
    uint8_t *raw_ring = smem + 2 * L.b_bytes;
    uint8_t *stage_base = raw_ring + STAGES * L.raw_bytes;
    uint64_t *landed = reinterpret_cast<uint64_t *>(stage_base + kEpilogueWarps * kStageBytes);
    uint64_t *smem_free = landed + STAGES, *full_t = smem_free + STAGES, *tmem_free = full_t + kTsSlots;
    uint64_t *acc_full = tmem_free + kTsSlots, *acc_empty = acc_full + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_empty + 2);
    float *s_bias = reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(landed) + kTsBarrierBytes);
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int cb = (int)blockIdx.x % p.nb, group = (int)blockIdx.x / p.nb;
    const int ncols = p.ncols[cb];
    const int un = ((ncols + 15) / 16) * 16;
    const float *__restrict__ Bm = p.B[cb];
    const int64_t ldb = p.ldb[cb];
    const bool tb = p.transb[cb] != 0;

    for (int i = t; i < kUN; i += kThreadsProj) s_bias[i] = (p.bias[cb] != nullptr && i < ncols) ? __ldg(p.bias[cb] + i) : 0.0f;
    if (t == 0) {
        for (int i = 0; i < STAGES; ++i) { mbar_init(&landed[i], kLoaderWarps * 32); mbar_init(&smem_free[i], kProducerWarps); }
        for (int i = 0; i < kTsSlots; ++i) { mbar_init(&full_t[i], kProducerWarps); mbar_init(&tmem_free[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], kEpilogueWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTsTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    {   // W_b: transpose + RNA split into the K-major core-matrix layout, once per CTA
        const int kchunks = (int)L.kpad8 / 4;
        const int total = un * kchunks;
        const uint32_t bh = smem_u32(b_hi_ptr), bl = smem_u32(b_lo_ptr);
        for (int c = t; c < total; c += kThreadsProj) {
            const int n8 = c & 7, kc = (c >> 3) % kchunks, ng = (c >> 3) / kchunks;
            const int n = ng * 8 + n8, k = kc * 4;
            float w[4] = {0.f, 0.f, 0.f, 0.f}, h[4], l[4];
            if (n < ncols) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (k + i < p.K) w[i] = __ldg(tb ? Bm + (int64_t)n * ldb + (k + i) : Bm + (int64_t)(k + i) * ldb + n);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) split_tf32(w[i], h[i], l[i]);
            st_shared_v4(bh + c * 16, h[0], h[1], h[2], h[3]);
            st_shared_v4(bl + c * 16, l[0], l[1], l[2], l[3]);
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int nkb = (int)(L.kpad8 + BK - 1) / BK;
    const int last_steps = ((int)L.kpad8 - (nkb - 1) * BK) / UMMA_K;
    const int my_tiles = group < p.tiles_m ? (p.tiles_m - 1 - group) / p.n_groups + 1 : 0;
    const int total_kb = my_tiles * nkb;

    if (warp >= kLoaderWarp0) {
        // ===================== loaders: raw k-blocks, row-major with the 16-byte chunks XOR-swizzled by row =====================
        const int tl = t - kLoaderWarp0 * 32;                                // 0..63
        const uint32_t ring_addr = smem_u32(raw_ring);
        const int kc = tl & 7, rsub = tl >> 3;                               // a warp covers 4 rows x 128 contiguous bytes
        constexpr int kPrefetchTiles = 4;
        const bool can_prefetch = (cb == 0) && (tl == 0) && p.lda <= 2 * (int64_t)p.K;
        auto prefetch_tile = [&](int it) {
            if (!can_prefetch || it >= my_tiles) return;
            const int64_t m0 = (int64_t)tile_index(p, group, it) * BM;
            const int part = p.n_parts > 1 ? (int)(m0 / p.part_rows) : 0;
            if (p.n_parts > 1 && part != p.local_part) return;
            const int64_t rows = min((int64_t)BM, (int64_t)p.M - m0);
            const float *src = p.A[part] + (m0 - (int64_t)part * p.part_rows) * p.lda;
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"((uint32_t)(rows * p.lda * 4)) : "memory");
        };
        for (int i = 0; i < kPrefetchTiles; ++i) prefetch_tile(i);
        for (int G = 0; G < total_kb; ++G) {
            const int stage = G % STAGES;
            mbar_wait(&smem_free[stage], (uint32_t)(((G / STAGES) & 1) ^ 1));
            const int tile = tile_index(p, group, G / nkb), kb = G % nkb;
            if (kb == 0) prefetch_tile(G / nkb + kPrefetchTiles);
            const int k = kb * BK + kc * 4;
            if (k < (int)L.kpad8) {
                const int64_t m0 = (int64_t)tile * BM;
                const int part = p.n_parts > 1 ? (int)(m0 / p.part_rows) : 0;
                const float *base = p.A[part] + (m0 - (int64_t)part * p.part_rows) * p.lda + k;
                const uint32_t kbytes = k < p.K ? (uint32_t)min(4, p.K - k) * 4u : 0u;
                const uint32_t dst0 = ring_addr + stage * L.raw_bytes;
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int rl = i * 8 + rsub;
                    const bool ok = m0 + rl < p.M;
                    cp_async16_zfill(dst0 + (uint32_t)rl * 128u + (uint32_t)((kc ^ (rl & 7)) * 16),
                                     ok ? base + (int64_t)rl * p.lda : p.A[0], ok ? kbytes : 0u);
                }
            }
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&landed[stage])) : "memory");
        }
    } else if (warp < kProducerWarps) {
        // ===================== converters: own row of a landed k-block -> (hi, lo) -> tensor memory =====================
        const uint32_t lane_field = (uint32_t)(warp * 32) << 16;             // this warp's TMEM lane quarter
        // software pipelined: the tensor-memory stores of k-block G are issued, and only after the shared-memory reads and
        // the split of k-block G+1 does the warp wait for them and publish G (tcgen05.wait::st latency off the critical path)
        int prev_slot = -1, prev_stage = -1;
        auto publish_prev = [&]() {
            if (prev_slot < 0) return;
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            __syncwarp();
            if (lane == 0) { mbar_arrive(&full_t[prev_slot]); mbar_arrive(&smem_free[prev_stage]); }
        };
        for (int G = 0; G < total_kb; ++G) {
            const int stage = G % STAGES, slot = G % kTsSlots, kb = G % nkb;
            mbar_wait(&landed[stage], (uint32_t)((G / STAGES) & 1));
            uint32_t hi[32], lo[32];
            const uint8_t *row = raw_ring + stage * L.raw_bytes + t * 128;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (kb * BK + c * 4 < (int)L.kpad8) v = *reinterpret_cast<const float4 *>(row + ((c ^ (t & 7)) * 16));
                const float a[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const uint32_t h = __float_as_uint(a[e]) & 0xFFFFE000u;
                    hi[c * 4 + e] = h;
                    lo[c * 4 + e] = __float_as_uint(a[e] - __uint_as_float(h));
                }
            }
            publish_prev();
            mbar_wait(&tmem_free[slot], (uint32_t)(((G / kTsSlots) & 1) ^ 1));      // MMAs of k-block G - 4 retired
            tc_fence_after();
            const uint32_t taddr = tmem_base + lane_field + (uint32_t)(kTsAcol0 + slot * 64);
            TFGK_ST32(taddr, hi);
            TFGK_ST32(taddr + 32u, lo);
            prev_slot = slot; prev_stage = stage;
        }
        publish_prev();
    } else if (warp == kProducerWarps + kEpilogueWarps) {
        // ===================== MMA issuer: A from tensor memory, W from shared memory =====================
        // The whole warp walks the loop with warp-uniform values and one elected lane issues: written as `if (lane == 0)`
        // the compiler wrapped every tcgen05.mma in an ELECT / BRA.U.ANY sequence and rebuilt both descriptors with integer
        // divisions per k-block - ~130 issue cycles per MMA against the 64 cycles the tensor core needs for it, which made
        // this single thread the critical path of the kernel (profiles/r2_notes.md).  Counters are carried, the W descriptors
        // advance by constants (the address field counts 16-byte units).
        const uint32_t idesc = make_idesc(un);
        const uint32_t sbo_b = (L.kpad8 / 4) * 128u;
        const uint64_t dbh0 = make_desc_sbo(smem_u32(b_hi_ptr), sbo_b), dbl0 = make_desc_sbo(smem_u32(b_lo_ptr), sbo_b);
        const uint32_t a_ring0 = tmem_base + (uint32_t)kTsAcol0;
        int slot = 0, kb = 0, it = 0;
        uint32_t slot_phase = 0;
        for (int G = 0; G < total_kb; ++G) {
            const int buf = it & 1;
            if (kb == 0) mbar_wait(&acc_empty[buf], (uint32_t)(((it >> 1) & 1) ^ 1));
            mbar_wait(&full_t[slot], slot_phase);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kUN);
            const uint32_t a_hi = a_ring0 + (uint32_t)(slot * 64);
            const uint64_t dbh = dbh0 + (uint64_t)(kb * 64), dbl = dbl0 + (uint64_t)(kb * 64);      // + kb * 1024 bytes
            const int steps = kb == nkb - 1 ? last_steps : BK / UMMA_K;
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < BK / UMMA_K; ++j) {
                    if (j < steps) {
                        const uint64_t bh = dbh + (uint64_t)(j * 16), bl = dbl + (uint64_t)(j * 16);           // + j * 256 bytes
                        const uint32_t ah = a_hi + (uint32_t)(j * UMMA_K), al = ah + 32u;
                        umma_tf32_ts(d_tmem, al, bh, idesc, (kb | j) != 0);
                        umma_tf32_ts(d_tmem, ah, bl, idesc, 1u);
                        umma_tf32_ts(d_tmem, ah, bh, idesc, 1u);
                    }
                }
                umma_commit(&tmem_free[slot]);
                if (kb == nkb - 1) umma_commit(&acc_full[buf]);
            }
            __syncwarp();
            if (++slot == kTsSlots) { slot = 0; slot_phase ^= 1u; }
            if (++kb == nkb) { kb = 0; ++it; }
        }
    } else {
        epilogue_loop(p, cb, group, un, ncols, tmem_base, stage_base, s_bias, acc_full, acc_empty, my_tiles, warp, lane);
    }
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTsTmemCols) : "memory");
    }
}

template <int STAGES>
static int launch_ts(const Params &p, int grid, uint32_t smem_bytes, cudaStream_t st) {
    static int configured[16] = {0};
    int dev = 0;
    TFGK_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16 || configured[dev] < (int)smem_bytes) {
        TFGK_CUDA(cudaFuncSetAttribute(gemm_proj_ts_kernel<STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        if (dev >= 0 && dev < 16) configured[dev] = (int)smem_bytes;
    }
    gemm_proj_ts_kernel<STAGES><<<grid, kThreadsProj, smem_bytes, st>>>(p);
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}

}  // namespace proj
}  // namespace tfgk

using namespace tfgk;

extern "C" int tfgk_gemm_proj_f32(const float *const *A_parts, int32_t n_parts, int64_t part_rows, int64_t lda,
                                  int32_t M, int32_t K, const tfgk_proj_block *blocks, int32_t n_blocks,
                                  int32_t first_part, int32_t max_ctas, void *stream) {
    TFGK_CHECK_ARG(A_parts != nullptr && blocks != nullptr, "gemm_proj: null argument");
    TFGK_CHECK_ARG(n_parts >= 1 && n_parts <= proj::kMaxParts, "gemm_proj: n_parts=%d not in [1, %d]", n_parts, proj::kMaxParts);
    TFGK_CHECK_ARG(n_blocks >= 1 && n_blocks <= proj::kMaxBlocks, "gemm_proj: n_blocks=%d not in [1, %d]", n_blocks, proj::kMaxBlocks);
    TFGK_CHECK_ARG(M >= 0 && K >= 1, "gemm_proj: bad size (M=%d, K=%d)", M, K);
    TFGK_CHECK_ARG(first_part >= 0 && first_part < n_parts, "gemm_proj: first_part=%d out of range", first_part);
    if (M == 0) return TFGK_OK;
    if (n_parts > 1)
        TFGK_CHECK_ARG(part_rows > 0 && part_rows % tc::BM == 0 && (int64_t)n_parts * part_rows >= M,
                       "gemm_proj: part_rows=%lld must be a positive multiple of %d covering M=%d", (long long)part_rows, tc::BM, M);
    if (K > 512 || (lda % 4) != 0 || lda < K) return TFGK_ERR_UNSUPPORTED;        // same accuracy bound as gemm_tc.cu
    proj::Params p;
    for (int i = 0; i < proj::kMaxParts; ++i) {
        p.A[i] = A_parts[i < n_parts ? i : 0];
        if (!aligned16(p.A[i]) || p.A[i] == nullptr) return i < n_parts && A_parts[i] == nullptr
            ? set_error(TFGK_ERR_INVALID_ARGUMENT, "gemm_proj: A part %d is null", i) : TFGK_ERR_UNSUPPORTED;
    }
    p.lda = lda; p.part_rows = n_parts > 1 ? part_rows : (int64_t)1 << 40; p.n_parts = n_parts;
    p.M = M; p.K = K; p.nb = n_blocks;
    p.tiles_m = (int)ceil_div64(M, tc::BM);
    p.first_tile = n_parts > 1 ? (int)((int64_t)first_part * part_rows / tc::BM) : 0;
    p.local_part = n_parts > 1 ? (first_part + n_parts - 1) % n_parts : 0;      // the walk starts one past the caller's own part
    if (p.first_tile >= p.tiles_m) p.first_tile = 0;
    for (int b = 0; b < proj::kMaxBlocks; ++b) {
        const tfgk_proj_block &blk = blocks[b < n_blocks ? b : 0];
        if (b < n_blocks) {
            TFGK_CHECK_ARG(blk.B != nullptr && blk.C != nullptr, "gemm_proj: block %d has a null operand", b);
            TFGK_CHECK_ARG(blk.ncols >= 1 && blk.ldb >= (blk.transB ? K : blk.ncols) && blk.ldc >= blk.ncols,
                           "gemm_proj: block %d has bad sizes", b);
            TFGK_CHECK_ARG(blk.act == TFGK_ACT_NONE || blk.act == TFGK_ACT_RELU, "gemm_proj: unknown activation %d", blk.act);
            if (blk.ncols > proj::kUN) return TFGK_ERR_UNSUPPORTED;
        }
        p.B[b] = blk.B; p.ldb[b] = blk.ldb; p.bias[b] = blk.bias; p.act[b] = blk.act; p.ncols[b] = blk.ncols;
        p.transb[b] = blk.transB;
        p.C[b] = blk.C; p.ldc[b] = blk.ldc;
    }
    // K <= 136, i.e. at least four raw stages next to the resident W: the range this kernel is tested and measured on.
    // Wider K (up to 512) goes to gemm_tc.cu through tfgk_gemm_f32's fallback on TFGK_ERR_UNSUPPORTED.
    const proj::PlanTS L(K);
    if (L.stages < 4) return TFGK_ERR_UNSUPPORTED;
    int dev = 0, sms = 0;
    TFGK_CUDA(cudaGetDevice(&dev));
    TFGK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (max_ctas > 0 && max_ctas < sms) sms = max_ctas;
    int n_groups = sms / n_blocks;
    if (n_groups < 1) n_groups = 1;
    if (n_groups > p.tiles_m) n_groups = p.tiles_m;
    p.n_groups = n_groups;
    const int grid = n_groups * n_blocks;
    cudaStream_t st = as_stream(stream);
    switch (L.stages) {
        case 6: return proj::launch_ts<6>(p, grid, L.total, st);
        case 5: return proj::launch_ts<5>(p, grid, L.total, st);
        default: return proj::launch_ts<4>(p, grid, L.total, st);
    }
}
