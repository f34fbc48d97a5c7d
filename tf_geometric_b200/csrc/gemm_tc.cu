// K4 (tensor-core path for the projections gemm_proj.cu does not take): C[M,N] = act(A[M,K] @ B[K,N] + bias) with
// 136 < K <= 512 and N <= 256, e.g. a 512-wide input projected to 16 columns.  tfgk_gemm_f32 tries tfgk_gemm_proj_f32
// first and comes here when that returns TFGK_ERR_UNSUPPORTED (non-transposed B only); everything else is the SIMT kernel.
//
//   * tcgen05.mma.cta_group::1.kind::tf32, UMMA 128 x UN x 8, fp32 accumulators in TMEM (2 x UN columns, double buffered)
//   * fp32-accurate via the 3xTF32 split: a = hi + lo with hi = rna_tf32(a), lo = a - hi (exact);
//     D += Ahi*Bhi + Ahi*Blo + Alo*Bhi  (the dropped lo*lo term is ~2^-22 relative)  => ~1e-6 relative error, well
//     inside the 1e-4 parity gate that single-pass TF32 (~1e-3) would fail (SURVEY.md section 7 "hard parts")
//   * A streams through a cp.async ring straight into the canonical K-major, no-swizzle UMMA layout (8-row x 16 B core
//     matrices; LBO = 128 B along K, SBO = 1024 B along M); the raw fp32 tile IS the hi operand (hardware truncation) and
//     only lo = a - trunc(a) is computed by the CUDA cores.  W ([K,N] row-major) is transposed, split and kept resident
//   * one elected thread issues the MMAs; tcgen05.commit -> mbarrier releases the smem stage / publishes the accumulator
//   * persistent CTAs: the epilogue of tile i (tcgen05.ld -> +bias -> act -> global) overlaps the MMAs of tile i+1
// The kernel is memory bound (4(MK+MN) bytes for ~6MNK tf32 flops at K~100): the tensor pipe is lightly loaded by design.
#include "common.cuh"
#include "tfgk_tc.cuh"

namespace tfgk {
namespace tc {

// ---- shared memory plan ------------------------------------------------------------------------------------------------
//   W resident for the whole kernel, already split:  Bhi | Blo, each UN x Kpad fp32 in K-major core-matrix order
//        element (n, k) at  (n/8)*SBO_B + (k/4)*128 + (n%8)*16 + (k%4)*4 ,  SBO_B = (Kpad/4)*128
//   A ring of S stages, one 128 x 32 k-block per stage:  Araw | Alo (16 KB each), chunk c = rg*64 + kc*8 + r8 at 16*c
//        Araw is written by cp.async straight from global memory and used AS the hi operand (the tensor core ignores the
//        low 13 mantissa bits of a tf32 operand, i.e. hi = trunc(a)); Alo = a - trunc(a) is produced in place by the thread
//        that issued the copy, so no cross-thread hand-off precedes the conversion.
struct SmemPlan {
    uint32_t kpad, b_bytes, a_stage_bytes, stages, total;
    __host__ __device__ SmemPlan(int un, int K) {
        kpad = (uint32_t)((K + BK - 1) / BK) * BK;
        b_bytes = (uint32_t)un * kpad * 4u;
        a_stage_bytes = 2u * BM * BK * 4u;
        const uint32_t budget = 227u * 1024u - 256u;
        stages = 0;
        for (uint32_t st = 3; st >= 2; --st)
            if (2u * b_bytes + st * a_stage_bytes + 128u + 1024u <= budget) { stages = st; break; }
        total = 2u * b_bytes + stages * a_stage_bytes + 128u + 1024u;      // + barriers + bias[UN] copy
    }
};

// ---- warp-specialised kernel ------------------------------------------------------------------------------------------
// The three phases run concurrently in different warps and hand over through mbarriers only (no __syncthreads in the
// steady state):
//   warps 0-3   producers : cp.async the next A k-block into the ring (after `empty[stage]`), convert lo for the k-block that
//                           has landed (own chunks only), fence.proxy.async, one arrive per warp on `full[stage]`
//   warps 4-11  epilogue  : wait `acc_full[buf]`, tcgen05.ld -> +bias -> act -> global, one arrive per warp on `acc_empty[buf]`
//   warp  12    MMA issuer: wait `full[stage]` (and `acc_empty[buf]` at the first k-block of a tile), 12 tcgen05.mma,
//                           tcgen05.commit -> `empty[stage]` (+ `acc_full[buf]` after the last k-block of the tile)
constexpr int kWsProducerWarps = 4, kWsEpilogueWarps = 8;
constexpr int kWsThreads = (kWsProducerWarps + kWsEpilogueWarps + 1) * 32;

template <int STAGES>
__global__ void __launch_bounds__(kWsThreads, 1) gemm_tf32x3_ws_kernel(const Params p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const SmemPlan L(p.un, p.K);
    uint8_t *b_hi_ptr = smem, *b_lo_ptr = smem + L.b_bytes;
    uint8_t *a_ring = smem + 2 * L.b_bytes;
    uint64_t *full = reinterpret_cast<uint64_t *>(a_ring + STAGES * L.a_stage_bytes);
    uint64_t *empty = full + STAGES, *acc_full = empty + STAGES, *acc_empty = acc_full + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_empty + 2);
    float *s_bias = reinterpret_cast<float *>(a_ring + STAGES * L.a_stage_bytes + 128);      // [UN], zeros when there is no bias
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    for (int i = t; i < p.un; i += kWsThreads) s_bias[i] = (p.bias != nullptr && i < p.N) ? __ldg(p.bias + i) : 0.0f;

    if (t == 0) {
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], kWsProducerWarps); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], kWsEpilogueWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    {   // W: transpose + RNA split, once per CTA, by everybody
        const int kchunks = (int)L.kpad / 4;
        const int total = p.un * kchunks;
        const uint32_t bh = smem_u32(b_hi_ptr), bl = smem_u32(b_lo_ptr);
        for (int cb = t; cb < total; cb += kWsThreads) {
            const int n8 = cb & 7, kc = (cb >> 3) % kchunks, ng = (cb >> 3) / kchunks;
            const int n = ng * 8 + n8, k = kc * 4;
            float w[4] = {0.f, 0.f, 0.f, 0.f}, h[4], l[4];
            if (n < p.N) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (k + i < p.K) w[i] = __ldg(p.B + (int64_t)(k + i) * p.ldb + n);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) split_tf32(w[i], h[i], l[i]);
            st_shared_v4(bh + cb * 16, h[0], h[1], h[2], h[3]);
            st_shared_v4(bl + cb * 16, l[0], l[1], l[2], l[3]);
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int nkb = (int)L.kpad / BK;
    const int my_tiles = blockIdx.x < p.tiles_m ? (p.tiles_m - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int total_kb = my_tiles * nkb;

    if (warp < kWsProducerWarps) {
        // ===================== producers =====================
        const uint32_t a_ring_addr = smem_u32(a_ring);
        constexpr int kChunksPerThread = (BM * BK / 4) / (kWsProducerWarps * 32);      // 8
        auto issue_load = [&](int G) {
            if (G < total_kb) {
                const int stage = G % STAGES;
                mbar_wait(&empty[stage], (uint32_t)(((G / STAGES) & 1) ^ 1));          // first use passes immediately
                const int tile = blockIdx.x + (G / nkb) * gridDim.x, kb = G % nkb;
                const int64_t m0 = (int64_t)tile * BM;
                const uint32_t dst0 = a_ring_addr + stage * L.a_stage_bytes;
#pragma unroll
                for (int i = 0; i < kChunksPerThread; ++i) {
                    const int c = t + kWsProducerWarps * 32 * i;
                    const int r8 = c & 7, kc = (c >> 3) & 7, rg = c >> 6;
                    const int64_t row = m0 + rg * 8 + r8;
                    const int k = kb * BK + kc * 4;
                    uint32_t bytes = 0;
                    const float *src = p.A;
                    if (row < p.M && k < p.K) {
                        bytes = (uint32_t)min(4, p.K - k) * 4u;
                        src = p.A + row * p.lda + k;
                    }
                    cp_async16_zfill(dst0 + c * 16, src, bytes);
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
#pragma unroll
        for (int G = 0; G < STAGES - 1; ++G) issue_load(G);
        for (int G = 0; G < total_kb; ++G) {
            issue_load(G + STAGES - 1);
            asm volatile("cp.async.wait_group %0;" ::"n"(STAGES - 1) : "memory");
            const int stage = G % STAGES;
            uint8_t *sraw = a_ring + stage * L.a_stage_bytes;
            uint8_t *slo = sraw + BM * BK * 4;
#pragma unroll
            for (int i = 0; i < kChunksPerThread; ++i) {
                const int c = t + kWsProducerWarps * 32 * i;
                const float4 v = *reinterpret_cast<const float4 *>(sraw + c * 16);
                float4 l;
                l.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
                l.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
                l.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
                l.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
                *reinterpret_cast<float4 *>(slo + c * 16) = l;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[stage]);
        }
    } else if (warp == kWsProducerWarps + kWsEpilogueWarps) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            const uint32_t idesc = make_idesc(p.un);
            const uint32_t sbo_b = (L.kpad / 4) * 128u;
            for (int G = 0; G < total_kb; ++G) {
                const int stage = G % STAGES, it = G / nkb, kb = G % nkb, buf = it & 1;
                if (kb == 0) mbar_wait(&acc_empty[buf], (uint32_t)(((it >> 1) & 1) ^ 1));   // epilogue drained this buffer
                mbar_wait(&full[stage], (uint32_t)((G / STAGES) & 1));
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kMaxUN);
                const uint32_t a_raw = smem_u32(a_ring + stage * L.a_stage_bytes), a_lo = a_raw + BM * BK * 4;
                const uint32_t b_hi = smem_u32(b_hi_ptr) + (uint32_t)kb * (BK / 4) * 128u, b_lo = b_hi + L.b_bytes;
#pragma unroll
                for (int j = 0; j < BK / UMMA_K; ++j) {
                    const uint32_t off = (uint32_t)j * 2u * 128u;
                    const uint64_t dah = make_desc_sbo(a_raw + off, 1024u), dal = make_desc_sbo(a_lo + off, 1024u);
                    const uint64_t dbh = make_desc_sbo(b_hi + off, sbo_b), dbl = make_desc_sbo(b_lo + off, sbo_b);
                    umma_tf32(d_tmem, dal, dbh, idesc, (kb | j) != 0);
                    umma_tf32(d_tmem, dah, dbl, idesc, 1u);
                    umma_tf32(d_tmem, dah, dbh, idesc, 1u);
                }
                umma_commit(&empty[stage]);
                if (kb == nkb - 1) umma_commit(&acc_full[buf]);
            }
        }
    } else {
        // ===================== epilogue =====================
        const int ew = warp - kWsProducerWarps;              // 0..7
        const int q = warp & 3, half = ew >> 2;              // TMEM lane quarter is fixed by warp_id % 4
        const int col_begin = half * (p.un / 2), col_end = (half + 1) * (p.un / 2);
        const bool vec_ok = (p.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
        for (int it = 0; it < my_tiles; ++it) {
            const int buf = it & 1;
            const int tile = blockIdx.x + it * gridDim.x;
            mbar_wait(&acc_full[buf], (uint32_t)((it >> 1) & 1));
            tc_fence_after();
            const int64_t row = (int64_t)tile * BM + q * 32 + lane;
            for (int c0 = col_begin; c0 < col_end; c0 += 8) {
                // 8 columns per TMEM round trip: measured faster than x32 reads (0.87 vs 1.06 ms), which stall the MMA pipe
                uint32_t r[8];
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * kMaxUN + c0);
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                             : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (row < p.M) {
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = apply_act(__uint_as_float(r[j]) + s_bias[c0 + j], p.act);
                    float *dst = p.C + row * p.ldc + c0;
                    if (vec_ok && c0 + 8 <= p.N) {
                        *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
                        *reinterpret_cast<float4 *>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (c0 + j < p.N) dst[j] = v[j];
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
    }
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}
}  // namespace tc
}  // namespace tfgk

using namespace tfgk;

extern "C" int tfgk_gemm_tc_f32(const float *A, int64_t lda, const float *B, int64_t ldb, const float *bias, int act,
                                int32_t M, int32_t N, int32_t K, float *C, int64_t ldc, void *stream) {
    // K <= 512: tensor-core accumulation truncates (round-toward-zero), so the error grows ~K^1.5; up to K = 512 it stays
    // below 5e-6 relative (tests/test_gpu_gemm_tc.py), beyond that the SIMT path is used.
    if (N > tc::kMaxUN || M < 1 || K < 1 || K > 512 || (int64_t)M * K < (1 << 14)) return TFGK_ERR_UNSUPPORTED;
    tc::Params p;
    p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.bias = bias; p.act = act;
    p.M = M; p.N = N; p.K = K; p.C = C; p.ldc = ldc;
    p.un = ((N + 15) / 16) * 16;
    p.tiles_m = (int)ceil_div64(M, tc::BM);
    if ((lda % 4 != 0) || !aligned16(A)) return TFGK_ERR_UNSUPPORTED;       // cp.async moves 16-byte chunks
    const tc::SmemPlan L(p.un, K);
    if (L.stages == 0) return TFGK_ERR_UNSUPPORTED;                         // W does not fit next to two A stages
    int dev = 0, sms = 0;
    TFGK_CUDA(cudaGetDevice(&dev));
    TFGK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int grid = p.tiles_m < sms ? p.tiles_m : sms;       // persistent: one CTA per SM
    if (L.stages == 3) {
        TFGK_CUDA(ensure_dynamic_smem(tc::gemm_tf32x3_ws_kernel<3>, L.total));
        tc::gemm_tf32x3_ws_kernel<3><<<grid, tc::kWsThreads, L.total, as_stream(stream)>>>(p);
    } else {
        TFGK_CUDA(ensure_dynamic_smem(tc::gemm_tf32x3_ws_kernel<2>, L.total));
        tc::gemm_tf32x3_ws_kernel<2><<<grid, tc::kWsThreads, L.total, as_stream(stream)>>>(p);
    }
    TFGK_LAUNCH_CHECK();
    return TFGK_OK;
}
