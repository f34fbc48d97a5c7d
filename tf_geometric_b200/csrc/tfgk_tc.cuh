// tcgen05 / mbarrier / UMMA-descriptor helpers shared by the tensor-core GEMM kernels (gemm_tc.cu, gemm_proj.cu).
#pragma once
#include "common.cuh"

namespace tfgk {
namespace tc {

constexpr int BM = 128;            // UMMA_M
constexpr int BK = 32;             // K elements per smem stage (8 core matrices of 16 B along K)
constexpr int UMMA_K = 8;          // tf32
constexpr int kMaxUN = 256;
constexpr int kTmemCols = 512;
constexpr uint32_t kSpinLimit = 1u << 28;

struct Params {
    const float *A; int64_t lda;
    const float *B; int64_t ldb;
    const float *bias; int act;
    int M, N, K;
    float *C; int64_t ldc;
    int un;            // UMMA_N: N rounded up to a multiple of 16
    int tiles_m;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (spin > kSpinLimit) __trap();      // never hang the GPU: a lost arrive becomes a launch failure
    }
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 64-bit shared-memory matrix descriptor: K-major, SWIZZLE_NONE, LBO = 128 B, SBO = 1024 B, descriptor version 1
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);          // start address,        bits [0,14)
    d |= (uint64_t)(128u >> 4) << 16;                  // leading byte offset,  bits [16,30)
    d |= (uint64_t)(1024u >> 4) << 32;                 // stride byte offset,   bits [32,46)
    d |= (uint64_t)1 << 46;                            // version = 1 (sm_100), bits [46,48)
    return d;                                          // base_offset 0, lbo_mode 0, layout_type 0 (no swizzle)
}

// 32-bit instruction descriptor: D = F32, A = B = TF32, both K-major, N = un, M = 128
__device__ __forceinline__ uint32_t make_idesc(int un) {
    uint32_t d = 0;
    d |= 1u << 4;                       // c_format  = F32
    d |= 2u << 7;                       // a_format  = TF32
    d |= 2u << 10;                      // b_format  = TF32
    d |= (uint32_t)(un >> 3) << 17;     // n_dim
    d |= (uint32_t)(BM >> 4) << 24;     // m_dim
    return d;
}

__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void split_tf32(float a, float &hi, float &lo) {
    uint32_t h;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(a));
    hi = __uint_as_float(h);
    lo = a - hi;
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, float x, float y, float z, float w) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}


__device__ __forceinline__ uint64_t make_desc_sbo(uint32_t saddr, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(128u >> 4) << 16;
    d |= (uint64_t)(sbo_bytes >> 4) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void *src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

}  // namespace tc
}  // namespace tfgk
