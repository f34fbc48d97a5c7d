// Shared helpers for the tfgk kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <float.h>
#include <mutex>
#include "tfgk.h"

namespace tfgk {

constexpr int kWarp = 32;

// thread-local error message, returned by tfgk_last_error()
char *error_buffer();
int set_error(int code, const char *fmt, ...);

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

#define TFGK_CHECK_ARG(cond, ...)                                              \
    do {                                                                       \
        if (!(cond)) return ::tfgk::set_error(TFGK_ERR_INVALID_ARGUMENT, __VA_ARGS__); \
    } while (0)

#define TFGK_CUDA(expr)                                                        \
    do {                                                                       \
        cudaError_t err__ = (expr);                                            \
        if (err__ != cudaSuccess)                                              \
            return ::tfgk::set_error(TFGK_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, \
                                     cudaGetErrorString(err__), __FILE__, __LINE__); \
    } while (0)

#define TFGK_LAUNCH_CHECK() TFGK_CUDA(cudaGetLastError())

inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// cudaFuncAttributeMaxDynamicSharedMemorySize once per (kernel, device) instead of on every launch (the attribute call costs
// microseconds - invisible next to a 10 ms aggregation, visible on Cora-sized graphs where a forward is a few launches).
// Only ever raises the limit; safe from several host threads (a repeated set is harmless).
template <typename Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, size_t bytes) {
    struct Entry { const void *fn; int dev; size_t bytes; };
    static Entry table[256];
    static int used = 0;
    static std::mutex guard;                  // launches may come from several host threads
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess) return err;
    std::lock_guard<std::mutex> lock(guard);
    const void *fn = reinterpret_cast<const void *>(kernel);
    const int n = used < 256 ? used : 256;
    for (int i = 0; i < n; ++i)
        if (table[i].fn == fn && table[i].dev == dev && table[i].bytes >= bytes) return cudaSuccess;
    err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (err == cudaSuccess && used < 256) {
        table[used].fn = fn; table[used].dev = dev; table[used].bytes = bytes;
        ++used;
    }
    return err;
}

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct alignas(64) TensorMap { uint64_t opaque[16]; };      // CUtensorMap (128 bytes), filled by the driver on the host

// Encodes a 2-D fp32 tensor map over n_rows rows of `width` columns (row stride ld floats) whose box is one row: the
// operand of TMA tile::gather4.  cuTensorMapEncodeTiled is reached through the runtime's driver entry point (no link-time
// dependency on libcuda).  Returns TFGK_ERR_UNSUPPORTED when the driver cannot encode the map, so callers fall back.
inline int make_row_tensor_map(TensorMap *out, const float *base, int64_t ld, int64_t n_rows, int32_t width) {
    typedef int (*EncodeTiledFn)(void *map, int dtype, uint32_t rank, void *base, const uint64_t *dims,
                                 const uint64_t *strides, const uint32_t *box, const uint32_t *elem_strides, int interleave,
                                 int swizzle, int l2promo, int oob_fill);
    static EncodeTiledFn encode = nullptr;
    if (encode == nullptr) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        TFGK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (fn == nullptr || qres != cudaDriverEntryPointSuccess)
            return set_error(TFGK_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled is not available from this driver");
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    const uint64_t dims[2] = {(uint64_t)width, (uint64_t)n_rows};
    const uint64_t strides[1] = {(uint64_t)ld * sizeof(float)};           // byte stride of dimension 1 (rows)
    const uint32_t box[2] = {(uint32_t)width, 1u};                        // gather4: 1 in the gathered dimension
    const uint32_t elem[2] = {1u, 1u};
    // CU_TENSOR_MAP_DATA_TYPE_FLOAT32 = 7, INTERLEAVE_NONE = 0, SWIZZLE_NONE = 0, L2_PROMOTION_L2_128B = 2, OOB_FILL_NONE = 0
    const int rc = encode(out, 7, 2, const_cast<float *>(base), dims, strides, box, elem, 0, 0, 2, 0);
    if (rc != 0) return set_error(TFGK_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled failed with CUresult %d", rc);
    return TFGK_OK;
}

// activation applied in every fused epilogue
__device__ __forceinline__ float apply_act(float v, int act) {
    return act == TFGK_ACT_RELU ? fmaxf(v, 0.0f) : v;
}

// streaming (read-once) loads: keep them out of L1 so gathered feature rows own the cache
__device__ __forceinline__ int ld_stream_i32(const int *p) {
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_stream_f32(const float *p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

}  // namespace tfgk
