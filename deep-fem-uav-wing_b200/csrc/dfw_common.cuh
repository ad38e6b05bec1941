// Shared helpers for libdfw_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/dfw_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libdfw_b200 is written for sm_100a (B200) only"
#endif

namespace dfw {

void set_error(const char* fmt, ...);

#define DFW_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            dfw::set_error(__VA_ARGS__);  \
            return 1;                     \
        }                                 \
    } while (0)

#define DFW_CUDA(expr)                                                                      \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            dfw::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                           __LINE__);                                                       \
            return 2;                                                                       \
        }                                                                                   \
    } while (0)

#define DFW_LAUNCH_CHECK() DFW_CUDA(cudaGetLastError())

constexpr int kNumSMs = 148;  // B200

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
__device__ __forceinline__ bool aligned16_dev(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- dtype helpers ---------------------------------------------------------------------
template <typename T>
struct Vec16;  // 16-byte vector of T
template <>
struct Vec16<float> {
    static constexpr int N = 4;
    float4 v;
    __device__ __forceinline__ void to_float(float* f) const {
        f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
    }
    __device__ __forceinline__ void from_float(const float* f) { v = make_float4(f[0], f[1], f[2], f[3]); }
};
template <>
struct Vec16<__nv_bfloat16> {
    static constexpr int N = 8;
    uint4 v;
    __device__ __forceinline__ void to_float(float* f) const {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            f[2 * i] = __uint_as_float(w[i] << 16);
            f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
    __device__ __forceinline__ void from_float(const float* f) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 p = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
            w[i] = *reinterpret_cast<uint32_t*>(&p);
        }
        v = make_uint4(w[0], w[1], w[2], w[3]);
    }
};

__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
template <typename T>
__device__ __forceinline__ T from_f32(float x);
template <>
__device__ __forceinline__ float from_f32<float>(float x) { return x; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }

// Counter-based dropout RNG: the keep-mask is a pure function of (seed, row, column), so the backward regenerates
// it instead of storing a mask.  Two levels, both the 32-bit "lowbias32" finaliser: a key per ROW (computed once by
// the thread or warp that owns the row) and ~9 integer instructions per element.  (The first version hashed a
// 64-bit element index with splitmix64: ~30 instructions per element, which made the thread-per-row epilogue of the
// tensor-core linear and the LayerNorm backward ALU bound.)
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16;
    x *= 0x21f0aaadu;
    x ^= x >> 15;
    x *= 0x735a2d97u;
    x ^= x >> 15;
    return x;
}
__device__ __forceinline__ uint32_t dropout_row_key(uint64_t seed, uint64_t row) {
    uint32_t k = mix32(static_cast<uint32_t>(row) ^ static_cast<uint32_t>(seed));
    k += static_cast<uint32_t>(row >> 32) * 0x85EBCA6Bu + static_cast<uint32_t>(seed >> 32);
    return mix32(k);
}
__device__ __forceinline__ uint32_t dropout_bits(uint32_t row_key, uint32_t col) { return mix32(row_key + col * 0x9E3779B9u); }
// seed given by value, or (DFW_EP_SEED_IS_PTR) read from device memory at kernel time
__device__ __forceinline__ uint64_t resolve_seed(uint64_t seed, int flags) {
    return (flags & DFW_EP_SEED_IS_PTR) ? *reinterpret_cast<const uint64_t*>(static_cast<uintptr_t>(seed)) : seed;
}
// keep iff bits >= threshold, threshold = p * 2^32
__host__ __device__ __forceinline__ uint32_t dropout_threshold(float p) {
    double t = static_cast<double>(p) * 4294967296.0;
    if (t < 0) t = 0;
    if (t > 4294967295.0) t = 4294967295.0;
    return static_cast<uint32_t>(t);
}

// The canonical CSR build of dfw_csr_build (dfw_csr.cu), shared with the vertex-normal build (dfw_screen.cu).  `gate`
// (nullable, device) skips every kernel when *gate == 0.  ws: dfw_csr_ws_bytes(E, N).
int csr_build_impl(const int64_t* edge_index, int64_t E, int64_t N, int by_src, int32_t* rowptr, int32_t* col,
                   int32_t* perm, float* inv_deg, int32_t* status, void* ws, size_t ws_bytes, dfw_stream_t stream,
                   const int32_t* gate);

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace dfw
