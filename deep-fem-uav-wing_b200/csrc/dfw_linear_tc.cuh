// Declarations shared between dfw_linear.cu (dispatch) and dfw_linear_tc.cu (tcgen05 kernels).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace dfw {
namespace tc {
struct Args {
    int64_t N;
    int Hout;        // logical output width
    int Npad;        // UMMA N (multiple of 16)
    int tmem_cols;   // power of two >= 32
    int nacc;        // fp32: number of hi*hi accumulators (cross terms use one more)
    int chunks[2];   // 128-byte K chunks per operand pair
    int stages;
    int flags;
    const float* bias; const float* gamma; const float* beta; float eps;
    const float* row_scale;
    const void* residual; uint32_t drop_thr; float drop_scale; uint64_t seed;
    void* out; void* pre_out; float* ln_stats;
    const float* rowdot_w; const float* rowdot_b; float* rowdot_out;
};
}  // namespace tc
size_t linear_tc_ws_bytes(int64_t Hout, int64_t k1, int64_t k2, int dtype);
bool linear_tc_eligible(int64_t N, int64_t Hout, int64_t k1, int64_t k2, int dtype, const void* a1, const void* a2);
int linear_tc_launch(const void* a1, const void* w1, int64_t k1, const void* a2, const void* w2, int64_t k2, int transpose_w,
                     tc::Args args, int dtype, void* ws, size_t ws_bytes, cudaStream_t s);
bool dw_tc_eligible(int64_t N, int64_t Hout, int64_t k1, int64_t k2, int dtype, const void* g, const void* a1, const void* a2);
int dw_tc_launch(const void* g_y, const void* a1, int64_t k1, const void* a2, int64_t k2, int64_t N, int64_t Hout, int dtype,
                 float* part, int splits, int64_t nodes_per_split, cudaStream_t s);
size_t colsum_ws_bytes(int64_t H);
int colsum_launch(const void* g_y, int64_t N, int64_t H, int dtype, float* part, float* dbias, int accumulate, cudaStream_t s);
}  // namespace dfw
