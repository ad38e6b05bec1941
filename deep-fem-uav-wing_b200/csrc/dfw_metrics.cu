// Evaluation metrics on the device (SURVEY 8f-2): MAE / RMSE / max error in the ORIGINAL stress scale for all
// nodes and for the masked nodes.
//
// Replaces the host-side numpy pass of compute_metrics (reference src/deep_fem_uav_wing/gnn/model.py:156-216):
// there, pred / target / mask are copied to the host in full (model.py:173-179), expm1'd (model.py:184-185) and
// reduced once per subset (model.py:190-204), once per validation batch (scripts/train_gnn.py:85-107).  Here one
// kernel reads the three arrays once and leaves 8 doubles on the device; the caller copies 64 bytes.
// Deterministic: fixed grid, fixed-order second pass, no float atomics.  Every max stage propagates NaN, so a NaN
// error makes mae, rmse and max_error of its subset NaN alike, as numpy does.
// Roofline: HBM, algorithmic bytes = N*C*2*b + N (mask); a 200k-node batch is launch-latency bound.
#include <algorithm>

#include "dfw_common.cuh"

namespace dfw {
namespace {

constexpr int kMetThreads = 256;
constexpr int kMetMaxBlocks = kNumSMs * 4;

struct Acc4 {
    double sum_abs, sum_sq;
    float mx;
    double cnt;
};

template <typename T>
__global__ void __launch_bounds__(kMetThreads) k_stress_metrics(const T* __restrict__ pred, const T* __restrict__ target,
                                                                const uint8_t* __restrict__ mask, int64_t N, int64_t C,
                                                                int log_scale, double* __restrict__ part /*[blocks][8]*/,
                                                                unsigned int* __restrict__ ticket, double* __restrict__ result) {
    __shared__ double sh[kMetThreads / 32][8];
    __shared__ bool last;
    // per thread: fp32 partials over a handful of elements, widened at the warp level
    float sa[2] = {0.f, 0.f}, sq[2] = {0.f, 0.f}, mx[2] = {0.f, 0.f}, cn[2] = {0.f, 0.f};
    const int64_t total = N * C;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        float p = to_f32(pred[i]), t = to_f32(target[i]);
        if (log_scale) {  // inverse of log1p (dataset.py:148-151)
            p = expm1f(p);
            t = expm1f(t);
        }
        const float e = fabsf(p - t);
        sa[0] += e; sq[0] = fmaf(e, e, sq[0]); mx[0] = max_nan(mx[0], e); cn[0] += 1.f;
        if (mask && mask[i / C]) {
            sa[1] += e; sq[1] = fmaf(e, e, sq[1]); mx[1] = max_nan(mx[1], e); cn[1] += 1.f;
        }
    }
    double v[8] = {(double)sa[0], (double)sq[0], (double)mx[0], (double)cn[0], (double)sa[1], (double)sq[1], (double)mx[1], (double)cn[1]};
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const double w = __shfl_xor_sync(0xffffffffu, v[k], o);
            v[k] = (k == 2 || k == 6) ? max_nan(v[k], w) : v[k] + w;
        }
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) sh[wid][k] = v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int w = 0; w < kMetThreads / 32; ++w)
            for (int k = 0; k < 8; ++k) a[k] = (k == 2 || k == 6) ? max_nan(a[k], sh[w][k]) : a[k] + sh[w][k];
        for (int k = 0; k < 8; ++k) part[8 * (int64_t)blockIdx.x + k] = a[k];
        __threadfence();
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last && threadIdx.x < 8) {  // fixed-order final reduction: thread k owns statistic k
        __threadfence();
        const int k = threadIdx.x;
        double a = 0.0;
        for (unsigned b = 0; b < gridDim.x; ++b) {
            const double w = part[8 * (int64_t)b + k];
            a = (k == 2 || k == 6) ? max_nan(a, w) : a + w;
        }
        sh[0][k] = a;
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        // [mae, rmse, max_error, count] for all nodes, then for the masked nodes; an empty subset reports zeros
        // (model.py:194-195).  Without a mask the masked statistics equal the all-node ones (model.py:207-210).
        for (int s = 0; s < 2; ++s) {
            const int src = (s == 1 && !mask) ? 0 : s;
            const double cnt = sh[0][4 * src + 3];
            result[4 * s + 0] = cnt > 0 ? sh[0][4 * src + 0] / cnt : 0.0;
            result[4 * s + 1] = cnt > 0 ? sqrt(sh[0][4 * src + 1] / cnt) : 0.0;
            result[4 * s + 2] = cnt > 0 ? sh[0][4 * src + 2] : 0.0;
            result[4 * s + 3] = cnt;
        }
        *ticket = 0u;
    }
}

}  // namespace
}  // namespace dfw

extern "C" size_t dfw_stress_metrics_ws_bytes(int64_t N, int64_t C) {
    (void)N; (void)C;
    return 256 + sizeof(double) * 8 * dfw::kMetMaxBlocks;
}

extern "C" int dfw_stress_metrics(const void* pred, const void* target, const uint8_t* mask, int64_t N, int64_t C, int log_scale,
                                  int dtype, double* result, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_stress_metrics: unknown dtype %d", dtype);
    DFW_REQUIRE(N >= 0 && C >= 1 && result, "dfw_stress_metrics: bad arguments");
    DFW_REQUIRE(N == 0 || (pred && target), "dfw_stress_metrics: null pointer");
    DFW_REQUIRE(ws && ws_bytes >= dfw_stress_metrics_ws_bytes(N, C), "dfw_stress_metrics: workspace too small");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(ws);
    double* part = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + 256);
    DFW_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s));
    const int64_t total = N * C;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((total + kMetThreads * 4 - 1) / (kMetThreads * 4), kMetMaxBlocks));
    if (dtype == DFW_F32)
        k_stress_metrics<float><<<blocks, kMetThreads, 0, s>>>((const float*)pred, (const float*)target, mask, N, C, log_scale, part, ticket, result);
    else
        k_stress_metrics<__nv_bfloat16><<<blocks, kMetThreads, 0, s>>>((const __nv_bfloat16*)pred, (const __nv_bfloat16*)target, mask, N, C,
                                                                       log_scale, part, ticket, result);
    DFW_LAUNCH_CHECK();
    return 0;
}
