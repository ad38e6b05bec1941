// (f1, second half) Node-feature assembly on the device (SURVEY 8f-1).
//
// Replaces the numpy block of build_graph_data (reference src/deep_fem_uav_wing/gnn/dataset.py:129-151):
//   x = [ (pos - min) / range  |  normal / |normal|  |  4 scaled global parameters ]   [N,10] fp32
//   y = log1p(stress_vm)                                                                [N,1]  fp32
// with the reference's guards (range < 1e-8 -> 1, dataset.py:135; |normal| < 1e-8 -> 1, dataset.py:140).
// The arithmetic is written with the non-contracting intrinsics (__fmul_rn / __fadd_rn / __fsqrt_rn / __fdiv_rn) in
// numpy's evaluation order, so x is BIT-IDENTICAL to the reference's float32 result (a zero may differ in sign: numpy's
// min over +0 and -0 depends on their order); y uses log1pf, within 1 ulp of the correctly rounded log1p.
// Two launches: a per-axis min/max reduction (fixed order: min/max are exact whatever the order) and one
// element-wise pass.  The min/max propagate NaN as numpy's pos.min(axis=0) does: a NaN coordinate makes that axis of
// its case NaN in every row.  HBM-bound; algorithmic bytes = 28 N read + 44 N written.
#include <algorithm>
#include <cfloat>

#include "dfw_common.cuh"

namespace dfw {
namespace {

constexpr int kFeatThreads = 256;
constexpr int kFeatMaxBlocks = kNumSMs * 4;

__global__ void __launch_bounds__(kFeatThreads) k_pos_minmax(const float* __restrict__ pos, int64_t N,
                                                             float* __restrict__ part /*[blocks][6]*/,
                                                             unsigned int* __restrict__ ticket, float* __restrict__ mm /*[6]*/) {
    __shared__ float sh[kFeatThreads / 32][6];
    __shared__ bool last;
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = pos[3 * i + a];
            lo[a] = min_nan(lo[a], v);
            hi[a] = max_nan(hi[a], v);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            lo[a] = min_nan(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = max_nan(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { sh[wid][a] = lo[a]; sh[wid][3 + a] = hi[a]; }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        const int k = threadIdx.x;
        float v = sh[0][k];
        for (int w = 1; w < kFeatThreads / 32; ++w) v = k < 3 ? min_nan(v, sh[w][k]) : max_nan(v, sh[w][k]);
        part[6 * (int64_t)blockIdx.x + k] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last && threadIdx.x < 6) {
        __threadfence();
        const int k = threadIdx.x;
        float v = part[k];
        for (unsigned b = 1; b < gridDim.x; ++b) v = k < 3 ? min_nan(v, part[6 * (int64_t)b + k]) : max_nan(v, part[6 * (int64_t)b + k]);
        mm[k] = v;
        if (k == 0) *ticket = 0u;
    }
}

struct FeatArgs {
    const float* pos; const float* normal; const float* stress; const float* mm;
    float gp[4];
    int normalize_pos, log_scale;
    float* x; float* y;
    int64_t N;
};

__global__ void __launch_bounds__(kFeatThreads) k_node_features(const FeatArgs p) {
    float mn[3] = {0.f, 0.f, 0.f}, rg[3] = {1.f, 1.f, 1.f};
    if (p.normalize_pos) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            mn[a] = p.mm[a];
            rg[a] = __fsub_rn(p.mm[3 + a], p.mm[a]);
            if (rg[a] < 1e-8f) rg[a] = 1.0f;  // dataset.py:135
        }
    }
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < p.N; i += (int64_t)gridDim.x * blockDim.x) {
        float* xo = p.x + 10 * i;
        const float px = p.pos[3 * i], py = p.pos[3 * i + 1], pz = p.pos[3 * i + 2];
        if (p.normalize_pos) {
            xo[0] = __fdiv_rn(__fsub_rn(px, mn[0]), rg[0]);
            xo[1] = __fdiv_rn(__fsub_rn(py, mn[1]), rg[1]);
            xo[2] = __fdiv_rn(__fsub_rn(pz, mn[2]), rg[2]);
        } else {
            xo[0] = px; xo[1] = py; xo[2] = pz;
        }
        const float nx = p.normal[3 * i], ny = p.normal[3 * i + 1], nz = p.normal[3 * i + 2];
        // numpy.linalg.norm(axis=1): sqrt(((x*x + y*y) + z*z)) in float32, no fused multiply-add
        float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(nx, nx), __fmul_rn(ny, ny)), __fmul_rn(nz, nz)));
        if (len < 1e-8f) len = 1.0f;  // dataset.py:140
        xo[3] = __fdiv_rn(nx, len);
        xo[4] = __fdiv_rn(ny, len);
        xo[5] = __fdiv_rn(nz, len);
        xo[6] = p.gp[0]; xo[7] = p.gp[1]; xo[8] = p.gp[2]; xo[9] = p.gp[3];
        if (p.y) {
            const float s = p.stress[i];
            p.y[i] = p.log_scale ? log1pf(s) : s;  // dataset.py:148-151
        }
    }
}

// ---- batched form: B cases concatenated (rows case_ptr[b] .. case_ptr[b+1]), per-case min/max and global parameters ----
// One launch pair for a whole inference launch of the design-screening loop (inference_gnn.py:380-398 builds one case at a
// time): the per-case kernels are tiny (20k nodes) and their 2 x B launches were host overhead, not GPU work.
__global__ void __launch_bounds__(kFeatThreads) k_pos_minmax_cases(const float* __restrict__ pos, const int64_t* __restrict__ case_ptr,
                                                                   float* __restrict__ mm /*[B][8]*/) {
    __shared__ float sh[kFeatThreads / 32][6];
    const int64_t r0 = case_ptr[blockIdx.x], r1 = case_ptr[blockIdx.x + 1];
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int64_t i = r0 + threadIdx.x; i < r1; i += blockDim.x) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = pos[3 * i + a];
            lo[a] = min_nan(lo[a], v);
            hi[a] = max_nan(hi[a], v);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            lo[a] = min_nan(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = max_nan(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { sh[wid][a] = lo[a]; sh[wid][3 + a] = hi[a]; }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        const int k = threadIdx.x;
        float v = sh[0][k];
        for (int w = 1; w < kFeatThreads / 32; ++w) v = k < 3 ? min_nan(v, sh[w][k]) : max_nan(v, sh[w][k]);
        mm[8 * (int64_t)blockIdx.x + k] = v;
    }
}

struct FeatCasesArgs {
    const float* pos; const float* normal; const float* stress; const float* mm; const float* gp; const int64_t* case_ptr;
    int normalize_pos, log_scale;
    float* x; float* y;
};

__global__ void __launch_bounds__(kFeatThreads) k_node_features_cases(const FeatCasesArgs p) {
    const int b = blockIdx.y;
    const int64_t r0 = p.case_ptr[b], r1 = p.case_ptr[b + 1];
    float mn[3] = {0.f, 0.f, 0.f}, rg[3] = {1.f, 1.f, 1.f};
    if (p.normalize_pos) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            mn[a] = p.mm[8 * b + a];
            rg[a] = __fsub_rn(p.mm[8 * b + 3 + a], p.mm[8 * b + a]);
            if (rg[a] < 1e-8f) rg[a] = 1.0f;  // dataset.py:135
        }
    }
    const float g0 = p.gp[4 * b], g1 = p.gp[4 * b + 1], g2 = p.gp[4 * b + 2], g3 = p.gp[4 * b + 3];
    for (int64_t i = r0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < r1; i += (int64_t)gridDim.x * blockDim.x) {
        float* xo = p.x + 10 * i;
        const float px = p.pos[3 * i], py = p.pos[3 * i + 1], pz = p.pos[3 * i + 2];
        if (p.normalize_pos) {
            xo[0] = __fdiv_rn(__fsub_rn(px, mn[0]), rg[0]);
            xo[1] = __fdiv_rn(__fsub_rn(py, mn[1]), rg[1]);
            xo[2] = __fdiv_rn(__fsub_rn(pz, mn[2]), rg[2]);
        } else {
            xo[0] = px; xo[1] = py; xo[2] = pz;
        }
        const float nx = p.normal[3 * i], ny = p.normal[3 * i + 1], nz = p.normal[3 * i + 2];
        float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(nx, nx), __fmul_rn(ny, ny)), __fmul_rn(nz, nz)));
        if (len < 1e-8f) len = 1.0f;  // dataset.py:140
        xo[3] = __fdiv_rn(nx, len);
        xo[4] = __fdiv_rn(ny, len);
        xo[5] = __fdiv_rn(nz, len);
        xo[6] = g0; xo[7] = g1; xo[8] = g2; xo[9] = g3;
        if (p.y) {
            const float s = p.stress[i];
            p.y[i] = p.log_scale ? log1pf(s) : s;  // dataset.py:148-151
        }
    }
}

}  // namespace
}  // namespace dfw

extern "C" size_t dfw_node_features_batched_ws_bytes(int64_t B) { return B > 0 ? (size_t)B * 8 * sizeof(float) : 0; }

extern "C" int dfw_node_features_batched(const float* pos, const float* normal, const float* stress, const float* global_params /*device [B,4]*/,
                                         const int64_t* case_ptr /*device [B+1]*/, int64_t B, int64_t max_case_rows, int normalize_pos, int log_scale,
                                         float* x, float* y, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(B >= 0 && max_case_rows >= 0, "dfw_node_features_batched: negative size");
    if (B == 0 || max_case_rows == 0) return 0;
    DFW_REQUIRE(B <= 65535, "dfw_node_features_batched: at most 65535 cases per call");
    DFW_REQUIRE(pos && normal && x && global_params && case_ptr, "dfw_node_features_batched: null pointer");
    DFW_REQUIRE((y == nullptr) || stress, "dfw_node_features_batched: y requested without stress");
    DFW_REQUIRE(ws && ws_bytes >= dfw_node_features_batched_ws_bytes(B), "dfw_node_features_batched: workspace too small");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    float* mm = static_cast<float*>(ws);
    if (normalize_pos) {
        k_pos_minmax_cases<<<(unsigned)B, kFeatThreads, 0, s>>>(pos, case_ptr, mm);
        DFW_LAUNCH_CHECK();
    }
    FeatCasesArgs a{};
    a.pos = pos; a.normal = normal; a.stress = stress; a.mm = mm; a.gp = global_params; a.case_ptr = case_ptr;
    a.normalize_pos = normalize_pos; a.log_scale = log_scale; a.x = x; a.y = y;
    const unsigned bx = (unsigned)std::max<int64_t>(1, std::min<int64_t>((max_case_rows + kFeatThreads - 1) / kFeatThreads, 64));
    k_node_features_cases<<<dim3(bx, (unsigned)B, 1), kFeatThreads, 0, s>>>(a);
    DFW_LAUNCH_CHECK();
    return 0;
}

extern "C" size_t dfw_node_features_ws_bytes(int64_t N) {
    (void)N;
    return 256 + 32 + sizeof(float) * 6 * dfw::kFeatMaxBlocks;
}

extern "C" int dfw_node_features(const float* pos, const float* normal, const float* stress, const float* global_params4,
                                 int normalize_pos, int log_scale, float* x, float* y, int64_t N, void* ws, size_t ws_bytes,
                                 dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(N >= 0, "dfw_node_features: negative N");
    if (N == 0) return 0;
    DFW_REQUIRE(pos && normal && x && global_params4, "dfw_node_features: null pointer");
    DFW_REQUIRE((y == nullptr) || stress, "dfw_node_features: y requested without stress");
    DFW_REQUIRE(ws && ws_bytes >= dfw_node_features_ws_bytes(N), "dfw_node_features: workspace too small");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(ws);
    float* mm = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + 256);
    float* part = mm + 8;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((N + kFeatThreads - 1) / kFeatThreads, kFeatMaxBlocks));
    if (normalize_pos) {
        DFW_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s));
        k_pos_minmax<<<blocks, kFeatThreads, 0, s>>>(pos, N, part, ticket, mm);
        DFW_LAUNCH_CHECK();
    }
    FeatArgs a{};
    a.pos = pos; a.normal = normal; a.stress = stress; a.mm = mm;
    for (int k = 0; k < 4; ++k) a.gp[k] = global_params4[k];  // host array: 4 floats by value
    a.normalize_pos = normalize_pos; a.log_scale = log_scale;
    a.x = x; a.y = y; a.N = N;
    k_node_features<<<blocks, kFeatThreads, 0, s>>>(a);
    DFW_LAUNCH_CHECK();
    return 0;
}
