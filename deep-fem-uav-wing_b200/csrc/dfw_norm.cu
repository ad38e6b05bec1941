// Row-wise pieces of the GraphSAGE backward and the masked loss.
//
//  dfw_epilogue_bwd : backward of  out = residual + dropout(relu(layernorm(y)))   (model.py:91-95)
//                     and of the decoder tail  relu -> dropout -> Linear(64,1)    (model.py:69-71).
//  dfw_masked_mse_* : MaskedMSELoss (model.py:126-153) without boolean indexing or host sync.
//  All HBM-bound, one warp per row with 128-bit accesses; column reductions (dgamma, dbeta, ...)
//  are two-pass and fixed-order (no float atomics).
#include <algorithm>
#include <cstdarg>
#include <cstring>

#include "dfw_common.cuh"

namespace dfw {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {

constexpr int kEbThreads = 256;
constexpr int kEbWarps = kEbThreads / 32;
constexpr int kEbMaxBlocks = kNumSMs * 4;

template <typename T>
__device__ __forceinline__ void ld4(const T* p, float* v) {
    if constexpr (sizeof(T) == 4) {
        float4 f = *reinterpret_cast<const float4*>(p);
        v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
    } else {
        uint2 u = *reinterpret_cast<const uint2*>(p);
        v[0] = __uint_as_float(u.x << 16); v[1] = __uint_as_float(u.x & 0xffff0000u);
        v[2] = __uint_as_float(u.y << 16); v[3] = __uint_as_float(u.y & 0xffff0000u);
    }
}
template <typename T>
__device__ __forceinline__ void st4(T* p, const float* v) {
    if constexpr (sizeof(T) == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
        __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]);
        __nv_bfloat162 p1 = __floats2bfloat162_rn(v[2], v[3]);
        *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1));
    }
}

struct EbArgs {
    const void* g_out; const float* g_rowdot; const float* rowdot_w;
    const void* pre_out; const float* ln_stats; const void* act;
    const float* gamma; const float* beta;
    uint32_t drop_thr; float drop_scale; uint64_t seed;
    void* g_y; float* part;  // [blocks][4][H] : (dgamma | d_rowdot_w), dbeta, (slot 2, col 0) = sum g_rowdot, colsum(g_y)
    int64_t N; int H; int flags;
};

// SPEC = 0: every option is a run-time flag.  SPEC = 1 / 3: the SAGE layer's tail (LayerNorm + ReLU, gradient from
// g_out; bit 1 = dropout) with the options folded at compile time - the generic kernel is issue bound (250 warp
// instructions per row, 63 % issue utilisation at 25 % occupancy, profiles/r01_ncu_summary_final.txt) and a good
// part of that was flag tests and the never-taken rowdot / act paths inside the row loop.
template <typename T, int VPL, int SPEC>
__global__ void __launch_bounds__(kEbThreads, VPL == 1 ? 2 : 1) k_epilogue_bwd(const EbArgs p) {
    constexpr int kMaxVPL = VPL;  // 16-byte column groups per lane: 1 (H <= 128) or 2 (H <= 256)
    __shared__ float red[kEbWarps][3][256 + 1];
    __shared__ float red_b[kEbWarps];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int H = p.H;
    const float invH = 1.f / (float)H;
    const bool ln = SPEC ? true : (bool)(p.flags & DFW_EP_LAYERNORM), relu = SPEC ? true : (bool)(p.flags & DFW_EP_RELU);
    const bool drop = SPEC ? (bool)(SPEC & 2) : (bool)(p.flags & DFW_EP_DROPOUT);
    const bool has_rowdot = SPEC ? false : p.g_rowdot != nullptr;
    const uint64_t seed_v = drop ? resolve_seed(p.seed, p.flags) : 0ull;
    const T* gout = (const T*)p.g_out;
    const T* pre = (const T*)p.pre_out;
    const T* act = SPEC ? nullptr : (const T*)p.act;
    T* gy = (T*)p.g_y;

    float gam[kMaxVPL][4], bet[kMaxVPL][4], rdw[kMaxVPL][4];
    float c0[kMaxVPL][4], c1[kMaxVPL][4];  // column partial sums
    bool vok[kMaxVPL];
#pragma unroll
    for (int v = 0; v < kMaxVPL; ++v) {
        const int c = (lane + v * 32) * 4;
        vok[v] = c < H;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            gam[v][j] = (p.gamma && vok[v]) ? __ldg(p.gamma + c + j) : 1.f;
            bet[v][j] = (p.beta && vok[v]) ? __ldg(p.beta + c + j) : 0.f;
            rdw[v][j] = (p.rowdot_w && vok[v]) ? __ldg(p.rowdot_w + c + j) : 0.f;
            c0[v][j] = 0.f;
            c1[v][j] = 0.f;
        }
    }
    float sum_gr = 0.f;

    float c2[kMaxVPL][4];  // column sums of g_y (= bias gradient of the producing linear)
#pragma unroll
    for (int v = 0; v < kMaxVPL; ++v)
#pragma unroll
        for (int j = 0; j < 4; ++j) c2[v][j] = 0.f;

    // kR rows per warp and iteration: all loads of the kR rows are issued before any arithmetic, so a warp
    // keeps 2*kR 512-byte requests in flight (one row at a time left the kernel latency-bound at 28 % of HBM).
    constexpr int kR = VPL == 1 ? 4 : 2;
    const int64_t warps = (int64_t)gridDim.x * kEbWarps;
    for (int64_t row0 = ((int64_t)blockIdx.x * kEbWarps + wid) * kR; row0 < p.N; row0 += warps * kR) {
        float g[kR][kMaxVPL][4], y[kR][kMaxVPL][4];
        float mean[kR], rstd[kR], gr[kR];
        bool rv[kR];
#pragma unroll
        for (int r = 0; r < kR; ++r) {
            const int64_t row = row0 + r;
            rv[r] = row < p.N;
            mean[r] = 0.f; rstd[r] = 1.f; gr[r] = 0.f;
            if (rv[r]) {
                if (ln) {
                    mean[r] = __ldg(p.ln_stats + 2 * row);
                    rstd[r] = __ldg(p.ln_stats + 2 * row + 1);
                }
                if (has_rowdot) gr[r] = __ldg(p.g_rowdot + row);
#pragma unroll
                for (int v = 0; v < kMaxVPL; ++v) {
                    if (!vok[v]) continue;
                    const int64_t off = row * H + (lane + v * 32) * 4;
                    if (!has_rowdot) ld4(gout + off, g[r][v]);
                    if (ln) ld4(pre + off, y[r][v]);
                    else if (act) ld4(act + off, y[r][v]);
                }
            }
        }
#pragma unroll
        for (int r = 0; r < kR; ++r) {
            if (!rv[r]) continue;  // warp-uniform
            const int64_t row = row0 + r;
            if (has_rowdot && lane == 0) sum_gr += gr[r];
            float xh[kMaxVPL][4];
            float s1 = 0.f, s2 = 0.f;
#pragma unroll
            for (int v = 0; v < kMaxVPL; ++v) {
                if (!vok[v]) continue;
                const int64_t off = row * H + (lane + v * 32) * 4;
                if (has_rowdot) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) g[r][v][j] = gr[r] * rdw[v][j];
                }
                float keep[4] = {1.f, 1.f, 1.f, 1.f};
                if (drop) {
                    const uint32_t row_key = dropout_row_key(seed_v, (uint64_t)row);
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        keep[j] = dropout_bits(row_key, (uint32_t)((lane + v * 32) * 4 + j)) >= p.drop_thr ? p.drop_scale : 0.f;
                }
                if (ln) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        xh[v][j] = (y[r][v][j] - mean[r]) * rstd[r];
                        const float z = xh[v][j] * gam[v][j] + bet[v][j];
                        float gg = g[r][v][j] * keep[j];
                        if (relu && !(z > 0.f)) gg = 0.f;
                        c0[v][j] += gg * xh[v][j];  // dgamma
                        c1[v][j] += gg;             // dbeta
                        gg *= gam[v][j];
                        g[r][v][j] = gg;
                        s1 += gg;
                        s2 += gg * xh[v][j];
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float a = act ? y[r][v][j] : 1.f;
                        if (has_rowdot) c0[v][j] += gr[r] * a;  // d_rowdot_w: `act` is the saved output, i.e. already post-ReLU AND post-dropout
                        float gg = g[r][v][j] * keep[j];
                        if (relu && !(a > 0.f)) gg = 0.f;
                        g[r][v][j] = gg;
                    }
                }
            }
            if (ln) {
                s1 = warp_sum(s1) * invH;
                s2 = warp_sum(s2) * invH;
            }
#pragma unroll
            for (int v = 0; v < kMaxVPL; ++v) {
                if (!vok[v]) continue;
                float o[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    o[j] = ln ? rstd[r] * (g[r][v][j] - s1 - xh[v][j] * s2) : g[r][v][j];
                    c2[v][j] += o[j];
                }
                st4(gy + row * H + (lane + v * 32) * 4, o);
            }
        }
    }

    if (!p.part) return;
    // block-level fixed-order reduction of the column partials -> part[block]
#pragma unroll
    for (int v = 0; v < kMaxVPL; ++v) {
        if (!vok[v]) continue;
        const int c = (lane + v * 32) * 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            red[wid][0][c + j] = c0[v][j];
            red[wid][1][c + j] = c1[v][j];
            red[wid][2][c + j] = c2[v][j];
        }
    }
    if (lane == 0) red_b[wid] = sum_gr;
    __syncthreads();
    for (int c = threadIdx.x; c < H; c += kEbThreads) {
        float a = 0.f, b = 0.f, d = 0.f;
#pragma unroll
        for (int w = 0; w < kEbWarps; ++w) {
            a += red[w][0][c];
            b += red[w][1][c];
            d += red[w][2][c];
        }
        p.part[((int64_t)blockIdx.x * 4 + 0) * H + c] = a;
        p.part[((int64_t)blockIdx.x * 4 + 1) * H + c] = b;
        p.part[((int64_t)blockIdx.x * 4 + 3) * H + c] = d;
    }
    if (threadIdx.x == 0) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kEbWarps; ++w) s += red_b[w];
        p.part[((int64_t)blockIdx.x * 4 + 2) * H] = s;
    }
}

// Backward of the LayerNorm-free epilogues (encoder linears: ReLU; decoder tail: ReLU + dropout + row-dot), i.e. the
// calls with no row statistics.  Purely element-wise plus column sums, so rows are PACKED: H/4 threads per row and
// 256/(H/4) rows per block step (the generic kernel above gives a row a whole warp and leaves half of its lanes idle
// at H = 64).  A thread's column group is fixed, so its column partials stay in registers; the row groups of a block
// are added in a fixed order.  Same `part` layout and second pass as the generic kernel.
template <typename T>
__global__ void __launch_bounds__(kEbThreads) k_act_bwd(const EbArgs p) {
    extern __shared__ float s_cols[];  // [3][rows_per_step][H]
    __shared__ float s_gr[kEbThreads];
    const int H = p.H, tpr = H / 4, rps = kEbThreads / tpr;
    const int rl = threadIdx.x / tpr, cl = (threadIdx.x % tpr) * 4;
    const bool active = rl < rps;
    const bool relu = p.flags & DFW_EP_RELU, drop = p.flags & DFW_EP_DROPOUT, has_rowdot = p.g_rowdot != nullptr;
    const uint64_t seed_v = drop ? resolve_seed(p.seed, p.flags) : 0ull;
    const T* gout = (const T*)p.g_out;
    const T* act = (const T*)p.act;
    T* gy = (T*)p.g_y;
    float rdw[4] = {0.f, 0.f, 0.f, 0.f};
    if (has_rowdot && active) {
#pragma unroll
        for (int j = 0; j < 4; ++j) rdw[j] = __ldg(p.rowdot_w + cl + j);
    }
    float c0[4] = {0.f, 0.f, 0.f, 0.f}, c2[4] = {0.f, 0.f, 0.f, 0.f};
    float sum_gr = 0.f;
    constexpr int kR = 4;  // rows in flight per thread
    const int64_t step = (int64_t)gridDim.x * rps;
    if (active) {
        for (int64_t row0 = (int64_t)blockIdx.x * rps + rl; row0 < p.N; row0 += step * kR) {
            float g[kR][4], y[kR][4], gr[kR];
            bool rv[kR];
#pragma unroll
            for (int r = 0; r < kR; ++r) {
                const int64_t row = row0 + r * step;
                rv[r] = row < p.N;
                gr[r] = 0.f;
                if (rv[r]) {
                    const int64_t off = row * H + cl;
                    if (has_rowdot) gr[r] = __ldg(p.g_rowdot + row);
                    else ld4(gout + off, g[r]);
                    if (act) ld4(act + off, y[r]);
                }
            }
#pragma unroll
            for (int r = 0; r < kR; ++r) {
                if (!rv[r]) continue;
                const int64_t row = row0 + r * step;
                if (has_rowdot && cl == 0) sum_gr += gr[r];
                float keep[4] = {1.f, 1.f, 1.f, 1.f};
                if (drop) {
                    const uint32_t row_key = dropout_row_key(seed_v, (uint64_t)row);
#pragma unroll
                    for (int j = 0; j < 4; ++j) keep[j] = dropout_bits(row_key, (uint32_t)(cl + j)) >= p.drop_thr ? p.drop_scale : 0.f;
                }
                float o[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float a = act ? y[r][j] : 1.f;
                    float gg = has_rowdot ? gr[r] * rdw[j] : g[r][j];
                    if (has_rowdot) c0[j] += gr[r] * a;  // d_rowdot_w: `act` is the saved output (post-ReLU, post-dropout)
                    gg *= keep[j];
                    if (relu && !(a > 0.f)) gg = 0.f;
                    o[j] = gg;
                    c2[j] += gg;
                }
                st4(gy + row * H + cl, o);
            }
        }
    }
    if (!p.part) return;
    float* sc0 = s_cols;
    float* sc2 = s_cols + (size_t)rps * H;
    if (active) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            sc0[rl * H + cl + j] = c0[j];
            sc2[rl * H + cl + j] = c2[j];
        }
    }
    s_gr[threadIdx.x] = (active && cl == 0) ? sum_gr : 0.f;
    __syncthreads();
    for (int c = threadIdx.x; c < H; c += kEbThreads) {
        float a = 0.f, d = 0.f;
        for (int q = 0; q < rps; ++q) {
            a += sc0[q * H + c];
            d += sc2[q * H + c];
        }
        p.part[((int64_t)blockIdx.x * 4 + 0) * H + c] = a;
        p.part[((int64_t)blockIdx.x * 4 + 1) * H + c] = 0.f;
        p.part[((int64_t)blockIdx.x * 4 + 3) * H + c] = d;
    }
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int q = 0; q < kEbThreads; ++q) t += s_gr[q];
        p.part[((int64_t)blockIdx.x * 4 + 2) * H] = t;
    }
}

// Second pass of the column reductions: one WARP per (slot, column); lanes stride over the per-block partials and
// a fixed shuffle tree combines them (deterministic).  A thread-per-column loop over ~600 partials is a chain of
// ~600 dependent L2 loads and took longer than the main kernel.
__global__ void __launch_bounds__(256) k_epilogue_bwd_reduce(const float* __restrict__ part, int blocks, int H, float* __restrict__ o0,
                                                              float* __restrict__ o1, float* __restrict__ o2, float* __restrict__ o3) {
    const int lane = threadIdx.x & 31;
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // warp id = slot * H + column
    if (w >= 4 * H) return;
    const int slot = w / H, c = w % H;
    float* out = slot == 0 ? o0 : (slot == 1 ? o1 : (slot == 2 ? o2 : o3));
    if (!out || (slot == 2 && c != 0)) return;
    float s = 0.f;
    for (int k = lane; k < blocks; k += 32) s += part[((int64_t)k * 4 + slot) * H + c];
    s = warp_sum(s);
    if (lane == 0) out[c] = s;
}

int eb_blocks(int64_t N) { return (int)std::max<int64_t>(1, std::min<int64_t>((N + kEbWarps * 4 - 1) / (kEbWarps * 4), kEbMaxBlocks)); }

// ---- masked MSE ----------------------------------------------------------------------------
constexpr int kMseThreads = 256;
constexpr int kMseMaxBlocks = kNumSMs * 4;

template <typename T>
__global__ void __launch_bounds__(kMseThreads) k_mse_fwd(const T* __restrict__ pred, const T* __restrict__ target,
                                                          const uint8_t* __restrict__ mask, int64_t N, int64_t C,
                                                          int mean, float* __restrict__ part /*[blocks][2]*/,
                                                          unsigned int* __restrict__ ticket, float* __restrict__ result) {
    __shared__ float ss[kMseThreads / 32], sc[kMseThreads / 32];
    __shared__ bool last;
    float s = 0.f, cnt = 0.f;
    const int64_t total = N * C;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / C;
        if (!mask || mask[r]) {
            const float d = to_f32(pred[i]) - to_f32(target[i]);
            s = fmaf(d, d, s);
            cnt += 1.f;
        }
    }
    s = warp_sum(s);
    cnt = warp_sum(cnt);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { ss[wid] = s; sc[wid] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, b = 0.f;
        for (int w = 0; w < kMseThreads / 32; ++w) { a += ss[w]; b += sc[w]; }
        part[2 * blockIdx.x] = a;
        part[2 * blockIdx.x + 1] = b;
        __threadfence();
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last) {  // fixed-order final reduction by the whole last block (a single-thread loop took ~25 us)
        __threadfence();
        double a = 0.0, b = 0.0;
        for (unsigned k = threadIdx.x; k < gridDim.x; k += blockDim.x) { a += (double)part[2 * k]; b += (double)part[2 * k + 1]; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        __shared__ double da[kMseThreads / 32], db[kMseThreads / 32];
        if (lane == 0) { da[wid] = a; db[wid] = b; }
        __syncthreads();
        if (threadIdx.x == 0) {
            a = 0.0; b = 0.0;
            for (int w = 0; w < kMseThreads / 32; ++w) { a += da[w]; b += db[w]; }
            result[0] = (float)(mean ? a / (b > 1.0 ? b : 1.0) : a);
            result[1] = (float)b;
            *ticket = 0u;
        }
    }
}

template <typename T>
__global__ void k_mse_bwd(const T* __restrict__ pred, const T* __restrict__ target, const uint8_t* __restrict__ mask,
                          const float* __restrict__ result, const float* __restrict__ g_loss, int64_t N, int64_t C,
                          int mean, T* __restrict__ g_pred) {
    const float cnt = result[1];
    const float scale = 2.f * g_loss[0] / (mean ? fmaxf(cnt, 1.f) : 1.f);
    const int64_t total = N * C;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / C;
        float g = 0.f;
        if (!mask || mask[r]) g = scale * (to_f32(pred[i]) - to_f32(target[i]));
        g_pred[i] = from_f32<T>(g);
    }
}

template <typename S, typename D>
__global__ void k_cast(const S* __restrict__ src, D* __restrict__ dst, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = from_f32<D>(to_f32(src[i]));
}

}  // namespace
}  // namespace dfw

extern "C" const char* dfw_last_error(void) { return dfw::g_err; }
extern "C" int dfw_abi_version(void) { return 1; }

extern "C" size_t dfw_epilogue_bwd_ws_bytes(int64_t N, int64_t Hout) {
    if (N < 0 || Hout < 1) return 0;
    return dfw::align_up(sizeof(float) * 4 * (size_t)Hout * dfw::eb_blocks(N), 256);
}

extern "C" int dfw_epilogue_bwd(const void* g_out, const float* g_rowdot, const float* rowdot_w, const void* pre_out,
                                const float* ln_stats, const void* act, const float* ln_gamma, const float* ln_beta,
                                float dropout_p, uint64_t seed, void* g_y, float* dgamma, float* dbeta,
                                float* d_rowdot_w, float* d_rowdot_b, float* d_bias, int64_t N, int64_t Hout, int flags,
                                int dtype, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_epilogue_bwd: unknown dtype %d", dtype);
    DFW_REQUIRE(N >= 0 && Hout >= 4 && Hout <= 256 && Hout % 4 == 0,
                "dfw_epilogue_bwd: Hout=%lld must be a multiple of 4 in [4,256]", (long long)Hout);
    DFW_REQUIRE((g_out != nullptr) != (g_rowdot != nullptr), "dfw_epilogue_bwd: exactly one of g_out / g_rowdot");
    DFW_REQUIRE(!g_rowdot || rowdot_w, "dfw_epilogue_bwd: g_rowdot needs rowdot_w");
    DFW_REQUIRE(g_y, "dfw_epilogue_bwd: null g_y");
    const bool ln = flags & DFW_EP_LAYERNORM;
    DFW_REQUIRE(!ln || (pre_out && ln_stats), "dfw_epilogue_bwd: LayerNorm backward needs pre_out and ln_stats");
    DFW_REQUIRE(ln || !(flags & DFW_EP_RELU) || act, "dfw_epilogue_bwd: ReLU backward needs act (or LayerNorm inputs)");
    DFW_REQUIRE(!(ln && g_rowdot), "dfw_epilogue_bwd: rowdot with LayerNorm is not a model configuration");
    if ((flags & DFW_EP_DROPOUT) && dropout_p == 0.f) flags &= ~DFW_EP_DROPOUT;
    const bool need_cols = (ln && (dgamma || dbeta)) || (g_rowdot && (d_rowdot_w || d_rowdot_b)) || d_bias;
    const int blocks = eb_blocks(N);
    if (need_cols) DFW_REQUIRE(ws && ws_bytes >= dfw_epilogue_bwd_ws_bytes(N, Hout), "dfw_epilogue_bwd: workspace too small");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    EbArgs a{};
    a.g_out = g_out; a.g_rowdot = g_rowdot; a.rowdot_w = rowdot_w; a.pre_out = pre_out; a.ln_stats = ln_stats; a.act = act;
    a.gamma = ln ? ln_gamma : nullptr; a.beta = ln ? ln_beta : nullptr;
    a.drop_thr = dropout_threshold(dropout_p); a.drop_scale = 1.f / (1.f - dropout_p); a.seed = seed;
    a.g_y = g_y; a.part = need_cols ? reinterpret_cast<float*>(ws) : nullptr;
    a.N = N; a.H = (int)Hout; a.flags = flags;
    if (N > 0) {
        if (!ln) {  // no row statistics: packed-row element-wise kernel
            const int tpr = (int)Hout / 4, rps = kEbThreads / tpr;
            const size_t smem = sizeof(float) * 2 * (size_t)rps * (size_t)Hout;
            if (dtype == DFW_F32) k_act_bwd<float><<<blocks, kEbThreads, smem, s>>>(a);
            else k_act_bwd<__nv_bfloat16><<<blocks, kEbThreads, smem, s>>>(a);
            DFW_LAUNCH_CHECK();
        } else {
        // the SAGE layer's tail gets the specialised instantiation
        const bool tail = ln && (flags & DFW_EP_RELU) && g_out && !g_rowdot;
        const int spec = tail ? ((flags & DFW_EP_DROPOUT) ? 3 : 1) : 0;
#define DFW_EB_GO(TT, V)                                                                     \
    do {                                                                                     \
        if (spec == 3) k_epilogue_bwd<TT, V, 3><<<blocks, kEbThreads, 0, s>>>(a);            \
        else if (spec == 1) k_epilogue_bwd<TT, V, 1><<<blocks, kEbThreads, 0, s>>>(a);       \
        else k_epilogue_bwd<TT, V, 0><<<blocks, kEbThreads, 0, s>>>(a);                      \
    } while (0)
        if (Hout <= 128) {
            if (dtype == DFW_F32) DFW_EB_GO(float, 1);
            else DFW_EB_GO(__nv_bfloat16, 1);
        } else {
            if (dtype == DFW_F32) DFW_EB_GO(float, 2);
            else DFW_EB_GO(__nv_bfloat16, 2);
        }
#undef DFW_EB_GO
        DFW_LAUNCH_CHECK();
        }
    }
    if (need_cols) {
        float* o0 = ln ? dgamma : d_rowdot_w;
        float* o1 = ln ? dbeta : nullptr;
        float* o2 = g_rowdot ? d_rowdot_b : nullptr;
        k_epilogue_bwd_reduce<<<(unsigned)((4 * Hout * 32 + 255) / 256), 256, 0, s>>>(a.part, N > 0 ? blocks : 0, (int)Hout, o0, o1, o2, d_bias);
        DFW_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" size_t dfw_masked_mse_ws_bytes(int64_t N, int64_t C) {
    (void)N; (void)C;
    return 256 + sizeof(float) * 2 * dfw::kMseMaxBlocks;
}

extern "C" int dfw_masked_mse_fwd(const void* pred, const void* target, const uint8_t* mask, int64_t N, int64_t C,
                                  int reduction_mean, int dtype, float* result, void* ws, size_t ws_bytes,
                                  dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_masked_mse_fwd: unknown dtype %d", dtype);
    DFW_REQUIRE(N >= 0 && C >= 1 && result, "dfw_masked_mse_fwd: bad arguments");
    DFW_REQUIRE(ws && ws_bytes >= dfw_masked_mse_ws_bytes(N, C), "dfw_masked_mse_fwd: workspace too small");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(ws);
    float* part = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + 256);
    DFW_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s));
    const int64_t total = N * C;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((total + kMseThreads - 1) / kMseThreads, kMseMaxBlocks));
    if (dtype == DFW_F32)
        k_mse_fwd<float><<<blocks, kMseThreads, 0, s>>>((const float*)pred, (const float*)target, mask, N, C, reduction_mean, part, ticket, result);
    else
        k_mse_fwd<__nv_bfloat16><<<blocks, kMseThreads, 0, s>>>((const __nv_bfloat16*)pred, (const __nv_bfloat16*)target, mask, N, C, reduction_mean, part, ticket, result);
    DFW_LAUNCH_CHECK();
    return 0;
}

extern "C" int dfw_masked_mse_bwd(const void* pred, const void* target, const uint8_t* mask, const float* result,
                                  const float* g_loss, int64_t N, int64_t C, int reduction_mean, int dtype, void* g_pred,
                                  dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_masked_mse_bwd: unknown dtype %d", dtype);
    DFW_REQUIRE(N >= 0 && C >= 1 && result && g_loss, "dfw_masked_mse_bwd: bad arguments");
    if (N == 0) return 0;  // an empty gradient has no storage: its pointer is null
    DFW_REQUIRE(g_pred, "dfw_masked_mse_bwd: null g_pred");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int64_t total = N * C;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, (int64_t)kNumSMs * 8));
    if (dtype == DFW_F32)
        k_mse_bwd<float><<<blocks, 256, 0, s>>>((const float*)pred, (const float*)target, mask, result, g_loss, N, C, reduction_mean, (float*)g_pred);
    else
        k_mse_bwd<__nv_bfloat16><<<blocks, 256, 0, s>>>((const __nv_bfloat16*)pred, (const __nv_bfloat16*)target, mask, result, g_loss, N, C, reduction_mean, (__nv_bfloat16*)g_pred);
    DFW_LAUNCH_CHECK();
    return 0;
}

extern "C" int dfw_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(n >= 0 && (n == 0 || (src && dst)), "dfw_cast: bad arguments");
    if (n == 0) return 0;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)kNumSMs * 8));
    if (src_dtype == DFW_F32 && dst_dtype == DFW_BF16)
        k_cast<float, __nv_bfloat16><<<blocks, 256, 0, s>>>((const float*)src, (__nv_bfloat16*)dst, n);
    else if (src_dtype == DFW_BF16 && dst_dtype == DFW_F32)
        k_cast<__nv_bfloat16, float><<<blocks, 256, 0, s>>>((const __nv_bfloat16*)src, (float*)dst, n);
    else if (src_dtype == DFW_F32 && dst_dtype == DFW_F32)
        k_cast<float, float><<<blocks, 256, 0, s>>>((const float*)src, (float*)dst, n);
    else if (src_dtype == DFW_BF16 && dst_dtype == DFW_BF16)
        k_cast<__nv_bfloat16, __nv_bfloat16><<<blocks, 256, 0, s>>>((const __nv_bfloat16*)src, (__nv_bfloat16*)dst, n);
    else {
        set_error("dfw_cast: unknown dtype pair %d -> %d", src_dtype, dst_dtype);
        return 1;
    }
    DFW_LAUNCH_CHECK();
    return 0;
}
