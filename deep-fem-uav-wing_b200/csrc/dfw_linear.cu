// (c)/(d) node-wise dense contractions of the GraphSAGE layer, SIMT-FP32 edition.
//
//   fwd : y = a1.w1^T (+ a2.w2^T) + bias ; out = residual + dropout(relu(layernorm(y)))
//         = SAGEConv's lin_l(mean) + lin_r(h) (PyG; reference call site model.py:90) with the
//           LayerNorm / ReLU / dropout / skip of model.py:91-95 fused into the epilogue, and the
//           encoder / decoder linears of model.py:52-57,67-72.
//   dx  : g_a = row_scale * (g_y . w) + addend
//   dw  : dW = g_y^T . a  (split over nodes, fixed-order second pass: no float atomics)
//
// One register-tiled kernel template serves the three contractions; only the tile loaders and
// the epilogue differ.  A CTA tile always spans the full output row (Hout <= 256), so the
// LayerNorm statistics are reduced inside the CTA with shuffles.  This is the exact-fp32
// path (FFMA); the tensor-core path lives in dfw_linear_tc.cu.
#include <algorithm>
#include <type_traits>

#include <cstdlib>

#include "dfw_common.cuh"
#include "dfw_linear_tc.cuh"

namespace dfw {
namespace {

bool force_simt() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DFW_FORCE_SIMT");
        v = (e && e[0] && e[0] != '0') ? 1 : 0;
    }
    return v == 1;
}

constexpr int BK = 16;
constexpr int PAD = 4;
constexpr int kThreads = 256;

enum Mode { MODE_FWD = 0, MODE_DX = 1, MODE_DW = 2 };

struct LinArgs {
    // operands (meaning depends on mode)
    const void* a1; const void* w1; int64_t k1;
    const void* a2; const void* w2; int64_t k2;
    const float* bias; const float* gamma; const float* beta; float eps;
    const void* residual; float dropout_p; uint32_t drop_thr; float drop_scale; uint64_t seed;
    void* out; void* pre_out; float* ln_stats;
    const float* rowdot_w; const float* rowdot_b; float* rowdot_out;
    const float* row_scale; const void* addend;
    int64_t N; int64_t Hout; int64_t K; int flags;
    // dW
    float* part; float* part_db; int splits; int64_t nodes_per_split; int tiles_i; int tiles_j1; int tiles_j2;
};

// ---- tile loaders --------------------------------------------------------------------------
// "Transposed" source: S[kk][idx] = M[idx_base+idx][k_base+kk]   (M row-major, leading dim ld)
template <typename T, int TILE>
struct TLoad {
    static constexpr int VE = 16 / sizeof(T);
    static constexpr int CH = BK / VE;
    static constexpr int ITEMS = TILE * CH;
    static constexpr int PER = (ITEMS + kThreads - 1) / kThreads;
    float r[PER][VE];
    __device__ __forceinline__ void load(const T* __restrict__ M, int64_t ld, int64_t idx_base, int64_t idx_lim,
                                         int64_t k_base, int64_t k_lim, bool vec_ok) {
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int item = threadIdx.x + p * kThreads;
            if (ITEMS % kThreads != 0 && item >= ITEMS) break;
            const int row = item / CH, ch = item % CH;
            const int64_t gi = idx_base + row, gk = k_base + ch * VE;
            if (gi < idx_lim && vec_ok && gk + VE <= k_lim) {
                Vec16<T> v;
                v.v = *reinterpret_cast<const decltype(v.v)*>(M + gi * ld + gk);
                v.to_float(r[p]);
            } else {
#pragma unroll
                for (int e = 0; e < VE; ++e)
                    r[p][e] = (gi < idx_lim && gk + e < k_lim) ? to_f32(M[gi * ld + gk + e]) : 0.f;
            }
        }
    }
    __device__ __forceinline__ void store(float* __restrict__ S) const {
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int item = threadIdx.x + p * kThreads;
            if (ITEMS % kThreads != 0 && item >= ITEMS) break;
            const int row = item / CH, ch = item % CH;
#pragma unroll
            for (int e = 0; e < VE; ++e) S[(ch * VE + e) * (TILE + PAD) + row] = r[p][e];
        }
    }
};

// "Direct" source: S[kk][idx] = M[k_base+kk][idx_base+idx]
template <typename T, int TILE>
struct DLoad {
    static constexpr int VE = 16 / sizeof(T);
    static constexpr int CH = TILE / VE;
    static constexpr int ITEMS = BK * CH;
    static constexpr int PER = (ITEMS + kThreads - 1) / kThreads;
    float r[PER][VE];
    __device__ __forceinline__ void load(const T* __restrict__ M, int64_t ld, int64_t idx_base, int64_t idx_lim,
                                         int64_t k_base, int64_t k_lim, bool vec_ok) {
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int item = threadIdx.x + p * kThreads;
            if (ITEMS % kThreads != 0 && item >= ITEMS) break;
            const int kk = item / CH, ch = item % CH;
            const int64_t gk = k_base + kk, gi = idx_base + ch * VE;
            if (gk < k_lim && vec_ok && gi + VE <= idx_lim) {
                Vec16<T> v;
                v.v = *reinterpret_cast<const decltype(v.v)*>(M + gk * ld + gi);
                v.to_float(r[p]);
            } else {
#pragma unroll
                for (int e = 0; e < VE; ++e)
                    r[p][e] = (gk < k_lim && gi + e < idx_lim) ? to_f32(M[gk * ld + gi + e]) : 0.f;
            }
        }
    }
    __device__ __forceinline__ void store(float* __restrict__ S) const {
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int item = threadIdx.x + p * kThreads;
            if (ITEMS % kThreads != 0 && item >= ITEMS) break;
            const int kk = item / CH, ch = item % CH;
            float* d = S + kk * (TILE + PAD) + ch * VE;
#pragma unroll
            for (int e = 0; e < VE; e += 4) *reinterpret_cast<float4*>(d + e) = make_float4(r[p][e], r[p][e + 1], r[p][e + 2], r[p][e + 3]);
        }
    }
};

template <int T_, int HALF>
__device__ __forceinline__ int tile_index(int t, int i) {
    // thread t owns T_ indices: [t*4, t*4+4) and, if T_==8, [HALF + t*4, HALF + t*4 + 4)
    return (i < 4) ? t * 4 + i : HALF + t * 4 + (i - 4);
}

template <typename T>
__device__ __forceinline__ void store_row4(T* __restrict__ base, int64_t row, int64_t ld, int c0, int64_t clim,
                                           const float* v, bool vec_ok) {
    if (vec_ok && c0 + 4 <= clim) {
        if constexpr (sizeof(T) == 4) {
            *reinterpret_cast<float4*>(base + row * ld + c0) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
            __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]);
            __nv_bfloat162 p1 = __floats2bfloat162_rn(v[2], v[3]);
            uint2 u = make_uint2(*reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1));
            *reinterpret_cast<uint2*>(base + row * ld + c0) = u;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (c0 + j < clim) base[row * ld + c0 + j] = from_f32<T>(v[j]);
    }
}

template <typename T>
__device__ __forceinline__ void load_row4(const T* __restrict__ base, int64_t row, int64_t ld, int c0, int64_t clim,
                                          float* v, bool vec_ok) {
    if (vec_ok && c0 + 4 <= clim) {
        if constexpr (sizeof(T) == 4) {
            float4 f = *reinterpret_cast<const float4*>(base + row * ld + c0);
            v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
        } else {
            uint2 u = *reinterpret_cast<const uint2*>(base + row * ld + c0);
            v[0] = __uint_as_float(u.x << 16); v[1] = __uint_as_float(u.x & 0xffff0000u);
            v[2] = __uint_as_float(u.y << 16); v[3] = __uint_as_float(u.y & 0xffff0000u);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (c0 + j < clim) ? to_f32(base[row * ld + c0 + j]) : 0.f;
    }
}

template <int TX>
__device__ __forceinline__ float row_group_sum(float v) {
#pragma unroll
    for (int o = TX / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- the kernel ----------------------------------------------------------------------------
template <typename T, int MODE, int BM, int BN, int TM, int TN>
__global__ void __launch_bounds__(kThreads) k_linear(const LinArgs p) {
    constexpr int TX = BN / TN, TY = BM / TM;
    static_assert(TX * TY == kThreads, "thread layout");
    static_assert(TX == 16 || TX == 32, "row reduction width");
    extern __shared__ __align__(16) float smem[];
    constexpr int A_STAGE = BK * (BM + PAD), B_STAGE = BK * (BN + PAD);
    float* const As0 = smem;
    float* const Bs0 = smem + 2 * A_STAGE;

    const int tx = threadIdx.x % TX, ty = threadIdx.x / TX;

    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    // ---- problem mapping ------------------------------------------------------------------
    // FWD: rows = nodes (M), cols = Hout, reduce over k1 then k2.   A: TLoad(a), B: TLoad(w)
    // DX : rows = nodes (M), cols = K (tile blockIdx.y), reduce over Hout.  A: TLoad(g_y), B: DLoad(w)
    // DW : rows = Hout (tile i), cols = K of a1 or a2 (tile j), reduce over a node range.
    //      A: DLoad(g_y), B: DLoad(a)
    int64_t m_base = 0, n_base = 0;
    int seg_count = 1;
    int tile_i = 0, tile_j = 0, split = 0, which = 0;
    int64_t red_begin = 0, red_end = 0;
    if (MODE == MODE_FWD) {
        m_base = (int64_t)blockIdx.x * BM;
        seg_count = p.a2 ? 2 : 1;
    } else if (MODE == MODE_DX) {
        m_base = (int64_t)blockIdx.x * BM;
        n_base = (int64_t)blockIdx.y * BN;
    } else {
        const int tiles_j = p.tiles_j1 + p.tiles_j2;
        const int tile = blockIdx.x;
        tile_i = tile / tiles_j;
        tile_j = tile % tiles_j;
        which = tile_j >= p.tiles_j1;
        if (which) tile_j -= p.tiles_j1;
        split = blockIdx.y;
        m_base = (int64_t)tile_i * BM;
        n_base = (int64_t)tile_j * BN;
        red_begin = (int64_t)split * p.nodes_per_split;
        red_end = min(p.N, red_begin + p.nodes_per_split);
    }

    float db_acc = 0.f;  // MODE_DW: column sum of g_y handled by thread (threadIdx.x < BM)

    for (int seg = 0; seg < seg_count; ++seg) {
        const T* Aop;
        const T* Bop;
        int64_t lda, ldb, a_idx_lim, b_idx_lim, k_begin, k_end;
        if (MODE == MODE_FWD) {
            Aop = (const T*)(seg == 0 ? p.a1 : p.a2);
            Bop = (const T*)(seg == 0 ? p.w1 : p.w2);
            const int64_t k = seg == 0 ? p.k1 : p.k2;
            lda = k; ldb = k; a_idx_lim = p.N; b_idx_lim = p.Hout; k_begin = 0; k_end = k;
        } else if (MODE == MODE_DX) {
            Aop = (const T*)p.a1;  // g_y [N,Hout]
            Bop = (const T*)p.w1;  // w [Hout,K]
            lda = p.Hout; ldb = p.K; a_idx_lim = p.N; b_idx_lim = p.K; k_begin = 0; k_end = p.Hout;
        } else {
            Aop = (const T*)p.a1;                      // g_y [N,Hout]
            Bop = (const T*)(which ? p.w2 : p.w1);     // a1 / a2 [N,k]
            lda = p.Hout; ldb = which ? p.k2 : p.k1; a_idx_lim = p.Hout; b_idx_lim = ldb;
            k_begin = red_begin; k_end = red_end;
        }
        const bool a_vec = (lda * sizeof(T)) % 16 == 0 && aligned16_dev(Aop);
        const bool b_vec = (ldb * sizeof(T)) % 16 == 0 && aligned16_dev(Bop);
        const int nsteps = (int)((k_end - k_begin + BK - 1) / BK);
        if (nsteps <= 0) continue;

        typename std::conditional<MODE == MODE_DW, DLoad<T, BM>, TLoad<T, BM>>::type la;
        typename std::conditional<MODE == MODE_FWD, TLoad<T, BN>, DLoad<T, BN>>::type lb;

        la.load(Aop, lda, m_base, a_idx_lim, k_begin, k_end, a_vec);
        lb.load(Bop, ldb, n_base, b_idx_lim, k_begin, k_end, b_vec);
        __syncthreads();  // previous segment's readers are done with buffer 0
        la.store(As0);
        lb.store(Bs0);
        __syncthreads();

        for (int t = 0; t < nsteps; ++t) {
            const int cur = t & 1;
            if (t + 1 < nsteps) {
                la.load(Aop, lda, m_base, a_idx_lim, k_begin + (int64_t)(t + 1) * BK, k_end, a_vec);
                lb.load(Bop, ldb, n_base, b_idx_lim, k_begin + (int64_t)(t + 1) * BK, k_end, b_vec);
            }
            const float* as = As0 + cur * A_STAGE;
            const float* bs = Bs0 + cur * B_STAGE;
#pragma unroll
            for (int kk = 0; kk < BK; ++kk) {
                float a[TM], b[TN];
                *reinterpret_cast<float4*>(a) = *reinterpret_cast<const float4*>(as + kk * (BM + PAD) + ty * 4);
                if (TM == 8) *reinterpret_cast<float4*>(a + 4) = *reinterpret_cast<const float4*>(as + kk * (BM + PAD) + BM / 2 + ty * 4);
                *reinterpret_cast<float4*>(b) = *reinterpret_cast<const float4*>(bs + kk * (BN + PAD) + tx * 4);
                if (TN == 8) *reinterpret_cast<float4*>(b + 4) = *reinterpret_cast<const float4*>(bs + kk * (BN + PAD) + BN / 2 + tx * 4);
#pragma unroll
                for (int i = 0; i < TM; ++i)
#pragma unroll
                    for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
            if (MODE == MODE_DW && p.part_db && tile_j == 0 && which == 0 && threadIdx.x < BM) {
#pragma unroll
                for (int kk = 0; kk < BK; ++kk) db_acc += as[kk * (BM + PAD) + threadIdx.x];
            }
            if (t + 1 < nsteps) {
                la.store(As0 + (cur ^ 1) * A_STAGE);
                lb.store(Bs0 + (cur ^ 1) * B_STAGE);
            }
            __syncthreads();
        }
    }

    // ---- epilogues ------------------------------------------------------------------------
    if (MODE == MODE_DW) {
        const int tiles = p.tiles_i * (p.tiles_j1 + p.tiles_j2);
        float* dst = p.part + ((int64_t)split * tiles + blockIdx.x) * (BM * BN);
#pragma unroll
        for (int i = 0; i < TM; ++i) {
            const int r = tile_index<TM, BM / 2>(ty, i);
#pragma unroll
            for (int jh = 0; jh < TN / 4; ++jh) {
                const int c = jh == 0 ? tx * 4 : BN / 2 + tx * 4;
                *reinterpret_cast<float4*>(dst + r * BN + c) =
                    make_float4(acc[i][jh * 4], acc[i][jh * 4 + 1], acc[i][jh * 4 + 2], acc[i][jh * 4 + 3]);
            }
        }
        if (p.part_db && tile_j == 0 && which == 0 && threadIdx.x < BM)
            p.part_db[((int64_t)split * p.tiles_i + tile_i) * BM + threadIdx.x] = db_acc;
        return;
    }

    const int64_t ncols = MODE == MODE_FWD ? p.Hout : p.K;
    const bool out_vec = ncols % 4 == 0;  // 16-byte (fp32) / 8-byte (bf16) aligned 4-element groups

    if (MODE == MODE_DX) {
        T* out = (T*)p.out;
        const T* addend = (const T*)p.addend;
#pragma unroll
        for (int i = 0; i < TM; ++i) {
            const int64_t r = m_base + tile_index<TM, BM / 2>(ty, i);
            if (r >= p.N) continue;
            const float sc = p.row_scale ? __ldg(p.row_scale + r) : 1.f;
#pragma unroll
            for (int jh = 0; jh < TN / 4; ++jh) {
                const int c = (int)n_base + (jh == 0 ? tx * 4 : BN / 2 + tx * 4);
                if (c >= ncols) continue;
                float v[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = acc[i][jh * 4 + j] * sc;
                if (addend) {
                    float ad[4];
                    load_row4(addend, r, ncols, c, ncols, ad, out_vec);
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] += ad[j];
                }
                store_row4(out, r, ncols, c, ncols, v, out_vec);
            }
        }
        return;
    }

    // MODE_FWD
    {
        const int64_t H = p.Hout;
        const float invH = 1.f / (float)H;
        T* out = (T*)p.out;
        T* pre = (T*)p.pre_out;
        const T* res = (const T*)p.residual;
        // per-thread column constants
        float bias[TN], gam[TN], bet[TN], rdw[TN];
        bool cok[TN];
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int c = tile_index<TN, BN / 2>(tx, j);
            cok[j] = c < H;
            bias[j] = (p.bias && cok[j]) ? __ldg(p.bias + c) : 0.f;
            gam[j] = (p.gamma && cok[j]) ? __ldg(p.gamma + c) : 1.f;
            bet[j] = (p.beta && cok[j]) ? __ldg(p.beta + c) : 0.f;
            rdw[j] = (p.rowdot_w && cok[j]) ? __ldg(p.rowdot_w + c) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < TM; ++i) {
            const int64_t r = m_base + tile_index<TM, BM / 2>(ty, i);
            const bool rok = r < p.N;  // no early exit: shuffles below need the whole row group
            float v[TN];
#pragma unroll
            for (int j = 0; j < TN; ++j) v[j] = cok[j] ? acc[i][j] + bias[j] : 0.f;
            if (pre && rok) {
#pragma unroll
                for (int jh = 0; jh < TN / 4; ++jh) {
                    const int c = jh == 0 ? tx * 4 : BN / 2 + tx * 4;
                    if (c < H) store_row4(pre, r, H, c, H, v + jh * 4, out_vec);
                }
            }
            if (p.flags & DFW_EP_LAYERNORM) {
                float s = 0.f;
#pragma unroll
                for (int j = 0; j < TN; ++j) s += v[j];
                const float mean = row_group_sum<TX>(s) * invH;
                float q = 0.f;
#pragma unroll
                for (int j = 0; j < TN; ++j) {
                    const float d = cok[j] ? v[j] - mean : 0.f;
                    q += d * d;
                }
                const float var = row_group_sum<TX>(q) * invH;
                const float rstd = rsqrtf(var + p.eps);
                if (p.ln_stats && rok && tx == 0) {
                    p.ln_stats[2 * r] = mean;
                    p.ln_stats[2 * r + 1] = rstd;
                }
#pragma unroll
                for (int j = 0; j < TN; ++j) v[j] = (v[j] - mean) * rstd * gam[j] + bet[j];
            }
            if (p.flags & DFW_EP_RELU) {
#pragma unroll
                for (int j = 0; j < TN; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            if (p.flags & DFW_EP_DROPOUT) {
#pragma unroll
                for (int j = 0; j < TN; ++j) {
                    const int c = tile_index<TN, BN / 2>(tx, j);
                    const uint32_t bits = dropout_bits(dropout_row_key(resolve_seed(p.seed, p.flags), (uint64_t)r), (uint32_t)c);
                    v[j] = bits >= p.drop_thr ? v[j] * p.drop_scale : 0.f;
                }
            }
            if (p.rowdot_out) {
                float s = 0.f;
#pragma unroll
                for (int j = 0; j < TN; ++j) s += cok[j] ? v[j] * rdw[j] : 0.f;
                s = row_group_sum<TX>(s);
                if (rok && tx == 0) p.rowdot_out[r] = s + (p.rowdot_b ? __ldg(p.rowdot_b) : 0.f);
            }
            if (out && rok) {
#pragma unroll
                for (int jh = 0; jh < TN / 4; ++jh) {
                    const int c = jh == 0 ? tx * 4 : BN / 2 + tx * 4;
                    if (c >= H) continue;
                    float w[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) w[j] = v[jh * 4 + j];
                    if (res) {
                        float rr[4];
                        load_row4(res, r, H, c, H, rr, out_vec);
#pragma unroll
                        for (int j = 0; j < 4; ++j) w[j] += rr[j];
                    }
                    store_row4(out, r, H, c, H, w, out_vec);
                }
            }
        }
    }
}

// second pass of dW: fixed-order sum over splits.  A block of 8 warps owns 32 consecutive outputs (one per lane, so
// every load is a coalesced 128-byte row segment of a partial tile); warp w sums splits w, w+8, w+16, ... and the
// eight partial sums are added in warp order.  (One thread per output walking all ~146 splits was a 15 us
// dependent-load chain for 19 MB of L2-resident partials.)
constexpr int kDwRedWarps = 8;
template <int BM, int BN>
__global__ void __launch_bounds__(kDwRedWarps * 32) k_dw_reduce(const float* __restrict__ part, const float* __restrict__ part_db, int splits,
                                                                int tiles_i, int tiles_j1, int tiles_j2, int64_t Hout, int64_t k1, int64_t k2,
                                                                float* __restrict__ dw1, float* __restrict__ dw2, float* __restrict__ dbias,
                                                                int accumulate) {
    __shared__ float red[kDwRedWarps][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t n1 = Hout * k1, n2 = Hout * k2;
    const int64_t total = n1 + n2 + (dbias ? Hout : 0);
    const int tiles = tiles_i * (tiles_j1 + tiles_j2);
    for (int64_t base = (int64_t)blockIdx.x * 32; base < total; base += (int64_t)gridDim.x * 32) {
        const int64_t idx = base + lane;
        float s = 0.f;
        float* dst = nullptr;
        if (idx < n1 + n2) {
            const bool second = idx >= n1;
            const int64_t e = second ? idx - n1 : idx;
            const int64_t k = second ? k2 : k1;
            const int64_t i = e / k, j = e % k;
            const int ti = (int)(i / BM), tj = (int)(j / BN) + (second ? tiles_j1 : 0);
            const int64_t off = (int64_t)(ti * (tiles_j1 + tiles_j2) + tj) * (BM * BN) + (i % BM) * BN + (j % BN);
            const int64_t st = (int64_t)tiles * (BM * BN);
            float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;  // four loads in flight, fixed association
            int sp = w;
            for (; sp + 3 * kDwRedWarps < splits; sp += 4 * kDwRedWarps) {
                q0 += part[(int64_t)sp * st + off];
                q1 += part[(int64_t)(sp + kDwRedWarps) * st + off];
                q2 += part[(int64_t)(sp + 2 * kDwRedWarps) * st + off];
                q3 += part[(int64_t)(sp + 3 * kDwRedWarps) * st + off];
            }
            for (; sp < splits; sp += kDwRedWarps) q0 += part[(int64_t)sp * st + off];
            s = (q0 + q1) + (q2 + q3);
            dst = (second ? dw2 : dw1) + e;
        } else if (idx < total) {
            const int64_t i = idx - n1 - n2;
            const int ti = (int)(i / BM);
            for (int sp = w; sp < splits; sp += kDwRedWarps) s += part_db[((int64_t)sp * tiles_i + ti) * BM + (i % BM)];
            dst = dbias + i;
        }
        red[w][lane] = s;
        __syncthreads();
        if (w == 0 && dst) {
            float t = red[0][lane];
#pragma unroll
            for (int k = 1; k < kDwRedWarps; ++k) t += red[k][lane];
            *dst = accumulate ? *dst + t : t;
        }
        __syncthreads();
    }
}

template <typename T, int MODE, int BM, int BN, int TM, int TN>
int launch_linear(const LinArgs& a, dim3 grid, cudaStream_t s) {
    constexpr size_t smem = sizeof(float) * 2 * BK * ((BM + PAD) + (BN + PAD));
    static_assert(smem <= 48 * 1024, "static-range shared memory");
    k_linear<T, MODE, BM, BN, TM, TN><<<grid, kThreads, smem, s>>>(a);
    DFW_LAUNCH_CHECK();
    return 0;
}

template <typename T, int MODE>
int dispatch_cols(const LinArgs& a, int64_t ncols_tile, dim3 grid64, dim3 grid128, dim3 grid256, cudaStream_t s) {
    if (ncols_tile <= 64) return launch_linear<T, MODE, 128, 64, 8, 4>(a, grid64, s);
    if (ncols_tile <= 128) return launch_linear<T, MODE, 128, 128, 8, 8>(a, grid128, s);
    return launch_linear<T, MODE, 64, 256, 8, 8>(a, grid256, s);
}

inline dim3 grid_rows(int64_t N, int BM, int64_t ytiles = 1) { return dim3((unsigned)((N + BM - 1) / BM), (unsigned)ytiles, 1); }

}  // namespace
}  // namespace dfw


// ---- tiny-K linears (the encoder's Linear(10, 64), model.py:53): pure streaming, no tiling needed ----------------
namespace dfw {
namespace {
constexpr int kSmallKMax = 16;

// partial dW[i, k] over the block's rows: thread = (output row i, k-slot), two-pass like the big kernels
// dW for a tiny reduction width K (the encoder's first layer, K = 10): dW[i, k] = sum_rows g[row, i] * x[row, k].
// A block owns a contiguous slice of rows; its 256 threads form 256/Hout row groups (thread = output feature i of
// one group), every thread keeps its K partial sums in registers and walks its group's rows four at a time (all
// loads of the four rows are issued before the FMAs), then the groups are summed in shared memory in a fixed order.
// (The first version used Hout threads per block and one row per iteration: a 338-deep dependent load chain on two
// warps per block - 250 us for a 60 MB read, 8 % of the training step.)
template <typename T>
__global__ void __launch_bounds__(256) k_linear_smallk_dw(const T* __restrict__ g, const T* __restrict__ x, float* __restrict__ part,
                                                           int64_t N, int K, int Hout) {
    extern __shared__ float s_red[];  // [groups][Hout * K]
    const int groups = 256 / Hout;    // Hout <= 256
    const int i = threadIdx.x % Hout, grp = threadIdx.x / Hout;
    const bool active = grp < groups;
    float acc[kSmallKMax];
#pragma unroll
    for (int k = 0; k < kSmallKMax; ++k) acc[k] = 0.f;
    const int64_t per = (N + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * per, r1 = min(N, r0 + per);
    if (active) {
        constexpr int U = 4;
        int64_t r = r0 + grp;
        for (; r + (int64_t)(U - 1) * groups < r1; r += (int64_t)U * groups) {
            float gv[U], xv[U][kSmallKMax];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t rr = r + (int64_t)u * groups;
                gv[u] = to_f32(g[rr * Hout + i]);
#pragma unroll
                for (int k = 0; k < kSmallKMax; ++k)
                    if (k < K) xv[u][k] = to_f32(x[rr * K + k]);
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int k = 0; k < kSmallKMax; ++k)
                    if (k < K) acc[k] = fmaf(gv[u], xv[u][k], acc[k]);
        }
        for (; r < r1; r += groups) {
            const float gv = to_f32(g[r * Hout + i]);
#pragma unroll
            for (int k = 0; k < kSmallKMax; ++k)
                if (k < K) acc[k] = fmaf(gv, to_f32(x[r * K + k]), acc[k]);
        }
#pragma unroll
        for (int k = 0; k < kSmallKMax; ++k)
            if (k < K) s_red[(grp * Hout + i) * K + k] = acc[k];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < Hout * K; e += 256) {
        float t = 0.f;
        for (int q = 0; q < groups; ++q) t += s_red[q * Hout * K + e];
        part[(int64_t)blockIdx.x * Hout * K + e] = t;
    }
}
// ---- tiled tiny-K kernels: x rows staged through shared memory ---------------------------------------------------
// The kernels above read the K <= 16 inputs of a row with K scalar loads per thread (two rows per warp instruction):
// 10-11 load instructions per 10-40 FMAs and a few KB in flight per SM - 47 us (forward) and 162 us (dW) for 59 MB
// passes.  Here a block stages a tile of kSmallTile rows of x with coalesced loads (zero-padded to KP columns), every
// thread owns four output features (one 16-byte vector of out / g) of kSmallTile / rows-per-pass rows of the tile and
// reads its rows' inputs as KP/4 broadcast LDS.128.
constexpr int kSmallTile = 128;

// The x tile of the NEXT iteration is fetched into registers before the current tile is worked on and written to the
// other shared-memory buffer afterwards: one barrier per tile, global latency under the arithmetic.
template <typename T, int KP>
struct SmallKStage {
    static constexpr int XR = (kSmallTile * KP + 255) / 256;  // staged elements per thread
    float xr[XR];
    __device__ __forceinline__ void fetch(const T* __restrict__ x, int64_t t0, int nr, int K) {
        const int n = nr * K;
        const T* src = x + t0 * K;
#pragma unroll
        for (int i = 0; i < XR; ++i) {
            const int e = threadIdx.x + i * 256;
            xr[i] = e < n ? to_f32(src[e]) : 0.f;
        }
    }
    __device__ __forceinline__ void commit(float* xs, int nr, int K) const {
        const int n = nr * K;
#pragma unroll
        for (int i = 0; i < XR; ++i) {
            const int e = threadIdx.x + i * 256;
            if (e < n) {
                const int r = e / K, k = e - r * K;
                xs[r * KP + k] = xr[i];
            }
        }
    }
};

template <typename T, int KP, typename TO = T>
__global__ void __launch_bounds__(256, 3) k_smallk_fwd_tiled(const T* __restrict__ x, const T* __restrict__ w, const float* __restrict__ bias,
                                                              TO* __restrict__ out, int64_t N, int K, int Hout, int relu) {
    __shared__ __align__(16) float xs[2][kSmallTile * KP];
    const int fq = Hout / 4;      // threads per row (<= 256)
    const int rpi = 256 / fq;     // rows per pass
    const int cq = threadIdx.x % fq, rl = threadIdx.x / fq;
    const bool active = rl < rpi;
    float wr[4][KP], b4[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        b4[j] = bias ? __ldg(bias + cq * 4 + j) : 0.f;
#pragma unroll
        for (int k = 0; k < KP; ++k) wr[j][k] = k < K ? to_f32(w[(int64_t)(cq * 4 + j) * K + k]) : 0.f;
    }
    for (int e = threadIdx.x; e < 2 * kSmallTile * KP; e += 256) (&xs[0][0])[e] = 0.f;  // the padding columns stay zero
    const int64_t stride = (int64_t)gridDim.x * kSmallTile;
    int64_t t0 = (int64_t)blockIdx.x * kSmallTile;
    SmallKStage<T, KP> st;
    int buf = 0;
    if (t0 < N) st.fetch(x, t0, (int)min((int64_t)kSmallTile, N - t0), K);
    __syncthreads();
    if (t0 < N) st.commit(xs[0], (int)min((int64_t)kSmallTile, N - t0), K);
    __syncthreads();
    for (; t0 < N; t0 += stride, buf ^= 1) {
        const int nr = (int)min((int64_t)kSmallTile, N - t0);
        const int64_t t1 = t0 + stride;
        const int nr1 = t1 < N ? (int)min((int64_t)kSmallTile, N - t1) : 0;
        if (nr1) st.fetch(x, t1, nr1, K);
        if (active) {
            const float* xt = xs[buf];
            for (int r = rl; r < nr; r += rpi) {
                float xv[KP];
#pragma unroll
                for (int k4 = 0; k4 < KP / 4; ++k4) {
                    const float4 f = *reinterpret_cast<const float4*>(xt + r * KP + k4 * 4);
                    xv[k4 * 4] = f.x; xv[k4 * 4 + 1] = f.y; xv[k4 * 4 + 2] = f.z; xv[k4 * 4 + 3] = f.w;
                }
                float o[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float a = b4[j];
#pragma unroll
                    for (int k = 0; k < KP; ++k) a = fmaf(xv[k], wr[j][k], a);
                    o[j] = relu ? fmaxf(a, 0.f) : a;
                }
                store_row4(out, t0 + r, (int64_t)Hout, cq * 4, (int64_t)Hout, o, true);
            }
        }
        if (nr1) st.commit(xs[buf ^ 1], nr1, K);
        __syncthreads();
    }
}

// part[block][i * K + k] = sum over the block's tiles of g[row, i] * x[row, k]; fixed tile -> block assignment and a
// fixed-order reduction over the row lanes: bit-reproducible.  Reduced over blocks by k_smallk_dw_reduce.
template <typename T, int KP>
__global__ void __launch_bounds__(256, 2) k_smallk_dw_tiled(const T* __restrict__ g, const T* __restrict__ x, float* __restrict__ part,
                                                             int64_t N, int K, int Hout) {
    __shared__ __align__(16) float xs[2][kSmallTile * KP];
    __shared__ float s_red[256 * KP];
    const int fq = Hout / 4;      // threads per row (Hout <= 256: <= 64)
    const int rpi = 256 / fq;     // row lanes (>= 4)
    const int cq = threadIdx.x % fq, rl = threadIdx.x / fq;
    const bool active = rl < rpi;
    float acc[4][KP];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < KP; ++k) acc[j][k] = 0.f;
    for (int e = threadIdx.x; e < 2 * kSmallTile * KP; e += 256) (&xs[0][0])[e] = 0.f;
    const int64_t stride = (int64_t)gridDim.x * kSmallTile;
    int64_t t0 = (int64_t)blockIdx.x * kSmallTile;
    SmallKStage<T, KP> st;
    int buf = 0;
    if (t0 < N) st.fetch(x, t0, (int)min((int64_t)kSmallTile, N - t0), K);
    __syncthreads();
    if (t0 < N) st.commit(xs[0], (int)min((int64_t)kSmallTile, N - t0), K);
    __syncthreads();
    for (; t0 < N; t0 += stride, buf ^= 1) {
        const int nr = (int)min((int64_t)kSmallTile, N - t0);
        const int64_t t1 = t0 + stride;
        const int nr1 = t1 < N ? (int)min((int64_t)kSmallTile, N - t1) : 0;
        if (nr1) st.fetch(x, t1, nr1, K);
        if (active) {
            const float* xt = xs[buf];
            constexpr int U = 8;  // rows of g in flight per thread
            for (int r = rl; r < nr; r += U * rpi) {
                float gv[U][4];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int rr = r + u * rpi;
                    if (rr < nr) {
                        load_row4(g, t0 + rr, (int64_t)Hout, cq * 4, (int64_t)Hout, gv[u], true);
                    } else {
                        gv[u][0] = gv[u][1] = gv[u][2] = gv[u][3] = 0.f;
                    }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int rr = min(r + u * rpi, nr - 1);  // rows past the tile carry g = 0
#pragma unroll
                    for (int k4 = 0; k4 < KP / 4; ++k4) {
                        const float4 f = *reinterpret_cast<const float4*>(xt + rr * KP + k4 * 4);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            acc[j][k4 * 4] = fmaf(gv[u][j], f.x, acc[j][k4 * 4]);
                            acc[j][k4 * 4 + 1] = fmaf(gv[u][j], f.y, acc[j][k4 * 4 + 1]);
                            acc[j][k4 * 4 + 2] = fmaf(gv[u][j], f.z, acc[j][k4 * 4 + 2]);
                            acc[j][k4 * 4 + 3] = fmaf(gv[u][j], f.w, acc[j][k4 * 4 + 3]);
                        }
                    }
                }
            }
        }
        if (nr1) st.commit(xs[buf ^ 1], nr1, K);
        __syncthreads();
    }
    // sum the row lanes, one of the four features per round (keeps the scratch at 256 * KP floats)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (active) {
#pragma unroll
            for (int k = 0; k < KP; ++k) s_red[(rl * fq + cq) * KP + k] = acc[j][k];
        }
        __syncthreads();
        for (int e = threadIdx.x; e < fq * KP; e += 256) {
            const int c = e / KP, k = e - c * KP;
            if (k < K) {
                float t = 0.f;
                for (int q = 0; q < rpi; ++q) t += s_red[(q * fq + c) * KP + k];
                part[(int64_t)blockIdx.x * Hout * K + (int64_t)(c * 4 + j) * K + k] = t;
            }
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) k_smallk_dw_reduce(const float* __restrict__ part, int blocks, int total, float* __restrict__ dw,
                                                           int accumulate) {
    const int lane = threadIdx.x & 31;
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // warp per output element, lanes stride over the partials
    if (e >= total) return;
    float s = 0.f;
    for (int b = lane; b < blocks; b += 32) s += part[(int64_t)b * total + e];
    s = warp_sum(s);
    if (lane == 0) dw[e] = accumulate ? dw[e] + s : s;
}
}  // namespace
}  // namespace dfw

extern "C" int dfw_linear_tc_eligible(int64_t N, int64_t Hout, int64_t k1, int64_t k2, int dtype) {
    // alignment of the operands is the caller's side of the contract (16-byte aligned rows): checked again at launch
    return (!dfw::force_simt() && dfw::linear_tc_eligible(N, Hout, k1, k2, dtype, nullptr, k2 > 0 ? reinterpret_cast<const void*>(16) : nullptr)) ? 1 : 0;
}

extern "C" int dfw_linear_fwd(const void* a1, const void* w1, int64_t k1, const void* a2, const void* w2, int64_t k2,
                              const float* bias, const float* ln_gamma, const float* ln_beta, float ln_eps,
                              const void* residual, float dropout_p, uint64_t seed, void* out, void* pre_out,
                              float* ln_stats, const float* rowdot_w, const float* rowdot_b, float* rowdot_out, int64_t N,
                              int64_t Hout, int flags, int dtype, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_linear_fwd: unknown dtype %d", dtype);
    DFW_REQUIRE(N >= 0 && Hout >= 1 && Hout <= 256, "dfw_linear_fwd: Hout=%lld must be in [1,256] (N=%lld)",
                (long long)Hout, (long long)N);
    DFW_REQUIRE(a1 && w1 && k1 >= 1, "dfw_linear_fwd: a1/w1 required");
    DFW_REQUIRE((a2 == nullptr) == (w2 == nullptr), "dfw_linear_fwd: a2 and w2 go together");
    DFW_REQUIRE(!a2 || k2 >= 1, "dfw_linear_fwd: k2 must be >= 1 with a2");
    DFW_REQUIRE(out || rowdot_out, "dfw_linear_fwd: no output requested");
    DFW_REQUIRE(!(flags & DFW_EP_RESIDUAL) || residual, "dfw_linear_fwd: DFW_EP_RESIDUAL without residual");
    DFW_REQUIRE((rowdot_w == nullptr) == (rowdot_out == nullptr), "dfw_linear_fwd: rowdot_w and rowdot_out go together");
    DFW_REQUIRE(!(flags & DFW_EP_DROPOUT) || (dropout_p >= 0.f && dropout_p < 1.f), "dfw_linear_fwd: dropout_p=%f not in [0,1)",
                (double)dropout_p);
    if (N == 0) return 0;
    if ((flags & DFW_EP_DROPOUT) && dropout_p == 0.f) flags &= ~DFW_EP_DROPOUT;
    DFW_REQUIRE(!(flags & DFW_EP_LAYERNORM) || (ln_gamma && ln_beta), "dfw_linear_fwd: DFW_EP_LAYERNORM needs gamma and beta");
    if (!(flags & DFW_EP_OUT_BF16) && ws && !force_simt() && linear_tc_eligible(N, Hout, k1, a2 ? k2 : 0, dtype, a1, a2) &&
        ws_bytes >= linear_tc_ws_bytes(Hout, k1, a2 ? k2 : 0, dtype) && aligned16(out ? out : a1) &&
        (!pre_out || aligned16(pre_out)) && (!residual || aligned16(residual))) {
        tc::Args t{};
        t.N = N; t.Hout = (int)Hout; t.flags = flags;
        t.bias = bias; t.gamma = ln_gamma; t.beta = ln_beta; t.eps = ln_eps; t.row_scale = nullptr;
        t.residual = (flags & DFW_EP_RESIDUAL) ? residual : nullptr;
        t.drop_thr = dropout_threshold(dropout_p); t.drop_scale = 1.f / (1.f - dropout_p); t.seed = seed;
        t.out = out; t.pre_out = pre_out; t.ln_stats = ln_stats;
        t.rowdot_w = rowdot_w; t.rowdot_b = rowdot_b; t.rowdot_out = rowdot_out;
        return linear_tc_launch(a1, w1, k1, a2, w2, k2, (flags & DFW_EP_TRANSPOSE_W) ? 1 : 0, t, dtype, ws, ws_bytes,
                                reinterpret_cast<cudaStream_t>(stream));
    }
    DFW_REQUIRE(!(flags & DFW_EP_TRANSPOSE_W), "dfw_linear_fwd: DFW_EP_TRANSPOSE_W needs a tensor-core eligible shape "
                "(ask dfw_linear_tc_eligible first)");
    const bool out_bf16 = flags & DFW_EP_OUT_BF16;
    flags &= ~DFW_EP_OUT_BF16;
    DFW_REQUIRE(!out_bf16 || (dtype == DFW_F32 && !a2 && k1 <= kSmallKMax && Hout % 4 == 0 && out && !pre_out && !rowdot_out &&
                              !(flags & ~DFW_EP_RELU) && aligned16(out) && !force_simt()),
                "dfw_linear_fwd: DFW_EP_OUT_BF16 is the tiny-K fp32 linear only (single operand, k1 <= %d, Hout %% 4 == 0, ReLU at most)", kSmallKMax);
    if (!force_simt() && !a2 && k1 <= kSmallKMax && Hout % 4 == 0 && Hout <= 1024 && out && !pre_out && !rowdot_out &&
        !(flags & ~DFW_EP_RELU) && aligned16(out)) {
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        const int64_t tiles = (N + kSmallTile - 1) / kSmallTile;
        const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(tiles, (int64_t)kNumSMs * 3));  // 3 resident blocks per SM
#define DFW_SK_FWD(TT, KPV)                                                                                              \
    k_smallk_fwd_tiled<TT, KPV><<<blocks, 256, 0, st>>>((const TT*)a1, (const TT*)w1, bias, (TT*)out, N, (int)k1, (int)Hout, \
                                                   flags & DFW_EP_RELU)
#define DFW_SK_FWD_K(TT)                                                                                                 \
    do {                                                                                                                 \
    if (k1 <= 4) DFW_SK_FWD(TT, 4); else if (k1 <= 8) DFW_SK_FWD(TT, 8); else if (k1 <= 12) DFW_SK_FWD(TT, 12);       \
    else DFW_SK_FWD(TT, 16);                                                                                         \
    } while (0)
        if (out_bf16) {
#define DFW_SK_FWD_MIX(KPV) \
    k_smallk_fwd_tiled<float, KPV, __nv_bfloat16><<<blocks, 256, 0, st>>>((const float*)a1, (const float*)w1, bias, (__nv_bfloat16*)out, N, (int)k1, \
                                                                           (int)Hout, flags & DFW_EP_RELU)
            if (k1 <= 4) DFW_SK_FWD_MIX(4); else if (k1 <= 8) DFW_SK_FWD_MIX(8); else if (k1 <= 12) DFW_SK_FWD_MIX(12); else DFW_SK_FWD_MIX(16);
#undef DFW_SK_FWD_MIX
        } else if (dtype == DFW_F32) DFW_SK_FWD_K(float); else DFW_SK_FWD_K(__nv_bfloat16);
#undef DFW_SK_FWD_K
#undef DFW_SK_FWD
        DFW_LAUNCH_CHECK();
        return 0;
    }
    LinArgs a{};
    a.a1 = a1; a.w1 = w1; a.k1 = k1; a.a2 = a2; a.w2 = w2; a.k2 = a2 ? k2 : 0;
    a.bias = bias; a.gamma = ln_gamma; a.beta = ln_beta; a.eps = ln_eps;
    a.residual = (flags & DFW_EP_RESIDUAL) ? residual : nullptr;
    a.dropout_p = dropout_p; a.drop_thr = dropout_threshold(dropout_p); a.drop_scale = 1.f / (1.f - dropout_p); a.seed = seed;
    a.out = out; a.pre_out = pre_out; a.ln_stats = ln_stats;
    a.rowdot_w = rowdot_w; a.rowdot_b = rowdot_b; a.rowdot_out = rowdot_out;
    a.N = N; a.Hout = Hout; a.flags = flags;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (dtype == DFW_F32)
        return dispatch_cols<float, MODE_FWD>(a, Hout, grid_rows(N, 128), grid_rows(N, 128), grid_rows(N, 64), s);
    return dispatch_cols<__nv_bfloat16, MODE_FWD>(a, Hout, grid_rows(N, 128), grid_rows(N, 128), grid_rows(N, 64), s);
}

extern "C" size_t dfw_linear_ws_bytes(int64_t Hout, int64_t k1, int64_t k2, int dtype) {
    if (Hout < 1 || k1 < 1 || k2 < 0) return 0;
    return dfw::linear_tc_ws_bytes(Hout, k1, k2, dtype);
}

extern "C" int dfw_linear_bwd_input(const void* g_y, const void* w, const float* row_scale, const void* addend,
                                    void* g_a, int64_t N, int64_t Hout, int64_t K, int dtype, void* ws, size_t ws_bytes,
                                    dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_linear_bwd_input: unknown dtype %d", dtype);
    DFW_REQUIRE(N >= 0 && Hout >= 1 && K >= 1, "dfw_linear_bwd_input: bad shape");
    DFW_REQUIRE(g_y && w && g_a, "dfw_linear_bwd_input: null pointer");
    if (N == 0) return 0;
    if (ws && !force_simt() && linear_tc_eligible(N, K, Hout, 0, dtype, g_y, nullptr) &&
        ws_bytes >= linear_tc_ws_bytes(K, Hout, 0, dtype) && aligned16(g_a) && (!addend || aligned16(addend))) {
        tc::Args t{};
        t.N = N; t.Hout = (int)K; t.flags = addend ? DFW_EP_RESIDUAL : 0;
        t.row_scale = row_scale; t.residual = addend; t.drop_scale = 1.f; t.out = g_a;
        return linear_tc_launch(g_y, w, Hout, nullptr, nullptr, 0, 1, t, dtype, ws, ws_bytes, reinterpret_cast<cudaStream_t>(stream));
    }
    LinArgs a{};
    a.a1 = g_y; a.w1 = w; a.row_scale = row_scale; a.addend = addend; a.out = g_a;
    a.N = N; a.Hout = Hout; a.K = K;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int64_t tile = K <= 64 ? 64 : (K <= 128 ? 128 : 256);
    const int64_t yt = (K + tile - 1) / tile;
    if (dtype == DFW_F32)
        return dispatch_cols<float, MODE_DX>(a, tile, grid_rows(N, 128, yt), grid_rows(N, 128, yt), grid_rows(N, 64, yt), s);
    return dispatch_cols<__nv_bfloat16, MODE_DX>(a, tile, grid_rows(N, 128, yt), grid_rows(N, 128, yt), grid_rows(N, 64, yt), s);
}

namespace dfw {
namespace {
struct DwPlan {
    int tiles_i, tiles_j1, tiles_j2, splits;
    int64_t nodes_per_split;
    size_t part_bytes, db_bytes;
};
constexpr int DW_BM = 128, DW_BN = 128;
DwPlan dw_plan(int64_t N, int64_t Hout, int64_t k1, int64_t k2) {
    DwPlan p;
    p.tiles_i = (int)((Hout + DW_BM - 1) / DW_BM);
    p.tiles_j1 = (int)((k1 + DW_BN - 1) / DW_BN);
    p.tiles_j2 = (int)((k2 + DW_BN - 1) / DW_BN);
    const int tiles = p.tiles_i * (p.tiles_j1 + p.tiles_j2);
    int64_t want = (2 * kNumSMs + tiles - 1) / tiles;
    int64_t max_splits = std::max<int64_t>(1, (N + 4 * BK - 1) / (4 * BK));
    int64_t splits = std::max<int64_t>(1, std::min(want, max_splits));
    int64_t per = (N + splits - 1) / splits;
    per = std::max<int64_t>(BK, (per + BK - 1) / BK * BK);  // N = 0 would give per = 0 and a division by zero below
    splits = std::max<int64_t>(1, (N + per - 1) / per);
    p.splits = (int)splits;
    p.nodes_per_split = per;
    p.part_bytes = align_up(sizeof(float) * (size_t)splits * tiles * DW_BM * DW_BN, 256);
    p.db_bytes = align_up(sizeof(float) * (size_t)splits * p.tiles_i * DW_BM, 256);
    return p;
}
// tensor-core variant: one CTA per [128 x 128] tile and node slice, ~one CTA per SM in total
DwPlan dw_plan_tc(int64_t N, int64_t Hout, int64_t k1, int64_t k2) {
    DwPlan p;
    p.tiles_i = (int)((Hout + 127) / 128);
    p.tiles_j1 = (int)((k1 + 127) / 128);
    p.tiles_j2 = (int)((k2 + 127) / 128);
    const int tiles = std::max(1, p.tiles_i * (p.tiles_j1 + p.tiles_j2));
    // ~2 CTAs per SM in total: short node slices keep the number of tensor-core accumulations per partial tile
    // small (their truncation bias grows linearly with it: 3.2e-6 -> ~1.6e-6 relative at 200k nodes, 0.9e-6 with 4 per SM)
    int64_t splits = std::max<int64_t>(1, 2 * kNumSMs / tiles);
    int64_t per = (N + splits - 1) / splits;
    per = std::max<int64_t>(32, (per + 31) / 32 * 32);
    splits = std::max<int64_t>(1, (N + per - 1) / per);
    p.splits = (int)splits;
    p.nodes_per_split = per;
    p.part_bytes = align_up(sizeof(float) * (size_t)splits * tiles * 128 * 128, 256);
    p.db_bytes = colsum_ws_bytes(Hout);
    return p;
}
}  // namespace
}  // namespace dfw

extern "C" size_t dfw_linear_bwd_weight_ws_bytes(int64_t N, int64_t Hout, int64_t k1, int64_t k2) {
    if (N < 0 || Hout < 1 || k1 < 1 || k2 < 0) return 0;
    dfw::DwPlan p = dfw::dw_plan(N, Hout, k1, k2);
    size_t need = p.part_bytes + p.db_bytes;
    if (Hout % 32 == 0 && k1 % 32 == 0 && k2 % 32 == 0) {
        dfw::DwPlan t = dfw::dw_plan_tc(N, Hout, k1, k2);
        need = std::max(need, t.part_bytes + t.db_bytes);
    }
    return need;
}

extern "C" int dfw_linear_bwd_weight(const void* g_y, const void* a1, int64_t k1, const void* a2, int64_t k2,
                                     float* dw1, float* dw2, float* dbias, int64_t N, int64_t Hout, int dtype,
                                     int accumulate, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_linear_bwd_weight: unknown dtype %d", dtype);
    DFW_REQUIRE(N >= 0 && Hout >= 1 && k1 >= 1, "dfw_linear_bwd_weight: bad shape");
    DFW_REQUIRE(g_y && a1 && dw1, "dfw_linear_bwd_weight: null pointer");
    DFW_REQUIRE((a2 == nullptr) == (dw2 == nullptr), "dfw_linear_bwd_weight: a2 and dw2 go together");
    if (!a2) k2 = 0;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (N > 0 && !force_simt() && dw_tc_eligible(N, Hout, k1, k2, dtype, g_y, a1, a2)) {
        DwPlan pt = dw_plan_tc(N, Hout, k1, k2);
        DFW_REQUIRE(ws && ws_bytes >= pt.part_bytes + pt.db_bytes, "dfw_linear_bwd_weight: workspace too small (%zu < %zu)",
                    ws_bytes, pt.part_bytes + pt.db_bytes);
        float* part = reinterpret_cast<float*>(ws);
        float* part_db = dbias ? reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + pt.part_bytes) : nullptr;
        int rc = dw_tc_launch(g_y, a1, k1, a2, k2, N, Hout, dtype, part, pt.splits, pt.nodes_per_split, s);
        if (rc) return rc;
        if (dbias && (rc = colsum_launch(g_y, N, Hout, dtype, part_db, dbias, accumulate, s))) return rc;
        const int64_t total = Hout * (k1 + k2);
        const int rgrid = (int)std::min<int64_t>((total + 31) / 32, (int64_t)kNumSMs * 8);
        k_dw_reduce<128, 128><<<rgrid, kDwRedWarps * 32, 0, s>>>(part, nullptr, pt.splits, pt.tiles_i, pt.tiles_j1, pt.tiles_j2, Hout, k1, k2, dw1,
                                                    dw2, nullptr, accumulate);
        DFW_LAUNCH_CHECK();
        return 0;
    }
    if (N > 0 && !force_simt() && !a2 && !dbias && k1 <= kSmallKMax && Hout <= 256) {
        int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((N + 255) / 256, (int64_t)kNumSMs * 4));
        const size_t need = sizeof(float) * (size_t)blocks * Hout * k1;
        if (ws && ws_bytes >= need && Hout % 4 == 0 && aligned16(g_y)) {
            blocks = (int)std::max<int64_t>(1, std::min<int64_t>((N + kSmallTile - 1) / kSmallTile, (int64_t)kNumSMs * 2));  // 2 resident blocks per SM
            float* part = reinterpret_cast<float*>(ws);
#define DFW_SK_DW(TT, KPV) k_smallk_dw_tiled<TT, KPV><<<blocks, 256, 0, s>>>((const TT*)g_y, (const TT*)a1, part, N, (int)k1, (int)Hout)
#define DFW_SK_DW_K(TT)                                                                                                 \
    do {                                                                                                                \
        if (k1 <= 4) DFW_SK_DW(TT, 4); else if (k1 <= 8) DFW_SK_DW(TT, 8); else if (k1 <= 12) DFW_SK_DW(TT, 12);         \
        else DFW_SK_DW(TT, 16);                                                                                         \
    } while (0)
            if (dtype == DFW_F32) DFW_SK_DW_K(float); else DFW_SK_DW_K(__nv_bfloat16);
#undef DFW_SK_DW_K
#undef DFW_SK_DW
            DFW_LAUNCH_CHECK();
            const int total = (int)(Hout * k1);
            k_smallk_dw_reduce<<<(total * 32 + 255) / 256, 256, 0, s>>>(part, blocks, total, dw1, accumulate);
            DFW_LAUNCH_CHECK();
            return 0;
        }
        if (ws && ws_bytes >= need) {
            float* part = reinterpret_cast<float*>(ws);
            const size_t red_bytes = sizeof(float) * (size_t)(256 / Hout) * Hout * k1;  // <= 16 KB
            if (dtype == DFW_F32) k_linear_smallk_dw<float><<<blocks, 256, red_bytes, s>>>((const float*)g_y, (const float*)a1, part, N, (int)k1, (int)Hout);
            else k_linear_smallk_dw<__nv_bfloat16><<<blocks, 256, red_bytes, s>>>((const __nv_bfloat16*)g_y, (const __nv_bfloat16*)a1, part, N, (int)k1, (int)Hout);
            DFW_LAUNCH_CHECK();
            const int total = (int)(Hout * k1);
            k_smallk_dw_reduce<<<(total * 32 + 255) / 256, 256, 0, s>>>(part, blocks, total, dw1, accumulate);
            DFW_LAUNCH_CHECK();
            return 0;
        }
    }
    DwPlan pl = dw_plan(N, Hout, k1, k2);
    DFW_REQUIRE(ws && ws_bytes >= pl.part_bytes + pl.db_bytes, "dfw_linear_bwd_weight: workspace too small (%zu < %zu)",
                ws_bytes, pl.part_bytes + pl.db_bytes);
    LinArgs a{};
    a.a1 = g_y; a.w1 = a1; a.w2 = a2; a.k1 = k1; a.k2 = k2; a.N = N; a.Hout = Hout;
    a.part = reinterpret_cast<float*>(ws);
    a.part_db = dbias ? reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + pl.part_bytes) : nullptr;
    a.splits = pl.splits; a.nodes_per_split = pl.nodes_per_split;
    a.tiles_i = pl.tiles_i; a.tiles_j1 = pl.tiles_j1; a.tiles_j2 = pl.tiles_j2;
    const int tiles = pl.tiles_i * (pl.tiles_j1 + pl.tiles_j2);
    dim3 grid((unsigned)tiles, (unsigned)pl.splits, 1);
    int rc;
    if (N == 0) {
        // nothing to reduce: the second pass writes zeros (or leaves dW untouched when accumulating)
        a.splits = 0;
        rc = 0;
    } else if (dtype == DFW_F32) {
        rc = launch_linear<float, MODE_DW, DW_BM, DW_BN, 8, 8>(a, grid, s);
    } else {
        rc = launch_linear<__nv_bfloat16, MODE_DW, DW_BM, DW_BN, 8, 8>(a, grid, s);
    }
    if (rc) return rc;
    const int64_t total = Hout * (k1 + k2) + (dbias ? Hout : 0);
    const int rgrid = (int)std::min<int64_t>((total + 31) / 32, (int64_t)kNumSMs * 8);
    k_dw_reduce<DW_BM, DW_BN><<<rgrid, kDwRedWarps * 32, 0, s>>>(a.part, a.part_db, a.splits, pl.tiles_i, pl.tiles_j1, pl.tiles_j2, Hout,
                                                    k1, k2, dw1, dw2, dbias, accumulate);
    DFW_LAUNCH_CHECK();
    return 0;
}
