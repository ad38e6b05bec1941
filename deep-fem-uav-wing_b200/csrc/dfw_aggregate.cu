// (b) deterministic segmented neighbour aggregation over a CSR (no atomics).
//
// Replaces PyG's  x.index_select(0, src) -> zeros.scatter_add_(0, dst, .) -> / clamp(count,1)
// behind SAGEConv(aggr='mean') (reference call site src/deep_fem_uav_wing/gnn/model.py:90),
// and - with the transposed CSR and row_scale = NULL - the backward of that mean.
//
// Design ("row-block edge streaming"):
//  * a group of LANES lanes (a full warp for 512-byte rows) owns a block of R consecutive destination
//    rows and STREAMS the block's contiguous edge range: column indices are fetched LANES at a time
//    (coalesced, L1-bypassing) and broadcast by shuffle; the source rows of U = 8 edges are requested
//    back to back (8 x 512 B in flight per warp whatever the degree) before any of them is consumed;
//  * row boundaries are group-uniform branches inside the stream, so short rows (degree ~6 surface
//    meshes) cost no extra dependent round trip: rowptr and col are each read once per block;
//  * every lane moves 16-byte vectors; fp32 accumulation in CSR order (bit-reproducible) using packed
//    FADD2 for fp32 rows and FHADD.BF16 (f32 += bf16, no unpack) for bf16 rows - the bf16 config is
//    instruction-issue bound, not bandwidth bound, on a naive kernel (profiles/r01_ncu_*_v1.csv).
// Roofline: HBM.  Algorithmic bytes per launch  A_min = 2*N*H*b + 4*E + 4*(N+1)  (DESIGN.md).
#include <algorithm>

#include "dfw_common.cuh"

namespace dfw {
namespace {


__device__ __forceinline__ uint4 ldg_nc_v4(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ int ldg_stream_s32(const int* p) {
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

__device__ __forceinline__ void stg_v4(void* p, const uint4& v) {
    asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// acc (fp32) += one 16-byte vector of T
template <typename T>
struct Acc;
template <>
struct Acc<float> {
    static constexpr int N = 4;
    uint64_t a[2];  // two packed f32x2
    __device__ __forceinline__ void zero() { a[0] = a[1] = 0ull; }
    __device__ __forceinline__ void add(const uint4& v) {
        uint64_t lo = ((uint64_t)v.y << 32) | v.x, hi = ((uint64_t)v.w << 32) | v.z;
        asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a[0]) : "l"(lo));
        asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a[1]) : "l"(hi));
    }
    __device__ __forceinline__ void fma(const uint4& v, float s) {  // acc += s * v (packed FFMA2)
        const uint64_t lo = ((uint64_t)v.y << 32) | v.x, hi = ((uint64_t)v.w << 32) | v.z;
        const uint64_t ss = ((uint64_t)__float_as_uint(s) << 32) | __float_as_uint(s);
        asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a[0]) : "l"(lo), "l"(ss));
        asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a[1]) : "l"(hi), "l"(ss));
    }
    __device__ __forceinline__ void get(float* f) const {
        f[0] = __uint_as_float((uint32_t)a[0]); f[1] = __uint_as_float((uint32_t)(a[0] >> 32));
        f[2] = __uint_as_float((uint32_t)a[1]); f[3] = __uint_as_float((uint32_t)(a[1] >> 32));
    }
};
template <>
struct Acc<__nv_bfloat16> {
    static constexpr int N = 8;
    float a[8];
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = 0.f;
    }
    __device__ __forceinline__ void add(const uint4& v) {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            unsigned short lo, hi;
            asm("mov.b32 {%0, %1}, %2;" : "=h"(lo), "=h"(hi) : "r"(w[i]));
            asm("add.rn.f32.bf16 %0, %1, %0;" : "+f"(a[2 * i]) : "h"(lo));      // FHADD.BF16: f32 += bf16
            asm("add.rn.f32.bf16 %0, %1, %0;" : "+f"(a[2 * i + 1]) : "h"(hi));
        }
    }
    __device__ __forceinline__ void fma(const uint4& v, float s) {  // acc += s * v
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            a[2 * i] = fmaf(__uint_as_float(w[i] << 16), s, a[2 * i]);
            a[2 * i + 1] = fmaf(__uint_as_float(w[i] & 0xffff0000u), s, a[2 * i + 1]);
        }
    }
    __device__ __forceinline__ void get(float* f) const {
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = a[i];
    }
};


// Persistent: one 32-warp CTA per SM.  Rows are cut into CHUNKS of 32 row-blocks; chunk k belongs to CTA
// k mod gridDim.x and a CTA's warps take the blocks of its chunks in order from a CTA-local counter.  So
//  * inside an SM, ~32*R neighbouring rows are in flight together; a warp walks R consecutive rows, whose
//    overlapping neighbourhoods hit L1 (34 % on the 2M-node lattice = exactly the row-to-next-row overlap: with
//    128 KB of gathers in flight per SM, L1 lines do not live long enough for reuse between warps);
//  * across the chip, all SMs advance through the node array as ONE wavefront (148 chunks wide), so the
//    longer-range reuse (neighbouring lattice planes) stays inside the 126 MB L2 and DRAM sees each row once
//    (ncu: DRAM traffic 2.2 GB = A_min).  (A contiguous band per SM loses this: DRAM reads tripled.)
//
// Inner loop, shaped by the ncu captures under profiles/ (r01):
//  * v1 spent 31 warp instructions per edge (79 % issue utilisation on a bf16 row).  Now an edge costs one
//    IMAD.WIDE (row address = column * row_bytes + opaque lane base; the other 16-byte vectors of the row are
//    immediate offsets when EXACT), the LDG.128s and the adds; column indices come kU at a time from ONE
//    broadcast LDS.128 of a shared-memory window (no SHFL per edge); row ends are tested once per batch of kU
//    edges and per edge only in batches holding one: 20 instructions per edge, 998 -> 710 us on cfg4.
//  * What bounds cfg4 now is the L2 -> SM fabric: 9.3 GB of L1 misses in 0.71 ms = 13 TB/s, the full-chip LTS
//    cap (~6300 B/clk).  Only more on-SM reuse (explicit de-duplication of a chunk's neighbours in shared
//    memory) can lift it further.
//  * 32 warps x one batch of kU rows in flight beat 16 warps x two software-pipelined batches (cfg4: 745 vs 956 us)
//    and 32 warps x two half batches (750 us): thread-level parallelism hides the per-block prologue
//    (rowptr -> col -> rows) best.
constexpr int kAggThreads = 1024;

template <typename T, int LANES, int VPL, bool HAS_ADD, bool EXACT, bool HAS_SRC>
__global__ void __launch_bounds__(kAggThreads, 1) k_aggregate(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                              const float* __restrict__ row_scale,
                                                              const float* __restrict__ src_scale /*per SOURCE row (HAS_SRC)*/,
                                                              const T* __restrict__ x,
                                                              const T* __restrict__ addend, T* __restrict__ out, int64_t N,
                                                              int nvec /*16B vectors per row*/, int R /*rows per group, < LANES*/) {
    using V = Vec16<T>;
    constexpr int EPV = V::N;
    constexpr int GROUPS = 32 / LANES;
    constexpr int kU0 = VPL >= 4 ? 2 : (VPL == 2 ? 4 : 8);  // source rows per batch (8 x 16 B per lane)
    constexpr int kU = kU0 < LANES ? kU0 : LANES;
    static_assert(LANES % kU == 0, "a column window holds whole batches");
    __shared__ int s_next;
    __shared__ __align__(16) int s_cols[kAggThreads / 32][2][32];
    __shared__ __align__(16) float s_scl[HAS_SRC ? kAggThreads / 32 : 1][2][32];  // the columns' source scales
    const int lane = threadIdx.x & 31;
    const int sub = lane % LANES;
    const unsigned gmask = LANES == 32 ? 0xffffffffu : (((1u << LANES) - 1u) << (lane / LANES * LANES));
    constexpr int kBPC = kAggThreads / 32;  // row-blocks (one per warp) per chunk
    const int64_t unit = (int64_t)R * GROUPS;  // rows per warp step
    if (threadIdx.x == 0) s_next = 0;
    __syncthreads();
    // Lanes past the end of a row (only when nvec < LANES*VPL) load a clamped, valid vector and never
    // store: every load below is UNCONDITIONAL, so the compiler keeps the requests of a batch in flight together.
    const uint32_t row_bytes = (uint32_t)nvec * 16u;
    bool vec_ok[VPL];
    uint32_t dlt[VPL];  // byte offset of vector v relative to vector 0 of this lane
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
        vec_ok[v] = EXACT || (sub + v * LANES) < nvec;
        dlt[v] = EXACT ? (uint32_t)(v * LANES * 16) : (uint32_t)(min(sub + v * LANES, nvec - 1) - min(sub, nvec - 1)) * 16u;
    }
    const uint32_t lane_off = (uint32_t)min(sub, nvec - 1) * 16u;
    // lane base pointers, made opaque so that a row address is ONE IMAD.WIDE (c * row_bytes + base) instead of
    // the compiler's re-association (c * row_bytes + lane_off) + x  (IMAD.WIDE + IADD3 + IADD3.X)
    uint64_t xl_ = reinterpret_cast<uint64_t>(x) + lane_off;
    uint64_t al_ = HAS_ADD ? reinterpret_cast<uint64_t>(addend) + lane_off : 0;
    uint64_t ol_ = reinterpret_cast<uint64_t>(out) + lane_off;
    asm volatile("" : "+l"(xl_), "+l"(al_), "+l"(ol_));
    const char* xl = reinterpret_cast<const char*>(xl_);
    const char* al = reinterpret_cast<const char*>(al_);
    char* ol = reinterpret_cast<char*>(ol_);
    int* const wcols = &s_cols[threadIdx.x >> 5][0][lane - sub];  // this group's slice of the two column windows
    float* const wscl = &s_scl[HAS_SRC ? threadIdx.x >> 5 : 0][0][lane - sub];

  for (;;) {
    int blk = 0;
    if (lane == 0) blk = atomicAdd(&s_next, 1);
    blk = __shfl_sync(0xffffffffu, blk, 0);
    const int64_t chunk = (int64_t)blockIdx.x + (int64_t)(blk / kBPC) * gridDim.x;
    const int64_t w0 = (chunk * kBPC + blk % kBPC) * unit;
    if (chunk * kBPC * unit >= N) break;  // this CTA's chunks are exhausted (warp-uniform)
    const int64_t r0 = w0 + (int64_t)(lane / LANES) * R;
    if (r0 >= N) continue;  // ragged end of the last chunk (group-uniform)
    const int nrows = (int)min((int64_t)R, N - r0);

    // rowptr[r0 .. r0+nrows] -> one value per lane
    const int rp = sub <= nrows ? __ldg(rowptr + r0 + sub) : 0;
    const float rsc = (row_scale && sub < nrows) ? __ldg(row_scale + r0 + sub) : 1.0f;  // one scale per lane, no load at flush time
    const int e_beg = __shfl_sync(gmask, rp, 0, LANES);
    const int e_end = __shfl_sync(gmask, rp, nrows, LANES);

    Acc<T> acc[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) acc[v].zero();
    uint4 ad[VPL];
    int cur = 0;                                          // current row inside the block
    int cur_end = __shfl_sync(gmask, rp, 1, LANES);       // its end edge; INT_MAX once every row is written
    auto fetch_addend = [&](int r) {
        if (HAS_ADD) {
            const char* p = al + (uint64_t)(r0 + r) * row_bytes;
#pragma unroll
            for (int v = 0; v < VPL; ++v) ad[v] = ldg_nc_v4(reinterpret_cast<const uint4*>(p + dlt[v]));
        }
    };
    auto flush = [&]() {  // write row `cur`, start the next one
        const float sc = __shfl_sync(gmask, rsc, cur, LANES);
        char* po = ol + (uint64_t)(r0 + cur) * row_bytes;
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
            float f[EPV];
            acc[v].get(f);
            if (HAS_ADD) {
                V a;
                a.v = *reinterpret_cast<decltype(a.v)*>(&ad[v]);
                float g[EPV];
                a.to_float(g);
#pragma unroll
                for (int i = 0; i < EPV; ++i) f[i] = fmaf(f[i], sc, g[i]);
            } else {
#pragma unroll
                for (int i = 0; i < EPV; ++i) f[i] *= sc;
            }
            V o;
            o.from_float(f);
            if (vec_ok[v]) stg_v4(po + dlt[v], *reinterpret_cast<uint4*>(&o.v));
            acc[v].zero();
        }
        ++cur;
        if (cur < nrows) {
            cur_end = __shfl_sync(gmask, rp, cur + 1, LANES);
            fetch_addend(cur);
        } else {
            cur_end = 0x7fffffff;  // the padding edges of the last batch fall into an accumulator nobody writes
        }
    };
    fetch_addend(0);

    const int ne = e_end - e_beg;
    const int nbatch = (ne + kU - 1) / kU;
    // lanes past the end of the edge range repeat the last valid column (a harmless L1 hit), so every slot of a
    // window holds a loadable column and a batch needs no bounds checks
    auto load_cols = [&](int j) { return ldg_stream_s32(col + e_beg + j + min(sub, min(LANES, ne - j) - 1)); };
    int mine = ne > 0 ? load_cols(0) : 0;
    // HAS_SRC: the scale of a column is a dependent load, so the columns run TWO windows ahead of the rows and the
    // scales one window ahead: neither round trip is waited for
    float smine = 0.f;
    int mine_nxt = 0;
    if (HAS_SRC && ne > 0) {
        smine = __ldg(src_scale + mine);
        if (LANES < ne) mine_nxt = load_cols(LANES);
    }
    // request the rows of batch b into `buf`; the first batch of a column window parks the window in shared memory
    // and requests the next window's columns
    float sb[HAS_SRC ? kU : 1];
    auto issue = [&](uint4 (&buf)[kU][VPL], int b) {
        const int j = b * kU;
        const int within = j & (LANES - 1);
        const int wsel = ((j / LANES) & 1) * 32;
        int* w = wcols + wsel;
        if (within == 0) {
            w[sub] = mine;
            if (HAS_SRC) wscl[wsel + sub] = smine;
            __syncwarp(gmask);
            const int nxt = j + LANES;
            if (HAS_SRC) {
                if (nxt < ne) {
                    mine = mine_nxt;
                    smine = __ldg(src_scale + mine);
                    if (nxt + LANES < ne) mine_nxt = load_cols(nxt + LANES);
                }
            } else if (nxt < ne) {
                mine = load_cols(nxt);
            }
        }
        if constexpr (HAS_SRC) {
            const float* ws_ = wscl + wsel + within;
            if constexpr (kU == 8) {
                const float4 s0 = *reinterpret_cast<const float4*>(ws_), s1 = *reinterpret_cast<const float4*>(ws_ + 4);
                sb[0] = s0.x; sb[1] = s0.y; sb[2] = s0.z; sb[3] = s0.w; sb[4] = s1.x; sb[5] = s1.y; sb[6] = s1.z; sb[7] = s1.w;
            } else if constexpr (kU == 4) {
                const float4 s0 = *reinterpret_cast<const float4*>(ws_);
                sb[0] = s0.x; sb[1] = s0.y; sb[2] = s0.z; sb[3] = s0.w;
            } else {
                const float2 s0 = *reinterpret_cast<const float2*>(ws_);
                sb[0] = s0.x; sb[1] = s0.y;
            }
        }
        uint32_t cb[kU];
        if constexpr (kU == 8) {
            const uint4 c0 = *reinterpret_cast<const uint4*>(w + within), c1 = *reinterpret_cast<const uint4*>(w + within + 4);
            cb[0] = c0.x; cb[1] = c0.y; cb[2] = c0.z; cb[3] = c0.w; cb[4] = c1.x; cb[5] = c1.y; cb[6] = c1.z; cb[7] = c1.w;
        } else if constexpr (kU == 4) {
            const uint4 c0 = *reinterpret_cast<const uint4*>(w + within);
            cb[0] = c0.x; cb[1] = c0.y; cb[2] = c0.z; cb[3] = c0.w;
        } else {
            const uint2 c0 = *reinterpret_cast<const uint2*>(w + within);
            cb[0] = c0.x; cb[1] = c0.y;
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
            const char* p = xl + (uint64_t)cb[u] * row_bytes;
#pragma unroll
            for (int v = 0; v < VPL; ++v) buf[u][v] = ldg_nc_v4(reinterpret_cast<const uint4*>(p + dlt[v]));
        }
    };
    auto consume = [&](uint4 (&buf)[kU][VPL], int b) {
        const int ebase = e_beg + b * kU;
        if (cur_end - ebase >= kU) {  // whole batch inside the current row
#pragma unroll
            for (int u = 0; u < kU; ++u) {
#pragma unroll
                for (int v = 0; v < VPL; ++v) {
                    if constexpr (HAS_SRC) acc[v].fma(buf[u][v], sb[u]);
                    else acc[v].add(buf[u][v]);
                }
            }
        } else {
#pragma unroll
            for (int u = 0; u < kU; ++u) {
                while (ebase + u == cur_end) flush();  // group-uniform; also steps over empty rows
#pragma unroll
                for (int v = 0; v < VPL; ++v) {
                    if constexpr (HAS_SRC) acc[v].fma(buf[u][v], sb[u]);
                    else acc[v].add(buf[u][v]);
                }
            }
        }
    };
    for (int b = 0; b < nbatch; ++b) {
        uint4 buf[kU][VPL];
        issue(buf, b);
        consume(buf, b);
    }
    while (cur < nrows) flush();  // last row and trailing empty rows
  }
}

// rows per group: about a dozen rows / <= 192 edges per group amortise the rowptr/col round trips of a block (the
// dependent prologue of every block is what the 32 warps have to hide); among the candidates take the one whose
// chunk count fills whole waves of 148 CTAs best (a 200k-row batch is only ~4 waves: 3.25 waves cost 4)
inline int pick_rows_per_group(int64_t N, int64_t E, int lanes, int groups) {
    const double deg = N > 0 ? (double)E / (double)N : 0.0;
    int hi = (int)(192.0 / (deg + 1.0));
    hi = std::max(1, std::min(hi, std::min(12, lanes - 1)));
    const int lo = std::max(1, (hi * 2 + 2) / 3);
    int best = hi;
    double best_eff = -1.0;
    for (int R = hi; R >= lo; --R) {
        const int64_t chunk_rows = (int64_t)R * groups * (kAggThreads / 32);
        const int64_t chunks = (N + chunk_rows - 1) / chunk_rows;
        const int64_t waves = (chunks + kNumSMs - 1) / kNumSMs;
        const double eff = (double)N / ((double)waves * kNumSMs * (double)chunk_rows);
        if (eff > best_eff + 0.02) {  // prefer larger R unless a smaller one is clearly better balanced
            best_eff = eff;
            best = R;
        }
    }
    return best;
}

template <typename T, int LANES, int VPL>
int launch(const int32_t* rowptr, const int32_t* col, const float* row_scale, const float* src_scale, const void* x,
           const void* addend, void* out, int64_t N, int64_t E, int nvec, cudaStream_t s) {
    constexpr int GROUPS = 32 / LANES;
    const int R = pick_rows_per_group(N, E, LANES, GROUPS);
    const int64_t chunk_rows = (int64_t)R * GROUPS * (kAggThreads / 32);
    const int64_t chunks = (N + chunk_rows - 1) / chunk_rows;
    const int64_t blocks = std::min<int64_t>(chunks, kNumSMs);
    if (blocks == 0) return 0;
    const bool exact = nvec == LANES * VPL;
#define DFW_AGG_GO(A, X, S)                                                                                                  \
    k_aggregate<T, LANES, VPL, A, X, S><<<(unsigned)blocks, kAggThreads, 0, s>>>(rowptr, col, row_scale, src_scale, (const T*)x, \
                                                                                (const T*)addend, (T*)out, N, nvec, R)
    if (src_scale) {  // (the scaled gather is only used without an addend: backward of the mean)
        if (exact) DFW_AGG_GO(false, true, true); else DFW_AGG_GO(false, false, true);
    } else if (exact) {
        if (addend) DFW_AGG_GO(true, true, false); else DFW_AGG_GO(false, true, false);
    } else {
        if (addend) DFW_AGG_GO(true, false, false); else DFW_AGG_GO(false, false, false);
    }
#undef DFW_AGG_GO
    DFW_LAUNCH_CHECK();
    return 0;
}

template <typename T>
int dispatch(const int32_t* rowptr, const int32_t* col, const float* row_scale, const float* src_scale, const void* x,
             const void* addend, void* out, int64_t N, int64_t E, int nvec, cudaStream_t s) {
#define DFW_AGG(L, V) return launch<T, L, V>(rowptr, col, row_scale, src_scale, x, addend, out, N, E, nvec, s)
    if (nvec <= 4) DFW_AGG(4, 1);
    if (nvec <= 8) DFW_AGG(8, 1);
    if (nvec <= 16) DFW_AGG(16, 1);
    if (nvec <= 32) DFW_AGG(32, 1);
    if (nvec <= 64) DFW_AGG(32, 2);
    if (nvec <= 128) DFW_AGG(32, 4);
#undef DFW_AGG
    set_error("dfw_sage_aggregate: row of %d x 16 bytes is wider than the supported 2048 bytes", nvec);
    return 1;
}

}  // namespace
}  // namespace dfw

static int aggregate_entry(const char* who, const int32_t* rowptr, const int32_t* col, const float* row_scale,
                           const float* src_scale, const void* x, const void* addend, void* out, int64_t N, int64_t E, int64_t H,
                           int dtype, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(N >= 0 && E >= 0 && H > 0, "%s: bad shape N=%lld E=%lld H=%lld", who, (long long)N, (long long)E, (long long)H);
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "%s: unknown dtype %d", who, dtype);
    const int64_t row_bytes = H * (dtype == DFW_F32 ? 4 : 2);
    DFW_REQUIRE(row_bytes % 16 == 0, "%s: H*sizeof(dtype) = %lld must be a multiple of 16", who, (long long)row_bytes);
    if (N == 0) return 0;
    DFW_REQUIRE(rowptr && (col || E == 0) && x && out, "%s: null pointer", who);
    DFW_REQUIRE(aligned16(x) && aligned16(out) && (!addend || aligned16(addend)), "%s: x/out/addend must be 16-byte aligned", who);
    DFW_REQUIRE(N * (row_bytes / 16) < (1LL << 40), "%s: tensor too large", who);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int nvec = (int)(row_bytes / 16);
    if (dtype == DFW_F32) return dispatch<float>(rowptr, col, row_scale, src_scale, x, addend, out, N, E, nvec, s);
    return dispatch<__nv_bfloat16>(rowptr, col, row_scale, src_scale, x, addend, out, N, E, nvec, s);
}

extern "C" int dfw_sage_aggregate(const int32_t* rowptr, const int32_t* col, const float* row_scale, const void* x,
                                  const void* addend, void* out, int64_t N, int64_t E, int64_t H, int dtype,
                                  dfw_stream_t stream) {
    return aggregate_entry("dfw_sage_aggregate", rowptr, col, row_scale, nullptr, x, addend, out, N, E, H, dtype, stream);
}

extern "C" int dfw_sage_aggregate_scaled(const int32_t* rowptr, const int32_t* col, const float* src_scale, const void* x,
                                         void* out, int64_t N, int64_t E, int64_t H, int dtype, dfw_stream_t stream) {
    if (N > 0 && !src_scale) {
        dfw::set_error("dfw_sage_aggregate_scaled: src_scale is NULL");
        return 1;
    }
    return aggregate_entry("dfw_sage_aggregate_scaled", rowptr, col, nullptr, src_scale, x, nullptr, out, N, E, H, dtype, stream);
}
