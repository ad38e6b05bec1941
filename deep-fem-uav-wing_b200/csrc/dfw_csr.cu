// (a) edge_index -> canonical CSR, built on the device.
//
// Replaces the per-call gather / scatter bookkeeping that PyG's SAGEConv performs on the raw
// COO edge list (reference call site: src/deep_fem_uav_wing/gnn/model.py:90; edge_index int64
// [2,E] in arbitrary order, gnn/dataset.py:39-63).  Result is bit-identical to
// numpy.lexsort((src, dst)) whatever the input order:
//     count (int atomics: order-independent) -> scan -> bucket fill (order inside a row is
//     arbitrary here) -> per-row sort of the 64-bit key (col << 32 | edge id) (canonical).
// HBM-bound integer work: every pass is a coalesced grid-stride sweep; the grid is a multiple
// of the SM count.
#include "dfw_common.cuh"

namespace dfw {
namespace {

constexpr int kScanThreads = 1024;
constexpr int kScanItems = 4;
constexpr int kScanChunk = kScanThreads * kScanItems;
constexpr int kBigRowSmemKeys = 4096;
constexpr int kWarpRowMax = 32;

struct CsrWs {
    uint64_t* keys;
    int32_t* cursor;
    int32_t* worklist;
    int32_t* blocksums;
    int32_t* counters;
    size_t bytes;
};

CsrWs carve(void* ws, int64_t E, int64_t N) {
    CsrWs w;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += align_up(bytes, 256);
        return o;
    };
    size_t o_keys = take(sizeof(uint64_t) * (size_t)(E > 0 ? E : 1));
    size_t o_cursor = take(sizeof(int32_t) * (size_t)(N + 1));
    size_t o_work = take(sizeof(int32_t) * (size_t)(E / (kWarpRowMax + 1) + 1));
    size_t nblk = (size_t)((N + 1 + kScanChunk - 1) / kScanChunk);
    size_t o_bs = take(sizeof(int32_t) * (nblk + 1));
    size_t o_cnt = take(sizeof(int32_t) * 4);
    char* base = reinterpret_cast<char*>(ws);
    w.keys = reinterpret_cast<uint64_t*>(base + o_keys);
    w.cursor = reinterpret_cast<int32_t*>(base + o_cursor);
    w.worklist = reinterpret_cast<int32_t*>(base + o_work);
    w.blocksums = reinterpret_cast<int32_t*>(base + o_bs);
    w.counters = reinterpret_cast<int32_t*>(base + o_cnt);
    w.bytes = off;
    return w;
}

__global__ void k_count(const int64_t* __restrict__ rows, const int64_t* __restrict__ cols, int64_t E,
                        int64_t N, int32_t* __restrict__ cnt_plus1, int32_t* __restrict__ status,
        const int32_t* __restrict__ gate) {
    if (gate && *gate == 0) return;  // dfw_csr_transpose: the graph turned out to be symmetric, nothing to build
    int bad = 0;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = rows[e], c = cols[e];
        if ((uint64_t)r >= (uint64_t)N || (uint64_t)c >= (uint64_t)N) {
            ++bad;
        } else {
            atomicAdd(&cnt_plus1[r + 1], 1);
        }
    }
    if (bad) atomicAdd(&status[0], bad);
}

// ---- 3-phase inclusive scan over a[0..n) (int32) ----------------------------------------
__device__ __forceinline__ int block_inclusive_scan(int v, int* smem /*32 ints*/) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    if (lane == 31) smem[wid] = v;
    __syncthreads();
    if (wid == 0) {
        int s = smem[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += t;
        }
        smem[lane] = s;
    }
    __syncthreads();
    if (wid > 0) v += smem[wid - 1];
    __syncthreads();
    return v;
}

__global__ void __launch_bounds__(kScanThreads) k_scan_partial(const int32_t* __restrict__ a, int64_t n,
                                                                int32_t* __restrict__ blocksums,
        const int32_t* __restrict__ gate) {
    if (gate && *gate == 0) return;  // dfw_csr_transpose: the graph turned out to be symmetric, nothing to build
    __shared__ int sm[32];
    int64_t base = (int64_t)blockIdx.x * kScanChunk + threadIdx.x * kScanItems;
    int s = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i)
        if (base + i < n) s += a[base + i];
    int incl = block_inclusive_scan(s, sm);
    if (threadIdx.x == kScanThreads - 1) blocksums[blockIdx.x] = incl;
}

__global__ void __launch_bounds__(kScanThreads) k_scan_blocksums(int32_t* __restrict__ blocksums, int nblk,
        const int32_t* __restrict__ gate) {
    if (gate && *gate == 0) return;  // dfw_csr_transpose: the graph turned out to be symmetric, nothing to build
    __shared__ int sm[32];
    __shared__ int carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < nblk; base += kScanThreads) {
        int i = base + threadIdx.x;
        int v = i < nblk ? blocksums[i] : 0;
        int incl = block_inclusive_scan(v, sm);
        int carry = carry_s;
        if (i < nblk) blocksums[i] = carry + incl - v;  // exclusive
        __syncthreads();
        if (threadIdx.x == kScanThreads - 1) carry_s = carry + incl;
        __syncthreads();
    }
}

// a = [0, deg_0, deg_1, ...] (length N+1) -> inclusive scan in place == rowptr.  Also emits
// cursor[i] = rowptr[i], inv_deg[i] = 1/max(deg_i,1), max degree.
__global__ void __launch_bounds__(kScanThreads) k_scan_apply(int32_t* __restrict__ a, int64_t n /*N+1*/,
                                                              const int32_t* __restrict__ blocksums,
                                                              int32_t* __restrict__ cursor, float* __restrict__ inv_deg,
                                                              int32_t* __restrict__ status,
        const int32_t* __restrict__ gate) {
    if (gate && *gate == 0) return;  // dfw_csr_transpose: the graph turned out to be symmetric, nothing to build
    __shared__ int sm[32];
    int64_t base = (int64_t)blockIdx.x * kScanChunk + threadIdx.x * kScanItems;
    int v[kScanItems];
    int s = 0, mx = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) {
        v[i] = (base + i < n) ? a[base + i] : 0;
        s += v[i];
        mx = max(mx, v[i]);
    }
    int incl = block_inclusive_scan(s, sm);
    int run = blocksums[blockIdx.x] + incl - s;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) {
        int64_t j = base + i;
        run += v[i];
        if (j < n) {
            a[j] = run;
            if (j < n - 1) cursor[j] = run;
            if (j >= 1 && inv_deg) inv_deg[j - 1] = 1.0f / (float)max(v[i], 1);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0 && mx > 0) atomicMax(&status[1], mx);
}

__global__ void k_fill(const int64_t* __restrict__ rows, const int64_t* __restrict__ cols, int64_t E, int64_t N,
                       int32_t* __restrict__ cursor, uint64_t* __restrict__ keys,
        const int32_t* __restrict__ gate) {
    if (gate && *gate == 0) return;  // dfw_csr_transpose: the graph turned out to be symmetric, nothing to build
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = rows[e], c = cols[e];
        if ((uint64_t)r < (uint64_t)N && (uint64_t)c < (uint64_t)N) {
            int pos = atomicAdd(&cursor[r], 1);
            keys[pos] = ((uint64_t)c << 32) | (uint64_t)(uint32_t)e;
        }
    }
}

// one warp per row, rank sort for deg <= 32 (keys are unique: the edge id is part of the key)
__global__ void __launch_bounds__(256) k_sort_rows_warp(const int32_t* __restrict__ rowptr, int64_t N,
                                                         const uint64_t* __restrict__ keys, int32_t* __restrict__ col,
                                                         int32_t* __restrict__ perm, int32_t* __restrict__ worklist,
                                                         int32_t* __restrict__ counters,
        const int32_t* __restrict__ gate) {
    if (gate && *gate == 0) return;  // dfw_csr_transpose: the graph turned out to be symmetric, nothing to build
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < N; row += warps) {
        const int beg = rowptr[row], deg = rowptr[row + 1] - beg;
        if (deg == 0) continue;
        if (deg > kWarpRowMax) {
            if (lane == 0) worklist[atomicAdd(&counters[0], 1)] = (int32_t)row;
            continue;
        }
        uint64_t k = lane < deg ? keys[beg + lane] : ~0ull;
        int rank = 0;
        for (int j = 0; j < deg; ++j) {
            uint64_t o = __shfl_sync(0xffffffffu, k, j);
            rank += (o < k);
        }
        if (lane < deg) {
            col[beg + rank] = (int32_t)(k >> 32);
            if (perm) perm[beg + rank] = (int32_t)(k & 0xffffffffu);
        }
    }
}

// ascending-only bitonic network (first step of every merge mirrors, the rest butterfly), so
// virtual +inf padding above `n` never moves: pairs whose upper index is >= n are skipped.
template <typename Ptr>
__device__ __forceinline__ void bitonic_ascending(Ptr a, int n) {
    int P = 1;
    while (P < n) P <<= 1;
    for (int k = 2; k <= P; k <<= 1) {
        for (int t = threadIdx.x; t < P / 2; t += blockDim.x) {  // mirror step
            int blk = t / (k / 2), off = t % (k / 2);
            int lo = blk * k + off, hi = blk * k + (k - 1 - off);
            if (hi < n) {
                uint64_t x = a[lo], y = a[hi];
                if (y < x) { a[lo] = y; a[hi] = x; }
            }
        }
        __syncthreads();
        for (int j = k / 4; j >= 1; j >>= 1) {
            for (int t = threadIdx.x; t < P / 2; t += blockDim.x) {
                int lo = (t / j) * (2 * j) + (t % j), hi = lo + j;
                if (hi < n) {
                    uint64_t x = a[lo], y = a[hi];
                    if (y < x) { a[lo] = y; a[hi] = x; }
                }
            }
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(256) k_sort_rows_big(const int32_t* __restrict__ rowptr, uint64_t* __restrict__ keys,
                                                        int32_t* __restrict__ col, int32_t* __restrict__ perm,
                                                        const int32_t* __restrict__ worklist,
                                                        const int32_t* __restrict__ counters,
        const int32_t* __restrict__ gate) {
    if (gate && *gate == 0) return;  // dfw_csr_transpose: the graph turned out to be symmetric, nothing to build
    __shared__ uint64_t sk[kBigRowSmemKeys];
    const int nwork = counters[0];
    for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int row = worklist[w];
        const int beg = rowptr[row], deg = rowptr[row + 1] - beg;
        if (deg <= kBigRowSmemKeys) {
            for (int i = threadIdx.x; i < deg; i += blockDim.x) sk[i] = keys[beg + i];
            __syncthreads();
            bitonic_ascending(sk, deg);
            for (int i = threadIdx.x; i < deg; i += blockDim.x) {
                uint64_t k = sk[i];
                col[beg + i] = (int32_t)(k >> 32);
                if (perm) perm[beg + i] = (int32_t)(k & 0xffffffffu);
            }
            __syncthreads();
        } else {
            bitonic_ascending(keys + beg, deg);  // in global memory; block-level syncs order the passes
            for (int i = threadIdx.x; i < deg; i += blockDim.x) {
                uint64_t k = keys[beg + i];
                col[beg + i] = (int32_t)(k >> 32);
                if (perm) perm[beg + i] = (int32_t)(k & 0xffffffffu);
            }
            __syncthreads();
        }
    }
}

}  // namespace
}  // namespace dfw

extern "C" size_t dfw_csr_ws_bytes(int64_t E, int64_t N) {
    if (E < 0 || N < 0) return 0;
    return dfw::carve(nullptr, E, N).bytes;
}

namespace dfw {
int csr_build_impl(const int64_t* edge_index, int64_t E, int64_t N, int by_src, int32_t* rowptr, int32_t* col,
                          int32_t* perm, float* inv_deg, int32_t* status, void* ws, size_t ws_bytes, dfw_stream_t stream,
                          const int32_t* gate = nullptr);
}

extern "C" int dfw_csr_build(const int64_t* edge_index, int64_t E, int64_t N, int by_src, int32_t* rowptr,
                             int32_t* col, int32_t* perm, float* inv_deg, int32_t* status, void* ws,
                             size_t ws_bytes, dfw_stream_t stream) {
    return dfw::csr_build_impl(edge_index, E, N, by_src, rowptr, col, perm, inv_deg, status, ws, ws_bytes, stream);
}

namespace dfw {
int csr_build_impl(const int64_t* edge_index, int64_t E, int64_t N, int by_src, int32_t* rowptr, int32_t* col,
                          int32_t* perm, float* inv_deg, int32_t* status, void* ws, size_t ws_bytes, dfw_stream_t stream,
                          const int32_t* gate) {
    DFW_REQUIRE(E >= 0 && N >= 0, "dfw_csr_build: negative size (E=%lld, N=%lld)", (long long)E, (long long)N);
    DFW_REQUIRE(E < 2147483647LL && N < 2147483647LL, "dfw_csr_build: E and N must be < 2^31 (E=%lld, N=%lld)",
                (long long)E, (long long)N);
    DFW_REQUIRE(rowptr && status && (col || E == 0), "dfw_csr_build: null output pointer");
    DFW_REQUIRE(edge_index || E == 0, "dfw_csr_build: null edge_index");
    CsrWs w = carve(ws, E, N);
    DFW_REQUIRE(ws && ws_bytes >= w.bytes, "dfw_csr_build: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);

    DFW_CUDA(cudaMemsetAsync(rowptr, 0, sizeof(int32_t) * (size_t)(N + 1), s));
    DFW_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t) * 2, s));
    DFW_CUDA(cudaMemsetAsync(w.counters, 0, sizeof(int32_t) * 4, s));

    const int64_t* rows = by_src ? edge_index : edge_index + E;
    const int64_t* cols = by_src ? edge_index + E : edge_index;
    const int threads = 256;
    const int grid_e = (int)std::max<int64_t>(1, std::min<int64_t>((E + threads - 1) / threads, (int64_t)kNumSMs * 16));
    if (E > 0) {
        k_count<<<grid_e, threads, 0, s>>>(rows, cols, E, N, rowptr, status, gate);
        DFW_LAUNCH_CHECK();
    }
    const int64_t n1 = N + 1;
    const int nblk = (int)((n1 + kScanChunk - 1) / kScanChunk);
    k_scan_partial<<<nblk, kScanThreads, 0, s>>>(rowptr, n1, w.blocksums, gate);
    DFW_LAUNCH_CHECK();
    k_scan_blocksums<<<1, kScanThreads, 0, s>>>(w.blocksums, nblk, gate);
    DFW_LAUNCH_CHECK();
    k_scan_apply<<<nblk, kScanThreads, 0, s>>>(rowptr, n1, w.blocksums, w.cursor, inv_deg, status, gate);
    DFW_LAUNCH_CHECK();
    if (E > 0) {
        k_fill<<<grid_e, threads, 0, s>>>(rows, cols, E, N, w.cursor, w.keys, gate);
        DFW_LAUNCH_CHECK();
        const int64_t warps_per_block = threads / 32;
        const int grid_r = (int)std::max<int64_t>(1, std::min<int64_t>((N + warps_per_block - 1) / warps_per_block, (int64_t)kNumSMs * 64));
        k_sort_rows_warp<<<grid_r, threads, 0, s>>>(rowptr, N, w.keys, col, perm, w.worklist, w.counters, gate);
        DFW_LAUNCH_CHECK();
        k_sort_rows_big<<<kNumSMs * 2, 256, 0, s>>>(rowptr, w.keys, col, perm, w.worklist, w.counters, gate);
        DFW_LAUNCH_CHECK();
    }
    return 0;
}
}  // namespace dfw

// ---- transposed CSR (rows = source) for the backward gather -------------------------------------------------
// Mesh graphs carry both directions of every edge (reference gnn/dataset.py:55-58), and then the CSR by source IS the
// CSR by destination.  dfw_csr_transpose checks that on the device (every edge (s -> d) of a duplicate-free CSR has its
// mirror (d -> s): one binary search per edge in the L2-resident col array) and either copies the CSR or runs the
// general build; the decision never leaves the device (the general build's kernels are gated on the flag), so the
// call is capturable in a CUDA graph and costs no host synchronisation.
namespace dfw {
namespace {
__global__ void __launch_bounds__(256) k_sym_check(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t N,
                                                    int32_t* __restrict__ asym) {
    for (int64_t d = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; d < N; d += (int64_t)gridDim.x * blockDim.x) {
        const int beg = rowptr[d], end = rowptr[d + 1];
        bool bad = false;
        for (int e = beg; e < end && !bad; ++e) {
            const int s = col[e];
            if (e + 1 < end && col[e + 1] == s) bad = true;  // duplicate edge: multiplicities would have to match too
            int lo = rowptr[s], hi = rowptr[s + 1];           // is d among the sources of row s ?
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (col[mid] < (int)d) lo = mid + 1; else hi = mid;
            }
            if (lo >= rowptr[s + 1] || col[lo] != (int)d) bad = true;
        }
        if (bad) *asym = 1;
    }
}
__global__ void __launch_bounds__(256) k_copy_if_symmetric(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t N,
                                                            int64_t E, int32_t* __restrict__ rowptr_t, int32_t* __restrict__ col_t,
                                                            const int32_t* __restrict__ asym) {
    if (*asym) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i <= N; i += stride) rowptr_t[i] = rowptr[i];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < E; i += stride) col_t[i] = col[i];
}
}  // namespace
}  // namespace dfw

extern "C" int dfw_csr_transpose(const int64_t* edge_index, int64_t E, int64_t N, const int32_t* rowptr, const int32_t* col,
                                 int32_t* rowptr_t, int32_t* col_t, int32_t* status, void* ws, size_t ws_bytes,
                                 dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(E >= 0 && N >= 0, "dfw_csr_transpose: negative size (E=%lld, N=%lld)", (long long)E, (long long)N);
    DFW_REQUIRE(rowptr && rowptr_t && status && ((col && col_t) || E == 0), "dfw_csr_transpose: null pointer");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    DFW_CUDA(cudaMemsetAsync(status + 2, 0, sizeof(int32_t), s));
    if (N > 0) {
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((N + 255) / 256, (int64_t)kNumSMs * 16));
        k_sym_check<<<grid, 256, 0, s>>>(rowptr, col, N, status + 2);
        DFW_LAUNCH_CHECK();
    }
    const int rc = csr_build_impl(edge_index, E, N, 1, rowptr_t, col_t, nullptr, nullptr, status, ws, ws_bytes, stream, status + 2);
    if (rc) return rc;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((std::max(E, N + 1) + 255) / 256, (int64_t)kNumSMs * 8));
    k_copy_if_symmetric<<<grid, 256, 0, s>>>(rowptr, col, N, E, rowptr_t, col_t, status + 2);
    DFW_LAUNCH_CHECK();
    return 0;
}

// =============================================================================================
// (f1) Graph construction from triangle faces, on the device (SURVEY 8f-1).
//
// Replaces the Python set loop of _faces_to_edge_index (reference src/deep_fem_uav_wing/gnn/dataset.py:26-63):
//   faces [F,3] of node IDS -> 0-based indices through node_id_to_idx (dataset.py:106), faces holding an unknown id
//   are skipped (dataset.py:43-46), the three undirected edges of every face are de-duplicated (dataset.py:49-52)
//   and emitted in both directions (dataset.py:55-58; a degenerate self pair (i,i) therefore appears twice).
// Here: expand to directed pairs -> the canonical CSR build above (rows sorted) -> per-row unique -> scan -> fill.
// Output is the CSR by destination the aggregation consumes, plus (optionally) the int64 edge_index in canonical
// (dst, src) order - the same edge SET as the reference, whose own order is Python-set iteration order.
// Integer work, bit-exact against oracle/sage_oracle.py:faces_to_edge_index_ref after canonical sorting.
// =============================================================================================
namespace dfw {
namespace {

// idx of `id` in the ascending array sorted_ids[0..N), or -1
__device__ __forceinline__ int64_t find_id(const int64_t* __restrict__ sorted_ids, int64_t N, int64_t id) {
    int64_t lo = 0, hi = N;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (sorted_ids[mid] < id) lo = mid + 1; else hi = mid;
    }
    return (lo < N && sorted_ids[lo] == id) ? lo : -1;
}

// one thread per face: 6 directed pairs into pairs[0][6f..] (src) / pairs[1][6f..] (dst); skipped faces write -1
__global__ void k_faces_expand(const int64_t* __restrict__ faces, int64_t F, const int64_t* __restrict__ sorted_ids,
                               const int64_t* __restrict__ id_perm, int64_t N, int64_t* __restrict__ pairs,
                               int32_t* __restrict__ status) {
    int skipped = 0;
    const int64_t E0 = 6 * F;
    for (int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; f < F; f += (int64_t)gridDim.x * blockDim.x) {
        int64_t v[3];
        bool ok = true;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int64_t id = faces[3 * f + k];
            int64_t idx;
            if (sorted_ids) {
                idx = find_id(sorted_ids, N, id);
                if (idx >= 0 && id_perm) idx = id_perm[idx];
            } else {
                idx = ((uint64_t)id < (uint64_t)N) ? id : -1;
            }
            v[k] = idx;
            ok = ok && idx >= 0;
        }
        skipped += !ok;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int64_t a = ok ? v[k] : -1, b = ok ? v[(k + 1) % 3] : -1;
            pairs[6 * f + 2 * k] = a;          pairs[E0 + 6 * f + 2 * k] = b;       // a -> b
            pairs[6 * f + 2 * k + 1] = b;      pairs[E0 + 6 * f + 2 * k + 1] = a;   // b -> a
        }
    }
    if (skipped) atomicAdd(&status[2], skipped);
}

// warp per row of the duplicate-holding CSR: cnt_plus1[r+1] = distinct columns (+1 if the row holds itself)
__global__ void __launch_bounds__(256) k_unique_count(const int32_t* __restrict__ rowptr0, const int32_t* __restrict__ col0,
                                                       int64_t N, int32_t* __restrict__ cnt_plus1) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < N; row += warps) {
        const int beg = rowptr0[row], end = rowptr0[row + 1];
        int n = 0;
        for (int base = beg; base < end; base += 32) {
            const int i = base + lane;
            bool first = false, self = false;
            if (i < end) {
                const int c = col0[i];
                first = (i == beg) || (col0[i - 1] != c);
                self = first && c == (int)row;
            }
            n += __popc(__ballot_sync(0xffffffffu, first)) + __popc(__ballot_sync(0xffffffffu, self));
        }
        if (lane == 0) cnt_plus1[row + 1] = n;
    }
}

__global__ void __launch_bounds__(256) k_unique_fill(const int32_t* __restrict__ rowptr0, const int32_t* __restrict__ col0,
                                                      const int32_t* __restrict__ rowptr, int64_t N, int32_t* __restrict__ col,
                                                      int64_t* __restrict__ edge_index, int64_t ei_stride) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < N; row += warps) {
        const int beg = rowptr0[row], end = rowptr0[row + 1];
        int out = rowptr[row];
        for (int base = beg; base < end; base += 32) {
            const int i = base + lane;
            bool first = false, self = false;
            int c = 0;
            if (i < end) {
                c = col0[i];
                first = (i == beg) || (col0[i - 1] != c);
                self = first && c == (int)row;
            }
            const unsigned mf = __ballot_sync(0xffffffffu, first), ms = __ballot_sync(0xffffffffu, self);
            const unsigned below = (1u << lane) - 1u;
            if (first) {
                const int pos = out + __popc(mf & below) + __popc(ms & below);
                const int copies = self ? 2 : 1;
                for (int k = 0; k < copies; ++k) {
                    col[pos + k] = c;
                    if (edge_index) {
                        edge_index[pos + k] = c;                    // source
                        edge_index[ei_stride + pos + k] = row;      // destination
                    }
                }
            }
            out += __popc(mf) + __popc(ms);
        }
    }
}

__global__ void k_store_count(const int32_t* __restrict__ rowptr, int64_t N, int64_t* __restrict__ num_edges) {
    if (threadIdx.x == 0 && blockIdx.x == 0) *num_edges = rowptr[N];
}

struct FacesWs {
    int64_t* pairs;    // [2, 6F]
    int32_t* rowptr0;  // [N+1]
    int32_t* col0;     // [6F]
    void* csr_ws;
    size_t csr_ws_bytes;
    size_t bytes;
};
FacesWs carve_faces(void* ws, int64_t F, int64_t N) {
    FacesWs w;
    const int64_t E0 = 6 * F;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += align_up(bytes, 256);
        return o;
    };
    const size_t o_pairs = take(sizeof(int64_t) * 2 * (size_t)(E0 > 0 ? E0 : 1));
    const size_t o_rp = take(sizeof(int32_t) * (size_t)(N + 1));
    const size_t o_col = take(sizeof(int32_t) * (size_t)(E0 > 0 ? E0 : 1));
    w.csr_ws_bytes = carve(nullptr, E0, N).bytes;
    const size_t o_csr = take(w.csr_ws_bytes);
    char* base = reinterpret_cast<char*>(ws);
    w.pairs = reinterpret_cast<int64_t*>(base + o_pairs);
    w.rowptr0 = reinterpret_cast<int32_t*>(base + o_rp);
    w.col0 = reinterpret_cast<int32_t*>(base + o_col);
    w.csr_ws = base + o_csr;
    w.bytes = off;
    return w;
}

}  // namespace
}  // namespace dfw

extern "C" size_t dfw_faces_ws_bytes(int64_t F, int64_t N) {
    if (F < 0 || N < 0) return 0;
    return dfw::carve_faces(nullptr, F, N).bytes;
}

extern "C" int dfw_faces_to_csr(const int64_t* faces, int64_t F, const int64_t* sorted_ids, const int64_t* id_perm, int64_t N,
                                int32_t* rowptr, int32_t* col, float* inv_deg, int64_t* edge_index, int64_t* num_edges,
                                int32_t* status, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(F >= 0 && N >= 0, "dfw_faces_to_csr: negative size (F=%lld, N=%lld)", (long long)F, (long long)N);
    DFW_REQUIRE(6 * F < 2147483647LL && N < 2147483647LL, "dfw_faces_to_csr: 6F and N must be < 2^31");
    DFW_REQUIRE(rowptr && status && num_edges && (col || F == 0), "dfw_faces_to_csr: null output pointer");
    DFW_REQUIRE(faces || F == 0, "dfw_faces_to_csr: null faces");
    FacesWs w = carve_faces(ws, F, N);
    DFW_REQUIRE(ws && ws_bytes >= w.bytes, "dfw_faces_to_csr: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int64_t E0 = 6 * F;
    const int threads = 256;
    DFW_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t) * 3, s));
    if (F > 0) {
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((F + threads - 1) / threads, (int64_t)kNumSMs * 16));
        k_faces_expand<<<grid, threads, 0, s>>>(faces, F, sorted_ids, id_perm, N, w.pairs, status);
        DFW_LAUNCH_CHECK();
    }
    // duplicate-holding CSR by destination (row 1 of `pairs`), columns sorted inside every row.  It clears
    // status[0..1] itself: [0] then counts the 6 placeholder pairs of every skipped face, [2] (ours) the faces.
    {
        // csr_build_impl zeroes status[0..1] only; keep status[2]
        const int rc = csr_build_impl(w.pairs, E0, N, 0, w.rowptr0, w.col0, nullptr, nullptr, status, w.csr_ws, w.csr_ws_bytes, stream);
        if (rc) return rc;
    }
    DFW_CUDA(cudaMemsetAsync(rowptr, 0, sizeof(int32_t) * (size_t)(N + 1), s));
    const int64_t warps_per_block = threads / 32;
    const int grid_r = (int)std::max<int64_t>(1, std::min<int64_t>((N + warps_per_block - 1) / warps_per_block, (int64_t)kNumSMs * 64));
    if (N > 0 && F > 0) {
        k_unique_count<<<grid_r, threads, 0, s>>>(w.rowptr0, w.col0, N, rowptr);
        DFW_LAUNCH_CHECK();
    }
    // scan -> rowptr, inv_deg, max degree (reuses the CSR build's scan; its cursor/blocksums live in the CSR workspace)
    CsrWs cw = carve(w.csr_ws, E0, N);
    DFW_CUDA(cudaMemsetAsync(status + 1, 0, sizeof(int32_t), s));
    const int64_t n1 = N + 1;
    const int nblk = (int)((n1 + kScanChunk - 1) / kScanChunk);
    k_scan_partial<<<nblk, kScanThreads, 0, s>>>(rowptr, n1, cw.blocksums, nullptr);
    DFW_LAUNCH_CHECK();
    k_scan_blocksums<<<1, kScanThreads, 0, s>>>(cw.blocksums, nblk, nullptr);
    DFW_LAUNCH_CHECK();
    k_scan_apply<<<nblk, kScanThreads, 0, s>>>(rowptr, n1, cw.blocksums, cw.cursor, inv_deg, status, nullptr);
    DFW_LAUNCH_CHECK();
    if (N > 0 && F > 0) {
        k_unique_fill<<<grid_r, threads, 0, s>>>(w.rowptr0, w.col0, rowptr, N, col, edge_index, E0);
        DFW_LAUNCH_CHECK();
    }
    k_store_count<<<1, 32, 0, s>>>(rowptr, N, num_edges);
    DFW_LAUNCH_CHECK();
    return 0;
}
