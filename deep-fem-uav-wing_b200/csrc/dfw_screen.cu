// Design screening on the device (BASELINE.json config 5): area-weighted vertex normals of a triangulated surface, so
// that a design needs no FEM output to be screened, and a per-case segmented reduction of the model's prediction into
// the few numbers a design is judged on.
//
// dfw_vertex_normals replaces the normal block of the reference's fem.py:390-424 (restated at synth.py:146-151):
//     fn = cross(p1 - p0, p2 - p0) per face;  normal[v] = sum of fn over the incidences (f, k) with faces[f, k] == v.
//   The vertex -> incidence lists come from the canonical CSR build of dfw_csr.cu (count -> scan -> fill -> per-row sort):
//   the incidence 3f + k is an "edge" of row faces[f, k] whose sort key is (v << 32 | 3f + k), so every row lists its
//   incidences in ascending order and one thread per vertex sums its face normals in that order.  No float atomics; the
//   sum of a vertex reads its own faces only, so concatenating cases cannot change it.
//
// dfw_case_stress_summary replaces the per-case host pass a screening run would otherwise make over the full prediction
// (the cfg5 block of bench.py brought back one torch mean per case).  Cases are cut into chunks of kChunkRows rows
// counted from the case's first row, so the chunking - and with it every partial and the order they are combined in -
// depends on the case's length only; the grid covers all chunks of all cases, so one 500k-node case shares a launch
// with 20k-node cases without serialising on one block.  fp64 partial sums, a fixed-order combine, no float atomics.
// Roofline: HBM; algorithmic bytes = N (pred) * sizeof(dtype) + 12 N (pos, the y column costs the cache lines) + N (mask).
#include <algorithm>
#include <cfloat>

#include "dfw_common.cuh"

namespace dfw {
namespace {

constexpr int kScrThreads = 256;
constexpr int kChunkRows = 2048;  // rows of a case per block-chunk: 8 per thread
constexpr int kScanBlock = 1024;
constexpr int64_t kNoRow = INT64_MAX;

// ---- vertex normals -------------------------------------------------------------------------------------------------
// one thread per face: incidence 3f + k becomes the pair (v, v) at column 3f + k of pairs [2, 3F]; a face that names an
// index outside [0, N) writes -1 for all three incidences (the CSR build drops them) and is counted in status[0]
__global__ void k_incidence_expand(const int64_t* __restrict__ faces, int64_t F, int64_t N, int64_t* __restrict__ pairs,
                                   int32_t* __restrict__ status) {
    int skipped = 0;
    const int64_t E = 3 * F;
    for (int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; f < F; f += (int64_t)gridDim.x * blockDim.x) {
        int64_t v[3];
        bool ok = true;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            v[k] = faces[3 * f + k];
            ok = ok && (uint64_t)v[k] < (uint64_t)N;
        }
        skipped += !ok;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int64_t r = ok ? v[k] : -1;
            pairs[3 * f + k] = r;
            pairs[E + 3 * f + k] = r;
        }
    }
    if (skipped) atomicAdd(&status[0], skipped);
}

// one thread per vertex: its face normals in ascending incidence order (perm of the CSR holds the incidence ids)
__global__ void __launch_bounds__(kScrThreads) k_vertex_normals(const float* __restrict__ pos, const int64_t* __restrict__ faces,
                                                                 const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm,
                                                                 int64_t N, float* __restrict__ normal) {
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < N; v += (int64_t)gridDim.x * blockDim.x) {
        float nx = 0.f, ny = 0.f, nz = 0.f;
        const int beg = rowptr[v], end = rowptr[v + 1];
        for (int j = beg; j < end; ++j) {
            const int64_t f = perm[j] / 3;
            const int64_t i0 = faces[3 * f], i1 = faces[3 * f + 1], i2 = faces[3 * f + 2];
            const float ox = pos[3 * i0], oy = pos[3 * i0 + 1], oz = pos[3 * i0 + 2];
            const float ax = __fsub_rn(pos[3 * i1], ox), ay = __fsub_rn(pos[3 * i1 + 1], oy), az = __fsub_rn(pos[3 * i1 + 2], oz);
            const float bx = __fsub_rn(pos[3 * i2], ox), by = __fsub_rn(pos[3 * i2 + 1], oy), bz = __fsub_rn(pos[3 * i2 + 2], oz);
            // numpy.cross order, no fused multiply-add: the same bits for the same face wherever it is summed
            nx = __fadd_rn(nx, __fsub_rn(__fmul_rn(ay, bz), __fmul_rn(az, by)));
            ny = __fadd_rn(ny, __fsub_rn(__fmul_rn(az, bx), __fmul_rn(ax, bz)));
            nz = __fadd_rn(nz, __fsub_rn(__fmul_rn(ax, by), __fmul_rn(ay, bx)));
        }
        normal[3 * v] = nx;
        normal[3 * v + 1] = ny;
        normal[3 * v + 2] = nz;
    }
}

struct NormalsWs {
    int64_t* pairs;     // [2, 3F]
    int32_t* rowptr;    // [N+1]
    int32_t* col;       // [3F]
    int32_t* perm;      // [3F]
    int32_t* csr_status;  // [2]
    void* csr_ws;
    size_t csr_ws_bytes;
    size_t bytes;
};
NormalsWs carve_normals(void* ws, int64_t F, int64_t N) {
    NormalsWs w;
    const int64_t E = 3 * F;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += align_up(bytes, 256);
        return o;
    };
    const size_t o_pairs = take(sizeof(int64_t) * 2 * (size_t)(E > 0 ? E : 1));
    const size_t o_rp = take(sizeof(int32_t) * (size_t)(N + 1));
    const size_t o_col = take(sizeof(int32_t) * (size_t)(E > 0 ? E : 1));
    const size_t o_perm = take(sizeof(int32_t) * (size_t)(E > 0 ? E : 1));
    const size_t o_st = take(sizeof(int32_t) * 2);
    w.csr_ws_bytes = dfw_csr_ws_bytes(E, N);
    const size_t o_csr = take(w.csr_ws_bytes);
    char* base = reinterpret_cast<char*>(ws);
    w.pairs = reinterpret_cast<int64_t*>(base + o_pairs);
    w.rowptr = reinterpret_cast<int32_t*>(base + o_rp);
    w.col = reinterpret_cast<int32_t*>(base + o_col);
    w.perm = reinterpret_cast<int32_t*>(base + o_perm);
    w.csr_status = reinterpret_cast<int32_t*>(base + o_st);
    w.csr_ws = base + o_csr;
    w.bytes = off;
    return w;
}

// ---- per-case stress summary ------------------------------------------------------------------------------------------
struct ChunkPart {
    double sum;       // sum of the finite screened stresses
    float mx;         // max over the finite screened stresses
    float mx_all;     // max over all finite stresses
    int64_t arg;      // row of mx within the case (kNoRow: none)
    int32_t n_scr;    // screened rows
    int32_t n_fin;    // screened rows with a finite stress
    int32_t n_over;   // finite screened stresses above the allowable
    int32_t n_bad;    // non-finite stresses
};

__device__ __forceinline__ void case_rows(const int64_t* __restrict__ case_ptr, int64_t b, int64_t N, int64_t& r0, int64_t& r1) {
    r0 = min(max(case_ptr[b], (int64_t)0), N);
    r1 = min(max(case_ptr[b + 1], r0), N);
}

// chunk_ptr[b] = sum over b' < b of ceil(len_b' / kChunkRows), capped at max_chunks (a malformed case_ptr cannot make the
// later kernels index past the workspace).  One block.
__global__ void __launch_bounds__(kScanBlock) k_chunk_scan(const int64_t* __restrict__ case_ptr, int64_t B, int64_t N, int64_t max_chunks,
                                                           int64_t* __restrict__ chunk_ptr) {
    __shared__ long long warp_tot[kScanBlock / 32];
    __shared__ long long carry_s;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int64_t base = 0; base < B; base += kScanBlock) {
        const int64_t b = base + threadIdx.x;
        long long c = 0;
        if (b < B) {
            int64_t r0, r1;
            case_rows(case_ptr, b, N, r0, r1);
            c = (r1 - r0 + kChunkRows - 1) / kChunkRows;
        }
        long long incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_tot[wid] = incl;
        __syncthreads();
        long long before = carry_s;
        for (int w = 0; w < wid; ++w) before += warp_tot[w];
        if (b < B) chunk_ptr[b] = min((long long)max_chunks, before + incl - c);
        __syncthreads();
        if (threadIdx.x == kScanBlock - 1) carry_s = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) chunk_ptr[B] = min((long long)max_chunks, carry_s);
}

// the case of chunk c: the last b with chunk_ptr[b] <= c (empty cases share their successor's chunk_ptr)
__device__ __forceinline__ int64_t chunk_case(const int64_t* __restrict__ chunk_ptr, int64_t B, int64_t c) {
    int64_t lo = 0, hi = B;  // answer in [0, B)
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (chunk_ptr[mid] <= c) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(kScrThreads) k_chunk_minmax_y(const float* __restrict__ pos, const int64_t* __restrict__ case_ptr,
                                                                 const int64_t* __restrict__ chunk_ptr, int64_t B, int64_t N,
                                                                 float* __restrict__ mm /*[chunks][2]*/) {
    __shared__ float sh[kScrThreads / 32][2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t total = chunk_ptr[B];
    for (int64_t c = blockIdx.x; c < total; c += gridDim.x) {
        const int64_t b = chunk_case(chunk_ptr, B, c);
        int64_t r0, r1;
        case_rows(case_ptr, b, N, r0, r1);
        const int64_t beg = r0 + (c - chunk_ptr[b]) * kChunkRows, end = min(beg + kChunkRows, r1);
        float lo = FLT_MAX, hi = -FLT_MAX;
        for (int64_t i = beg + threadIdx.x; i < end; i += blockDim.x) {
            const float y = pos[3 * i + 1];
            lo = fminf(lo, y);
            hi = fmaxf(hi, y);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (lane == 0) { sh[wid][0] = lo; sh[wid][1] = hi; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < kScrThreads / 32; ++w) { lo = fminf(lo, sh[w][0]); hi = fmaxf(hi, sh[w][1]); }
            mm[2 * c] = lo;
            mm[2 * c + 1] = hi;
        }
        __syncthreads();
    }
}

__device__ __forceinline__ void take_max(float& mx, int64_t& arg, float o_mx, int64_t o_arg) {
    if (o_mx > mx || (o_mx == mx && o_arg < arg)) { mx = o_mx; arg = o_arg; }  // ties: the lowest row wins
}

struct SummaryArgs {
    const void* pred; const float* pos; const uint8_t* mask; const int64_t* case_ptr; const int64_t* chunk_ptr; const float* mm;
    ChunkPart* part;
    int64_t B, N;
    double root_band, allowable;
    int log_scale;
};

// The screened-row rule of a case, shared by every per-case reduction over the model output: mask[row] != 0 when a mask
// is given, else the root band pos_y > root_band * (max_y - min_y) of the row's own case (fem.py:637-640,
// synth.py:154-155), from the per-chunk y ranges of k_chunk_minmax_y.  band_threshold is called by the whole block
// (it synchronises); its scratch is a block-shared [kScrThreads / 32][2] float array.
__device__ __forceinline__ double band_threshold(const float* __restrict__ mm, int64_t c0, int64_t c1, double root_band,
                                                 float (*sh)[2], double* thr_s) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    float lo = FLT_MAX, hi = -FLT_MAX;
    for (int64_t k = c0 + threadIdx.x; k < c1; k += blockDim.x) { lo = fminf(lo, mm[2 * k]); hi = fmaxf(hi, mm[2 * k + 1]); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) { sh[wid][0] = lo; sh[wid][1] = hi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kScrThreads / 32; ++w) { lo = fminf(lo, sh[w][0]); hi = fmaxf(hi, sh[w][1]); }
        *thr_s = root_band * ((double)hi - (double)lo);
    }
    __syncthreads();
    return *thr_s;
}

__device__ __forceinline__ bool screened_row(const uint8_t* __restrict__ mask, const float* __restrict__ pos, int64_t i, double thr) {
    return mask ? mask[i] != 0 : (double)pos[3 * i + 1] > thr;
}

template <typename T>
__global__ void __launch_bounds__(kScrThreads) k_chunk_stats(const SummaryArgs p) {
    __shared__ double sh_sum[kScrThreads / 32];
    __shared__ float sh_f[kScrThreads / 32][4];
    __shared__ float sh_band[kScrThreads / 32][2];
    __shared__ int64_t sh_arg[kScrThreads / 32];
    __shared__ int sh_n[kScrThreads / 32][4];
    __shared__ double thr_s;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const T* __restrict__ pred = static_cast<const T*>(p.pred);
    const int64_t total = p.chunk_ptr[p.B];
    for (int64_t c = blockIdx.x; c < total; c += gridDim.x) {
        const int64_t b = chunk_case(p.chunk_ptr, p.B, c);
        int64_t r0, r1;
        case_rows(p.case_ptr, b, p.N, r0, r1);
        const int64_t c0 = p.chunk_ptr[b], c1 = p.chunk_ptr[b + 1];
        const double thr = p.mask ? 0.0 : band_threshold(p.mm, c0, c1, p.root_band, sh_band, &thr_s);
        const int64_t beg = r0 + (c - c0) * kChunkRows, end = min(beg + kChunkRows, r1);
        double sum = 0.0;
        float mx = -INFINITY, mx_all = -INFINITY;
        int64_t arg = kNoRow;
        int n_scr = 0, n_fin = 0, n_over = 0, n_bad = 0;
        for (int64_t i = beg + threadIdx.x; i < end; i += blockDim.x) {  // ascending rows per thread: strict > keeps the lowest
            float v = to_f32(pred[i]);
            if (p.log_scale) v = expm1f(v);  // inverse of log1p (dataset.py:148-151), as dfw_stress_metrics
            const bool fin = isfinite(v);
            const bool scr = screened_row(p.mask, p.pos, i, thr);
            n_bad += !fin;
            n_scr += scr;
            if (fin) {
                mx_all = fmaxf(mx_all, v);
                if (scr) {
                    ++n_fin;
                    sum += (double)v;
                    if (v > mx) { mx = v; arg = i - r0; }
                    n_over += (p.allowable > 0.0 && (double)v > p.allowable);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, o);
            mx_all = fmaxf(mx_all, __shfl_xor_sync(0xffffffffu, mx_all, o));
            take_max(mx, arg, __shfl_xor_sync(0xffffffffu, mx, o), __shfl_xor_sync(0xffffffffu, arg, o));
            n_scr += __shfl_xor_sync(0xffffffffu, n_scr, o);
            n_fin += __shfl_xor_sync(0xffffffffu, n_fin, o);
            n_over += __shfl_xor_sync(0xffffffffu, n_over, o);
            n_bad += __shfl_xor_sync(0xffffffffu, n_bad, o);
        }
        if (lane == 0) {
            sh_sum[wid] = sum;
            sh_f[wid][2] = mx; sh_f[wid][3] = mx_all;
            sh_arg[wid] = arg;
            sh_n[wid][0] = n_scr; sh_n[wid][1] = n_fin; sh_n[wid][2] = n_over; sh_n[wid][3] = n_bad;
        }
        __syncthreads();
        if (threadIdx.x == 0) {  // warps in a fixed order
            for (int w = 1; w < kScrThreads / 32; ++w) {
                sum += sh_sum[w];
                mx_all = fmaxf(mx_all, sh_f[w][3]);
                take_max(mx, arg, sh_f[w][2], sh_arg[w]);
                n_scr += sh_n[w][0]; n_fin += sh_n[w][1]; n_over += sh_n[w][2]; n_bad += sh_n[w][3];
            }
            ChunkPart q;
            q.sum = sum; q.mx = mx; q.mx_all = mx_all; q.arg = arg;
            q.n_scr = n_scr; q.n_fin = n_fin; q.n_over = n_over; q.n_bad = n_bad;
            p.part[c] = q;
        }
        __syncthreads();
    }
}

// one thread per case: its chunks in ascending order
__global__ void k_case_finalize(const int64_t* __restrict__ case_ptr, const int64_t* __restrict__ chunk_ptr, const ChunkPart* __restrict__ part,
                                int64_t B, int64_t N, double* __restrict__ out) {
    for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
        int64_t r0, r1;
        case_rows(case_ptr, b, N, r0, r1);
        double sum = 0.0;
        float mx = -INFINITY, mx_all = -INFINITY;
        int64_t arg = kNoRow, n_scr = 0, n_fin = 0, n_over = 0, n_bad = 0;
        for (int64_t c = chunk_ptr[b]; c < chunk_ptr[b + 1]; ++c) {
            const ChunkPart q = part[c];
            sum += q.sum;
            mx_all = fmaxf(mx_all, q.mx_all);
            take_max(mx, arg, q.mx, q.arg);
            n_scr += q.n_scr; n_fin += q.n_fin; n_over += q.n_over; n_bad += q.n_bad;
        }
        double* o = out + 8 * b;
        o[0] = (double)(r1 - r0);
        o[1] = (double)n_scr;
        o[2] = n_fin ? (double)mx : 0.0;
        o[3] = n_fin ? (double)arg : -1.0;
        o[4] = n_fin ? sum / (double)n_fin : 0.0;
        o[5] = mx_all > -INFINITY ? (double)mx_all : 0.0;
        o[6] = (double)n_over;
        o[7] = (double)n_bad;
    }
}

int64_t max_chunks(int64_t N, int64_t B) { return (N + kChunkRows - 1) / kChunkRows + B; }

struct SummaryWs {
    int64_t* chunk_ptr;  // [B+1]
    float* mm;           // [max_chunks][2]
    ChunkPart* part;     // [max_chunks]
    size_t bytes;
};
SummaryWs carve_summary(void* ws, int64_t N, int64_t B) {
    SummaryWs w;
    const int64_t mc = max_chunks(N, B);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += align_up(bytes, 256);
        return o;
    };
    const size_t o_cp = take(sizeof(int64_t) * (size_t)(B + 1));
    const size_t o_mm = take(sizeof(float) * 2 * (size_t)std::max<int64_t>(mc, 1));
    const size_t o_part = take(sizeof(ChunkPart) * (size_t)std::max<int64_t>(mc, 1));
    char* base = reinterpret_cast<char*>(ws);
    w.chunk_ptr = reinterpret_cast<int64_t*>(base + o_cp);
    w.mm = reinterpret_cast<float*>(base + o_mm);
    w.part = reinterpret_cast<ChunkPart*>(base + o_part);
    w.bytes = off;
    return w;
}

// ---- per-case KS aggregate of the screened prediction and its seed gradient -------------------------------------------
// Both reductions below reuse the summary's chunk plan and workspace: their per-chunk partials fit in its ChunkPart slots.
struct KsPart {
    double m;   // max of u over the chunk's set (after k_case_ks, in the case's first slot: over the case's set)
    double s;   // sum over the set of exp(rho (u - m)); a row with u == m counts 1 (also when u = m = -inf)
    int64_t n;  // rows in the set (0: m and s are meaningless)
};
static_assert(sizeof(KsPart) <= sizeof(ChunkPart) && alignof(KsPart) <= alignof(ChunkPart), "KS partials use the summary's slots");

constexpr int kRowsPerThread = kChunkRows / kScrThreads;

struct KsArgs {
    const void* pred; const float* pos; const uint8_t* mask; const int64_t* case_ptr; const int64_t* chunk_ptr; const float* mm;
    KsPart* part; float* seed;
    int64_t B, N;
    double root_band, rho;
};

__device__ __forceinline__ double ks_term(double rho, double u, double m) { return u == m ? 1.0 : exp(rho * (u - m)); }

// the KS set S_b: screened rows whose fp32 stress expm1f(u) is finite - the rows behind max_stress_pa of the summary
template <typename T>
__device__ __forceinline__ void ks_load(const KsArgs& p, int64_t beg, int64_t end, double thr, float (&u)[kRowsPerThread],
                                        bool (&in)[kRowsPerThread]) {
    const T* __restrict__ pred = static_cast<const T*>(p.pred);
#pragma unroll
    for (int k = 0; k < kRowsPerThread; ++k) {
        const int64_t i = beg + threadIdx.x + (int64_t)k * kScrThreads;
        u[k] = 0.f;
        in[k] = false;
        if (i < end) {
            u[k] = to_f32(pred[i]);
            in[k] = isfinite(expm1f(u[k])) && screened_row(p.mask, p.pos, i, thr);
        }
    }
}

// per chunk: its max m and sum exp(rho (u - m)) in fp64; rows in ascending order per thread, lanes by a fixed butterfly,
// warps in index order
template <typename T>
__global__ void __launch_bounds__(kScrThreads) k_chunk_ks(const KsArgs p) {
    __shared__ float sh_band[kScrThreads / 32][2];
    __shared__ float sh_m[kScrThreads / 32];
    __shared__ int sh_n[kScrThreads / 32];
    __shared__ double sh_s[kScrThreads / 32];
    __shared__ double thr_s;
    __shared__ float m_s;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t total = p.chunk_ptr[p.B];
    for (int64_t c = blockIdx.x; c < total; c += gridDim.x) {
        const int64_t b = chunk_case(p.chunk_ptr, p.B, c);
        int64_t r0, r1;
        case_rows(p.case_ptr, b, p.N, r0, r1);
        const int64_t c0 = p.chunk_ptr[b], c1 = p.chunk_ptr[b + 1];
        const double thr = p.mask ? 0.0 : band_threshold(p.mm, c0, c1, p.root_band, sh_band, &thr_s);
        const int64_t beg = r0 + (c - c0) * kChunkRows, end = min(beg + kChunkRows, r1);
        float u[kRowsPerThread];
        bool in[kRowsPerThread];
        ks_load<T>(p, beg, end, thr, u, in);
        float mx = -INFINITY;
        int n = 0;
#pragma unroll
        for (int k = 0; k < kRowsPerThread; ++k) {
            if (in[k]) { mx = fmaxf(mx, u[k]); ++n; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            n += __shfl_xor_sync(0xffffffffu, n, o);
        }
        if (lane == 0) { sh_m[wid] = mx; sh_n[wid] = n; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < kScrThreads / 32; ++w) { mx = fmaxf(mx, sh_m[w]); n += sh_n[w]; }
            m_s = mx;
        }
        __syncthreads();
        const double m = (double)m_s;
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < kRowsPerThread; ++k) {
            if (in[k]) s += ks_term(p.rho, (double)u[k], m);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) sh_s[wid] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < kScrThreads / 32; ++w) s += sh_s[w];
            KsPart q;
            q.m = m; q.s = s; q.n = n;
            p.part[c] = q;
        }
        __syncthreads();
    }
}

// one thread per case: its chunks in ascending order, each rescaled to the running max; the case's (m, s, n) goes back
// into its first chunk slot for k_chunk_ks_seed.  out[b] = [KS_b = m + ln(s) / rho, n]; [0, 0] for an empty set.
__global__ void k_case_ks(const int64_t* __restrict__ chunk_ptr, KsPart* __restrict__ part, int64_t B, double rho,
                          double* __restrict__ out) {
    for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
        double m = -INFINITY, s = 0.0;
        int64_t n = 0;
        const int64_t c0 = chunk_ptr[b], c1 = chunk_ptr[b + 1];
        for (int64_t c = c0; c < c1; ++c) {
            const KsPart q = part[c];
            if (q.n == 0) continue;
            if (n == 0) {
                m = q.m; s = q.s;
            } else if (q.m > m) {
                s = s * ks_term(rho, m, q.m) + q.s;
                m = q.m;
            } else {
                s += q.s * ks_term(rho, q.m, m);
            }
            n += q.n;
        }
        out[2 * b] = n ? m + log(s) / rho : 0.0;
        out[2 * b + 1] = (double)n;
        if (c0 < c1) {
            KsPart q;
            q.m = m; q.s = s; q.n = n;
            part[c0] = q;
        }
    }
}

// one write per row: w = exp(rho (u - m_b)) / s_b on S_b, computed in fp64 and rounded to fp32 once; 0 elsewhere
template <typename T>
__global__ void __launch_bounds__(kScrThreads) k_chunk_ks_seed(const KsArgs p) {
    __shared__ float sh_band[kScrThreads / 32][2];
    __shared__ double thr_s;
    const int64_t total = p.chunk_ptr[p.B];
    for (int64_t c = blockIdx.x; c < total; c += gridDim.x) {
        const int64_t b = chunk_case(p.chunk_ptr, p.B, c);
        int64_t r0, r1;
        case_rows(p.case_ptr, b, p.N, r0, r1);
        const int64_t c0 = p.chunk_ptr[b], c1 = p.chunk_ptr[b + 1];
        const double thr = p.mask ? 0.0 : band_threshold(p.mm, c0, c1, p.root_band, sh_band, &thr_s);
        const int64_t beg = r0 + (c - c0) * kChunkRows, end = min(beg + kChunkRows, r1);
        const KsPart q = p.part[c0];
        float u[kRowsPerThread];
        bool in[kRowsPerThread];
        ks_load<T>(p, beg, end, thr, u, in);
#pragma unroll
        for (int k = 0; k < kRowsPerThread; ++k) {
            const int64_t i = beg + threadIdx.x + (int64_t)k * kScrThreads;
            if (i < end) p.seed[i] = (in[k] && q.n > 0) ? __double2float_rn(ks_term(p.rho, (double)u[k], q.m) / q.s) : 0.f;
        }
    }
}

// ---- per-case column sums ----------------------------------------------------------------------------------------------
constexpr int kColGroup = (int)(sizeof(ChunkPart) / sizeof(double));  // columns per pass: one ChunkPart slot of doubles

// per chunk: fp64 sums of columns [col0, col0 + ng) of a fp32 [N, C]; same fixed order as k_chunk_ks
__global__ void __launch_bounds__(kScrThreads) k_chunk_colsum(const float* __restrict__ a, int64_t C, int64_t col0, int ng,
                                                               const int64_t* __restrict__ case_ptr, const int64_t* __restrict__ chunk_ptr,
                                                               int64_t B, int64_t N, double* __restrict__ part /*[chunks][kColGroup]*/) {
    __shared__ double sh[kScrThreads / 32][kColGroup];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t total = chunk_ptr[B];
    for (int64_t c = blockIdx.x; c < total; c += gridDim.x) {
        const int64_t b = chunk_case(chunk_ptr, B, c);
        int64_t r0, r1;
        case_rows(case_ptr, b, N, r0, r1);
        const int64_t beg = r0 + (c - chunk_ptr[b]) * kChunkRows, end = min(beg + kChunkRows, r1);
        double acc[kColGroup];
#pragma unroll
        for (int j = 0; j < kColGroup; ++j) acc[j] = 0.0;
        for (int64_t i = beg + threadIdx.x; i < end; i += blockDim.x) {
            const float* __restrict__ row = a + i * C + col0;
#pragma unroll
            for (int j = 0; j < kColGroup; ++j)
                if (j < ng) acc[j] += (double)row[j];
        }
#pragma unroll
        for (int j = 0; j < kColGroup; ++j) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o);
        }
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < kColGroup; ++j) sh[wid][j] = acc[j];
        }
        __syncthreads();
        if (threadIdx.x < ng) {  // one thread per column, warps in index order
            const int j = threadIdx.x;
            double t = sh[0][j];
            for (int w = 1; w < kScrThreads / 32; ++w) t += sh[w][j];
            part[c * kColGroup + j] = t;
        }
        __syncthreads();
    }
}

// one thread per (case, column): the case's chunks in ascending order
__global__ void k_case_colsum(const int64_t* __restrict__ chunk_ptr, const double* __restrict__ part, int64_t B, int ng,
                              int64_t nc, int64_t j0, double* __restrict__ out) {
    const int64_t total = B * ng;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = t / ng;
        const int j = (int)(t % ng);
        double sum = 0.0;
        for (int64_t c = chunk_ptr[b]; c < chunk_ptr[b + 1]; ++c) sum += part[c * kColGroup + j];
        out[b * nc + j0 + j] = sum;
    }
}

}  // namespace
}  // namespace dfw

extern "C" size_t dfw_vertex_normals_ws_bytes(int64_t F, int64_t N) {
    if (F < 0 || N < 0) return 0;
    return dfw::carve_normals(nullptr, F, N).bytes;
}

extern "C" int dfw_vertex_normals(const float* pos, int64_t N, const int64_t* faces, int64_t F, float* normal, int32_t* status,
                                  void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(F >= 0 && N >= 0, "dfw_vertex_normals: negative size (F=%lld, N=%lld)", (long long)F, (long long)N);
    DFW_REQUIRE(3 * F < 2147483647LL && N < 2147483647LL, "dfw_vertex_normals: 3F and N must be < 2^31");
    DFW_REQUIRE(status && (normal || N == 0), "dfw_vertex_normals: null output pointer");
    DFW_REQUIRE((pos || N == 0) && (faces || F == 0), "dfw_vertex_normals: null input pointer");
    NormalsWs w = carve_normals(ws, F, N);
    DFW_REQUIRE(ws && ws_bytes >= w.bytes, "dfw_vertex_normals: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int64_t E = 3 * F;
    DFW_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t), s));
    if (F > 0) {
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((F + 255) / 256, (int64_t)kNumSMs * 16));
        k_incidence_expand<<<grid, 256, 0, s>>>(faces, F, N, w.pairs, status);
        DFW_LAUNCH_CHECK();
    }
    const int rc = csr_build_impl(w.pairs, E, N, 0, w.rowptr, w.col, w.perm, nullptr, w.csr_status, w.csr_ws, w.csr_ws_bytes, stream,
                                  nullptr);
    if (rc) return rc;
    if (N > 0) {
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((N + kScrThreads - 1) / kScrThreads, (int64_t)kNumSMs * 16));
        k_vertex_normals<<<grid, kScrThreads, 0, s>>>(pos, faces, w.rowptr, w.perm, N, normal);
        DFW_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" size_t dfw_case_stress_summary_ws_bytes(int64_t N, int64_t B) {
    if (N < 0 || B < 0) return 0;
    return dfw::carve_summary(nullptr, N, B).bytes;
}

extern "C" int dfw_case_stress_summary(const void* pred, int dtype, const float* pos, const uint8_t* mask, const int64_t* case_ptr,
                                       int64_t B, int64_t N, double root_band, double allowable_pa, int log_scale, double* out,
                                       void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_case_stress_summary: unknown dtype %d", dtype);
    DFW_REQUIRE(B >= 0 && N >= 0, "dfw_case_stress_summary: negative size (B=%lld, N=%lld)", (long long)B, (long long)N);
    if (B == 0) return 0;
    DFW_REQUIRE(case_ptr && out, "dfw_case_stress_summary: null case_ptr or output");
    DFW_REQUIRE(N == 0 || (pred && pos), "dfw_case_stress_summary: null pred or pos");
    SummaryWs w = carve_summary(ws, N, B);
    DFW_REQUIRE(ws && ws_bytes >= w.bytes, "dfw_case_stress_summary: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int64_t mc = max_chunks(N, B);
    k_chunk_scan<<<1, kScanBlock, 0, s>>>(case_ptr, B, N, mc, w.chunk_ptr);
    DFW_LAUNCH_CHECK();
    // every chunk of every case: the grid follows the total row count, not the largest case
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(mc, (int64_t)kNumSMs * 8));
    if (!mask) {
        k_chunk_minmax_y<<<grid, kScrThreads, 0, s>>>(pos, case_ptr, w.chunk_ptr, B, N, w.mm);
        DFW_LAUNCH_CHECK();
    }
    SummaryArgs a{};
    a.pred = pred; a.pos = pos; a.mask = mask; a.case_ptr = case_ptr; a.chunk_ptr = w.chunk_ptr; a.mm = w.mm; a.part = w.part;
    a.B = B; a.N = N; a.root_band = root_band; a.allowable = allowable_pa; a.log_scale = log_scale;
    if (dtype == DFW_F32)
        k_chunk_stats<float><<<grid, kScrThreads, 0, s>>>(a);
    else
        k_chunk_stats<__nv_bfloat16><<<grid, kScrThreads, 0, s>>>(a);
    DFW_LAUNCH_CHECK();
    const int fgrid = (int)std::max<int64_t>(1, std::min<int64_t>((B + 127) / 128, (int64_t)kNumSMs * 4));
    k_case_finalize<<<fgrid, 128, 0, s>>>(case_ptr, w.chunk_ptr, w.part, B, N, out);
    DFW_LAUNCH_CHECK();
    return 0;
}

extern "C" int dfw_case_ks_seed(const void* pred, int dtype, const float* pos, const uint8_t* mask, const int64_t* case_ptr, int64_t B,
                                int64_t N, double root_band, double rho, double* out, float* seed, void* ws, size_t ws_bytes,
                                dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_case_ks_seed: unknown dtype %d", dtype);
    DFW_REQUIRE(B >= 0 && N >= 0, "dfw_case_ks_seed: negative size (B=%lld, N=%lld)", (long long)B, (long long)N);
    DFW_REQUIRE(rho > 0.0 && rho < INFINITY, "dfw_case_ks_seed: rho must be positive and finite (got %g)", rho);
    if (B == 0) return 0;
    DFW_REQUIRE(case_ptr && out, "dfw_case_ks_seed: null case_ptr or output");
    DFW_REQUIRE(N == 0 || (pred && seed && (pos || mask)), "dfw_case_ks_seed: null pred, seed or pos");
    SummaryWs w = carve_summary(ws, N, B);
    DFW_REQUIRE(ws && ws_bytes >= w.bytes, "dfw_case_ks_seed: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int64_t mc = max_chunks(N, B);
    k_chunk_scan<<<1, kScanBlock, 0, s>>>(case_ptr, B, N, mc, w.chunk_ptr);
    DFW_LAUNCH_CHECK();
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(mc, (int64_t)kNumSMs * 8));
    if (!mask) {
        k_chunk_minmax_y<<<grid, kScrThreads, 0, s>>>(pos, case_ptr, w.chunk_ptr, B, N, w.mm);
        DFW_LAUNCH_CHECK();
    }
    KsArgs a{};
    a.pred = pred; a.pos = pos; a.mask = mask; a.case_ptr = case_ptr; a.chunk_ptr = w.chunk_ptr; a.mm = w.mm;
    a.part = reinterpret_cast<KsPart*>(w.part); a.seed = seed;
    a.B = B; a.N = N; a.root_band = root_band; a.rho = rho;
    if (dtype == DFW_F32)
        k_chunk_ks<float><<<grid, kScrThreads, 0, s>>>(a);
    else
        k_chunk_ks<__nv_bfloat16><<<grid, kScrThreads, 0, s>>>(a);
    DFW_LAUNCH_CHECK();
    const int fgrid = (int)std::max<int64_t>(1, std::min<int64_t>((B + 127) / 128, (int64_t)kNumSMs * 4));
    k_case_ks<<<fgrid, 128, 0, s>>>(w.chunk_ptr, a.part, B, rho, out);
    DFW_LAUNCH_CHECK();
    if (dtype == DFW_F32)
        k_chunk_ks_seed<float><<<grid, kScrThreads, 0, s>>>(a);
    else
        k_chunk_ks_seed<__nv_bfloat16><<<grid, kScrThreads, 0, s>>>(a);
    DFW_LAUNCH_CHECK();
    return 0;
}

extern "C" int dfw_case_column_sums(const float* a, int64_t N, int64_t C, int64_t c0, int64_t nc, const int64_t* case_ptr, int64_t B,
                                    double* out, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(N >= 0 && C >= 0 && c0 >= 0 && nc >= 0 && B >= 0,
                "dfw_case_column_sums: negative size (N=%lld, C=%lld, c0=%lld, nc=%lld, B=%lld)", (long long)N, (long long)C,
                (long long)c0, (long long)nc, (long long)B);
    DFW_REQUIRE(c0 + nc <= C, "dfw_case_column_sums: columns [%lld, %lld) outside the %lld columns of a", (long long)c0,
                (long long)(c0 + nc), (long long)C);
    if (B == 0 || nc == 0) return 0;
    DFW_REQUIRE(case_ptr && out, "dfw_case_column_sums: null case_ptr or output");
    DFW_REQUIRE(N == 0 || a, "dfw_case_column_sums: null input");
    SummaryWs w = carve_summary(ws, N, B);
    DFW_REQUIRE(ws && ws_bytes >= w.bytes, "dfw_case_column_sums: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int64_t mc = max_chunks(N, B);
    k_chunk_scan<<<1, kScanBlock, 0, s>>>(case_ptr, B, N, mc, w.chunk_ptr);
    DFW_LAUNCH_CHECK();
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(mc, (int64_t)kNumSMs * 8));
    double* part = reinterpret_cast<double*>(w.part);
    for (int64_t j0 = 0; j0 < nc; j0 += kColGroup) {  // the chunk slots hold kColGroup columns: one pass per group
        const int ng = (int)std::min<int64_t>(kColGroup, nc - j0);
        k_chunk_colsum<<<grid, kScrThreads, 0, s>>>(a, C, c0 + j0, ng, case_ptr, w.chunk_ptr, B, N, part);
        DFW_LAUNCH_CHECK();
        const int fgrid = (int)std::max<int64_t>(1, std::min<int64_t>((B * ng + 127) / 128, (int64_t)kNumSMs * 4));
        k_case_colsum<<<fgrid, 128, 0, s>>>(w.chunk_ptr, part, B, ng, nc, j0, out);
        DFW_LAUNCH_CHECK();
    }
    return 0;
}
