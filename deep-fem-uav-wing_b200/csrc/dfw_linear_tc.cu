// (c) fused node-wise linear on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
//   y = a1.w1^T (+ a2.w2^T) + bias ; out = residual + dropout(relu(layernorm(row_scale * y)))
//
// = SAGEConv's lin_l(mean) + lin_r(h) (PyG; reference call site model.py:90) with the epilogue of
// model.py:91-95, and - with transposed weights - the input-gradient contraction of the backward.
//
// Design (one CTA = one 128-row tile, full output row => LayerNorm stays inside the CTA):
//   warp 0   : TMA producer  - cp.async.bulk.tensor 2D boxes [128 rows x 128 B] of the activations and
//              [Hout rows x 128 B] of the weights, SWIZZLE_128B, into a ring of smem stages (mbarrier full/empty)
//   warp 1   : MMA issuer    - one elected thread issues tcgen05.mma (M=128, N=Hout, K=32 B) with the
//              accumulator in TMEM; tcgen05.commit releases the stage / signals the epilogue
//   warps 2-5: epilogue      - tcgen05.ld, one thread per output row: bias, LayerNorm (two-pass, the row
//              lives in that thread's TMEM lane: no cross-thread reduction), ReLU, dropout, residual, store.
//              In fp32 mode the same warps first act as CONVERTERS (see below).
//   bf16 : kind::f16, operands straight from TMA.
//   fp32 : 3xTF32 error-compensated split (kind::tf32): a = a_hi + a_lo, w = w_hi + w_lo with
//          x_hi = tf32(x), x_lo = tf32(x - x_hi);  D += a_lo.w_hi + a_hi.w_lo + a_hi.w_hi.  (weights: round to
//          nearest, pre-split; activations: the hardware's own truncation, see tf32_lo)
//          Per-element error ~2^-22, so results stay inside the 1e-5 fp32 parity bound where a single
//          TF32 pass (2^-11) would not.  Weights are pre-split by a tiny kernel; the activation split is
//          done in shared memory, in place, by the converter warps between the TMA and the MMA.
// Roofline: HBM (intensity 4H/(3b) flop/B is below the tensor ridge for H <= 256): DESIGN.md.
#include <cuda.h>

#include <algorithm>

#include <cstdlib>
#include <cstring>

#include "dfw_common.cuh"
#include "dfw_linear_tc.cuh"
#include "dfw_tc_common.cuh"

namespace dfw {
namespace tc {

constexpr int kThreads = 192;
constexpr int kTileM = 128;
constexpr int kMaxStages = 6;

struct Maps {
    CUtensorMap a[2];
    CUtensorMap w_hi[2];
    CUtensorMap w_lo[2];
    CUtensorMap res;  // the residual [N, Hout] tensor, boxes of [128 rows x 128 B]
};


// smem carve-up (all offsets from a 1024-aligned base)
struct Smem {
    uint32_t a_hi, a_lo, w_hi, w_lo, stage_bytes;
    uint32_t res, staging, nbuf;  // epilogue regions alias the pipeline stages (free once the last MMA has retired)
    uint32_t cvec, bars, total;
};
__host__ __device__ inline Smem carve(bool tf32, int Npad, int stages, int out_boxes) {
    Smem s;
    const uint32_t cb = tf32 ? 64u : 128u;                      // K bytes per pipeline stage (see kernel)
    const uint32_t a = kTileM * cb;                             // activation tile: 8 KB (fp32) / 16 KB (bf16)
    const uint32_t w = ((uint32_t)Npad * cb + 1023u) / 1024u * 1024u;
    const uint32_t box = kTileM * kChunkBytes;                  // epilogue boxes stay [128 rows x 128 B]
    s.a_hi = 0;
    s.a_lo = a;
    s.w_hi = tf32 ? 2 * a : a;
    s.w_lo = s.w_hi + w;
    s.stage_bytes = tf32 ? 2 * a + 2 * w : a + w;
    const uint32_t pipe = s.stage_bytes * stages;
    s.res = 0;
    s.staging = (uint32_t)out_boxes * box;
    const uint32_t left = pipe > s.staging ? (pipe - s.staging) / box : 0;
    s.nbuf = left > 4 ? 4 : left;
    s.cvec = pipe;
    s.bars = s.cvec + 4 * 256 * 4;
    s.total = s.bars + 8 * (3 * kMaxStages + 2) + 16;
    return s;
}

template <typename T, bool TF32>
__global__ void __launch_bounds__(kThreads) k_linear_tc(const __grid_constant__ Maps maps, const Args p) {
    constexpr int EPC = kChunkBytes / (int)sizeof(T);  // elements (columns) per 128-byte epilogue box: 32 fp32 / 64 bf16
    // Main-loop K chunk: 128 B (SWIZZLE_128B) for bf16, 64 B (SWIZZLE_64B) for fp32.  The fp32 stage holds four
    // tiles (a_hi, a_lo, w_hi, w_lo); with 64-byte chunks a stage is 32 KB, three stages fit in < 110 KB and TWO
    // CTAs share an SM, so the epilogue of one tile overlaps the main loop of another (one CTA per SM leaves the
    // epilogue latency - ~7 us per tile - fully exposed; measured with %globaltimer probes).
    constexpr int CB = TF32 ? 64 : 128;
    constexpr int KPC = CB / (int)sizeof(T);           // K elements per chunk
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment as an OFFSET into the shared window: the pointer keeps its address space, so the compiler
    // emits LDS/STS instead of generic LD/ST for the converters and the epilogue staging
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int out_boxes = p.Hout / EPC;
    const Smem L = carve(TF32, p.Npad, p.stages, out_boxes);
    float* cvec = reinterpret_cast<float*>(smem + L.cvec);  // [4][256]: bias, gamma, beta, rowdot_w
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + L.bars);
    uint64_t* empty = full + kMaxStages;
    uint64_t* conv = empty + kMaxStages;
    uint64_t* accum_full = conv + kMaxStages;
    uint64_t* res_full = accum_full + 1;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(res_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t m_base = (int64_t)blockIdx.x * kTileM;
    const int total_chunks = p.chunks[0] + p.chunks[1];
    // One chunk = one pipeline stage: the activation box of this CTA's rows plus the weight boxes of the same K range.
    // Every CTA loads its own weights: multicasting them over a thread-block cluster was measured slower (DESIGN.md section 4).
    const uint32_t stage_tx = (uint32_t)(kTileM * CB + p.Npad * CB * (TF32 ? 2 : 1));
    auto issue_chunk = [&](int c, int stage) {
        const int seg = c >= p.chunks[0];
        const int kc = (seg ? c - p.chunks[0] : c) * KPC;
        uint8_t* st = smem + (size_t)stage * L.stage_bytes;
        mbar_arrive_expect_tx(&full[stage], stage_tx);
        tma_load_2d(st + L.a_hi, &maps.a[seg], &full[stage], kc, (int)m_base);
        tma_load_2d(st + L.w_hi, &maps.w_hi[seg], &full[stage], kc, 0);
        if (TF32) tma_load_2d(st + L.w_lo, &maps.w_lo[seg], &full[stage], kc, 0);
    };
    int prefilled = 0;  // producer thread: chunks requested before the setup barrier
    if (warp == 0 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
            mbar_init(&conv[s], 128);
        }
        mbar_init(accum_full, 1);
        mbar_init(res_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // The first ring of loads needs neither TMEM nor the per-column constants: request it NOW, so the ~1 us of DRAM
        // latency runs under the rest of the setup (TMEM allocation, constant loads, the block-wide barrier) instead of
        // after it.
        prefilled = total_chunks < p.stages ? total_chunks : p.stages;
        for (int c = 0; c < prefilled; ++c) issue_chunk(c, c);
        prefetch_tmap(&maps.w_hi[0]);
        if (p.chunks[1]) {
            prefetch_tmap(&maps.a[1]);
            prefetch_tmap(&maps.w_hi[1]);
        }
        if (p.residual) prefetch_tmap(&maps.res);
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"((uint32_t)p.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (warp >= 2) {  // per-column constants -> smem (read back as broadcasts)
        for (int c = threadIdx.x - 64; c < p.Hout; c += 128) {
            cvec[c] = p.bias ? __ldg(p.bias + c) : 0.f;
            cvec[256 + c] = p.gamma ? __ldg(p.gamma + c) : 1.f;
            cvec[512 + c] = p.beta ? __ldg(p.beta + c) : 0.f;
            cvec[768 + c] = p.rowdot_w ? __ldg(p.rowdot_w + c) : 0.f;
        }
    }
    fence_tc_before();
    __syncthreads();
    fence_tc_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = prefilled == p.stages ? 0 : prefilled;
            uint32_t phase = prefilled == p.stages ? 1u : 0u;
            for (int c = prefilled; c < total_chunks; ++c) {
                mbar_wait(&empty[stage], phase ^ 1);
                issue_chunk(c, stage);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            if (p.residual) {
                // the pipeline stages are free once the last MMA has retired: reuse them for the residual tile
                mbar_wait(accum_full, 0);
                mbar_arrive_expect_tx(res_full, (uint32_t)(out_boxes * kTileM * kChunkBytes));
                for (int b = 0; b < out_boxes; ++b)
                    tma_load_2d(smem + L.res + (size_t)b * kTileM * kChunkBytes, &maps.res, res_full, b * EPC, (int)m_base);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            // cute::UMMA::InstrDescriptor: c_format F32 (1<<4) | a/b format (BF16=1, TF32=2) at [7,10)/[10,13) |
            // K-major A and B | N>>3 at [17,23) | M>>4 at [24,29)
            const uint32_t fmt = TF32 ? 2u : 1u;
            const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(p.Npad >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
            int stage = 0;
            uint32_t phase = 0;
            uint32_t accumulate = 0;
            // fp32: hi*hi products alternate between `nacc` accumulators, all cross terms go to one more
            // (see tmem_combine); bf16: a single accumulator
            uint32_t acc_main[2] = {0u, 0u}, acc_cross = 0u;
            const uint32_t t_cross = tmem_base + (uint32_t)(p.nacc * p.Npad);
            const uint64_t dbase = make_desc_k<CB>(0);  // every field but the 14-bit start address
            const bool stacked = TF32 && p.nacc == 1 && 2 * p.Npad <= 256 && L.w_lo == L.w_hi + (uint32_t)p.Npad * CB;
            const uint32_t idesc2 = (idesc & ~(0x3Fu << 17)) | ((uint32_t)((2 * p.Npad) >> 3) << 17);
            int kstep = 0;
            for (int c = 0; c < total_chunks; ++c) {
                mbar_wait(TF32 ? &conv[stage] : &full[stage], phase);
                fence_tc_after();
                const uint32_t st = smem_u32(smem + (size_t)stage * L.stage_bytes);
#pragma unroll
                for (int k = 0; k < CB / 32; ++k) {  // UMMA_K = 32 bytes (16 bf16 / 8 tf32); +32 B = +2 in the address field
                    const uint64_t a_hi = dbase + ((st + L.a_hi + k * 32) >> 4);
                    const uint64_t w_hi = dbase + ((st + L.w_hi + k * 32) >> 4);
                    if (TF32) {
                        const uint64_t a_lo = dbase + ((st + L.a_lo + k * 32) >> 4);
                        const uint64_t w_lo = dbase + ((st + L.w_lo + k * 32) >> 4);
                        if (stacked) {
                            // tcgen05.mma costs ~140 cycles per instruction here whatever N is (measured: issue/latency
                            // bound, not MAC bound), so use fewer, wider instructions: w_lo sits right behind w_hi in
                            // shared memory, hence ONE N = 2*Npad MMA yields a_hi.w_hi (columns [0,Npad): main accumulator)
                            // and a_hi.w_lo (columns [Npad,2Npad): cross accumulator); a second N = Npad MMA adds a_lo.w_hi.
                            umma<TF32>(tmem_base, a_hi, w_hi, idesc2, acc_cross);
                            umma<TF32>(t_cross, a_lo, w_hi, idesc, 1u);
                            acc_cross = 1u;
                        } else {
                            const int m = kstep % p.nacc;
                            umma<TF32>(t_cross, a_lo, w_hi, idesc, acc_cross);
                            umma<TF32>(t_cross, a_hi, w_lo, idesc, 1u);
                            umma<TF32>(tmem_base + (uint32_t)(m * p.Npad), a_hi, w_hi, idesc, acc_main[m]);
                            acc_cross = 1u;
                            acc_main[m] = 1u;
                            ++kstep;
                        }
                    } else {
                        umma<TF32>(tmem_base, a_hi, w_hi, idesc, accumulate);
                    }
                    accumulate = 1u;
                }
                umma_commit(&empty[stage]);  // frees the smem stage once these MMAs have read it
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            umma_commit(accum_full);
        }
    } else {
        // ===== converter (fp32 only) then epilogue: warps 2..5 =====
        const int et = threadIdx.x - 64;  // 0..127
        if (TF32) {
            int stage = 0;
            uint32_t phase = 0;
            for (int c = 0; c < total_chunks; ++c) {
                mbar_wait(&full[stage], phase);
                uint8_t* st = smem + (size_t)stage * L.stage_bytes;
                float4* hi = reinterpret_cast<float4*>(st + L.a_hi);
                float4* lo = reinterpret_cast<float4*>(st + L.a_lo);
#pragma unroll
                for (int i = 0; i < (kTileM * CB / 16) / 128; ++i) {  // position-preserving: swizzle-agnostic
                    const int idx = et + i * 128;
                    lo[idx] = tf32_lo(hi[idx]);
                }
                fence_proxy_async();  // generic-proxy writes -> visible to the tensor core's async proxy
                mbar_arrive(&conv[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }

        mbar_wait(accum_full, 0);
        fence_tc_after();
        const int q = warp & 3;  // TMEM lane quarter this warp may access
        const int r_in_tile = q * 32 + lane;
        const int64_t row = m_base + r_in_tile;
        const bool rok = row < p.N;
        const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16);
        const int H = p.Hout;
        const int n32 = H / 32;
        const float rs = (p.row_scale && rok) ? __ldg(p.row_scale + row) : 1.f;
        const bool ln = p.flags & DFW_EP_LAYERNORM;
        const bool relu = p.flags & DFW_EP_RELU, drop = p.flags & DFW_EP_DROPOUT;
        const uint32_t row_key = drop ? dropout_row_key(resolve_seed(p.seed, p.flags), (uint64_t)row) : 0u;
        const float4* bias4 = reinterpret_cast<const float4*>(cvec);
        const float4* gam4 = reinterpret_cast<const float4*>(cvec + 256);
        const float4* bet4 = reinterpret_cast<const float4*>(cvec + 512);
        const float4* rdw4 = reinterpret_cast<const float4*>(cvec + 768);
        uint8_t* stg = smem + L.staging;
        float mean = 0.f, rstd = 1.f;

        // y = (acc + bias) * row_scale for the 32 columns starting at c0
        auto finish_y = [&](int c0, float* v) {
#pragma unroll
            for (int g = 0; g < 8; ++g) {
                const float4 b = bias4[c0 / 4 + g];
                v[4 * g] = (v[4 * g] + b.x) * rs;
                v[4 * g + 1] = (v[4 * g + 1] + b.y) * rs;
                v[4 * g + 2] = (v[4 * g + 2] + b.z) * rs;
                v[4 * g + 3] = (v[4 * g + 3] + b.w) * rs;
            }
        };
        // write 32 fp32 values of this thread's row into a staging box (converted to T) at column c_in_box
        auto stage_row = [&](uint8_t* box, int c_in_box, const float* v) {
            if constexpr (sizeof(T) == 4) {
#pragma unroll
                for (int g = 0; g < 8; ++g)
                    *reinterpret_cast<float4*>(box + box_off(r_in_tile, c_in_box / 4 + g)) =
                        make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
            } else {
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    Vec16<T> u;
                    u.from_float(v + 8 * g);
                    *reinterpret_cast<uint4*>(box + box_off(r_in_tile, c_in_box / 8 + g)) = u.v;
                }
            }
        };
        // Output path: every epilogue warp owns tile rows q*32 .. q*32+31 end to end.  Its threads stage their rows in the
        // warp's PRIVATE 4 KB slice of one swizzled [128 rows x 128 B] box (conflict-free), then the warp writes the slice out
        // with coalesced 16-byte stores (8 lanes = one 128-byte segment of one row, 4 rows per instruction).  No TMA store, no
        // proxy fence, no barrier between the epilogue warps.  (Round 1 pushed every box through cp.async.bulk.tensor stores:
        // a [128 x 128 B] box is 128 separate row writes for the TMA unit and cost ~0.5 us of acquire / store per 32-column
        // group on the tile's critical path, profiles/r01c_lin_fwd_fp32_ncu_summary.txt.)
        const uint32_t out_row_bytes = (uint32_t)H * (uint32_t)sizeof(T);
        auto acquire_box = [&]() -> uint8_t* {
            __syncwarp();  // the read-back of this warp's slice for the previous box is done
            return stg;
        };
        auto release_box = [&](void* gbase, uint8_t* box, int col0) {
            __syncwarp();
            uint8_t* g = static_cast<uint8_t*>(gbase) + (size_t)col0 * sizeof(T) + (size_t)(lane & 7) * 16;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int r = q * 32 + it * 4 + (lane >> 3);
                const uint4 v = *reinterpret_cast<const uint4*>(box + box_off(r, lane & 7));
                if (m_base + r < p.N) *reinterpret_cast<uint4*>(g + (size_t)(m_base + r) * out_row_bytes) = v;
            }
        };
        // Every pass walks the row 32 columns at a time with the TMEM load of the NEXT group in flight while the
        // current one is worked on (the values are copied out of the load's registers first, so one register set per
        // region is enough).

        // ---- pass 1: sum the accumulator regions (3xTF32: hi*hi [+ hi*hi] + cross, round-to-nearest), y = (acc + bias) *
        // row_scale written BACK to region 0 (passes 2 and 3 read finished values), row sum for LayerNorm, and the
        // pre-activation tensor ----
        // Without LayerNorm and without a pre-activation output there is nothing to do between the passes: pass 3 sums the
        // regions itself (input-gradient, encoder and decoder linears: one TMEM round trip less).
        const int regions = TF32 ? p.nacc + 1 : 1;
        const bool y_in_tmem = ln || p.pre_out;
        if (y_in_tmem) {
            float s = 0.f;
            uint32_t ra[32], rb[32];
            tmem_ld32_issue(t_row, ra);
            if (regions > 1) tmem_ld32_issue(t_row + p.Npad, rb);
            uint8_t* box = nullptr;
            for (int g = 0; g < n32; ++g) {
                const int c0 = g * 32;
                float v[32];
                tmem_ld_wait(ra);
                if (regions > 1) {
                    tmem_ld_wait(rb);
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(ra[j]) + __uint_as_float(rb[j]);
                    if (regions > 2) {
                        float w[32];
                        tmem_ld32(t_row + 2 * p.Npad + c0, w);
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] += w[j];
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(ra[j]);
                }
                if (g + 1 < n32) {
                    tmem_ld32_issue(t_row + c0 + 32, ra);
                    if (regions > 1) tmem_ld32_issue(t_row + p.Npad + c0 + 32, rb);
                }
                finish_y(c0, v);
#pragma unroll
                for (int j = 0; j < 32; ++j) s += v[j];
                tmem_st32_nowait(t_row + c0, v);
                if (p.pre_out) {
                    if (c0 % EPC == 0) box = acquire_box();  // as late as possible: the store that used this buffer has had the whole group's math to finish reading it
                    stage_row(box, c0 % EPC, v);
                    if ((c0 + 32) % EPC == 0) release_box(p.pre_out, box, c0 / EPC * EPC);
                }
            }
            tmem_st_wait();
            mean = s / (float)H;
        }
        // ---- pass 2: variance around the mean (two-pass, like torch) ----
        if (ln) {
            float qs = 0.f;
            uint32_t ra[32];
            tmem_ld32_issue(t_row, ra);
            for (int g = 0; g < n32; ++g) {
                float v[32];
                tmem_ld_wait(ra);
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(ra[j]);
                if (g + 1 < n32) tmem_ld32_issue(t_row + (g + 1) * 32, ra);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float d = v[j] - mean;
                    qs = fmaf(d, d, qs);
                }
            }
            rstd = rsqrtf(qs / (float)H + p.eps);
            if (p.ln_stats && rok) {
                p.ln_stats[2 * row] = mean;
                p.ln_stats[2 * row + 1] = rstd;
            }
        }
        // ---- pass 3: normalise, ReLU, dropout, row-dot, residual, store ----
        if (p.residual) mbar_wait(res_full, 0);
        float dot = 0.f;
        {
            const bool sum_here = !y_in_tmem && regions > 1;
            uint32_t ra[32], rb[32];
            tmem_ld32_issue(t_row, ra);
            if (sum_here) tmem_ld32_issue(t_row + p.Npad, rb);
            uint8_t* box = nullptr;
            for (int g = 0; g < n32; ++g) {
                const int c0 = g * 32;
                const int ob = c0 / EPC, h = (c0 % EPC) / 32;
                const uint8_t* rbox = smem + L.res + (size_t)ob * kTileM * kChunkBytes;
                float v[32];
                tmem_ld_wait(ra);
                if (sum_here) {
                    tmem_ld_wait(rb);
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(ra[j]) + __uint_as_float(rb[j]);
                    if (regions > 2) {
                        float w[32];
                        tmem_ld32(t_row + 2 * p.Npad + c0, w);
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] += w[j];
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(ra[j]);
                }
                if (g + 1 < n32) {
                    tmem_ld32_issue(t_row + c0 + 32, ra);
                    if (sum_here) tmem_ld32_issue(t_row + p.Npad + c0 + 32, rb);
                }
                if (!y_in_tmem) finish_y(c0, v);
                if (ln) {
#pragma unroll
                    for (int g4 = 0; g4 < 8; ++g4) {
                        const float4 ga = gam4[c0 / 4 + g4], be = bet4[c0 / 4 + g4];
                        v[4 * g4] = (v[4 * g4] - mean) * rstd * ga.x + be.x;
                        v[4 * g4 + 1] = (v[4 * g4 + 1] - mean) * rstd * ga.y + be.y;
                        v[4 * g4 + 2] = (v[4 * g4 + 2] - mean) * rstd * ga.z + be.z;
                        v[4 * g4 + 3] = (v[4 * g4 + 3] - mean) * rstd * ga.w + be.w;
                    }
                }
                if (relu) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
                }
                if (drop) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const uint32_t bits = dropout_bits(row_key, (uint32_t)(c0 + j));
                        v[j] = bits >= p.drop_thr ? v[j] * p.drop_scale : 0.f;
                    }
                }
                if (p.rowdot_out) {
#pragma unroll
                    for (int g4 = 0; g4 < 8; ++g4) {
                        const float4 w = rdw4[c0 / 4 + g4];
                        dot = fmaf(v[4 * g4], w.x, dot);
                        dot = fmaf(v[4 * g4 + 1], w.y, dot);
                        dot = fmaf(v[4 * g4 + 2], w.z, dot);
                        dot = fmaf(v[4 * g4 + 3], w.w, dot);
                    }
                }
                if (p.residual) {
                    if constexpr (sizeof(T) == 4) {
#pragma unroll
                        for (int g4 = 0; g4 < 8; ++g4) {
                            const float4 r4 = *reinterpret_cast<const float4*>(rbox + box_off(r_in_tile, h * 8 + g4));
                            v[4 * g4] += r4.x; v[4 * g4 + 1] += r4.y; v[4 * g4 + 2] += r4.z; v[4 * g4 + 3] += r4.w;
                        }
                    } else {
#pragma unroll
                        for (int g4 = 0; g4 < 4; ++g4) {
                            Vec16<T> u;
                            u.v = *reinterpret_cast<const uint4*>(rbox + box_off(r_in_tile, h * 4 + g4));
                            float f[8];
                            u.to_float(f);
#pragma unroll
                            for (int i = 0; i < 8; ++i) v[8 * g4 + i] += f[i];
                        }
                    }
                }
                if (p.out) {
                    if (c0 % EPC == 0) box = acquire_box();
                    stage_row(box, h * 32, v);
                    if ((c0 + 32) % EPC == 0) release_box(p.out, box, ob * EPC);
                }
            }
        }
        if (p.rowdot_out && rok) p.rowdot_out[row] = dot + (p.rowdot_b ? __ldg(p.rowdot_b) : 0.f);
    }

    fence_tc_before();
    __syncthreads();
    if (warp == 2) {
        fence_tc_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

// The three epilogue passes of one 128-row tile for ONE thread (= tile row `q*32 + lane`, whose accumulator lives in TMEM lane
// `q*32 + lane` from column `t_row`): y = (acc + bias) * row_scale, LayerNorm, ReLU, dropout, row-dot, residual, stores through the
// warp's private staging slice.  Used by the persistent kernel k_linear_tcp.
// Written lean on purpose: knock-out timing (DESIGN.md section 4) + the ncu source page showed the epilogue warps, not the main loop, pacing the
// persistent kernel (epilogue alone 114 us of the 134 us SAGE forward;
// main loop alone 77 us): ~6.4k warp instructions per tile and warp at ~0.2 IPC, a third of them address / predicate / branch
// overhead of the write-back (64-bit row bound checks and a reconvergence region per store, register copies of the prefetched
// residual, special registers re-read per round), and a quarter of the stall samples on the residual loads, requested one
// 64-byte round (~200 clk) ahead.  Here: FULL tiles carry no row predicates, every address is a per-tile lane pointer plus
// compile-time multiples of one step, the residual of a whole 32-column group is requested BEFORE the group's TMEM load and
// math (no copies: each round owns its registers), and main + cross accumulators are loaded with one wait
// (fp32 SAGE forward 134 -> 118 us, bf16 H = 256 on 2 M rows 1129 -> 986 us).
template <typename T, bool TF32, bool FULL>
__device__ __forceinline__ void epilogue_tile(const Args& p, const float* cvec, int HP, uint8_t* slice, uint32_t t_row, int64_t m_base, int q, int lane) {
    constexpr int SCOLS = 64 / (int)sizeof(T);  // columns per 64-byte staging round: 16 fp32 / 32 bf16
    constexpr int ROUNDS = 32 / SCOLS;          // rounds per 32-column group
    constexpr int EPS = 16 / (int)sizeof(T);    // elements per 16-byte slot
    const int H = p.Hout;
    const int n32 = H / 32;
    const bool ln = p.flags & DFW_EP_LAYERNORM, relu = p.flags & DFW_EP_RELU, drop = p.flags & DFW_EP_DROPOUT;
    const float4* bias4 = reinterpret_cast<const float4*>(cvec);
    const float4* gam4 = reinterpret_cast<const float4*>(cvec + HP);
    const float4* bet4 = reinterpret_cast<const float4*>(cvec + 2 * HP);
    const float4* rdw4 = reinterpret_cast<const float4*>(cvec + 3 * HP);
    const uint32_t row_bytes = (uint32_t)H * (uint32_t)sizeof(T);
    const bool y_in_tmem = ln || p.pre_out;
    // thread-per-row domain (TMEM lane = tile row)
    const int64_t row = m_base + q * 32 + lane;
    const bool rok = FULL || row < p.N;
    const bool has_rs = p.row_scale != nullptr;
    const float rs = (has_rs && rok) ? __ldg(p.row_scale + row) : 1.f;
    const uint32_t row_key = drop ? dropout_row_key(resolve_seed(p.seed, p.flags), (uint64_t)row) : 0u;
    // write-back domain: 4 lanes = one 64-byte row piece; iteration `it` handles warp row it*8 + (lane >> 2)
    const int jj = lane & 3, rr0 = lane >> 2;
    const int64_t wrow = m_base + q * 32 + rr0;
    const int nvalid = FULL ? 32 : (int)min((int64_t)32, max((int64_t)0, p.N - wrow));  // iteration `it` is in range iff it*8 < nvalid
    const size_t lane_off = (size_t)wrow * row_bytes + (size_t)jj * 16;
    const size_t step = (size_t)8 * row_bytes;
    uint8_t* const sts_row = slice + lane * 64;
    const int sts_sw = (lane >> 1) & 3;
    const uint8_t* const lds_ptr = slice + rr0 * 64 + ((jj ^ ((lane >> 3) & 3)) << 4);  // + it * 512 (the swizzle term does not depend on `it`)
    uint8_t* const out_lane = p.out ? static_cast<uint8_t*>(p.out) + lane_off : nullptr;
    uint8_t* const pre_lane = p.pre_out ? static_cast<uint8_t*>(p.pre_out) + lane_off : nullptr;
    const uint8_t* const res_lane = p.residual ? static_cast<const uint8_t*>(p.residual) + lane_off : nullptr;
    const bool has_res = res_lane != nullptr;
    // bf16: the residual is added to the fp32 epilogue value BEFORE the one rounding to bf16, as in the classic and SIMT kernels
    // (added after the packing it would round twice: up to 1.5 ulp).  So it is read in the thread-per-row domain, 64 contiguous
    // bytes of the thread's own row per round.  fp32 packs exactly, so it keeps the coalesced read of the write-back domain.
    constexpr bool kResInRow = sizeof(T) == 2;
    const uint8_t* const res_row = (kResInRow && has_res && rok) ? static_cast<const uint8_t*>(p.residual) + (size_t)row * row_bytes : nullptr;

    auto load_res = [&](const uint8_t* src, uint4 (&dst)[4]) {
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            if (FULL || it * 8 < nvalid) dst[it] = *reinterpret_cast<const uint4*>(src + it * step);
            else dst[it] = make_uint4(0u, 0u, 0u, 0u);
        }
    };
    // 64 bytes of this thread's row (pk) -> staging -> coalesced global store, + residual piece (rv) if given
    auto stage_and_store = [&](uint8_t* dst, const uint4 (&pk)[4], const uint4* rv) {
        __syncwarp();  // the previous round's read-back is done
#pragma unroll
        for (int j = 0; j < 4; ++j) *reinterpret_cast<uint4*>(sts_row + ((j ^ sts_sw) << 4)) = pk[j];
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            uint4 v = *reinterpret_cast<const uint4*>(lds_ptr + it * 512);
            if (rv) {
                const uint4 r4 = rv[it];
                if constexpr (sizeof(T) == 4) {
                    v.x = __float_as_uint(__uint_as_float(v.x) + __uint_as_float(r4.x));
                    v.y = __float_as_uint(__uint_as_float(v.y) + __uint_as_float(r4.y));
                    v.z = __float_as_uint(__uint_as_float(v.z) + __uint_as_float(r4.z));
                    v.w = __float_as_uint(__uint_as_float(v.w) + __uint_as_float(r4.w));
                } else {
                    Vec16<T> a, b;
                    a.v = v;
                    b.v = r4;
                    float fa[8], fb[8];
                    a.to_float(fa);
                    b.to_float(fb);
#pragma unroll
                    for (int e8 = 0; e8 < 8; ++e8) fa[e8] += fb[e8];
                    a.from_float(fa);
                    v = a.v;
                }
            }
            if (FULL || it * 8 < nvalid) *reinterpret_cast<uint4*>(dst + it * step) = v;
        }
    };
    auto pack = [&](const float* src, uint4 (&pk)[4]) {  // SCOLS values -> 64 bytes
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if constexpr (sizeof(T) == 4) {
                pk[j] = make_uint4(__float_as_uint(src[4 * j]), __float_as_uint(src[4 * j + 1]), __float_as_uint(src[4 * j + 2]), __float_as_uint(src[4 * j + 3]));
            } else {
                Vec16<T> u;
                u.from_float(src + EPS * j);
                pk[j] = u.v;
            }
        }
    };
    auto load_acc = [&](int c0, float* v) {  // hi*hi + cross terms, summed in round-to-nearest fp32 (see tmem_combine)
        if (TF32) {
            uint32_t ra[32], rb[32];
            tmem_ld32_issue(t_row + c0, ra);
            tmem_ld32_issue(t_row + p.Npad + c0, rb);
            tmem_ld_wait(ra);
            tmem_ld_wait(rb);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(ra[j]) + __uint_as_float(rb[j]);
        } else {
            tmem_ld32(t_row + c0, v);
        }
    };
    // y = (acc + bias) * row_scale for the 32 columns starting at c0
    auto finish_y = [&](int c0, float* v) {
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            const float4 b = bias4[c0 / 4 + g];
            v[4 * g] += b.x;
            v[4 * g + 1] += b.y;
            v[4 * g + 2] += b.z;
            v[4 * g + 3] += b.w;
        }
        if (has_rs) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= rs;
        }
    };
    float mean = 0.f, rstd = 1.f;
    // ---- pass 1: y written back to region 0, row sum, pre-activation tensor ----
    if (y_in_tmem) {
        float s = 0.f;
        for (int g = 0; g < n32; ++g) {
            const int c0 = g * 32;
            float v[32];
            load_acc(c0, v);
            finish_y(c0, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) s += v[j];
            tmem_st32_nowait(t_row + c0, v);
            if (pre_lane) {
#pragma unroll
                for (int h = 0; h < ROUNDS; ++h) {
                    uint4 pk[4];
                    pack(v + h * SCOLS, pk);
                    stage_and_store(pre_lane + (size_t)(c0 + h * SCOLS) * sizeof(T), pk, nullptr);
                }
            }
        }
        tmem_st_wait();
        mean = s / (float)H;
    }
    // ---- pass 2: variance around the mean (two-pass, like torch) ----
    if (ln) {
        float qs = 0.f;
        for (int g = 0; g < n32; ++g) {
            float v[32];
            tmem_ld32(t_row + g * 32, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const float d = v[j] - mean;
                qs = fmaf(d, d, qs);
            }
        }
        rstd = rsqrtf(qs / (float)H + p.eps);
        if (p.ln_stats && rok) {
            p.ln_stats[2 * row] = mean;
            p.ln_stats[2 * row + 1] = rstd;
        }
    }
    // ---- pass 3: normalise, ReLU, dropout, row-dot, (+ residual in the write-back), store ----
    float dot = 0.f;
    for (int g = 0; g < n32; ++g) {
        const int c0 = g * 32;
        uint4 rv[ROUNDS][4];
        if (has_res) {
            if constexpr (kResInRow) {
#pragma unroll
                for (int h = 0; h < ROUNDS; ++h)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        rv[h][j] = res_row ? *reinterpret_cast<const uint4*>(res_row + (size_t)(c0 + h * SCOLS) * sizeof(T) + j * 16)
                                           : make_uint4(0u, 0u, 0u, 0u);
            } else {
#pragma unroll
                for (int h = 0; h < ROUNDS; ++h) load_res(res_lane + (size_t)(c0 + h * SCOLS) * sizeof(T), rv[h]);
            }
        }
        float v[32];
        if (y_in_tmem) {
            tmem_ld32(t_row + c0, v);
        } else {
            load_acc(c0, v);
            finish_y(c0, v);
        }
        if (ln) {
#pragma unroll
            for (int g4 = 0; g4 < 8; ++g4) {
                const float4 ga = gam4[c0 / 4 + g4], be = bet4[c0 / 4 + g4];
                v[4 * g4] = (v[4 * g4] - mean) * rstd * ga.x + be.x;
                v[4 * g4 + 1] = (v[4 * g4 + 1] - mean) * rstd * ga.y + be.y;
                v[4 * g4 + 2] = (v[4 * g4 + 2] - mean) * rstd * ga.z + be.z;
                v[4 * g4 + 3] = (v[4 * g4 + 3] - mean) * rstd * ga.w + be.w;
            }
        }
        if (relu) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (drop) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const uint32_t bits = dropout_bits(row_key, (uint32_t)(c0 + j));
                v[j] = bits >= p.drop_thr ? v[j] * p.drop_scale : 0.f;
            }
        }
        if (p.rowdot_out) {
#pragma unroll
            for (int g4 = 0; g4 < 8; ++g4) {
                const float4 w = rdw4[c0 / 4 + g4];
                dot = fmaf(v[4 * g4], w.x, dot);
                dot = fmaf(v[4 * g4 + 1], w.y, dot);
                dot = fmaf(v[4 * g4 + 2], w.z, dot);
                dot = fmaf(v[4 * g4 + 3], w.w, dot);
            }
        }
        if constexpr (kResInRow) {
            if (has_res) {
#pragma unroll
                for (int h = 0; h < ROUNDS; ++h)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        Vec16<T> u;
                        u.v = rv[h][j];
                        float f[EPS];
                        u.to_float(f);
#pragma unroll
                        for (int i = 0; i < EPS; ++i) v[h * SCOLS + j * EPS + i] += f[i];
                    }
            }
        }
        if (out_lane) {
#pragma unroll
            for (int h = 0; h < ROUNDS; ++h) {
                uint4 pk[4];
                pack(v + h * SCOLS, pk);
                uint8_t* dst = out_lane + (size_t)(c0 + h * SCOLS) * sizeof(T);
                if (has_res && !kResInRow) stage_and_store(dst, pk, rv[h]);
                else stage_and_store(dst, pk, nullptr);
            }
        }
    }
    if (p.rowdot_out && rok) p.rowdot_out[row] = dot + (p.rowdot_b ? __ldg(p.rowdot_b) : 0.f);
}

// =====================================================================================================================
// Persistent variant: one CTA per SM loops over 128-row tiles.
//   * K chunks of 128 bytes (SWIZZLE_128B) for fp32 too: the TMA unit retires ~one box ROW per 2 clk whatever its width
//     (tools/probes/tma_rate_probe.cu: the SAGE-layer operand stream takes 72 us with 64-byte rows, 40 us with 128-byte rows),
//     so the 64-byte chunks that let two CTAs share an SM in k_linear_tc also capped its main loop.
//   * the accumulator is double-buffered in TMEM (2 x (main + cross) x Npad columns <= 512): two epilogue warpgroups take
//     alternate tiles, so a tile's three epilogue passes (~10 us) run under the main loops of the next TWO tiles, and no
//     wave quantisation is left (1563 tiles on 296 CTA slots were 5.28 -> 6 rounds).
//   * per-column constants are loaded once per CTA; outputs leave through per-warp staging slices and coalesced stores, the
//     residual is read (coalesced) in the same write-back loop instead of being re-staged through shared memory.
// Warps: 0 TMA producer, 1 MMA issuer, 2 TMEM owner, 4-7 / 8-11 epilogue warpgroups (even / odd tiles), 12-15 converters (fp32).
// =====================================================================================================================
constexpr int kPThreads = 512;
constexpr int kPStagesMax = 4;

struct PLayout {
    uint32_t a_hi, a_lo, w_hi, w_lo, stage_bytes, staging, cvec, bars, total;
};
__host__ __device__ inline PLayout pcarve(bool tf32, int Npad, int Hout, int stages) {
    PLayout L;
    const uint32_t a = kTileM * 128u;                                    // 16 KB activation box
    const uint32_t w = ((uint32_t)Npad * 128u + 1023u) / 1024u * 1024u;  // weight box of one 128-byte K chunk
    L.a_hi = 0;
    L.a_lo = a;
    L.w_hi = tf32 ? 2 * a : a;
    L.w_lo = L.w_hi + w;
    L.stage_bytes = tf32 ? 2 * a + 2 * w : a + w;
    L.staging = L.stage_bytes * (uint32_t)stages;    // 8 epilogue warps x [32 rows x 64 B]
    L.cvec = L.staging + 8u * 2048u;
    L.bars = L.cvec + 4u * (uint32_t)((Hout + 31) / 32 * 32) * 4u;
    L.total = L.bars + 8u * (3 * kPStagesMax + 4) + 16u;
    return L;
}

template <typename T, bool TF32>
__global__ void __launch_bounds__(kPThreads, 1) k_linear_tcp(const __grid_constant__ Maps maps, const Args p, const int num_tiles) {
    constexpr int KPC = 128 / (int)sizeof(T);   // K elements per 128-byte chunk
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const PLayout L = pcarve(TF32, p.Npad, p.Hout, p.stages);
    const int HP = (p.Hout + 31) / 32 * 32;
    float* cvec = reinterpret_cast<float*>(smem + L.cvec);  // [4][HP]: bias, gamma, beta, rowdot_w
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + L.bars);
    uint64_t* empty = full + kPStagesMax;
    uint64_t* conv = empty + kPStagesMax;
    uint64_t* acc_full = conv + kPStagesMax;   // [2]
    uint64_t* acc_empty = acc_full + 2;        // [2]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total_chunks = p.chunks[0] + p.chunks[1];
    const int nmine = ((int)blockIdx.x < num_tiles) ? (num_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int regions = TF32 ? 2 : 1;
    const uint32_t buf_cols = (uint32_t)(regions * p.Npad);

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
            mbar_init(&conv[s], 4);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        prefetch_tmap(&maps.a[0]);
        prefetch_tmap(&maps.w_hi[0]);
        if (p.chunks[1]) {
            prefetch_tmap(&maps.a[1]);
            prefetch_tmap(&maps.w_hi[1]);
        }
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int c = threadIdx.x; c < p.Hout; c += kPThreads) {
        cvec[c] = p.bias ? __ldg(p.bias + c) : 0.f;
        cvec[HP + c] = p.gamma ? __ldg(p.gamma + c) : 1.f;
        cvec[2 * HP + c] = p.beta ? __ldg(p.beta + c) : 0.f;
        cvec[3 * HP + c] = p.rowdot_w ? __ldg(p.rowdot_w + c) : 0.f;
    }
    fence_tc_before();
    __syncthreads();
    fence_tc_after();
    const uint32_t tmem_base = *tmem_ptr;

    // Register budget per warpgroup (512 threads x 128 at launch): the producer / MMA / converter warpgroups give registers back,
    // the two epilogue warpgroups take 168 each (setmaxnreg sits at the head of each role's branch so that ptxas allocates the
    // branch against the new limit).
    if (warp < 4) {
      if constexpr (TF32) asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
      if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            const uint32_t stage_tx = (uint32_t)(kTileM * 128 + p.Npad * 128 * (TF32 ? 2 : 1));
            int stage = 0;
            uint32_t phase = 0;
            for (int i = 0; i < nmine; ++i) {
                const int m_base = ((int)blockIdx.x + i * (int)gridDim.x) * kTileM;
                for (int c = 0; c < total_chunks; ++c) {
                    const int seg = c >= p.chunks[0];
                    const int kc = (seg ? c - p.chunks[0] : c) * KPC;
                    mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t* st = smem + (size_t)stage * L.stage_bytes;
                    mbar_arrive_expect_tx(&full[stage], stage_tx);
                    tma_load_2d(st + L.a_hi, &maps.a[seg], &full[stage], kc, m_base);
                    tma_load_2d(st + L.w_hi, &maps.w_hi[seg], &full[stage], kc, 0);
                    if (TF32) tma_load_2d(st + L.w_lo, &maps.w_lo[seg], &full[stage], kc, 0);
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
            }
        }
      } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            const uint32_t fmt = TF32 ? 2u : 1u;
            const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(p.Npad >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
            const uint32_t idesc2 = (idesc & ~(0x3Fu << 17)) | ((uint32_t)((2 * p.Npad) >> 3) << 17);  // [w_hi | w_lo] in one instruction
            const uint64_t dbase = make_desc_k<128>(0);
            int stage = 0;
            uint32_t phase = 0;
            for (int i = 0; i < nmine; ++i) {
                const int ab = i & 1;
                mbar_wait(&acc_empty[ab], (uint32_t)(((i >> 1) & 1) ^ 1));
                fence_tc_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)ab * buf_cols;
                uint32_t accumulate = 0;
                for (int c = 0; c < total_chunks; ++c) {
                    mbar_wait(TF32 ? &conv[stage] : &full[stage], phase);
                    fence_tc_after();
                    const uint32_t st = smem_u32(smem + (size_t)stage * L.stage_bytes);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {  // UMMA_K = 32 bytes
                        const uint64_t a_hi = dbase + ((st + L.a_hi + k * 32) >> 4);
                        const uint64_t w_hi = dbase + ((st + L.w_hi + k * 32) >> 4);
                        if (TF32) {
                            const uint64_t a_lo = dbase + ((st + L.a_lo + k * 32) >> 4);
                            umma<TF32>(d_tmem, a_hi, w_hi, idesc2, accumulate);            // main = a_hi.w_hi | cross = a_hi.w_lo
                            umma<TF32>(d_tmem + (uint32_t)p.Npad, a_lo, w_hi, idesc, 1u);  // cross += a_lo.w_hi
                        } else {
                            umma<TF32>(d_tmem, a_hi, w_hi, idesc, accumulate);
                        }
                        accumulate = 1u;
                    }
                    umma_commit(&empty[stage]);
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
                umma_commit(&acc_full[ab]);
            }
        }
      }
    } else if (warp >= 12) {
        // ===== converters (fp32): a_lo = a - trunc_tf32(a), in place beside the TMA tile =====
        if constexpr (TF32) asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
        if (TF32) {
            const int ct = threadIdx.x - 384;
            int stage = 0;
            uint32_t phase = 0;
            const int nchunks = nmine * total_chunks;
            for (int g = 0; g < nchunks; ++g) {
                mbar_wait(&full[stage], phase);
                uint8_t* st = smem + (size_t)stage * L.stage_bytes;
                const float4* hi = reinterpret_cast<const float4*>(st + L.a_hi);
                float4* lo = reinterpret_cast<float4*>(st + L.a_lo);
#pragma unroll
                for (int j = 0; j < (kTileM * 128 / 16) / 128; ++j) lo[ct + j * 128] = tf32_lo(hi[ct + j * 128]);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&conv[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        // ===== epilogue warpgroups: WG0 (warps 4-7) takes even tiles, WG1 (warps 8-11) odd tiles =====
        if constexpr (TF32) asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");  // (bf16 measured 8 % slower with the re-balancing: left alone)
        const int wg = (warp - 4) >> 2;
        const int q = warp & 3;  // TMEM lane quarter
        uint8_t* slice = smem + L.staging + (size_t)(warp - 4) * 2048;  // this warp's [32 rows x 64 B]

        for (int i = wg; i < nmine; i += 2) {
            const int64_t m_base = (int64_t)((int)blockIdx.x + i * (int)gridDim.x) * kTileM;
            const int ab = i & 1;
            mbar_wait(&acc_full[ab], (uint32_t)((i >> 1) & 1));
            fence_tc_after();
            const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)ab * buf_cols;

            if (m_base + kTileM <= p.N) epilogue_tile<T, TF32, true>(p, cvec, HP, slice, t_row, m_base, q, lane);
            else epilogue_tile<T, TF32, false>(p, cvec, HP, slice, t_row, m_base, q, lane);
            fence_tc_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[ab]);
        }
    }

    fence_tc_before();
    __syncthreads();
    if (warp == 2) {
        fence_tc_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

// ---- weight preparation: (optional transpose) + TF32 hi/lo split, or plain copy/transpose for bf16 ----
// One launch prepares BOTH operands' weights (blockIdx.y = operand): the per-call preparation used to be two
// ~3 us launches in front of every linear.
struct PrepArgs {
    const void* w[2];
    void* hi[2];
    void* lo[2];
    int rows[2], cols[2];
};
template <typename T>
__global__ void k_prep_weight(const PrepArgs a, int transpose, int split) {
    const int op = blockIdx.y;
    const T* __restrict__ w = static_cast<const T*>(a.w[op]);
    T* __restrict__ hi = static_cast<T*>(a.hi[op]);
    T* __restrict__ lo = static_cast<T*>(a.lo[op]);
    const int rows = a.rows[op], cols = a.cols[op];
    const int64_t n = (int64_t)rows * cols;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        // output index i over [orow, ocol] where out = transpose ? w^T : w
        const int ocols = transpose ? rows : cols;
        const int64_t orow = i / ocols, ocol = i % ocols;
        const T val = transpose ? w[ocol * cols + orow] : w[i];
        if constexpr (sizeof(T) == 4) {
            if (split) {
                const float h = __uint_as_float(rna_tf32(val));
                hi[i] = h;
                lo[i] = __uint_as_float(rna_tf32(val - h));
            } else {
                hi[i] = val;
            }
        } else {
            hi[i] = val;
        }
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

// 2D row-major [rows, cols] tensor, box = [box_rows x 128 bytes], SWIZZLE_128B
int make_map(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int elt, int box_rows, int mode) {
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return 1;
    }
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)cols * elt};
    const int inner_bytes = mode == kMapSw64 ? 64 : kChunkBytes;
    cuuint32_t box[2] = {(cuuint32_t)(inner_bytes / elt), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, elt == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim,
                     gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     mode == kMapSw128Atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : (mode == kMapSw64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B),
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld elt=%d box_rows=%d)", (int)r, (long long)rows,
                  (long long)cols, elt, box_rows);
        return 1;
    }
    return 0;
}

}  // namespace tc

// Called by dfw_linear_fwd / dfw_linear_bwd_input.  Returns -1 if the shape is not eligible for the
// tensor-core path (caller falls back to the SIMT kernel), 0 on success, >0 on error.
size_t linear_tc_ws_bytes(int64_t Hout, int64_t k1, int64_t k2, int dtype) {
    const size_t e = dtype == DFW_F32 ? 4 : 2;
    const size_t per = align_up((size_t)Hout * (size_t)(k1 > 0 ? k1 : 0) * e, 1024) + align_up((size_t)Hout * (size_t)(k2 > 0 ? k2 : 0) * e, 1024);
    return 2 * per + 1024;
}

bool linear_tc_eligible(int64_t N, int64_t Hout, int64_t k1, int64_t k2, int dtype, const void* a1, const void* a2) {
    const int e = dtype == DFW_F32 ? 4 : 2;
    if (N < 1 || Hout < 16 || Hout > 256 || Hout % 16 || (Hout * e) % 128) return false;
    if (k1 < 1 || (k1 * e) % 16 || (a2 && (k2 < 1 || (k2 * e) % 16))) return false;
    if (!aligned16(a1) || (a2 && !aligned16(a2))) return false;
    if (N >= (1LL << 31)) return false;
    return true;
}

// w1/w2 are given in [Hout, k] layout (transpose_w = 0) or [k, Hout] layout to be transposed (transpose_w = 1,
// used by the input-gradient contraction where the reduction runs over the weight's FIRST index).
int linear_tc_launch(const void* a1, const void* w1, int64_t k1, const void* a2, const void* w2, int64_t k2, int transpose_w,
                     tc::Args args, int dtype, void* ws, size_t ws_bytes, cudaStream_t s) {
    using namespace tc;
    const bool tf32 = dtype == DFW_F32;
    const int e = tf32 ? 4 : 2;
    const int64_t Hout = args.Hout;
    if (ws_bytes < linear_tc_ws_bytes(Hout, k1, a2 ? k2 : 0, dtype)) {
        set_error("linear_tc: workspace too small");
        return 1;
    }
    // carve the prepared-weight workspace
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~uintptr_t(1023));
    const size_t sz1 = align_up((size_t)Hout * k1 * e, 1024), sz2 = a2 ? align_up((size_t)Hout * k2 * e, 1024) : 0;
    void* hi[2] = {base, base + sz1};
    void* lo[2] = {base + sz1 + sz2, base + 2 * sz1 + sz2};
    const void* wsrc[2] = {w1, w2};
    const int64_t ks[2] = {k1, a2 ? k2 : 0};
    const void* wuse[2] = {w1, w2};
    if (tf32 || transpose_w) {
        const int nops = a2 ? 2 : 1;
        PrepArgs pa{};
        int64_t nmax = 0;
        for (int i = 0; i < nops; ++i) {
            pa.w[i] = wsrc[i];
            pa.hi[i] = hi[i];
            pa.lo[i] = lo[i];
            pa.rows[i] = transpose_w ? (int)ks[i] : (int)Hout;
            pa.cols[i] = transpose_w ? (int)Hout : (int)ks[i];
            nmax = std::max<int64_t>(nmax, (int64_t)pa.rows[i] * pa.cols[i]);
            wuse[i] = hi[i];
        }
        const dim3 pgrid((unsigned)std::min<int64_t>((nmax + 255) / 256, kNumSMs * 4), (unsigned)nops, 1);
        if (tf32) k_prep_weight<float><<<pgrid, 256, 0, s>>>(pa, transpose_w, 1);
        else k_prep_weight<__nv_bfloat16><<<pgrid, 256, 0, s>>>(pa, transpose_w, 0);
        DFW_LAUNCH_CHECK();
    }

    // ---- persistent variant (one CTA per SM, 128-byte K chunks, double-buffered accumulator) where its TMEM budget fits ----
    {
        // Measured A/B (tools/lin_ab.py, profiles/r02_linear_persistent_ab.json; us, classic -> persistent, L2 flushed):
        //   fp32 H=128 (config 2): SAGE forward train 140 -> 132, inference 116 -> 105, input gradient 107 -> 97, single operand 73 -> 64
        //   bf16 H=128 (config 5): 111 -> 104, 91 -> 77, 79 -> 69, 55 -> 44;  bf16 H=256, 2 M rows (config 4): 1128 -> 1131, 911 -> 821,
        //   790 -> 777, 548 -> 519;  fp32 H=64: 87 -> 81, 73 -> 63, 66 -> 56, 50 -> 42.
        // (Its first version lost 2-14 % on the two-operand shapes: the residual was read on demand inside the write-back loop,
        // ~1 us of exposed latency per 64-byte round; it is now requested one round ahead.)  DFW_TC_PERSIST=0 forces the classic kernel.
        static const int env_persist = [] { const char* e = getenv("DFW_TC_PERSIST"); return e ? atoi(e) : 1; }();
        const int Npad = (int)((Hout + 15) / 16 * 16);
        const int regions = tf32 ? 2 : 1;
        const int64_t tiles64 = (args.N + kTileM - 1) / kTileM;
        const bool want = env_persist != 0;
        if (want && 2 * regions * Npad <= 512 && Hout % 32 == 0 && tiles64 >= 2) {
            Maps pm;
            memset(&pm, 0, sizeof(pm));
            args.Npad = Npad;
            args.nacc = 1;
            int cols = 32;
            while (cols < 2 * regions * Npad) cols <<= 1;
            args.tmem_cols = cols;
            const void* as2[2] = {a1, a2};
            for (int i = 0; i < (a2 ? 2 : 1); ++i) {
                if (make_map(&pm.a[i], as2[i], args.N, ks[i], e, kTileM, kMapSw128)) return 1;
                if (make_map(&pm.w_hi[i], wuse[i], Hout, ks[i], e, Npad, kMapSw128)) return 1;
                if (tf32 && make_map(&pm.w_lo[i], lo[i], Hout, ks[i], e, Npad, kMapSw128)) return 1;
                args.chunks[i] = (int)((ks[i] * e + 127) / 128);
            }
            if (!a2) args.chunks[1] = 0;
            int stages = kPStagesMax;
            while (stages > 2 && pcarve(tf32, Npad, (int)Hout, stages).total + 1024 > 227 * 1024) --stages;
            if (pcarve(tf32, Npad, (int)Hout, stages).total + 1024 <= 227 * 1024) {
                args.stages = stages;
                const size_t psmem = pcarve(tf32, Npad, (int)Hout, stages).total + 1024;
                const unsigned grid = (unsigned)std::min<int64_t>(tiles64, kNumSMs);
                if (tf32) {
                    auto kern = k_linear_tcp<float, true>;
                    DFW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
                    kern<<<grid, kPThreads, psmem, s>>>(pm, args, (int)tiles64);
                } else {
                    auto kern = k_linear_tcp<__nv_bfloat16, false>;
                    DFW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
                    kern<<<grid, kPThreads, psmem, s>>>(pm, args, (int)tiles64);
                }
                DFW_LAUNCH_CHECK();
                return 0;
            }
        }
    }

    Maps maps;
    memset(&maps, 0, sizeof(maps));
    args.Npad = (int)((Hout + 15) / 16 * 16);
    // one hi*hi accumulator + one cross accumulator when that keeps TMEM <= 256 columns (two CTAs per SM);
    // two hi*hi accumulators otherwise if they fit (halves the truncation bias, see tmem_combine)
    args.nacc = !tf32 ? 1 : (2 * args.Npad <= 256 ? 1 : (3 * args.Npad <= 512 ? 2 : 1));
    const int acc_cols = tf32 ? (args.nacc + 1) * args.Npad : args.Npad;
    int cols = 32;
    while (cols < acc_cols) cols <<= 1;
    args.tmem_cols = cols;
    const void* as[2] = {a1, a2};
    for (int i = 0; i < (a2 ? 2 : 1); ++i) {
        const int mm = tf32 ? kMapSw64 : kMapSw128;  // main-loop chunk: 64 B for fp32, 128 B for bf16
        const int cb = tf32 ? 64 : 128;
        if (make_map(&maps.a[i], as[i], args.N, ks[i], e, kTileM, mm)) return 1;
        if (make_map(&maps.w_hi[i], wuse[i], Hout, ks[i], e, args.Npad, mm)) return 1;
        if (tf32 && make_map(&maps.w_lo[i], lo[i], Hout, ks[i], e, args.Npad, mm)) return 1;
        args.chunks[i] = (int)((ks[i] * e + cb - 1) / cb);
    }
    if (!a2) args.chunks[1] = 0;
    if (args.residual && make_map(&maps.res, args.residual, args.N, Hout, e, kTileM)) return 1;
    const int out_boxes = (int)(Hout * e / kChunkBytes);

    // stages: as many as fit; prefer <= ~110 KB so that two CTAs share an SM (epilogue of one overlaps the mainloop of the other)
    const int total_chunks = args.chunks[0] + args.chunks[1];
    // the epilogue aliases the pipeline: it needs room for the residual tile plus >= 1 staging box
    auto fits = [&](int st, size_t budget) {
        Smem L = carve(tf32, args.Npad, st, out_boxes);
        return L.total + 1024 <= budget && L.nbuf >= 1;
    };
    int stages = kMaxStages;
    while (stages > 2 && !fits(stages, 110 * 1024)) --stages;
    if (!fits(stages, 110 * 1024)) {
        stages = kMaxStages;
        while (stages > 2 && !fits(stages, 225 * 1024)) --stages;
    }
    if (!fits(stages, 225 * 1024)) {
        set_error("linear_tc: no shared-memory configuration for Hout=%lld", (long long)Hout);
        return 1;
    }
    // not more stages than K chunks, but keep enough bytes for the epilogue aliases
    while (stages > 2 && stages > total_chunks && fits(stages - 1, 225 * 1024)) --stages;
    args.stages = stages;
    const size_t smem = carve(tf32, args.Npad, stages, out_boxes).total + 1024;
    const unsigned tiles = (unsigned)((args.N + kTileM - 1) / kTileM);
    if (tf32) {
        auto kern = k_linear_tc<float, true>;
        DFW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<tiles, kThreads, smem, s>>>(maps, args);
    } else {
        auto kern = k_linear_tc<__nv_bfloat16, false>;
        DFW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<tiles, kThreads, smem, s>>>(maps, args);
    }
    DFW_LAUNCH_CHECK();
    return 0;
}

}  // namespace dfw
