// (b') neighbour aggregation of bf16 rows as a BLOCK-SPARSE product on the 5th-generation tensor cores.
//
// Same contract as dfw_sage_aggregate (PyG's index_select -> scatter_add_ -> / clamp(count, 1) behind SAGEConv(aggr='mean'),
// reference call site src/deep_fem_uav_wing/gnn/model.py:90), for the refined-mesh case (BASELINE.json config 4: 2 M nodes,
// 27 M edges, 512-byte bf16 rows) where the gather kernel is NOT bound by HBM: ncu (profiles/r01_ncu_summary_final.txt) shows
// DRAM traffic = A_min but 5x A_min crossing the L2 -> SM fabric, the L1 data pipe 80 % busy and 69 % issue utilisation -
// every edge moves a 512-byte row through the LSU and costs 8 FHADD per lane, so even a perfectly staged SIMT kernel stays
// near 0.31 ms of issue + 0.38 ms of LDS per launch against an HBM floor of 0.33 ms.
//
// Design: rows are cut into blocks of 128 consecutive destination rows.  A one-time plan (dfw_agg_plan_build) lists, per block,
// the ascending DISTINCT source rows it needs (S of them: 2.5 - 4.2 per output row on the config-4 lattice against 13.7 edges)
// and a 16-bit slot per edge.  Per block the mean is then the dense product
//        OUT[128, H] = ADJ[128, S] . X_staged[S, H]          (fp32 accumulation in TMEM, 1/deg applied in the epilogue)
// with ADJ the block's 0/1 (multiplicity) matrix.  Every staged row crosses the L2 -> SM fabric and the LSU ONCE per block
// (cp.async straight into the UMMA operand layout), the accumulation costs no SIMT instruction at all, and exactness is
// kept: ADJ entries are small integers and the products of a bf16 row with them are exact, sums are fp32 (the result differs
// from the CSR-order fp32 sum only by the association order: <= 1 bf16 ulp after the final rounding, tests/).
//
// One persistent CTA per SM, blocks taken in order blockIdx.x + i * gridDim.x (all SMs sweep the node array as one wavefront,
// so neighbouring blocks' shared sources hit L2).  Warp roles, all decoupled by mbarriers:
//   warp 0      loader    - 1-D bulk copies (cp.async.bulk) of the plan: per block its record (row offsets, S) and slots, per
//                           64-source chunk its 64 row indices into an 8-deep index ring
//   warp 1      MMA       - one thread: tcgen05.mma kind::f16, M = 128, N = H, K = 16 x 4 per chunk; A = ADJ chunk (K-major,
//                           SWIZZLE_128B), B = staged rows in their natural [node][feature] order = MN-major SWIZZLE_128B
//                           (the same layout dfw_linear_dw_tc.cu consumes); accumulator double-buffered in TMEM
//   warps 4-7   epilogue  - tcgen05.ld, * row_scale, -> bf16 -> swizzled staging box -> TMA store (block i drains while block
//                           i+1 accumulates)
//   warps 8-11  adjacency - thread m writes row m of the ADJ chunk (zero line + one 2-byte store per edge whose slot falls
//                           in the chunk)
//   warps 12-19 producers - cp.async 16 B per lane: 8 source rows per warp per chunk, written at the swizzled position
// Measured alternatives for the gather (config 4, k-d order, profiles/r02_aggregate_tc_notes.md): cp.async 16 B per lane (this
// version) 537-550 us; LDG.128 -> registers -> STS.128 with 16 producer warps 1184 us; TMA tile::gather4 (four rows x one
// 128-byte box column per instruction, tools/probes/gather4_probe.cu) 1481 us - the TMA unit retires one gather4 per ~70 clk.
// What bounds this version is the shared-memory / L1 data path: per 64-row chunk ~1000 LSU wavefronts (LDGSTS read + write
// sides 512, ADJ zeroing 128, epilogue staging 260, ADJ entries ~70) plus the tensor core's own operand reads (~380) in
// ~1650 clk (ncu r02f: l1tex data pipe 61 %, tensor pipe 32 %, DRAM traffic = A_min).
// Roofline: HBM.  Algorithmic bytes per launch  A_min = 2*N*H*2 + 4*E + 4*(N+1)  (SURVEY 8d; the plan actually reads
// 2 B per edge + 4 B per staged row instead of the CSR's 4 B per edge).
#include <cuda.h>

#include <algorithm>
#include <cstring>

#include "dfw_common.cuh"
#include "dfw_tc_common.cuh"

namespace dfw {
namespace tcagg {

using namespace tc;

constexpr int kBlockRows = 128;
constexpr int kChunk = 64;        // staged source rows (K) per pipeline stage
constexpr int kRecU16 = 136;      // uint16 per block record: S, #entries, chunk pointers [2 .. 2 + nchunks]; 272 B
constexpr int kPlanCap = 3072;    // edges per block the plan (and the kernel's slot buffer) can hold: mean degree <= 24
constexpr int kSortCap = 4096;    // power of two >= kPlanCap (bitonic sort in the plan build)
constexpr int kIdxRing = 8;
constexpr int kThreads = 640;
constexpr int kProducerWarps = 8;
constexpr int kOwnChunks = kBlockRows / kChunk;  // a block's first 128 staged rows are its own rows (plan slots 0 .. 127)
constexpr int kMaxStages = 3;      // measured on config 4 (k-d order): 2 / 3 / 4 stages = 638 / 537 / 549 us - not latency bound beyond 3
constexpr int kStagingBoxes = 1;  // shared memory goes to the pipeline (bytes in flight bound this kernel), not to the epilogue

struct Params {
    const int4* blk_meta;      // [nblocks] {src_off, S, slot_off, number of adjacency entries}
    const int32_t* plan_src;   // block b: plan_src[src_off .. src_off + round_up(max(S,1), 64))
    const uint16_t* plan_rec;  // [nblocks][kRecU16]
    const uint16_t* plan_slot; // block b: adjacency entries plan_slot[slot_off .. slot_off + nent), ordered by chunk
    const float* row_scale;    // fp32 [N] or NULL
    const uint8_t* x;          // bf16 [N, H]
    uint8_t* out;              // bf16 [N, H]
    int64_t N;
    int nblocks;
    int H;
    int stages;
};

struct Layout {
    uint32_t b_bytes, a_bytes, stage, staging, blkbuf, blkbuf_bytes, idx, flags, bars, total;
};
__host__ __device__ inline Layout carve(int H, int stages) {
    Layout L;
    L.b_bytes = (uint32_t)kChunk * (uint32_t)H * 2u;  // H/64 boxes of [64 rows x 128 B]
    L.a_bytes = kBlockRows * 128u;                    // [128 rows x 64 k] bf16
    L.stage = L.b_bytes + L.a_bytes;
    L.staging = L.stage * (uint32_t)stages;           // kStagingBoxes boxes [128 rows x 128 B] for the TMA stores
    L.blkbuf = L.staging + (uint32_t)kStagingBoxes * kBlockRows * 128u;
    L.blkbuf_bytes = 288u + kPlanCap * 2u;            // record (272 B, padded) + slots
    L.idx = L.blkbuf + 2u * L.blkbuf_bytes;
    L.flags = L.idx + kIdxRing * kChunk * 4u;
    L.bars = L.flags + kIdxRing * 8u;
    L.total = L.bars + 8u * (3 * kMaxStages + 2 * kIdxRing + 8) + 16u;
    return L;
}

__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ uint64_t make_desc_mn128(uint32_t saddr, uint32_t lbo_bytes) {  // bf16, MN-major, SWIZZLE_128B
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(1024 >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ int chunks_of(int S) { return (max(S, kBlockRows) + kChunk - 1) / kChunk; }
// mbarrier wait whose try_wait carries a suspend-time hint: the warp sleeps in hardware until the phase completes (or the
// hint expires) instead of spinning through issue slots - 16 of this kernel's 20 warps are waiting at any time, and the
// plain spin loop took half of all issue cycles (ncu r02c: 24 M + 19 M loop iterations per launch).
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t ok, spins = 0;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(addr), "r"(parity), "r"(20000u)
            : "memory");
        if (!ok && ++spins > (1u << 20)) {
            printf("dfw_aggregate_tc: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x, addr, parity);
            __trap();
        }
    } while (!ok);
}
#define mbar_wait mbar_wait_sleep

__global__ void __launch_bounds__(kThreads, 1) k_aggregate_tc(const __grid_constant__ CUtensorMap map_x, const Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const Layout L = carve(p.H, p.stages);
    int2* idx_flag = reinterpret_cast<int2*>(smem + L.flags);  // .x: 0 = end of stream, 1 = gathered chunk (64 indices in the ring slot), 2 = the block's OWN rows .y .. .y+63
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + L.bars);       // [stages]  producers (8) + adjacency warps (4)
    uint64_t* empty = full + kMaxStages;                               // [stages]  tcgen05.commit
    uint64_t* zfull = empty + kMaxStages;                              // [stages]  the ADJ tile of the stage has been zero-filled (TMA)
    uint64_t* idx_full = zfull + kMaxStages;                           // [ring]    loader (tx bytes)
    uint64_t* idx_empty = idx_full + kIdxRing;                         // [ring]    producer warps (8) + the tile producer
    uint64_t* blk_full = idx_empty + kIdxRing;                         // [2]       loader (tx bytes)
    uint64_t* blk_empty = blk_full + 2;                                // [2]       adjacency warps (4)
    uint64_t* acc_full = blk_empty + 2;                                // [2]       tcgen05.commit
    uint64_t* acc_empty = acc_full + 2;                                // [2]       epilogue threads (128)
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int H = p.H;
    const int nmine = ((int)blockIdx.x < p.nblocks) ? (p.nblocks - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const uint32_t tmem_cols = H > 128 ? 512u : (H > 64 ? 256u : 128u);

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full[s], kProducerWarps * 32 + 4 + 1);  // every producer lane (cp.async completion), the adjacency warps, the tile producer
            mbar_init(&empty[s], 1);
            mbar_init(&zfull[s], 1);
        }
        for (int r = 0; r < kIdxRing; ++r) {
            mbar_init(&idx_full[r], 1);
            mbar_init(&idx_empty[r], kProducerWarps + 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&blk_full[b], 1);
            mbar_init(&blk_empty[b], 4);
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], 128);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        prefetch_tmap(&map_x);
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_tc_before();
    __syncthreads();
    fence_tc_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===================== loader: plan -> shared memory (bulk copies, one thread) =====================
        if (lane == 0 && nmine > 0) {
            int g = 0;  // chunk counter of this CTA
            int4 meta_next = __ldg(p.blk_meta + blockIdx.x);
            for (int i = 0; i < nmine; ++i) {
                const int b = (int)blockIdx.x + i * (int)gridDim.x;
                const int4 meta = meta_next;
                if (i + 1 < nmine) meta_next = __ldg(p.blk_meta + b + gridDim.x);
                const int bb = i & 1;
                mbar_wait(&blk_empty[bb], (uint32_t)(((i >> 1) & 1) ^ 1));
                uint8_t* buf = smem + L.blkbuf + (size_t)bb * L.blkbuf_bytes;
                const uint32_t slot_bytes = ((uint32_t)meta.w * 2u + 15u) & ~15u;
                mbar_arrive_expect_tx(&blk_full[bb], kRecU16 * 2u + slot_bytes);
                bulk_g2s(buf, p.plan_rec + (size_t)b * kRecU16, kRecU16 * 2u, &blk_full[bb]);
                if (slot_bytes) bulk_g2s(buf + 288, p.plan_slot + meta.z, slot_bytes, &blk_full[bb]);
                const int nch = chunks_of(meta.y);
                for (int c = 0; c < nch; ++c, ++g) {
                    const int r = g % kIdxRing;
                    mbar_wait(&idx_empty[r], (uint32_t)(((g / kIdxRing) & 1) ^ 1));
                    if (c < kOwnChunks) {  // the block's own rows: consecutive, fetched as plain TMA tiles by the tile producer
                        idx_flag[r] = make_int2(2, b * kBlockRows + c * kChunk);
                        mbar_arrive(&idx_full[r]);
                    } else {
                        idx_flag[r] = make_int2(1, 0);
                        mbar_arrive_expect_tx(&idx_full[r], kChunk * 4u);
                        bulk_g2s(smem + L.idx + (size_t)r * kChunk * 4, p.plan_src + (size_t)meta.x + (size_t)c * kChunk, kChunk * 4u, &idx_full[r]);
                    }
                }
            }
            const int r = g % kIdxRing;  // end of stream
            mbar_wait(&idx_empty[r], (uint32_t)(((g / kIdxRing) & 1) ^ 1));
            idx_flag[r] = make_int2(0, 0);
            mbar_arrive(&idx_full[r]);
        } else if (lane == 0) {
            idx_flag[0] = make_int2(0, 0);
            mbar_arrive(&idx_full[0]);
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0 && nmine > 0) {
            // c_format F32 | A, B = BF16 | A K-major, B MN-major (bit 16) | N = H | M = 128
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(H >> 3) << 17) | ((uint32_t)(kBlockRows >> 4) << 24);
            const uint64_t abase = make_desc_k<128>(0);
            int stage = 0;
            uint32_t phase = 0;
            int s_next = __ldg(reinterpret_cast<const int*>(p.blk_meta + blockIdx.x) + 1);
            for (int i = 0; i < nmine; ++i) {
                const int b = (int)blockIdx.x + i * (int)gridDim.x;
                const int nch = chunks_of(s_next);
                if (i + 1 < nmine) s_next = __ldg(reinterpret_cast<const int*>(p.blk_meta + b + gridDim.x) + 1);
                const int ab = i & 1;
                mbar_wait(&acc_empty[ab], (uint32_t)(((i >> 1) & 1) ^ 1));
                fence_tc_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(ab * H);
                for (int c = 0; c < nch; ++c) {
                    mbar_wait(&full[stage], phase);
                    fence_proxy_async();
                    fence_tc_after();
                    const uint32_t st = smem_u32(smem + (size_t)stage * L.stage);
#pragma unroll
                    for (int ks = 0; ks < kChunk / 16; ++ks) {
                        const uint64_t adesc = abase + ((st + L.b_bytes + ks * 32) >> 4);
                        const uint64_t bdesc = make_desc_mn128(st + ks * 16 * 128, kChunk * 128);
                        umma<false>(d_tmem, adesc, bdesc, idesc, (c | ks) ? 1u : 0u);
                    }
                    umma_commit(&empty[stage]);
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
                umma_commit(&acc_full[ab]);
            }
        }
    } else if (warp == 3) {
        // ===================== tile producer (one thread, TMA only) =====================
        // Per chunk: (1) zero-fills the stage's ADJ tile with two fully out-of-bounds tile loads (the TMA unit writes zeros, no
        // global read, no LSU traffic - the adjacency warps used to spend 8 STS.128 + a named barrier per chunk on this);
        // (2) for the block's own rows (chunks 0, 1) loads the 64 consecutive rows as ordinary [64 rows x 128 B] tiles - a
        // third of all staged rows never touches the LSU.
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            const int nbox = H >> 6;
            const int oob_row = (int)min((int64_t)0x7ffffff0, p.N + 4096);
            for (int g = 0;; ++g) {
                const int r = g & (kIdxRing - 1);
                mbar_wait(&idx_full[r], (uint32_t)((g / kIdxRing) & 1));
                const int2 f = idx_flag[r];
                if (f.x == 0) break;
                mbar_wait(&empty[stage], phase ^ 1);
                uint8_t* st = smem + (size_t)stage * L.stage;
                mbar_arrive_expect_tx(&zfull[stage], L.a_bytes);
                tma_load_2d(st + L.b_bytes, &map_x, &zfull[stage], 0, oob_row);
                tma_load_2d(st + L.b_bytes + kChunk * 128, &map_x, &zfull[stage], 0, oob_row);
                if (f.x == 2) {
                    mbar_arrive_expect_tx(&full[stage], L.b_bytes);
                    for (int bx = 0; bx < nbox; ++bx) tma_load_2d(st + (size_t)bx * (kChunk * 128), &map_x, &full[stage], bx * 64, f.y);
                } else {
                    mbar_arrive(&full[stage]);
                }
                mbar_arrive(&idx_empty[r]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp >= 4 && warp < 8) {
        // ===================== epilogue =====================
        // Each warp owns TMEM lanes / block rows q*32 .. q*32+31 end to end: thread-per-row TMEM loads, a PRIVATE 4 KB slice
        // of the staging box (swizzled, conflict-free), then the warp writes the rows back out with fully coalesced
        // 16-byte stores (8 lanes = one 128-byte segment of one row).  No TMA store, no cross-warp barrier: the first version
        // pushed every [128 rows x 128 B] box through cp.async.bulk.tensor stores and spent ~12 us per block in the
        // epilogue (ncu r02c) - a box is 128 separate 128-byte row writes for the TMA unit.
        const int q = warp & 3;
        const int m = q * 32 + lane;
        uint8_t* box = smem + L.staging;
        const uint32_t row_bytes = (uint32_t)H * 2u;
        for (int i = 0; i < nmine; ++i) {
            const int b = (int)blockIdx.x + i * (int)gridDim.x;
            const int64_t row0 = (int64_t)b * kBlockRows;
            const int64_t row = row0 + m;
            const float rs = (row < p.N) ? (p.row_scale ? __ldg(p.row_scale + row) : 1.f) : 0.f;
            const int ab = i & 1;
            mbar_wait(&acc_full[ab], (uint32_t)((i >> 1) & 1));
            fence_tc_after();
            const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * H);
            uint32_t ra[32], rb[32];
            tmem_ld32_issue(t_row, ra);
            for (int cb = 0; cb < H / 64; ++cb) {
                tmem_ld32_issue(t_row + cb * 64 + 32, rb);
                __syncwarp();  // the read-back of the previous box is done
                tmem_ld_wait(ra);
#pragma unroll
                for (int g4 = 0; g4 < 4; ++g4) {
                    float f[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) f[j] = __uint_as_float(ra[8 * g4 + j]) * rs;
                    Vec16<__nv_bfloat16> u;
                    u.from_float(f);
                    *reinterpret_cast<uint4*>(box + box_off(m, g4)) = u.v;
                }
                if (cb + 1 < H / 64) tmem_ld32_issue(t_row + (cb + 1) * 64, ra);
                tmem_ld_wait(rb);
#pragma unroll
                for (int g4 = 0; g4 < 4; ++g4) {
                    float f[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) f[j] = __uint_as_float(rb[8 * g4 + j]) * rs;
                    Vec16<__nv_bfloat16> u;
                    u.from_float(f);
                    *reinterpret_cast<uint4*>(box + box_off(m, 4 + g4)) = u.v;
                }
                __syncwarp();
                uint8_t* orow = p.out + (size_t)cb * 128 + (size_t)(lane & 7) * 16;
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    const int r = q * 32 + it * 4 + (lane >> 3);
                    const uint4 v = *reinterpret_cast<const uint4*>(box + box_off(r, lane & 7));
                    if (row0 + r < p.N) *reinterpret_cast<uint4*>(orow + (size_t)(row0 + r) * row_bytes) = v;
                }
            }
            fence_tc_before();
            mbar_arrive(&acc_empty[ab]);
        }
    } else if (warp >= 8 && warp < 12) {
        // ===================== adjacency builder =====================
        // Per chunk: once the tile producer's TMA zero fill of the ADJ tile has landed, the chunk's plan entries (one per distinct
        // (source, row) pair, already ordered by chunk) are applied flat, one 2-byte store each - no per-row walk, no
        // divergence, no clearing by the LSU.  (The first version let thread m walk row m's slots with
        // data-dependent loops: ~900 clk per chunk, the bottleneck of the whole kernel - ncu r02e.)
        const int m = threadIdx.x - 256;
        int stage = 0;
        uint32_t phase = 0;
        for (int i = 0; i < nmine; ++i) {
            const int bb = i & 1;
            mbar_wait(&blk_full[bb], (uint32_t)((i >> 1) & 1));
            const uint8_t* buf = smem + L.blkbuf + (size_t)bb * L.blkbuf_bytes;
            const uint16_t* rec = reinterpret_cast<const uint16_t*>(buf);
            const uint16_t* ent = reinterpret_cast<const uint16_t*>(buf + 288);
            const int nch = chunks_of((int)rec[0]);
            for (int c = 0; c < nch; ++c) {
                mbar_wait(&zfull[stage], phase);  // the tile is free (its MMAs retired) AND zero-filled
                uint8_t* tile = smem + (size_t)stage * L.stage + L.b_bytes;
                const int t_end = rec[3 + c];
                for (int t = (int)rec[2 + c] + m; t < t_end; t += 128) {
                    const uint32_t e = ent[t];
                    const uint32_t kk = e & 63u, row = (e >> 6) & 127u, cnt = (e >> 13) + 1u;
                    const __nv_bfloat16 v = __float2bfloat16_rn((float)cnt);
                    *reinterpret_cast<__nv_bfloat16*>(tile + row * 128u + (((kk >> 3) ^ (row & 7u)) << 4) + (kk & 7u) * 2u) = v;
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&full[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&blk_empty[bb]);
        }
    } else if (warp >= 12) {
        // ===================== producers: staged rows -> MN-major SWIZZLE_128B boxes =====================
        const int pw = warp - 12;
        const int lpr = H >> 3;            // lanes per row (16-byte vectors per row): 32 / 16 / 8
        const int rpi = 32 / lpr;          // rows per warp instruction
        const int c16 = lane % lpr;        // this lane's 16-byte vector of the row
        const int rsub = lane / lpr;
        const uint32_t dcol = (uint32_t)(c16 >> 3) * (kChunk * 128u);  // feature box
        const uint32_t row_bytes = (uint32_t)H * 2u;
        const uint8_t* xl = p.x + (size_t)c16 * 16;
        int stage = 0;
        uint32_t phase = 0;
        for (int g = 0;; ++g) {
            const int r = g & (kIdxRing - 1);
            mbar_wait(&idx_full[r], (uint32_t)((g / kIdxRing) & 1));
            const int kind = idx_flag[r].x;
            if (kind == 0) break;
            if (kind == 2) {  // own rows: the tile producer fetches them; this lane only accounts for its arrival - in the
                // barrier's NEW phase: the stage's previous use must have been consumed first
                mbar_wait(&empty[stage], phase ^ 1);
                mbar_arrive(&full[stage]);
                __syncwarp();
                if (lane == 0) mbar_arrive(&idx_empty[r]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
                continue;
            }
            mbar_wait(&empty[stage], phase ^ 1);
            const int32_t* idx = reinterpret_cast<const int32_t*>(smem + L.idx + (size_t)r * kChunk * 4);
            const uint32_t sb = smem_u32(smem + (size_t)stage * L.stage) + dcol;
            for (int it = 0; it < 8 / rpi; ++it) {
                const int k = pw * 8 + it * rpi + rsub;
                const int src = idx[k];
                cp_async16(sb + (uint32_t)k * 128u + (uint32_t)(((c16 & 7) ^ (k & 7)) << 4), xl + (size_t)src * row_bytes);
            }
            // completion is signalled by the copy engine itself: every lane's arrive fires when ITS copies of this chunk have
            // landed (.noinc: it counts as one of the expected arrivals), so the warp never waits for data and all `stages`
            // chunks can be in flight.  (A first version waited with cp.async.wait_group 1 before arriving: at most two chunks
            // in flight whatever the stage count, ~1 us per chunk = the load latency / 2.)
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&full[stage])) : "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&idx_empty[r]);
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
    }

    fence_tc_before();
    __syncthreads();
    if (warp == 2) {
        fence_tc_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

// -------------------------------------------------------------------------------------------------------------------------
// plan build (one-time per graph)
// -------------------------------------------------------------------------------------------------------------------------
__global__ void k_plan_sizes(const int32_t* __restrict__ rowptr, int64_t N, int nblocks, int32_t* __restrict__ sz /*[2][nblocks]*/) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const int64_t r0 = (int64_t)b * kBlockRows, r1 = min(N, r0 + kBlockRows);
    const int ne = rowptr[r1] - rowptr[r0];
    sz[b] = (kBlockRows + ne + kChunk - 1) / kChunk * kChunk;  // own rows (always 128 slots) + at most one halo source per edge
    sz[nblocks + b] = (ne + 7) & ~7;
}
// exclusive scan of the two size arrays into blk_meta.x / .z (one CTA walks the blocks with a running carry)
__global__ void __launch_bounds__(1024) k_plan_scan(const int32_t* __restrict__ sz, int nblocks, int4* __restrict__ meta) {
    __shared__ int64_t warp_tot[2][32];
    __shared__ int64_t carry[2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x < 2) carry[threadIdx.x] = 0;
    __syncthreads();
    for (int base = 0; base < nblocks; base += 1024) {
        const int b = base + threadIdx.x;
        int64_t v[2] = {b < nblocks ? (int64_t)sz[b] : 0, b < nblocks ? (int64_t)sz[nblocks + b] : 0};
        int64_t inc[2] = {v[0], v[1]};
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t0 = __shfl_up_sync(0xffffffffu, inc[0], o), t1 = __shfl_up_sync(0xffffffffu, inc[1], o);
            if (lane >= o) { inc[0] += t0; inc[1] += t1; }
        }
        if (lane == 31) { warp_tot[0][wid] = inc[0]; warp_tot[1][wid] = inc[1]; }
        __syncthreads();
        int64_t off[2] = {carry[0], carry[1]};
        for (int w = 0; w < wid; ++w) { off[0] += warp_tot[0][w]; off[1] += warp_tot[1][w]; }
        if (b < nblocks) {
            int4 mm = meta[b];
            mm.x = (int)(off[0] + inc[0] - v[0]);
            mm.z = (int)(off[1] + inc[1] - v[1]);
            meta[b] = mm;
        }
        __syncthreads();
        if (threadIdx.x == 1023) { carry[0] = off[0] + inc[0]; carry[1] = off[1] + inc[1]; }
        __syncthreads();
    }
}
// one CTA per block: sort the block's edges by (own/halo, source, row), number the sources, emit the source list, the
// chunk-sorted adjacency entries and the record
//   slots     : the block's OWN rows always hold slots 0 .. 127 (slot = row - first row, used or not: the kernel fetches them as
//               two plain TMA tiles), the distinct HALO sources follow in ascending order from slot 128
//   plan_src  : source row of every slot, padded to a multiple of 64 with the last one (finite rows under zero ADJ columns)
//   plan_slot : one uint16 ENTRY per distinct (source, row) pair, ordered by (slot, row):  (count-1) << 13 | row << 6 | slot % 64
//               - exactly the stores the kernel's adjacency warps perform, chunk c = entries [cptr[c], cptr[c+1])
//   plan_rec  : [0] = S = 128 + #halo sources, [1] = number of entries, [2 .. 2 + nchunks] = cptr
__global__ void __launch_bounds__(256) k_plan_block(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t N, int4* __restrict__ meta,
                                                     int32_t* __restrict__ plan_src, uint16_t* __restrict__ plan_rec, uint16_t* __restrict__ plan_slot,
                                                     unsigned long long* __restrict__ status /*[0] max edges of a block, [1] sum of S*/) {
    __shared__ unsigned long long key[kSortCap];
    __shared__ uint16_t rowoff[kBlockRows + 1];
    __shared__ int wsum[2][8];
    __shared__ int s_total[2];
    __shared__ int cmin[kRecU16];
    const int b = blockIdx.x;
    const int64_t r0 = (int64_t)b * kBlockRows;
    const int nr = (int)min((int64_t)kBlockRows, N - r0);
    const int e0 = rowptr[r0];
    const int ne = rowptr[r0 + nr] - e0;
    int4 mm = meta[b];
    uint16_t* rec = plan_rec + (size_t)b * kRecU16;
    if (ne > kPlanCap) {  // the plan cannot hold this block: flag it (the caller keeps the gather kernel)
        if (threadIdx.x == 0) {
            atomicMax(status, (unsigned long long)ne);
            mm.y = 0;
            mm.w = 0;
            meta[b] = mm;
        }
        for (int t = threadIdx.x; t < kRecU16; t += 256) rec[t] = 0;
        return;
    }
    if (threadIdx.x == 0) atomicMax(status, (unsigned long long)ne);
    for (int t = threadIdx.x; t <= kBlockRows; t += 256) rowoff[t] = (uint16_t)(rowptr[r0 + min(t, nr)] - e0);
    for (int t = threadIdx.x; t < kRecU16; t += 256) {
        rec[t] = 0;
        cmin[t] = 0x7fffffff;
    }
    int P = 2;
    while (P < ne) P <<= 1;
    const unsigned long long kHalo = 1ull << 62;
    for (int t = threadIdx.x; t < P; t += 256) {
        unsigned long long k = ~0ull;
        if (t < ne) {
            const int c = col[e0 + t];
            const bool own = c >= r0 && c < r0 + nr;
            k = (own ? 0ull : kHalo) | ((unsigned long long)(uint32_t)c << 16) | (unsigned long long)t;
        }
        key[t] = k;
    }
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < P; t += 256) {
                const int u = t ^ j;
                if (u > t) {
                    const unsigned long long a = key[t], c = key[u];
                    const bool asc = (t & k) == 0;
                    if ((a > c) == asc) { key[t] = c; key[u] = a; }
                }
            }
            __syncthreads();
        }
    }
    // local edge index -> row of the block (the sort key's low half keeps CSR order, so equal sources come row by row)
    auto row_of = [&](int idx) {
        int lo = 0, hi = kBlockRows;  // largest r with rowoff[r] <= idx
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if ((int)rowoff[mid] <= idx) lo = mid; else hi = mid;
        }
        return lo;
    };
    auto src_of = [&](int t) { return (int)((key[t] >> 16) & 0xffffffffull); };
    auto is_halo = [&](int t) { return (key[t] & kHalo) != 0; };
    auto src_head = [&](int t) { return t == 0 || (key[t] >> 16) != (key[t - 1] >> 16); };
    auto ent_head = [&](int t) { return src_head(t) || row_of((int)(key[t] & 0xffffu)) != row_of((int)(key[t - 1] & 0xffffu)); };
    // two exclusive scans in one pass: distinct HALO sources (slot numbers from 128) and distinct (source, row) pairs (entry positions)
    const int per = (P + 255) / 256;
    const int t0 = threadIdx.x * per, t1 = min(t0 + per, ne);
    int local[2] = {0, 0};
    for (int t = t0; t < t1; ++t) {
        local[0] += (is_halo(t) && src_head(t)) ? 1 : 0;
        local[1] += ent_head(t) ? 1 : 0;
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc[2] = {local[0], local[1]};
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v0 = __shfl_up_sync(0xffffffffu, inc[0], o), v1 = __shfl_up_sync(0xffffffffu, inc[1], o);
        if (lane >= o) { inc[0] += v0; inc[1] += v1; }
    }
    if (lane == 31) { wsum[0][wid] = inc[0]; wsum[1][wid] = inc[1]; }
    __syncthreads();
    int off[2] = {inc[0] - local[0], inc[1] - local[1]};
    for (int w = 0; w < wid; ++w) { off[0] += wsum[0][w]; off[1] += wsum[1][w]; }
    if (threadIdx.x == 255) { s_total[0] = off[0] + local[0]; s_total[1] = off[1] + local[1]; }
    int hslot = off[0] - 1, epos = off[1] - 1;
    for (int t = t0; t < t1; ++t) {
        const bool halo = is_halo(t);
        if (halo && src_head(t)) {
            ++hslot;
            plan_src[(size_t)mm.x + kBlockRows + hslot] = src_of(t);
        }
        if (ent_head(t)) {
            ++epos;
            const int slot = halo ? kBlockRows + hslot : src_of(t) - (int)r0;
            const int row = row_of((int)(key[t] & 0xffffu));
            int cnt = 1;  // multiplicity of a duplicate edge: the run of equal (source, row) may continue into the next thread's piece
            for (int u = t + 1; u < ne && !ent_head(u); ++u) ++cnt;
            if (cnt > 8) atomicMax(status, 1ull << 40);  // more than the 3-bit field holds: the plan is unusable
            plan_slot[(size_t)mm.z + epos] = (uint16_t)((min(cnt, 8) - 1) << 13 | row << 6 | (slot & (kChunk - 1)));
            atomicMin(&cmin[slot / kChunk], epos);  // first entry of chunk slot / 64
        }
    }
    // own rows: slot i <-> row r0 + i (clamped inside the tensor for the ragged last block: those ADJ columns are empty)
    for (int t = threadIdx.x; t < kBlockRows; t += 256) plan_src[(size_t)mm.x + t] = (int32_t)min(r0 + t, N - 1);
    __syncthreads();
    const int S = kBlockRows + s_total[0], nent = s_total[1];
    const int padded = (S + kChunk - 1) / kChunk * kChunk;
    const int32_t fill = s_total[0] > 0 ? src_of(ne - 1) : (int32_t)min(r0 + kBlockRows - 1, N - 1);
    for (int t = S + threadIdx.x; t < padded; t += 256) plan_src[(size_t)mm.x + t] = fill;
    if (threadIdx.x == 0) {
        const int nch = padded / kChunk;
        int nxt = nent;  // chunks without entries (own rows nobody in the block points at) start where the next chunk starts
        rec[2 + nch] = (uint16_t)nent;
        for (int c = nch - 1; c >= 0; --c) {
            if (cmin[c] != 0x7fffffff) nxt = cmin[c];
            rec[2 + c] = (uint16_t)nxt;
        }
        rec[0] = (uint16_t)S;
        rec[1] = (uint16_t)nent;
        mm.y = S;
        mm.w = nent;
        meta[b] = mm;
        atomicAdd(status + 1, (unsigned long long)S);
    }
}

}  // namespace tcagg
}  // namespace dfw

// ---- C ABI -----------------------------------------------------------------------------------------------------------------
extern "C" int dfw_agg_plan_sizes(int64_t N, int64_t E, int64_t* nblocks, int64_t* src_cap, int64_t* slot_cap) {
    using namespace dfw;
    DFW_REQUIRE(N >= 0 && E >= 0 && nblocks && src_cap && slot_cap, "dfw_agg_plan_sizes: bad arguments");
    const int64_t nb = (N + tcagg::kBlockRows - 1) / tcagg::kBlockRows;
    *nblocks = nb;
    *src_cap = E + (tcagg::kBlockRows + tcagg::kChunk) * nb + tcagg::kChunk;
    *slot_cap = E + 8 * nb + 8;
    return 0;
}

extern "C" int dfw_agg_plan_build(const int32_t* rowptr, const int32_t* col, int64_t N, int64_t E, int32_t* blk_meta, int32_t* plan_src,
                                  uint16_t* plan_rec, uint16_t* plan_slot, uint64_t* status, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    using namespace dfw::tcagg;
    DFW_REQUIRE(N >= 0 && E >= 0, "dfw_agg_plan_build: negative size");
    DFW_REQUIRE(N < (1LL << 31) - 256 && E < (1LL << 31) - 256, "dfw_agg_plan_build: N and E must be < 2^31");
    if (N == 0) return 0;
    DFW_REQUIRE(rowptr && (col || E == 0) && blk_meta && plan_src && plan_rec && plan_slot && status, "dfw_agg_plan_build: null pointer");
    const int64_t nb = (N + kBlockRows - 1) / kBlockRows;
    DFW_REQUIRE(ws && ws_bytes >= (size_t)(2 * nb * 4), "dfw_agg_plan_build: workspace too small (need 8 bytes per block)");
    DFW_REQUIRE(aligned16(blk_meta) && aligned16(plan_src) && aligned16(plan_rec) && aligned16(plan_slot), "dfw_agg_plan_build: plan arrays must be 16-byte aligned");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    DFW_CUDA(cudaMemsetAsync(status, 0, 16, s));
    k_plan_sizes<<<(unsigned)((nb + 255) / 256), 256, 0, s>>>(rowptr, N, (int)nb, static_cast<int32_t*>(ws));
    DFW_LAUNCH_CHECK();
    k_plan_scan<<<1, 1024, 0, s>>>(static_cast<const int32_t*>(ws), (int)nb, reinterpret_cast<int4*>(blk_meta));
    DFW_LAUNCH_CHECK();
    k_plan_block<<<(unsigned)nb, 256, 0, s>>>(rowptr, col, N, reinterpret_cast<int4*>(blk_meta), plan_src, plan_rec, plan_slot,
                                              reinterpret_cast<unsigned long long*>(status));
    DFW_LAUNCH_CHECK();
    return 0;
}

extern "C" int dfw_agg_plan_max_block_edges(void) { return dfw::tcagg::kPlanCap; }

extern "C" int dfw_sage_aggregate_tc(const int32_t* blk_meta, const int32_t* plan_src, const uint16_t* plan_rec, const uint16_t* plan_slot,
                                     const float* row_scale, const void* x, void* out, int64_t N, int64_t H, int dtype, dfw_stream_t stream) {
    using namespace dfw;
    using namespace dfw::tcagg;
    DFW_REQUIRE(N >= 0, "dfw_sage_aggregate_tc: negative N");
    DFW_REQUIRE(dtype == DFW_BF16, "dfw_sage_aggregate_tc: bf16 rows only (dtype %d); fp32 rows use dfw_sage_aggregate", dtype);
    DFW_REQUIRE(H == 64 || H == 128 || H == 256, "dfw_sage_aggregate_tc: H must be 64, 128 or 256 (got %lld)", (long long)H);
    if (N == 0) return 0;
    DFW_REQUIRE(blk_meta && plan_src && plan_rec && plan_slot && x && out, "dfw_sage_aggregate_tc: null pointer");
    DFW_REQUIRE(aligned16(x) && aligned16(out), "dfw_sage_aggregate_tc: x/out must be 16-byte aligned");
    const int64_t nb = (N + kBlockRows - 1) / kBlockRows;
    Params p{};
    p.blk_meta = reinterpret_cast<const int4*>(blk_meta);
    p.plan_src = plan_src;
    p.plan_rec = plan_rec;
    p.plan_slot = plan_slot;
    p.row_scale = row_scale;
    p.x = static_cast<const uint8_t*>(x);
    p.N = N;
    p.nblocks = (int)nb;
    p.H = (int)H;
    int stages = kMaxStages;
    while (stages > 2 && carve((int)H, stages).total + 1024 > 227 * 1024) --stages;
    p.stages = stages;
    const size_t smem = carve((int)H, stages).total + 1024;
    p.out = static_cast<uint8_t*>(out);
    CUtensorMap map;
    memset(&map, 0, sizeof(map));
    if (tc::make_map(&map, x, N, H, 2, kChunk)) return 1;  // [64 rows x 64 features] tiles of x: the blocks' own rows + the zero fill
    auto kern = k_aggregate_tc;
    DFW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)std::min<int64_t>(nb, kNumSMs);
    kern<<<grid, kThreads, smem, reinterpret_cast<cudaStream_t>(stream)>>>(map, p);
    DFW_LAUNCH_CHECK();
    return 0;
}
