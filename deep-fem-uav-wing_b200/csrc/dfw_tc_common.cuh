// Device + host helpers shared by the tcgen05 kernels (dfw_linear_tc.cu, dfw_linear_dw_tc.cu).
#pragma once
#include <cuda.h>

#include "dfw_common.cuh"

namespace dfw {
namespace tc {

constexpr int kChunkBytes = 128;  // one SWIZZLE_128B atom row

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// try_wait carries a suspend-time hint: the warp sleeps in hardware until the phase completes (or the hint expires) instead of
// polling every ~50 ns - the plain loop of the waiting warps took a third of the persistent linear's issue slots, which its
// epilogue needs (ncu r02: 4.3 M polls x ~5 instructions against 40 M epilogue instructions per launch).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t ok;
    uint32_t spins = 0;
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
        if (!ok && ++spins > (1u << 20)) {  // a legitimate wait lasts microseconds (a failed try_wait sleeps up to 20 us): protocol bug, fail loudly
            printf("dfw_linear_tc: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x, addr, parity);
            __trap();
        }
    } while (!ok);
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
// start>>4 [0,14) | LBO>>4 [16,30) (=1, unused for swizzled K-major) | SBO>>4 [32,46) (8 rows x 128 B = 1024 B)
// | version=1 [46,48) | layout_type=2 (SWIZZLE_128B) [61,64)
// K-major descriptor for a tile whose rows are CBYTES bytes (= the swizzle span): 128 -> SWIZZLE_128B (layout 2,
// 8 rows = 1024 B), 64 -> SWIZZLE_64B (layout 4, 8 rows = 512 B)
template <int CBYTES>
__device__ __forceinline__ uint64_t make_desc_k(uint32_t saddr) {
    constexpr uint64_t sbo = CBYTES * 8, layout = CBYTES == 128 ? 2 : 4;
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((sbo >> 4) << 32) | ((uint64_t)1 << 46) | (layout << 61);
}

template <bool TF32>
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (TF32) {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, "
        "[%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
        "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
        "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
        "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
        "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// Split form of tmem_ld32 for software pipelining: issue the load of the NEXT 32 columns, work on the current ones, and
// only then wait.  The wait names the destination registers as in/out operands, so no use of them can be scheduled
// above it.
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, "
        "[%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                   "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]),
                   "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]),
                   "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_st32_nowait(uint32_t taddr, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
        "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
        "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
        "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
        "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Sum `regions` accumulator regions (each `pitch` columns apart) into region 0, 32 columns at a time.
// The tensor core adds into its fp32 accumulator with truncation, so error grows linearly with the number of
// accumulations (measured: ~2e-8 relative per tcgen05.mma).  The 3xTF32 kernels therefore keep the large
// hi*hi products in one or two accumulators and all small cross terms in another, and combine them here in
// round-to-nearest fp32 (tools/tc_accuracy.py).
__device__ __forceinline__ void tmem_combine(uint32_t t_row, int ncols, int regions, int pitch) {
    for (int c0 = 0; c0 < ncols; c0 += 32) {
        float v[32];
        tmem_ld32(t_row + c0, v);
        for (int r = 1; r < regions; ++r) {
            float w[32];
            tmem_ld32(t_row + r * pitch + c0, w);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += w[j];
        }
        tmem_st32(t_row + c0, v);
    }
}
__device__ __forceinline__ void fence_tc_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_tc_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Low half of the 3xTF32 split of an ACTIVATION.  The tensor core reads an fp32 word as tf32 by ignoring the low 13
// mantissa bits, so the raw tile already IS a_hi = trunc_tf32(a): only a_lo = a - a_hi has to be written (exact in
// fp32; its own truncation to tf32 leaves a relative error <= 2^-21).  Saves the converter warps a third of their
// shared-memory traffic and the cvt.rna instructions (the converters' LDS/STS were 54 % of the L1 data pipe in dW).
__device__ __forceinline__ float4 tf32_lo(const float4& a) {
    float4 l;
    l.x = a.x - __uint_as_float(__float_as_uint(a.x) & 0xffffe000u);
    l.y = a.y - __uint_as_float(__float_as_uint(a.y) & 0xffffe000u);
    l.z = a.z - __uint_as_float(__float_as_uint(a.z) & 0xffffe000u);
    l.w = a.w - __uint_as_float(__float_as_uint(a.w) & 0xffffe000u);
    return l;
}

__device__ __forceinline__ uint32_t rna_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}

// One [128 rows x 128 B] box in SWIZZLE_128B layout: 16-byte chunk j of row r lives at r*128 + ((j ^ (r & 7)) << 4).
// A thread that owns row r touches 8 distinct bank groups per quarter-warp: conflict-free.
__device__ __forceinline__ uint32_t box_off(int r, int j) { return (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4)); }


enum { kMapSw128 = 0, kMapSw128Atom32 = 1, kMapSw64 = 2 };
int make_map(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int elt, int box_rows, int mode = kMapSw128);

}  // namespace tc
}  // namespace dfw
