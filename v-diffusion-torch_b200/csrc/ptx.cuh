// Thin inline-PTX layer for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA, TMEM
// alloc / ld / st, commit, fences) and the shared-memory / instruction descriptors UMMA consumes.
// Hand-written; no CUTLASS/CuTe dependency.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cuda.h>          // CUtensorMap (type only; the encoder is fetched at run time, no -lcuda)
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace vdt {

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier --------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a launch failure, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {   // ~2 s at 2 GHz
            printf("vdt: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", (int)blockIdx.x,
                   (int)threadIdx.x, smem_u32(bar), parity);
            __trap();
        }
    }
}

// ---- proxies / fences --------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {   // generic-proxy smem writes -> async proxy (UMMA/TMA)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMA ---------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
        "[%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3)
        : "memory");
}

// 2-D tile load delivered to the same smem offset of every CTA in `cta_mask` of the cluster; each
// destination CTA's mbarrier (same offset) receives the complete_tx for the bytes it got.
__device__ __forceinline__ void tma_load_2d_multicast(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                                      uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster "
        "[%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask)
        : "memory");
}

// CTA-pair (cta_group::2) TMA loads: data lands in the executing CTA's smem, the complete_tx goes to the
// mbarrier at the same offset in the pair's leader (even-ranked) CTA: clearing bit 24 of a shared::cluster
// address selects the leader's window.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ void tma_load_2d_2cta(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_2cta(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                                 int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], "
        "[%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1),
        "r"(c2), "r"(c3)
        : "memory");
}
// Arrive on the mbarrier at this smem offset in CTA `cta` of the cluster, without release semantics: no memory barrier
// is generated.  For hand-offs whose payload is not generic-proxy memory (e.g. "this warp's tcgen05.ld of the
// accumulator have completed": ordered by tcgen05.wait::ld and tcgen05.fence::before_thread_sync), where a release
// fence would only make the warp wait for its own global stores.
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint64_t* bar, uint32_t cta) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(smem_u32(bar)), "r"(cta)
        : "memory");
}
// 16-byte shared-memory accesses by 32-bit shared address (a pointer that went through integer arithmetic loses its
// address space and would be accessed with generic LD / ST, which take the slow path for shared memory)
__device__ __forceinline__ void sts_v4(uint32_t addr, const float4& v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds_v4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// One lane of a converged warp.  tcgen05.mma / tcgen05.commit are issued by one thread, but from warp-uniform code:
// when the whole warp walks the issue loop and only the instruction itself sits under `if (elect_one())`, the
// descriptors stay in uniform registers and each MMA costs a handful of instructions.  Under `if (lane == 0)` the
// compiler must assume divergence and wraps every UTCHMMA in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop (~20
// instructions per MMA), which bounds kernels whose MMAs are short (attention's 128x64x16: 32 cycles each).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred px;\n\t"
        "elect.sync _|px, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, px;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---- clusters ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---- TMEM --------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem, uint32_t ncols) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {          // same warp as alloc
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* slot_in_smem, uint32_t ncols) {   // same warp in both CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp receives lane (base_lane + i).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]),
        "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]),
        "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}

// ---- UMMA --------------------------------------------------------------------------------------
// Shared-memory matrix descriptor for a K-major bf16 tile stored as rows of 128 bytes (64 elements)
// with the 128-byte swizzle TMA writes (8-row / 1024-byte atoms): start>>4 | LBO(16B)=1 | SBO=1024B |
// version 1 (Blackwell) | layout SWIZZLE_128B.  Advancing K by 16 elements = +32 bytes = +2 in the
// start-address field.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// Same for an MN-major operand (the MMA's N -- or M -- index is the contiguous one in memory, e.g. V [key][d] as the
// B operand of P V): tiles of 64 MN-elements (one 128-byte swizzle row) x 8 K-rows = 1024 bytes; SBO = distance
// between consecutive groups of 8 K-rows (1024 B when the rows of one 64-wide chunk are stored back to back),
// LBO = distance between consecutive 64-element MN chunks.  Advancing K by 16 rows = +2048 bytes.
__device__ __forceinline__ uint64_t umma_desc_sw128_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// Instruction descriptor, kind::f16: D fp32, A/B both fp16 (format 0) or both bf16 (format 1), both
// K-major, M x N.
__host__ __device__ constexpr uint32_t umma_idesc_16(int m, int n, int fp16) {
    return (1u << 4) | ((fp16 ? 0u : 1u) << 7) | ((fp16 ? 0u : 1u) << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
           (static_cast<uint32_t>(m >> 4) << 24);
}
constexpr uint32_t kIdescBMajorMN = 1u << 16;   // B operand is MN-major (bit 15 would be the A operand)
__device__ __forceinline__ void umma_16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrives on the mbarrier once every previously issued MMA of this thread has completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// Same, arriving on the mbarrier at this smem offset in every CTA of `cta_mask`.
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask)
                 : "memory");
}

// CTA-pair MMA: D (2 x 128 rows, one half per CTA's TMEM) += A (each CTA's 128 rows) * B^T (each CTA holds
// half of the N rows).  Issued by one thread of the leader CTA; descriptors are CTA-relative.
__device__ __forceinline__ void umma_16_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask)
                 : "memory");
}

// 128-bit coherent global load.  Unlike ld.global.nc, neither nvcc nor ptxas may sink it below a later store
// that might alias, so a batch of these issued before the first store of a loop stays a batch in flight.
__device__ __forceinline__ float4 ldg_nc_v4_issue(const float* p) {
    float4 v;
    asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void compiler_fence() { asm volatile("" ::: "memory"); }

// ---- counter RNG ---------------------------------------------------------------------------------
// Philox4x32-10: four 32-bit words per (counter, key); used for on-device ancestral noise and for training dropout.
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += 0x9E3779B9u; key.y += 0xBB67AE85u;
    }
    return ctr;
}

// ---- small math --------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {   // 2^x, one MUFU op (max rel. error 2^-22), flushes denormals
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + __expf(-x)); }
// fp32 pair -> packed 16-bit operand pair.  fp16 saturates at +-65504 instead of overflowing to inf.
__device__ __forceinline__ uint32_t pack_16(float lo, float hi, int fp16) {
    if (fp16) {                                      // one F2FP.SATFINITE.F16.F32.PACK_AB: overflow clamps to +-65504
        uint32_t r;
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
        return r;
    }
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
// same without the saturation, for values known to be in range (softmax probabilities, normalised activations)
__device__ __forceinline__ uint32_t pack_16_inrange(float lo, float hi, int fp16) {
    if (fp16) {
        __half2 v = __floats2half2_rn(lo, hi);
        return *reinterpret_cast<uint32_t*>(&v);
    }
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint16_t cvt_16(float x, int fp16) {
    if (fp16) {
        uint16_t r;
        asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(r) : "f"(x));
        return r;
    }
    __nv_bfloat16 v = __float2bfloat16(x);
    return *reinterpret_cast<uint16_t*>(&v);
}

}  // namespace vdt
