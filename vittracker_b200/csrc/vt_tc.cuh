// Thin inline-PTX wrappers for the Blackwell (sm_100a) primitives the tensor-core kernels use:
// mbarrier, bulk async copy, TMEM allocation, tcgen05.ld / st / mma / commit and the shared-memory
// and instruction descriptors.  Field layouts follow the PTX ISA "tcgen05" chapter (cross-checked
// against the bit-field definitions in CUTLASS' cute/arch/mma_sm100_desc.hpp).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

namespace vt {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier -------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_inval(uint64_t* bar) { asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
    return ok != 0;
}
#ifdef VT_TC_WATCHDOG
// Development aid: a wait that does not return within ~2^22 polls records (block, warp, barrier address, parity, caller tag) and raises a
// global abort flag that makes every later wait return at once, so that a deadlocked kernel terminates and the records can be read.
__device__ int g_wd_abort;
__device__ int g_wd_n;
__device__ int g_wd_rec[256][6];
__device__ int g_wd_tag[40];           // per-warp progress tags of block 0 (set by the kernels)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    unsigned n = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (*reinterpret_cast<volatile int*>(&g_wd_abort)) return;
        if (++n == (1u << 22)) {
            if ((threadIdx.x & 31) == 0) {
                const int k = atomicAdd(&g_wd_n, 1);
                if (k < 256) {
                    g_wd_rec[k][0] = blockIdx.x; g_wd_rec[k][1] = threadIdx.x >> 5; g_wd_rec[k][2] = (int)smem_u32(bar);
                    g_wd_rec[k][3] = (int)parity; g_wd_rec[k][4] = (int)clock(); g_wd_rec[k][5] = 0;
                }
                __threadfence();
            }
        }
        if (n == (1u << 23)) { *reinterpret_cast<volatile int*>(&g_wd_abort) = 1; __threadfence(); return; }
    }
}
#else
// Spin on try_wait (a hardware-bounded suspend per try).  A suspend-time hint (mbarrier.try_wait ..., hint -> TRYWAIT + NANOSLEEP.SYNCS)
// was measured: every tcgen05 kernel got 1 - 3 % SLOWER (wake-up latency), so the plain spin stays.
// The loop doubles as an always-on watchdog: a wait that outlasts 2^26 tries (seconds; every legitimate wait here is far below a
// millisecond) is a protocol deadlock - the kernel traps (the launch fails with an error the host sees) instead of hanging the GPU.
#ifndef VT_MBAR_WATCHDOG_TRIES
#define VT_MBAR_WATCHDOG_TRIES (1u << 26)
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t n = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++n > VT_MBAR_WATCHDOG_TRIES) __trap();
    }
}
#endif

// ---- bulk async copy global -> shared (completes on an mbarrier with complete_tx) ---------------------
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMEM allocation (one full warp executes these) --------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ---- fences around thread synchronisation ------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- TMEM <-> registers, shape 32x32b: lane i of the warp <-> TMEM lane (base + i), N consecutive columns --
// A warp may only touch the lane quarter 32*(warp_id % 4) .. +31; taddr = base | lane << 16 | column.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&r)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&r)[4]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3])
                 : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
        "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
                 "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}

// width-generic forms (N = 4, 8 or 16 consecutive columns)
template <int N> __device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&r)[N]) {
    static_assert(N == 4 || N == 8 || N == 16, "tmem_ld width");
    if constexpr (N == 4) tmem_ld4(taddr, r);
    else if constexpr (N == 8) tmem_ld8(taddr, r);
    else tmem_ld16(taddr, r);
}
template <int N> __device__ __forceinline__ void tmem_st(uint32_t taddr, const uint32_t (&r)[N]) {
    static_assert(N == 4 || N == 8 || N == 16, "tmem_st width");
    if constexpr (N == 4) tmem_st4(taddr, r);
    else if constexpr (N == 8) tmem_st8(taddr, r);
    else tmem_st16(taddr, r);
}

// ---- descriptors -------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, SWIZZLE_NONE.  Addresses / offsets are encoded >> 4 (16-byte units).
//   K-major  operand (rows = M or N, 16-bit elements): element (r, k) lives at
//       start + (r / 8) * SBO + (r % 8) * 16 + (k / 8) * LBO + (k % 8) * 2
//   MN-major operand: element (mn, k) lives at
//       start + (mn / 8) * SBO + (mn % 8) * 2 + (k / 8) * LBO + (k % 8) * 16
__device__ __forceinline__ uint64_t smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;          // descriptor version 1 (Blackwell)
    return d;                        // base_offset 0, lbo_mode 0, layout_type 0 (no swizzle)
}
// Instruction descriptor for kind::f16: fp16 A and B, fp32 accumulate, M x N, A K-major.
__device__ __forceinline__ uint32_t instr_desc_f16(int M, int N, bool b_mn_major) {
    return (1u << 4)                          // c_format  = F32
           | (0u << 7) | (0u << 10)           // a_format = b_format = F16
           | (0u << 15)                       // a_major   = K
           | ((b_mn_major ? 1u : 0u) << 16)   // b_major
           | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- MMA issue (single thread) -----------------------------------------------------------------------
// D[tmem] (+)= A[smem desc] * B[smem desc]^T
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]^T     (A: lane = row, one 32-bit column holds K elements 2c, 2c+1)
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}
// Arrive on `bar` once every tcgen05 operation issued so far by this thread has completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- warp-convergent variants: every lane executes the statement, one elected lane performs it -----------
// (issuing from inside `if (lane == 0)` makes the compiler wrap each UTCHMMA in a per-lane waterfall loop)
__device__ __forceinline__ void mma_ts_elect(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mma_ss_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mma_commit_elect(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar))
        : "memory");
}
// arm `bar` with `bytes` and start the bulk copy, both by the elected lane
__device__ __forceinline__ void bulk_g2s_elect(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t.reg .b64 st;\n\telect.sync _|q, 0xffffffff;\n\t"
        "@q mbarrier.arrive.expect_tx.shared::cta.b64 st, [%3], %2;\n\t"
        "@q cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t}" ::"r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// for a stage that is many copies: arm the barrier ONCE with the stage's total, then start the copies (bulk_g2s, a copy per lane)
// (an mbarrier.arrive.expect_tx per copy costs the issuing warp ~200 cycles per copy: conv4's control warp spent more than half of
// an item's time arming 24 copies)
__device__ __forceinline__ void mbar_arrive_expect_tx_elect(uint64_t* bar, uint32_t bytes) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t.reg .b64 st;\n\telect.sync _|q, 0xffffffff;\n\t"
        "@q mbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
        : "memory");
}
// ---- fp32 -> fp16 hi/lo split ------------------------------------------------------------------------
// v ~= hi + lo with hi = fp16(v), lo = fp16(v - hi): ~22 significant bits for |v| well inside fp16 range.
// Two instructions per element: one packed conversion gives both hi halves, one mixed-precision FMA per element (sm_100
// fma.rn.f32.f16: an fp16 product accumulated onto an fp32 addend, exact here) gives v - hi without unpacking, one packed conversion
// gives both lo halves.
__device__ __forceinline__ void split_pack2(float v0, float v1, uint32_t& hi, uint32_t& lo) {
    float l0, l1;
    asm("{\n\t.reg .b16 h0, h1, m;\n\t"
        "cvt.rn.f16x2.f32 %0, %4, %3;\n\t"
        "mov.b32 {h0, h1}, %0;\n\t"
        "mov.b16 m, 0xBC00;\n\t"                       // -1.0
        "fma.rn.f32.f16 %1, h0, m, %3;\n\t"
        "fma.rn.f32.f16 %2, h1, m, %4;\n\t}"
        : "=&r"(hi), "=f"(l0), "=f"(l1)
        : "f"(v0), "f"(v1));
    asm("cvt.rn.f16x2.f32 %0, %2, %1;" : "=r"(lo) : "f"(l0), "f"(l1));
}

// The same split on the host, for the weight packers: fp16 bit patterns of hi and lo.
inline void split_f16(float v, uint16_t* hi, uint16_t* lo) {
    const __half h = __float2half_rn(v);
    const __half l = __float2half_rn(v - __half2float(h));
    memcpy(hi, &h, 2);
    memcpy(lo, &l, 2);
}
// Host: element (n, k) of a no-swizzle K-major UMMA operand [k/8][N][8], split into the hi and lo images
inline void put_kmajor_f16(uint8_t* hi, uint8_t* lo, int N, int n, int k, float v) {
    uint16_t h, l;
    split_f16(v, &h, &l);
    const size_t off = ((size_t)(k / 8) * N + n) * 16 + (k % 8) * 2;
    memcpy(hi + off, &h, 2);
    memcpy(lo + off, &l, 2);
}

}  // namespace tc
}  // namespace vt
