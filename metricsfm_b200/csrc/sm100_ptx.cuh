// sm100_ptx.cuh — thin inline-PTX wrappers for the Blackwell (sm_100a) features the matcher uses:
// mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05 (alloc / mma.kind::i8 / commit / ld / fences).
#pragma once
#include <cstdint>
#include <cuda.h>

namespace msfm {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// The value, as something the compiler cannot re-derive: a loop-invariant address computed once before a loop stays in
// a register instead of being rematerialised (shared-window base, warp-index arithmetic) in every iteration.
__device__ __forceinline__ uint32_t opaque(uint32_t x) {
    asm volatile("mov.b32 %0, %0;" : "+r"(x));
    return x;
}

__device__ __forceinline__ uint32_t lane_id() {
    uint32_t l;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
    return l;
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- shared-memory access by 32-bit shared address
// (keeps the compiler from falling back to generic LD/ST with 64-bit address arithmetic)
__device__ __forceinline__ int lds_s32(uint32_t addr) {
    int v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ int4 lds_v4(uint32_t addr) {
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint2 lds_v2_volatile(uint32_t addr) {
    uint2 v;
    asm volatile("ld.volatile.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_v2_volatile(uint32_t addr, uint32_t x, uint32_t y) {
    asm volatile("st.volatile.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(x), "r"(y) : "memory");
}

// ---------------------------------------------------------------- mbarrier (by 32-bit shared address)
__device__ __forceinline__ bool mbar_try_wait_a(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
    while (!mbar_try_wait_a(bar, parity)) {
    }
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// Polling wait with back-off for the single-lane producer / MMA-issuer roles, so that their spinning does not steal
// issue slots from the epilogue warps that share the SM sub-partition.
template <unsigned kSleepNs = 20>
__device__ __forceinline__ void mbar_wait_backoff(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) __nanosleep(kSleepNs);
}

// Register re-balancing between warpgroups (4 consecutive, 4-aligned warps execute it together).
template <uint32_t kRegs>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegs)); }
template <uint32_t kRegs>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegs)); }

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tensormap(const void *tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
// 2-D tiled load: coordinates (c0 = innermost/byte column, c1 = row).
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const void *tmap, uint64_t *bar, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// 1-D bulk copy global -> shared (bytes multiple of 16, both addresses 16-byte aligned).
__device__ __forceinline__ void bulk_load_1d(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_result) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, 8-bit integer operands, int32 accumulate.
__device__ __forceinline__ void mma_i8_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Same, taking the low words of the two shared-memory descriptors (address >> 4; the high words are the constant
// SW128 / 1024-byte-stride fields): keeps the issuing loop free of 64-bit descriptor arithmetic.
template <bool kAccumulate>
__device__ __forceinline__ void mma_i8_ss_lo(uint32_t tmem_d, uint32_t desc_a_lo, uint32_t desc_b_lo, uint32_t idesc) {
    constexpr uint32_t kHi = (1024u >> 4) | (1u << 14) | (2u << 29);  // bits 32.. of make_smem_desc_sw128()
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %4};\n\t"
        "mov.b64 db, {%2, %4};\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], da, db, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(desc_a_lo), "r"(desc_b_lo), "r"(idesc), "r"(kHi), "n"(kAccumulate ? 1 : 0)
        : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes x 32 columns of 32-bit accumulators -> 32 registers per thread (thread = lane/row, register = column).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle, rows of exactly 128 bytes
// (one swizzle atom wide): 8-row groups are 1024 bytes apart (SBO), LBO unused.
//   bits [0,14)  start address >> 4        bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4   bits [46,48) descriptor version (1 on sm_100)
//   bits [61,64) layout type (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Instruction descriptor for kind::i8: u8 x u8 -> s32, both operands K-major, dense, no saturation.
//   [4,6) c_format = 2 (S32)   [7,10) a_format (0 = u8, 1 = s8)   [10,13) b_format
//   [15] a_major = 0 (K)  [16] b_major = 0 (K)  [17,23) N >> 3  [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_i8(uint32_t m, uint32_t n, uint32_t a_signed, uint32_t b_signed) {
    return (2u << 4) | (a_signed << 7) | (b_signed << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

}  // namespace ptx
}  // namespace msfm
