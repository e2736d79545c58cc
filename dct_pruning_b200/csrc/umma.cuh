// Thin inline-PTX layer for sm_100a tensor-core work: mbarrier, tcgen05.{alloc,mma,commit,ld,fence},
// cp.async.bulk, shared-memory matrix descriptors and the kind::f16 instruction descriptor.
//
// Field layouts follow the PTX ISA "tcgen05 matrix descriptor / instruction descriptor" tables:
//   smem descriptor : [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1
//                     | [49,52) base_offset | [61,64) swizzle (0 none, 2 128B, 4 64B, 6 32B)
//   instr descriptor: [4,6) D fmt (1=f32) | [7,10) A fmt (1=bf16) | [10,13) B fmt | [15] A MN-major
//                     | [16] B MN-major | [17,23) N>>3 | [24,29) M>>4
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace dctp {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// One probe: mbarrier.try_wait blocks in hardware until the phase completes or an implementation-defined time limit passes.
// (No suspend-time hint: with one, ptxas follows the probe with NANOSLEEP.SYNCS, which any barrier event of the CTA wakes up - in
//  a warp-specialised kernel with a barrier event every few hundred cycles the waiting warps then spin through ~10 instructions
//  per event: 40 % of the instructions score_stack_kernel executed, profiles/r02_ncu_stack_56x56.md.  Measured on one box, same
//  build otherwise: without the hint 56x56 3.71 vs 3.67 TB/s, 28x28 3.41 vs 3.35; a nanosleep of 20 or 60 ns between probes changes
//  nothing: the polls are not what bounds these kernels.)
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a descriptor or pipeline bug must not hang the GPU.  Legitimate waits are microseconds;
// after 2 s of wall clock (%globaltimer) the wait gives up and returns false (the caller records it in
// the status word and carries on to the exit path).
__device__ __forceinline__ uint64_t global_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return true;
    const uint64_t t0 = global_ns();
#pragma unroll 1
    for (;;) {
#pragma unroll 1
        for (int spin = 0; spin < 16; ++spin) {
#if defined(DCTP_POLL_NS) && DCTP_POLL_NS > 0
            __nanosleep(DCTP_POLL_NS);
#endif
            if (mbar_try_wait(bar, parity)) return true;
        }
        if (global_ns() - t0 > 2000000000ull) return false;
    }
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 1-D bulk async copy global -> shared (TMA engine, no tensor map): bytes % 16 == 0, both 16-B aligned
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Programmatic dependent launch: `launch_dependents` lets the next kernel of the stream (if it was launched with the
// programmatic-serialization attribute) start its prologue while this grid is still running; `grid_dependency_wait`
// blocks until the preceding grid has completed and its memory is visible.  Both are no-ops in a plain launch.
__device__ __forceinline__ void launch_dependents() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void grid_dependency_wait() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// 16-byte asynchronous copy global -> shared (LDGSTS, L2 only), grouped; the issuing thread sees the data after the wait
__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() {
    asm volatile("cp.async.commit_group;" ::: "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void cp_async_wait_but_one() {          // all groups but the most recent one have completed
    asm volatile("cp.async.wait_group 1;" ::: "memory");
}

// generic-proxy smem writes -> visible to the async proxy (tensor core operand reads)
__device__ __forceinline__ void fence_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// one lane of a converged warp (the compiler keeps the body on the uniform datapath)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem) {   // one full warp
    static_assert(kCols >= 32 && kCols <= 512 && (kCols & (kCols - 1)) == 0, "power of two in [32,512]");
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {          // same warp that allocated
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp receives lane (base_lane + i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {     // 32 lanes x 32 consecutive fp32 columns
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, "
        "%27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
          "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
          "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns, registers -> TMEM (thread i of the warp writes lane base_lane + i)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
        "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[16]) {   // first 8 registers -> 8 columns
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
                 "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// 16 lanes x 16 consecutive fp32 columns in the mma-fragment arrangement (probe P1, tools/probe_r2.cu): with t the thread
// index in the warp, v[4g + 0,1] = (lane base + t/4,     column 8g + 2(t%4) + 0,1)
//                    v[4g + 2,3] = (lane base + t/4 + 8, column 8g + 2(t%4) + 0,1)      (lane base: a multiple of 16)
__device__ __forceinline__ void tmem_ld_frag16(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_frag8(uint32_t taddr, uint32_t (&v)[4]) {      // 16 lanes x 8 columns
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x1.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
                 : "r"(taddr)
                 : "memory");
}
// registers -> 16 lanes x 8 (x2) / 4 (x1) consecutive 32-bit columns: v[2g + 0] = (lane base + t/4, column 4g + t%4),
// v[2g + 1] = (lane base + t/4 + 8, same column)   (probe P7)
__device__ __forceinline__ void tmem_st_frag8(uint32_t taddr, const uint32_t (&v)[4]) {
    asm volatile("tcgen05.st.sync.aligned.16x128b.x2.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_frag4(uint32_t taddr, uint32_t v0, uint32_t v1) {
    asm volatile("tcgen05.st.sync.aligned.16x128b.x1.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(v0), "r"(v1) : "memory");
}
// 2-D tiled TMA load (tensor map in kernel parameter space / __grid_constant__): box -> dense rows in shared memory,
// out-of-bounds rows arrive as zeros and still count towards the transaction bytes (probe P6)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
// named barrier over `threads` threads (ids 1..15; 0 is __syncthreads)
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// ---------------------------------------------------------------- descriptors
enum : uint32_t { SWIZZLE_NONE = 0, SWIZZLE_128B = 2, SWIZZLE_64B = 4, SWIZZLE_32B = 6 };

__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                   uint32_t swizzle) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= static_cast<uint64_t>(1) << 46;                 // descriptor version for sm_100
    d |= static_cast<uint64_t>(swizzle & 7) << 61;
    return d;
}
// advance the 14-bit start-address field by `bytes` (stays inside the same swizzle atom row / next atom)
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) {
    return desc + static_cast<uint64_t>(bytes >> 4);
}

// the 14-bit start-address field sits in the low word: advancing by `bytes` never carries out of it here
__device__ __forceinline__ uint64_t desc_with_lo(uint64_t desc, uint32_t lo) {
    return (desc & 0xFFFFFFFF00000000ull) | lo;
}

__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t M, uint32_t N, bool a_mn_major, bool b_mn_major) {
    return (1u << 4)                        // D = f32
           | (1u << 7)                      // A = bf16
           | (1u << 10)                     // B = bf16
           | ((a_mn_major ? 1u : 0u) << 15)
           | ((b_mn_major ? 1u : 0u) << 16)
           | ((N >> 3) << 17)
           | ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread for the CTA
__device__ __forceinline__ void mma_bf16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T : A is a 128-lane x K operand held in TMEM as packed bf16 pairs
// (column c of lane m holds A[m][2c], A[m][2c+1]), so it costs no shared-memory bandwidth
__device__ __forceinline__ void mma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when they have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------- bf16 hi/lo split
// x ~= hi + lo with hi = rn_bf16(x), lo = rn_bf16(x - hi): residual <= 2^-17 |x|
__device__ __forceinline__ void split2_packed(uint64_t ab, uint32_t& hi, uint32_t& lo);
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    // (the packed form: when a and b sit in an even/odd register pair - two components of a 128-bit load - the residuals cost
    //  one FADD2 instead of two FADDs; the bits are the same)
    split2_packed((static_cast<uint64_t>(__float_as_uint(b)) << 32) | __float_as_uint(a), hi, lo);
}

// the same split for an fp32 pair held in a 64-bit register pair (a in the low word): the residual comes from one packed
// subtraction (FADD2 on sm_100)
__device__ __forceinline__ void split2_packed(uint64_t ab, uint32_t& hi, uint32_t& lo) {
    const float a = __uint_as_float(static_cast<uint32_t>(ab)), b = __uint_as_float(static_cast<uint32_t>(ab >> 32));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
    const uint64_t h2 = (static_cast<uint64_t>(hi & 0xFFFF0000u) << 32) | static_cast<uint64_t>(hi << 16);
    uint64_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(ab), "l"(h2));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(__uint_as_float(static_cast<uint32_t>(r >> 32))), "f"(__uint_as_float(static_cast<uint32_t>(r))));
}
__device__ __forceinline__ uint64_t add2_packed(uint64_t x, uint64_t y) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(x), "l"(y));
    return r;
}
__device__ __forceinline__ uint64_t sub2_packed(uint64_t x, uint64_t y) {
    uint64_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(x), "l"(y));
    return r;
}
__device__ __forceinline__ uint64_t pack2(uint32_t lo_word, uint32_t hi_word) {
    return (static_cast<uint64_t>(hi_word) << 32) | lo_word;
}

}  // namespace umma
}  // namespace dctp
