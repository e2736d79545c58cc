// What the tcgen05 score kernels share, on top of the inline-PTX layer (umma.cuh): the device status codes, the element types of
// the activation, the bf16 operand layouts and MMA issue helpers, the fp64 energy of a non-finite map, and the table of the
// activations a multi-site launch scores.  Each kernel header includes this one and no other score_*.cuh.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include "umma.cuh"

namespace dctp {

struct FastDiv {            // q = n / d for n < 2^32 / d
    uint32_t mul, d;
    __host__ void set(uint32_t div) { d = div; mul = static_cast<uint32_t>(0x100000000ull / div) + 1u; }
    __device__ __forceinline__ uint32_t div(uint32_t n) const { return d == 1 ? n : __umulhi(n, mul); }
};

enum : int { DCTP_DEV_OK = 0, DCTP_DEV_MMA_TIMEOUT = 1, DCTP_DEV_SMEM_ALIGN = 2 };

// element type of the activation a score kernel reads (the values of DCTP_DTYPE_* in include/dctp.h)
constexpr int IN_F32 = 0, IN_BF16 = 1, IN_F16 = 2;
__host__ __device__ constexpr int in_bytes(int in) { return in == IN_F32 ? 4 : 2; }

// element i of a 16-bit stream as fp32 (exact)
template <int IN>
__device__ __forceinline__ float in16_to_float(const uint16_t* x, long long i) {
    if constexpr (IN == IN_BF16) return __uint_as_float(static_cast<uint32_t>(x[i]) << 16);
    else return __half2float(__ushort_as_half(x[i]));
}
// two packed fp16 values (the first in the low half) as fp32
__device__ __forceinline__ float2 f16x2_to_float2(uint32_t p) {
    __half2 h;
    memcpy(&h, &p, 4);
    return __half22float2(h);
}

// A <= 64-row bf16 operand without swizzle (the stage-2 basis of score_stack.cuh, the Kronecker basis of score_kron.cuh): the
// 8-element k-chunk c of row n at c * LBO + n * 16 (LBO = 64 rows of 16 bytes + 16: the chunks of one row spread over the banks),
// BYTES for the hi or the lo part of a 64-deep operand
struct OperandImage64 {
    static constexpr uint32_t LBO = 64 * 16 + 16;
    static constexpr uint32_t BYTES = 8 * LBO;                           // 8320
};

namespace detail {

// byte offset of bf16 element (row, k) in a K-major SWIZZLE_128B operand with `rows` rows
__host__ __device__ __forceinline__ uint32_t kmajor_off(uint32_t row, uint32_t k, uint32_t rows) {
    uint32_t kb = k >> 6, kk = k & 63;
    return kb * (rows * 128u) + (row >> 3) * 1024u + (row & 7) * 128u + ((((kk >> 3) ^ row) & 7) << 4) + ((kk & 7) << 1);
}

__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// one float4 of the dense stream -> hi/lo operand bytes, scattered through the table entry
template <int VPE> struct Scatter;
template <> struct Scatter<1> {
    using Entry = uint16_t;
    __device__ static __forceinline__ void st(uint8_t* hi, uint8_t* lo, Entry e, const float4& v) {
        uint32_t h0, l0, h1, l1;
        umma::split2(v.x, v.y, h0, l0);
        umma::split2(v.z, v.w, h1, l1);
        *reinterpret_cast<uint2*>(hi + e) = make_uint2(h0, h1);
        *reinterpret_cast<uint2*>(lo + e) = make_uint2(l0, l1);
    }
};
template <> struct Scatter<2> {
    using Entry = uint32_t;        // two uint16 offsets
    __device__ static __forceinline__ void st(uint8_t* hi, uint8_t* lo, Entry e, const float4& v) {
        uint32_t h0, l0, h1, l1;
        umma::split2(v.x, v.y, h0, l0);
        umma::split2(v.z, v.w, h1, l1);
        const uint32_t o0 = e & 0xFFFFu, o1 = e >> 16;
        *reinterpret_cast<uint32_t*>(hi + o0) = h0;
        *reinterpret_cast<uint32_t*>(lo + o0) = l0;
        *reinterpret_cast<uint32_t*>(hi + o1) = h1;
        *reinterpret_cast<uint32_t*>(lo + o1) = l1;
    }
};
template <> struct Scatter<4> {
    using Entry = uint2;           // four uint16 offsets
    __device__ static __forceinline__ void st(uint8_t* hi, uint8_t* lo, Entry e, const float4& v) {
        uint32_t h0, l0, h1, l1;
        umma::split2(v.x, v.y, h0, l0);
        umma::split2(v.z, v.w, h1, l1);
        *reinterpret_cast<uint16_t*>(hi + (e.x & 0xFFFFu)) = static_cast<uint16_t>(h0);
        *reinterpret_cast<uint16_t*>(lo + (e.x & 0xFFFFu)) = static_cast<uint16_t>(l0);
        *reinterpret_cast<uint16_t*>(hi + (e.x >> 16)) = static_cast<uint16_t>(h0 >> 16);
        *reinterpret_cast<uint16_t*>(lo + (e.x >> 16)) = static_cast<uint16_t>(l0 >> 16);
        *reinterpret_cast<uint16_t*>(hi + (e.y & 0xFFFFu)) = static_cast<uint16_t>(h1);
        *reinterpret_cast<uint16_t*>(lo + (e.y & 0xFFFFu)) = static_cast<uint16_t>(l1);
        *reinterpret_cast<uint16_t*>(hi + (e.y >> 16)) = static_cast<uint16_t>(h1 >> 16);
        *reinterpret_cast<uint16_t*>(lo + (e.y >> 16)) = static_cast<uint16_t>(l1 >> 16);
    }
};

// three passes x KS k-steps of D (+)= A[smem] * B[smem]^T, straight-line (a runtime issue loop costs ~100 cycles of
// dependent uniform-datapath work per MMA, three times what the tensor core needs for it).
//   pass 0: A hi x B hi, pass 1: A lo x B hi, pass 2: A hi x B lo
// MN_MAJOR_A: the A operand advances 2048 B per k-step (MN-major), else 32 B inside / one slab across 64-element K blocks.
template <int KS, int KP, bool MN_MAJOR_A>
__device__ __forceinline__ void issue_ss3(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, uint64_t desc_a,
                                          uint64_t desc_b, uint32_t idesc, bool acc0 = false) {
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
        const uint32_t la = pass == 1 ? a_lo : a_hi, lb = pass == 2 ? b_lo : b_hi;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks)
            umma::mma_bf16_ss(d, umma::desc_with_lo(desc_a, la + (MN_MAJOR_A ? ks * 128 : (ks >> 2) * 1024 + (ks & 3) * 2)),
                              umma::desc_with_lo(desc_b, lb + (ks >> 2) * (KP * 8) + (ks & 3) * 2), idesc, acc0 || (pass | ks) != 0);
    }
}
template <int KP, bool MN_MAJOR_A>
__device__ __forceinline__ void issue_ss3_n(int ks, uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                            uint64_t desc_a, uint64_t desc_b, uint32_t idesc, bool acc0 = false) {
    switch (ks) {
        case 1: issue_ss3<1, KP, MN_MAJOR_A>(d, a_hi, a_lo, b_hi, b_lo, desc_a, desc_b, idesc, acc0); break;
        case 2: issue_ss3<2, KP, MN_MAJOR_A>(d, a_hi, a_lo, b_hi, b_lo, desc_a, desc_b, idesc, acc0); break;
        case 3: issue_ss3<3, KP, MN_MAJOR_A>(d, a_hi, a_lo, b_hi, b_lo, desc_a, desc_b, idesc, acc0); break;
        case 4: issue_ss3<4, KP, MN_MAJOR_A>(d, a_hi, a_lo, b_hi, b_lo, desc_a, desc_b, idesc, acc0); break;
        case 5: if constexpr (KP > 64) issue_ss3<5, KP, MN_MAJOR_A>(d, a_hi, a_lo, b_hi, b_lo, desc_a, desc_b, idesc, acc0); break;
        case 6: if constexpr (KP > 64) issue_ss3<6, KP, MN_MAJOR_A>(d, a_hi, a_lo, b_hi, b_lo, desc_a, desc_b, idesc, acc0); break;
        case 7: if constexpr (KP > 64) issue_ss3<7, KP, MN_MAJOR_A>(d, a_hi, a_lo, b_hi, b_lo, desc_a, desc_b, idesc, acc0); break;
        default: if constexpr (KP > 64) issue_ss3<8, KP, MN_MAJOR_A>(d, a_hi, a_lo, b_hi, b_lo, desc_a, desc_b, idesc, acc0); break;
    }
}

// one pass (one hi/lo operand pair) of a <= 64-deep product: ks k-steps, straight-line for each count
template <int KS, bool MN_MAJOR_A>
__device__ __forceinline__ void issue_ss_pass(uint32_t d, uint32_t la, uint32_t lb, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              bool acc_first) {
#pragma unroll
    for (int ks = 0; ks < KS; ++ks)
        umma::mma_bf16_ss(d, umma::desc_with_lo(desc_a, la + (MN_MAJOR_A ? ks * 128 : ks * 2)), umma::desc_with_lo(desc_b, lb + ks * 2), idesc,
                          acc_first || ks != 0);
}
template <bool MN_MAJOR_A>
__device__ __forceinline__ void issue_ss_pass_n(int ks, uint32_t d, uint32_t la, uint32_t lb, uint64_t desc_a, uint64_t desc_b,
                                                uint32_t idesc, bool acc_first) {
    switch (ks) {
        case 1: issue_ss_pass<1, MN_MAJOR_A>(d, la, lb, desc_a, desc_b, idesc, acc_first); break;
        case 2: issue_ss_pass<2, MN_MAJOR_A>(d, la, lb, desc_a, desc_b, idesc, acc_first); break;
        case 3: issue_ss_pass<3, MN_MAJOR_A>(d, la, lb, desc_a, desc_b, idesc, acc_first); break;
        default: issue_ss_pass<4, MN_MAJOR_A>(d, la, lb, desc_a, desc_b, idesc, acc_first); break;
    }
}

// one pass of a <= 64-deep product with the A operand in TMEM (packed bf16 pairs, 8 columns per k-step)
template <int KS>
__device__ __forceinline__ void issue_ts_pass(uint32_t d, uint32_t a_col, uint32_t lb, uint64_t desc_b, uint32_t idesc, bool acc_first) {
#pragma unroll
    for (int ks = 0; ks < KS; ++ks)
        umma::mma_bf16_ts(d, a_col + 8 * ks, umma::desc_with_lo(desc_b, lb + ks * 2), idesc, acc_first || ks != 0);
}
__device__ __forceinline__ void issue_ts_pass_n(int ks, uint32_t d, uint32_t a_col, uint32_t lb, uint64_t desc_b, uint32_t idesc,
                                                bool acc_first) {
    switch (ks) {
        case 1: issue_ts_pass<1>(d, a_col, lb, desc_b, idesc, acc_first); break;
        case 2: issue_ts_pass<2>(d, a_col, lb, desc_b, idesc, acc_first); break;
        case 3: issue_ts_pass<3>(d, a_col, lb, desc_b, idesc, acc_first); break;
        default: issue_ts_pass<4>(d, a_col, lb, desc_b, idesc, acc_first); break;
    }
}

// The fp64 energy of one map, recomputed from global memory.  The tensor-core kernels call it only when the fp32 energy they
// computed is not finite; a finite map gives a finite value unless its fp32 energy overflows, so clean inputs never get here.
// Kernels that put several maps into one MMA keep them apart with zero blocks in an operand, and 0 * NaN and 0 * Inf are NaN:
// a non-finite map turns the energies of the other maps of its tile non-finite too.  This tells the two apart: NaN if the
// N x N map at x (rows N floats apart) holds a NaN or an Inf - it is the culprit -, otherwise its sum of squares (Parseval: the
// orthonormal DCT keeps it), exactly 0 for a dead map.
__device__ __forceinline__ double map_energy64(const float* x, int N) {
    double s = 0.0;
#pragma unroll 1
    for (int i = 0; i < N * N; ++i) {
        const double e = x[i];
        if (!isfinite(e)) return __longlong_as_double(0x7FF8000000000000ll);
        s = fma(e, e, s);
    }
    return s;
}

}  // namespace detail

// detail::map_energy64 of map m of a dense stream of element type IN (x: the stream's first element)
template <int IN>
__device__ __forceinline__ double map_energy64_in(const void* x, long long m, int NN, int N) {
    if constexpr (IN == IN_F32) {
        return detail::map_energy64(static_cast<const float*>(x) + m * NN, N);
    } else {
        const uint16_t* p = static_cast<const uint16_t*>(x) + m * NN;
        double s = 0.0;
#pragma unroll 1
        for (int i = 0; i < N * N; ++i) {
            const double e = in16_to_float<IN>(p, i);
            if (!isfinite(e)) return __longlong_as_double(0x7FF8000000000000ll);
            s = fma(e, e, s);
        }
        return s;
    }
}

constexpr int SCORE_MAX_SEG = 16;   // activations (hook sites of the same map side) one launch can score

// One dense activation of a launch: all its scored maps back to back.  A launch walks the tiles of its segments in order;
// tile t belongs to segment s with tile0[s] <= t < tile0[s + 1].  (In score_large.cuh a tile is a work item (map, v-chunk):
// a segment holds a whole number of maps' items, so item % NVC is still the v-chunk.)
struct ScoreSegments {
    int n_seg;
    int tile0[SCORE_MAX_SEG + 1];
    int n_maps[SCORE_MAX_SEG], c_count[SCORE_MAX_SEG];
    long long total_elems[SCORE_MAX_SEG];                // n_maps * NN
    const void* x[SCORE_MAX_SEG];                        // first scored element (of the kernel's IN type), 16-B aligned
    double* accum[SCORE_MAX_SEG];                        // fp64 [c_count] of the site
};
struct ScoreTensorMaps { CUtensorMap m[SCORE_MAX_SEG]; };

// moves the segment cursor sg on to the segment of `tile` (each role of a kernel walks its tiles in increasing order)
__device__ __forceinline__ void advance_segment(const ScoreSegments& seg, int tile, int& sg) {
    while (tile >= seg.tile0[sg + 1]) ++sg;
}

}  // namespace dctp
