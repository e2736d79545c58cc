// Fused DCT-score hook kernel on 5th-gen tensor cores (tcgen05 + TMEM), bf16x3 split precision.
//
// Replaces, for one hooked activation, the per-slice Python loop of
// /root/reference/utils/common.py:262-277 (dct_2d per (image, channel) -> sum of squared
// coefficients -> per-channel batch sum).  One launch reads every scored map from HBM exactly
// once, keeps the cosine basis resident in shared memory, runs C_N * X * C_N^T on tensor cores
// and reduces the coefficients to energies straight out of TMEM: no coefficient tensor is ever
// written to HBM (unless the debug `dump` pointer asks for it).
//
// Tile = 128 TMEM lanes x KP contraction columns, packed with G x J square maps of side N:
//   Ms = N rounded up to 8            lanes (and contraction columns) one map occupies
//   G  = 128 / Ms  lane groups,  J = KP / Ms  column groups,  map t of the tile sits at (g, j) = (t / J, t % J)
//
//   stage 0   HBM -> registers (128-bit loads, all of a tile's loads in flight at once) -> bf16 hi/lo -> A1
//   stage 1   D1[(g,h), (j,v)] = sum_{(j',w)} A1[(g,h), (j',w)] * B[(j,v), (j',w)]
//             A1[(g,h),(j,w)] = X_{g,j}[h,w]   K-major;  B = I_J (x) C_N  (block diagonal, zero padded)
//             -> D1[(g,h),(j,v)] = Y_{g,j}[h,v] = (X C^T)[h,v]
//   epi   1   D1 -> bf16 hi/lo -> A2_q[(g,v), k]   MN-major (transpose-free: a lane writes along M)
//   stage 2   per column group q:  D2[(g,v), q*N2 + u] = sum_h A2_q[(g,v), h] * C[u, h] = Z_{g,j}[u,v]
//             (the top-left corner of B is C itself, so stage 2 re-uses the resident basis;
//              for Ms == 8 two column groups share one K=16 step: q = j/2, k = (j%2)*8 + h)
//   epi   2   energy_{g,j} = sum_{u,v} D2^2  (fixed-order fp32 tree) -> one fp64 atomicAdd per map
//
// Every product runs as three bf16 MMAs: hi*hi + lo*hi + hi*lo (fp32 accumulate in TMEM).
// Operands live in shared memory in the canonical SWIZZLE_128B layouts (8-row x 128-byte atoms).
// A2 re-uses A1's storage (stage 1 has completed when epilogue 1 runs).  Positions of A1/A2 that a
// tile does not write hold finite bf16 leftovers; they only ever meet zero entries of B.  (Nothing but
// bf16 operand data may ever be stored there: an arbitrary bit pattern can read as NaN, and NaN * 0
// would leak into live lanes.)
//
// Everything that is the same for every tile is computed once: the scatter table (where each loaded
// vector lands in the swizzled operand: built on the host, staged into shared memory), the operand
// descriptors, each lane's A2 store offsets.  Latency is hidden twice over: the loads of tile t+1 are
// issued into registers right after tile t's stage-1 MMAs (they land while the tensor core and the
// epilogues run), and several CTAs share an SM (4 at KP = 64).
#pragma once
#include "umma.cuh"

namespace dctp {

struct FastDiv {            // q = n / d for n < 2^32 / d
    uint32_t mul, d;
    __host__ void set(uint32_t div) { d = div; mul = static_cast<uint32_t>(0x100000000ull / div) + 1u; }
    __device__ __forceinline__ uint32_t div(uint32_t n) const { return d == 1 ? n : __umulhi(n, mul); }
};

enum : int { DCTP_DEV_OK = 0, DCTP_DEV_MMA_TIMEOUT = 1, DCTP_DEV_SMEM_ALIGN = 2 };

// how stage 0 reaches the maps
enum : int {
    LOAD_DENSE1 = 0,   // scored maps form one contiguous fp32 stream; N % 4 == 0: one 8-byte store per float4
    LOAD_DENSE2 = 1,   //   "   N even: two 4-byte stores per float4
    LOAD_DENSE4 = 2,   //   "   any N : four 2-byte stores per float4 (+ scalar tail)
    LOAD_GEN4 = 3,     // per-map base pointers (channel windows, strided batches), 128-bit loads
    LOAD_GEN2 = 4,     //   "   64-bit loads
    LOAD_GEN1 = 5      //   "   32-bit loads
};

struct UmmaScoreArgs {
    const float* x;                 // activation base pointer (fp32, maps contiguous: stride_h = N, stride_w = 1)
    long long stride_b, stride_c;   // in elements
    int c_begin, c_count;           // scored channel window (DenseNet: last 12)
    int n_maps;                     // B * c_count
    int N, NN;                      // map side (H == W), N*N
    int Ms, G, J, MT;               // lanes per map, lane groups, column groups, maps per tile (G*J)
    int num_tiles;
    int K1;                         // stage-1 k-steps (16 columns each) = ceil(J*Ms / 16)
    int N1;                         // stage-1 output columns = 16*K1
    int NQ, K2S, N2;                // stage-2: groups, k-steps per group, output columns per group
    int TPM, tpm_shift;             // threads per map in the final reduction (power of two <= 32, TPM*MT <= 128), its log2
    int chan_step;                  // (gridDim.x * MT) mod c_count: channel advance between a CTA's consecutive tiles
    uint32_t idesc1, idesc2;
    uint32_t a2_lbo, a2_group_bytes;
    FastDiv div_vpm, div_n, div_ms, div_j;
    // dense modes
    const float* x_dense;           // first scored element (x + c_begin*stride_c)
    long long total_elems;          // n_maps * NN
    int tile_vec;                   // float4 vectors per full tile = MT*NN/4
    const uint16_t* scatter;        // [tile_vec][vpe] byte offsets into the K-major A1 operand
    uint32_t var_bytes;             // bytes of `scatter` (dense) / of the map-pointer array (generic)
    uint32_t red_bytes;             // bytes of the epilogue-2 reduction scratch: J * 128 floats
    const uint16_t* basis_hi;       // [KP x KP] bf16 bits of I_J (x) C_N, row = output index, col = contraction index
    const uint16_t* basis_lo;
    double* accum;                  // [c_count] per-channel energy sums (fp64)
    float* energy_out;              // optional [n_maps] per-(image,channel) energies
    float* dump;                    // optional [n_maps x NN] DCT coefficients Z[u][v] (parity of the transform itself)
    int* status;                    // device status word (DCTP_DEV_*)
};

namespace detail {

// byte offset of bf16 element (row, k) in a K-major SWIZZLE_128B operand with `rows` rows
__host__ __device__ __forceinline__ uint32_t kmajor_off(uint32_t row, uint32_t k, uint32_t rows) {
    uint32_t kb = k >> 6, kk = k & 63;
    return kb * (rows * 128u) + (row >> 3) * 1024u + (row & 7) * 128u + ((((kk >> 3) ^ row) & 7) << 4) + ((kk & 7) << 1);
}
// byte offset of bf16 element (m, k) in an MN-major SWIZZLE_128B operand; lbo = stride between 64-wide M blocks
__device__ __forceinline__ uint32_t mnmajor_off(uint32_t m, uint32_t k, uint32_t lbo) {
    return (m >> 6) * lbo + (k >> 3) * 1024u + (k & 7) * 128u + (((((m & 63) >> 3) ^ k) & 7) << 4) + ((m & 7) << 1);
}

__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

template <int VEC> struct Ld;
template <> struct Ld<4> {
    __device__ static __forceinline__ void ld(const float* p, float (&v)[4]) {
        asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "l"(p));
    }
    __device__ static __forceinline__ void st(uint8_t* hi, uint8_t* lo, uint32_t off, const float (&v)[4]) {
        uint32_t h0, l0, h1, l1;
        umma::split2(v[0], v[1], h0, l0);
        umma::split2(v[2], v[3], h1, l1);
        *reinterpret_cast<uint2*>(hi + off) = make_uint2(h0, h1);
        *reinterpret_cast<uint2*>(lo + off) = make_uint2(l0, l1);
    }
};
template <> struct Ld<2> {
    __device__ static __forceinline__ void ld(const float* p, float (&v)[2]) {
        asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "l"(p));
    }
    __device__ static __forceinline__ void st(uint8_t* hi, uint8_t* lo, uint32_t off, const float (&v)[2]) {
        uint32_t h0, l0;
        umma::split2(v[0], v[1], h0, l0);
        *reinterpret_cast<uint32_t*>(hi + off) = h0;
        *reinterpret_cast<uint32_t*>(lo + off) = l0;
    }
};
template <> struct Ld<1> {
    __device__ static __forceinline__ void ld(const float* p, float (&v)[1]) {
        asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v[0]) : "l"(p));
    }
    __device__ static __forceinline__ void st(uint8_t* hi, uint8_t* lo, uint32_t off, const float (&v)[1]) {
        uint32_t h0, l0;
        umma::split2(v[0], 0.f, h0, l0);
        *reinterpret_cast<uint16_t*>(hi + off) = static_cast<uint16_t>(h0 & 0xFFFFu);
        *reinterpret_cast<uint16_t*>(lo + off) = static_cast<uint16_t>(l0 & 0xFFFFu);
    }
};

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

template <int KP>
struct UmmaScoreSmem {
    static_assert(KP == 64 || KP == 128, "contraction width");
    static constexpr uint32_t KB = KP / 64;                        // 64-element K blocks
    static constexpr uint32_t A_BYTES = KB * 128u * 128u;          // one 128-row operand (hi or lo); A2 aliases it
    static constexpr uint32_t B_BYTES = KB * KP * 128u;
    static constexpr uint32_t OFF_A_HI = 0;
    static constexpr uint32_t OFF_A_LO = OFF_A_HI + A_BYTES;
    static constexpr uint32_t OFF_B_HI = OFF_A_LO + A_BYTES;
    static constexpr uint32_t OFF_B_LO = OFF_B_HI + B_BYTES;
    static constexpr uint32_t OFF_CTRL = OFF_B_LO + B_BYTES;       // mbarrier + TMEM slot
    static constexpr uint32_t OFF_VAR = OFF_CTRL + 64;             // reduction scratch, then scatter table (dense) or map pointers (generic)
    static constexpr uint32_t FIXED = OFF_VAR;
    static constexpr uint32_t TMEM_COLS = 2 * KP;                  // D1 | D2
    __host__ __device__ static constexpr uint32_t total(uint32_t red_bytes, uint32_t var_bytes) {
        return FIXED + red_bytes + ((var_bytes + 15u) & ~15u);
    }
};

constexpr int UMMA_PF_SLOTS = 13;          // prefetch registers: 13 float4 per thread = a 1568-vector tile (56^2, 28^2, 14^2, 7^2)

// PF: keep the next tile's loads in flight (in registers) across this tile's tensor and epilogue phases.
template <int KP, int MODE, bool PF>
__global__ void __launch_bounds__(128, KP == 64 ? 4 : 1) score_umma_kernel(const UmmaScoreArgs a) {
    using S = UmmaScoreSmem<KP>;
    using namespace umma;
    constexpr bool DENSE = MODE <= LOAD_DENSE4;
    static_assert(DENSE || !PF, "prefetch goes with the dense load path");
    constexpr int VPE = MODE == LOAD_DENSE1 ? 1 : MODE == LOAD_DENSE2 ? 2 : 4;
    constexpr int VEC = MODE == LOAD_GEN4 ? 4 : MODE == LOAD_GEN2 ? 2 : 1;
    constexpr int NCHUNK = KP / 8;                                 // 8-column chunks of a D1 row
    constexpr int SLOTS = PF ? UMMA_PF_SLOTS : 1;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* a_hi = smem + S::OFF_A_HI;
    uint8_t* a_lo = smem + S::OFF_A_LO;
    uint8_t* b_hi = smem + S::OFF_B_HI;
    uint8_t* b_lo = smem + S::OFF_B_LO;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::OFF_CTRL);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::OFF_CTRL + 8);
    float* red = reinterpret_cast<float*>(smem + S::OFF_VAR);     // epilogue-2 scratch, [<= 8 rows][128 lanes]
    const float** mptr = reinterpret_cast<const float**>(smem + S::OFF_VAR + a.red_bytes);   // generic modes
    const typename detail::Scatter<VPE>::Entry* scat =
        reinterpret_cast<const typename detail::Scatter<VPE>::Entry*>(smem + S::OFF_VAR + a.red_bytes);  // dense modes

    const uint32_t tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // (shuffle: the compiler then knows it is warp-uniform)
    if ((smem_u32(smem) & 1023u) != 0) {                           // SWIZZLE_128B atoms need 1024-B alignment
        if (tid == 0) atomicExch(a.status, DCTP_DEV_SMEM_ALIGN);
        return;
    }

    // ---- register prefetch of a tile's stream
    [[maybe_unused]] float4 pf[SLOTS];
    [[maybe_unused]] uint32_t pf_full = 0;
    auto tile_vectors = [&](int tile) -> uint32_t {                // whole float4 vectors of this tile's stream
        const long long left = a.total_elems - static_cast<long long>(tile) * a.MT * a.NN;
        return static_cast<uint32_t>(min(static_cast<long long>(a.tile_vec), left >> 2));
    };
    auto prefetch = [&](int tile) {
        pf_full = tile_vectors(tile);
        const float4* src = reinterpret_cast<const float4*>(a.x_dense + static_cast<long long>(tile) * a.MT * a.NN) + tid;
#pragma unroll
        for (int u = 0; u < SLOTS; ++u)
            if (tid + u * 128 < pf_full) pf[u] = detail::ldg_stream(src + u * 128);
    };
    // ---- one-time setup: zero the operand area, stage basis and scatter table, TMEM, barrier.  None of it touches
    //      the activation, so under a programmatic dependent launch it overlaps the tail of the preceding kernel.
    for (uint32_t off = tid * 16; off < S::OFF_B_HI; off += 128 * 16)
        *reinterpret_cast<uint4*>(smem + off) = make_uint4(0, 0, 0, 0);
    for (uint32_t i = tid; i < KP * (KP / 8); i += 128) {
        uint32_t n = i / (KP / 8), c8 = i % (KP / 8);
        uint4 vh = *reinterpret_cast<const uint4*>(a.basis_hi + n * KP + c8 * 8);
        uint4 vl = *reinterpret_cast<const uint4*>(a.basis_lo + n * KP + c8 * 8);
        uint32_t off = detail::kmajor_off(n, c8 * 8, KP);
        *reinterpret_cast<uint4*>(b_hi + off) = vh;
        *reinterpret_cast<uint4*>(b_lo + off) = vl;
    }
    if constexpr (DENSE) {
        const uint4* src = reinterpret_cast<const uint4*>(a.scatter);
        uint4* dst = reinterpret_cast<uint4*>(smem + S::OFF_VAR + a.red_bytes);
        for (uint32_t i = tid; i < (a.var_bytes + 15) / 16; i += 128) dst[i] = src[i];
    }
    if (warp == 0) tmem_alloc<S::TMEM_COLS>(tmem_slot);
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_init_fence();
    }
    fence_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tmem_lane = tmem + ((warp * 32u) << 16);

    // operand descriptors: high words are per layout, low words (start address) advance per k-step / group
    // (the low word carries the start address in bits [0,14) and the leading-dimension offset in [16,30))
    const uint64_t desc_k = make_smem_desc(0, 16, 1024, SWIZZLE_128B);            // K-major A1 and B
    const uint64_t desc_mn = make_smem_desc(0, a.a2_lbo, 1024, SWIZZLE_128B);     // MN-major A2
    const uint32_t k_lo = static_cast<uint32_t>(desc_k), mn_lo = static_cast<uint32_t>(desc_mn);
    const uint32_t lo_a_hi = smem_u32(a_hi) >> 4, lo_a_lo = smem_u32(a_lo) >> 4;
    const uint32_t lo_b_hi = smem_u32(b_hi) >> 4, lo_b_lo = smem_u32(b_lo) >> 4;

    auto issue_stage1 = [&]() {                                    // one elected thread; D1 = A1 * B^T
        tc_fence_after_sync();
        detail::issue_ss3_n<KP, false>(a.K1, tmem, k_lo + lo_a_hi, k_lo + lo_a_lo, k_lo + lo_b_hi, k_lo + lo_b_lo, desc_k, desc_k, a.idesc1);
        mma_commit(bar);
    };
    auto issue_stage2 = [&]() {                                    // per column group: D2 = A2_q * C^T
        tc_fence_after_sync();
#pragma unroll 1
        for (uint32_t q = 0; q < (uint32_t)a.NQ; ++q) {
            const uint32_t qoff = q * (a.a2_group_bytes >> 4);
            detail::issue_ss3_n<KP, true>(a.K2S, tmem + KP + q * a.N2, mn_lo + lo_a_hi + qoff, mn_lo + lo_a_lo + qoff, k_lo + lo_b_hi,
                                          k_lo + lo_b_lo, desc_mn, desc_k, a.idesc2);
        }
        mma_commit(bar);
    };

    // this thread's TMEM lane as (lane group, row in map), and where its D1 chunks go in A2
    const uint32_t my_g = a.div_ms.div(tid);
    const uint32_t my_r = tid - my_g * a.Ms;
    const bool lane_in_map = my_g < (uint32_t)a.G && my_r < (uint32_t)a.N;
    const uint32_t used_cols = a.J * a.Ms;
    const bool ms8 = a.Ms == 8;
    const uint32_t col_lim = ms8 ? 16u : (uint32_t)a.Ms;           // meaningful D2 columns per stage-2 group
    const uint32_t blocks_per_q = a.N2 >> 4;                       // x16 column blocks per stage-2 group
    const uint32_t n_blocks = a.NQ * blocks_per_q;                 // x16 column blocks holding coefficients
    // D2 columns in [Ms, N2) are exact zeros unless a neighbouring map's basis block reaches into them
    const bool mask_cols = !ms8 && a.J > 1 && (a.Ms & 15) != 0;
    uint32_t a2off[NCHUNK];
#pragma unroll
    for (int ci = 0; ci < NCHUNK; ++ci) {
        const uint32_t c = ci * 8;
        const uint32_t j = a.div_ms.div(c), v0 = c - j * a.Ms;
        const uint32_t q = ms8 ? (j >> 1) : j;
        const uint32_t k = ms8 ? ((j & 1) * 8 + my_r) : my_r;
        a2off[ci] = q * a.a2_group_bytes + detail::mnmajor_off(my_g * a.Ms + v0, k, a.a2_lbo);
    }
    uint32_t phase = 0;
    bool alive = true;

    // ---- phases of one tile.  Software pipeline across tiles (one mbarrier, strictly alternating phases):
    //        stage0(t+1) and MMA1(t+1) are issued as soon as MMA2(t) has released the operand buffer, so
    //        epilogue 2 and the reduction of tile t run while the tensor core already works on tile t+1.
    auto stage0 = [&](int tile) {
        const int map0 = tile * a.MT;
        [[maybe_unused]] const int maps_here = min(a.MT, a.n_maps - map0);
        // HBM -> registers -> bf16 hi/lo -> A1 (each scored map is read exactly once)
        if constexpr (DENSE) {
            const long long elem0 = static_cast<long long>(map0) * a.NN;
            uint32_t n_full;
            if constexpr (PF) {
                n_full = pf_full;
#pragma unroll
                for (int u = 0; u < SLOTS; ++u)
                    if (tid + u * 128 < n_full) detail::Scatter<VPE>::st(a_hi, a_lo, scat[tid + u * 128], pf[u]);
            } else {
                n_full = tile_vectors(tile);
                const float4* src = reinterpret_cast<const float4*>(a.x_dense + elem0);
                constexpr int U = 8;                               // 8 x 16 B in flight per thread; x 4 CTAs covers the HBM latency
#pragma unroll 1
                for (uint32_t base = tid; base < n_full; base += 128 * U) {
                    float4 v[U];
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (base + u * 128 < n_full) v[u] = detail::ldg_stream(src + base + u * 128);
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (base + u * 128 < n_full) detail::Scatter<VPE>::st(a_hi, a_lo, scat[base + u * 128], v[u]);
                }
            }
            if constexpr (VPE == 4) {                              // odd sizes: the stream may end inside a float4
                const long long left = a.total_elems - elem0;
                const uint32_t tail = static_cast<uint32_t>(min(static_cast<long long>(a.tile_vec) * 4, left)) - n_full * 4;
                if (tid < tail && n_full < (uint32_t)a.tile_vec) {
                    const float x = a.x_dense[elem0 + n_full * 4 + tid];
                    const uint2 e = scat[n_full];
                    const uint32_t o = tid == 0 ? (e.x & 0xFFFFu) : tid == 1 ? (e.x >> 16) : (e.y & 0xFFFFu);
                    uint32_t h, l;
                    split2(x, 0.f, h, l);
                    *reinterpret_cast<uint16_t*>(a_hi + o) = static_cast<uint16_t>(h);
                    *reinterpret_cast<uint16_t*>(a_lo + o) = static_cast<uint16_t>(l);
                }
            }
        } else {
            if ((int)tid < maps_here) {
                int m = map0 + (int)tid;
                int b = m / a.c_count, c = m - b * a.c_count;
                mptr[tid] = a.x + b * a.stride_b + (long long)(a.c_begin + c) * a.stride_c;
            }
            __syncthreads();
            const uint32_t vpm = a.NN / VEC;             // vectors per map
            const uint32_t total = maps_here * vpm;
            constexpr int U = VEC == 4 ? 8 : 4;
#pragma unroll 1
            for (uint32_t base = 0; base < total; base += 128 * U) {
                float v[U][VEC];
                uint32_t off[U];
                bool ok[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    uint32_t idx = base + u * 128 + tid;
                    ok[u] = idx < total;
                    if (ok[u]) {
                        uint32_t t = a.div_vpm.div(idx);
                        uint32_t e = (idx - t * vpm) * VEC;
                        uint32_t g = a.div_j.div(t), j = t - g * a.J;
                        uint32_t h = a.div_n.div(e), w = e - h * a.N;
                        detail::Ld<VEC>::ld(mptr[t] + e, v[u]);
                        off[u] = detail::kmajor_off(g * a.Ms + h, j * a.Ms + w, 128);
                    }
                }
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (ok[u]) detail::Ld<VEC>::st(a_hi, a_lo, off[u], v[u]);
            }
        }
        fence_async_smem();
        __syncthreads();
        if (warp == 0) {
            if (elect_one()) issue_stage1();
            __syncwarp();
        }
        if constexpr (PF) {                                        // the following tile's loads go out now and land
            const int next = tile + (int)gridDim.x;                // while the tensor core and the epilogues work
            if (next < a.num_tiles) prefetch(next);
        }
    };
    auto epilogue1 = [&]() {
        // D1 row (g,h) -> bf16 hi/lo -> A2_q[(g, v), k]   (MN-major operand, aliases A1)
#pragma unroll
        for (int part = 0; part < KP / 32; ++part) {               // 32 columns at a time keeps the register footprint small
            if ((uint32_t)(part * 32) < (uint32_t)a.N1) {
                uint32_t r[2][16];
                tmem_ld16(tmem_lane + part * 32, r[0]);
                if ((uint32_t)(part * 32 + 16) < (uint32_t)a.N1) tmem_ld16(tmem_lane + part * 32 + 16, r[1]);
                tmem_ld_wait();
                if (lane_in_map) {
#pragma unroll
                    for (int ci = 0; ci < 4; ++ci) {
                        if ((uint32_t)(part * 32 + ci * 8) < used_cols) {
                            uint32_t h4[4], l4[4];
#pragma unroll
                            for (int p = 0; p < 4; ++p)
                                split2(__uint_as_float(r[ci >> 1][(ci & 1) * 8 + 2 * p]),
                                       __uint_as_float(r[ci >> 1][(ci & 1) * 8 + 2 * p + 1]), h4[p], l4[p]);
                            const uint32_t off = a2off[part * 4 + ci];
                            *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(h4[0], h4[1], h4[2], h4[3]);
                            *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(l4[0], l4[1], l4[2], l4[3]);
                        }
                    }
                }
            }
        }
        tc_fence_before_sync();
        fence_async_smem();
        __syncthreads();
        if (warp == 0) {
            if (elect_one()) issue_stage2();
            __syncwarp();
        }
    };
    // final reduction roles, fixed for the whole kernel
    const uint32_t tpm = a.TPM;
    const uint32_t red_t = tid >> a.tpm_shift, red_sub = tid & (tpm - 1);
    const uint32_t red_g = a.div_j.div(min(red_t, (uint32_t)a.MT - 1)), red_j = min(red_t, (uint32_t)a.MT - 1) - red_g * a.J;
    const uint32_t red_rows = ms8 ? 1u : blocks_per_q;
    const float* red_row = red + (ms8 ? red_j : red_j * blocks_per_q) * 128 + red_g * a.Ms;
    uint32_t chan = (uint32_t)((static_cast<long long>(blockIdx.x) * a.MT + red_t) % a.c_count);

    auto epilogue2 = [&](int tile) {
        const int map0 = tile * a.MT;
        const int maps_here = min(a.MT, a.n_maps - map0);
        // coefficients -> energy, never leaving the SM.  Lane = (g, v); x16 block = (q, 16 columns).
        //      red[row][lane]: one row per block (two per block when Ms == 8: the block holds two maps)
        {
            uint32_t q = 0, in_q = 0;                              // group of the current block, block index inside it
#pragma unroll
            for (int part = 0; part < KP / 32; ++part) {
                if ((uint32_t)(part * 2) < n_blocks) {
                    uint32_t r[2][16];
                    tmem_ld16(tmem_lane + KP + part * 32, r[0]);
                    if ((uint32_t)(part * 2 + 1) < n_blocks) tmem_ld16(tmem_lane + KP + part * 32 + 16, r[1]);
                    tmem_ld_wait();
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        if ((uint32_t)(part * 2 + b) < n_blocks) {
                            float e0 = 0.f, e1 = 0.f;
                            if (mask_cols) {                       // leftovers past the group's own map: masked
#pragma unroll
                                for (int i = 0; i < 8; ++i) {
                                    float z0 = in_q * 16 + i < col_lim ? __uint_as_float(r[b][i]) : 0.f;
                                    float z1 = in_q * 16 + 8 + i < col_lim ? __uint_as_float(r[b][8 + i]) : 0.f;
                                    e0 = fmaf(z0, z0, e0);
                                    e1 = fmaf(z1, z1, e1);
                                }
                            } else {
#pragma unroll
                                for (int i = 0; i < 8; ++i) {
                                    float z0 = __uint_as_float(r[b][i]), z1 = __uint_as_float(r[b][8 + i]);
                                    e0 = fmaf(z0, z0, e0);
                                    e1 = fmaf(z1, z1, e1);
                                }
                            }
                            if (ms8) {
                                red[(2 * (part * 2 + b)) * 128 + tid] = e0;
                                red[(2 * (part * 2 + b) + 1) * 128 + tid] = e1;
                            } else {
                                red[(part * 2 + b) * 128 + tid] = e0 + e1;
                            }
                            if (a.dump != nullptr) {
                                if (lane_in_map) {
#pragma unroll 1
                                    for (int i = 0; i < 16; ++i) {
                                        uint32_t n = in_q * 16 + i;
                                        uint32_t j = ms8 ? (2 * q + (n >> 3)) : q;
                                        uint32_t u = ms8 ? (n & 7) : n;
                                        int t = (int)(my_g * a.J + j);
                                        float z = 0.f;
#pragma unroll
                                        for (int s = 0; s < 16; ++s) z = s == i ? __uint_as_float(r[b][s]) : z;
                                        if (u < (uint32_t)a.N && j < (uint32_t)a.J && t < maps_here)
                                            a.dump[(long long)(map0 + t) * a.NN + u * a.N + my_r] = z;
                                    }
                                }
                            }
                            if (++in_q == blocks_per_q) { in_q = 0; ++q; }
                        }
                    }
                }
            }
        }
        tc_fence_before_sync();
        __syncthreads();
        {
            // TPM threads per map, fixed summation order -> bit-reproducible per-map energy
            float s = 0.f;
            const bool live = (int)red_t < maps_here;
            if (live) {
                for (uint32_t row = 0; row < red_rows; ++row) {
                    const float* rp = red_row + row * 128;
                    for (uint32_t v = red_sub; v < (uint32_t)a.N; v += tpm) s += rp[v];
                }
            }
#pragma unroll
            for (uint32_t o = 16; o > 0; o >>= 1)
                if (o < tpm) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (live && red_sub == 0) {
                double e = s;
                if (!isfinite(s)) {                                // a non-finite map in the tile (rare: see map_energy64)
                    const int m = map0 + (int)red_t, b = m / a.c_count;
                    const float* xm = DENSE ? a.x_dense + static_cast<long long>(m) * a.NN
                                            : a.x + b * a.stride_b + static_cast<long long>(a.c_begin + m - b * a.c_count) * a.stride_c;
                    e = detail::map_energy64(xm, a.N);
                    s = static_cast<float>(e);
                }
                atomicAdd(a.accum + chan, e);
                if (a.energy_out) a.energy_out[map0 + (int)red_t] = s;
            }
            chan += a.chan_step;                                   // (map0 + red_t) mod c_count, without the division
            if (chan >= (uint32_t)a.c_count) chan -= a.c_count;
        }
    };

    // Dependents may start only now that this CTA holds its TMEM columns: a later kernel's CTA that grabbed TMEM first
    // and then waited for this grid to finish would deadlock against a CTA of this grid still waiting for columns.
    launch_dependents();
    grid_dependency_wait();                                        // the activation (written by the preceding kernel) is complete
    if constexpr (PF) {
        if ((int)blockIdx.x < a.num_tiles) prefetch(blockIdx.x);
    }
    int tile = blockIdx.x;
    if (tile < a.num_tiles) stage0(tile);
    while (tile < a.num_tiles) {
        const int next = tile + (int)gridDim.x;
        if (!mbar_wait(bar, phase)) { alive = false; break; }      // MMA1(tile)
        phase ^= 1;
        tc_fence_after_sync();
        epilogue1();
        if (!mbar_wait(bar, phase)) { alive = false; break; }      // MMA2(tile): operand buffer and D1 are free again
        phase ^= 1;
        tc_fence_after_sync();
        if (next < a.num_tiles) stage0(next);
        epilogue2(tile);                                           // overlaps MMA1(next)
        tile = next;
    }

    if (!alive && tid == 0) {                                      // a hand-over never came: flag it and poison the result
        atomicExch(a.status, DCTP_DEV_MMA_TIMEOUT);
        for (int c = 0; c < a.c_count; ++c) a.accum[c] = __longlong_as_double(0x7FF8000000000000ll);
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc<S::TMEM_COLS>(tmem);
}

}  // namespace dctp
