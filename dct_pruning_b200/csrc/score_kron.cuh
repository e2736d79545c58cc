// Fused DCT-score hook kernel for small maps (dense tensors, side 1..8): single-stage Kronecker formulation.
//
// Same contract as the other score kernels (/root/reference/utils/common.py:262-277).  For N <= 8 the separable
// two-stage form wastes the tensor core (a 7x7 map fills 7 of the 16 rows a k-step wants, twice) and needs the
// intermediate rewritten as an operand.  Here a map is one row of a plain GEMM:
//
//   Z_flat[map, (u,v)] = sum_{(h,w)} X_flat[map, (h,w)] * Kr[(u,v), (h,w)],      Kr = C_N (x) C_N   (N^2 x N^2, <= 64 x 64)
//
//   A   = X_flat (bf16 hi | lo) in TMEM: lane = map (128 maps per sub-tile), K2 = N^2 rounded up to 16 contraction columns
//   B   = Kr (bf16 hi, lo) resident in shared memory, K-major, N2 = K2 rows
//   D   = 128 lanes x N2 fp32 columns; three passes hi*hi + lo*hi + hi*lo; 12 MMAs of M128 N64 K16 = 384 tensor cycles per
//         128 maps of 7x7 (25 KB, 1113 cycles of HBM time at the measured 6.55 TB/s)
//   epi   thread = lane = map: sum of squares of its own N2 columns -> one fp64 atomicAdd; no second stage, no scatter table,
//         no cross-lane reduction
//
// Warp specialised, one CTA per SM, 18 warps: warps 0-7 = two groups of converters (thread = map: fp32 row -> bf16 hi/lo -> tcgen05.st;
// group g takes the 128-map sub-tiles g, g + 2, ... of the CTA), warps 8-15 = two groups of epilogue warps (likewise), warp 16 = TMA
// producer (ring of 3 tiles), warp 17 = MMA issuer.  TMEM: A ring 4 x 64 columns | D ring 4 x 64 columns.  (One group of each, 10
// warps, ran the 7x7 layers at 3.7 TB/s with 42 % of the issue slots and 21 % of the tensor pipe busy: a latency chain.)
// EVEN sides: 2-D tensor map over [n_maps, N^2] whose box is a few floats wider than a row (the excess is out of bounds and
// arrives as zeros), so that a thread's 128-bit reads of its own row are free of bank conflicts.  ODD sides: rows are not
// 16-byte multiples; the stream is viewed as [rows, 32 floats] (as in score_stack.cuh) and read with 32-bit loads (odd stride).
// 16-bit input (IN, score_stack.cuh): the row layout (EVEN) needs a row pitch of whole 16-byte units, which 16-bit maps have at sides
// 4 and 8 only (box width padded to an odd number of 16-byte units); every other side uses the flat [rows, 32 elements] view.  bf16
// maps are their own hi part: A_lo is not written and the MMA issuer runs the hi*hi and hi*lo passes only; fp16 is split as fp32.
#pragma once
#include <cuda.h>
#include "score_stack.cuh"

namespace dctp {

struct KronArgs {
    ScoreSegments seg;              // the activations of the launch (score_stack.cuh)
    int N, NN;
    int sub_tiles;                  // 128-map sub-tiles per TMA tile (1, 2 or 4)
    int row_elems;                  // shared-memory stride of a map's row in elements (EVEN: box width, ODD: NN)
    int tile_maps, num_tiles;
    uint32_t tile_bytes;            // bytes one TMA tile lands
    int box_rows;                   // second box dimension (EVEN: maps per tile, ODD: 128-byte rows per tile)
    uint32_t idesc;
    const uint8_t* k_hi;            // Kr operand images (StackSmem::LBO2 layout)
    const uint8_t* k_lo;
    float* energy_out;              // optional, single-segment launches only
    float* dump;                    // optional, single-segment launches only
    int* status;
};

struct KronSmem {
    static constexpr uint32_t NSTG = 3, STG_STRIDE = 36 * 1024;
    static constexpr uint32_t OFF_K = NSTG * STG_STRIDE;
    static constexpr uint32_t OFF_BARS = OFF_K + 2 * StackSmem::C2_HALF;
    static constexpr uint32_t OFF_SLOT = OFF_BARS + 256;
    static constexpr uint32_t TOTAL = OFF_SLOT + 128;
};

constexpr int KRON_NT = 576, KRON_W_PROD = 16, KRON_W_MMA = 17;

template <int K2, bool EVEN, int IN = IN_F32>
__global__ void __launch_bounds__(KRON_NT, 1) score_kron_kernel(const __grid_constant__ ScoreTensorMaps tmaps, const __grid_constant__ KronArgs a) {
    using S = KronSmem;
    using namespace umma;
    constexpr int KS = K2 / 16;
    constexpr uint32_t LBO = StackSmem::LBO2, HALF = StackSmem::C2_HALF, STEP = (2 * LBO) >> 4;
    constexpr uint32_t TM_A = 0, TM_D = 256;

    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;   // (shuffle: known warp-uniform)
    uint8_t* stg = smem;
    uint8_t* kr = smem + S::OFF_K;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BARS);
    uint64_t* stg_full = bars;            // [3] TMA landed
    uint64_t* stg_free = bars + 3;        // [3] 8 converter warps
    uint64_t* a_full = bars + 6;          // [4] 4 converter warps
    uint64_t* a_free = bars + 10;         // [4] the MMAs that read the slot have completed
    uint64_t* d_full = bars + 14;         // [4]
    uint64_t* d_free = bars + 18;         // [4] 4 epilogue warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::OFF_SLOT);

    // barriers and TMEM first: the producer warp then has tiles on their way while the other warps stage the Kronecker basis
    if (warp == KRON_W_MMA) tmem_alloc<512>(tmem_slot);
    if (tid == 0) {
        for (int s = 0; s < 3; ++s) { mbar_init(stg_full + s, 1); mbar_init(stg_free + s, 8); }
        for (int s = 0; s < 4; ++s) { mbar_init(a_full + s, 4); mbar_init(a_free + s, 1); mbar_init(d_full + s, 1); mbar_init(d_free + s, 4); }
        mbar_init_fence();
    }
    if (warp == KRON_W_PROD && lane == 0) tma_prefetch_desc(&tmaps.m[0]);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    launch_dependents();
    if (warp != KRON_W_PROD) {
        const uint32_t ptid = tid < KRON_W_PROD * 32 ? tid : tid - 32;
        for (uint32_t off = ptid * 16; off < HALF; off += (KRON_NT - 32) * 16) {
            *reinterpret_cast<uint4*>(kr + off) = *reinterpret_cast<const uint4*>(a.k_hi + off);
            *reinterpret_cast<uint4*>(kr + HALF + off) = *reinterpret_cast<const uint4*>(a.k_lo + off);
        }
        fence_async_smem();
        named_bar_sync(6, KRON_NT - 32);
    }
    grid_dependency_wait();

    const int first = blockIdx.x, stride = gridDim.x;
    bool dead = false;
    auto seg_of = [&](int tile, int& sg) {
        while (tile >= a.seg.tile0[sg + 1]) ++sg;
    };
    auto is_tail = [&](int tile, int sg) {               // (ODD) a stream that does not end on a 32-element row: last tile from global memory
        return !EVEN && tile == a.seg.tile0[sg + 1] - 1 && (a.seg.total_elems[sg] & 31) != 0;
    };
#define KRON_WAIT(bar, par)                          \
    if (!mbar_wait((bar), (par))) {                  \
        dead = true;                                 \
        break;                                       \
    }

    if (warp == KRON_W_PROD) {
        // ================================================================ TMA producer
        if (elect_one()) {
            uint32_t it = 0;
            int sg = 0;
            for (int tile = first; tile < a.num_tiles; tile += stride) {
                seg_of(tile, sg);
                if (is_tail(tile, sg)) continue;
                const uint32_t s = it % S::NSTG;
                if (it >= S::NSTG) KRON_WAIT(stg_free + s, ((it / S::NSTG) - 1u) & 1u);
                mbar_arrive_expect_tx(stg_full + s, a.tile_bytes);
                tma_load_2d(stg + s * S::STG_STRIDE, &tmaps.m[sg], 0, (tile - a.seg.tile0[sg]) * a.box_rows, stg_full + s);
                ++it;
            }
        }
        __syncwarp();
    } else if (warp == KRON_W_MMA) {
        // ================================================================ MMA issuer
        if (elect_one()) {
            const uint64_t desc = make_smem_desc(0, LBO, 128, SWIZZLE_NONE);
            const uint32_t lo_hi = static_cast<uint32_t>(desc) + (smem_u32(kr) >> 4), lo_lo = lo_hi + (HALF >> 4);
            uint32_t j = 0;
            for (int tile = first; tile < a.num_tiles && !dead; tile += stride)
                for (int st = 0; st < a.sub_tiles; ++st, ++j) {
                    const uint32_t sl = j & 3u;
                    KRON_WAIT(a_full + sl, (j >> 2) & 1u);
                    if (j >= 4) KRON_WAIT(d_free + sl, ((j >> 2) - 1u) & 1u);
                    tc_fence_after_sync();
                    const uint32_t ahi = tmem + TM_A + sl * 64, alo = ahi + K2 / 2, d = tmem + TM_D + sl * 64;
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
                        if (IN == IN_BF16 && pass == 1) continue;                // bf16 input: A_lo = 0
#pragma unroll
                        for (int ks = 0; ks < KS; ++ks)
                            mma_bf16_ts(d, (pass == 1 ? alo : ahi) + 8 * ks, desc_with_lo(desc, (pass == 2 ? lo_lo : lo_hi) + ks * STEP), a.idesc,
                                        (pass | ks) != 0);
                    }
                    mma_commit(d_full + sl);
                    mma_commit(a_free + sl);
                }
        }
        __syncwarp();
    } else if (warp < 8) {
        // ================================================================ converters: thread = map, fp32 row -> bf16 hi | lo -> A (TMEM)
        const uint32_t grp = warp >> 2, gt = tid & 127u;                   // group, thread within it = map within a sub-tile
        const uint32_t lane_bits = ((warp & 3u) * 32u) << 16;
        uint32_t it = 0, j = 0;
        int sg = 0;
        for (int tile = first; tile < a.num_tiles && !dead; tile += stride) {
            seg_of(tile, sg);
            const bool from_global = is_tail(tile, sg);
            uint32_t s = 0;
            if (!from_global) {
                s = it % S::NSTG;
                KRON_WAIT(stg_full + s, (it / S::NSTG) & 1u);
            }
            for (int st = 0; st < a.sub_tiles; ++st, ++j) {
                if ((j & 1u) != grp) continue;                            // the other group's sub-tile
                const uint32_t sl = j & 3u;
                if (j >= 4) KRON_WAIT(a_free + sl, ((j >> 2) - 1u) & 1u);
                tc_fence_after_sync();
                const uint32_t ahi = tmem + TM_A + sl * 64 + lane_bits, alo = ahi + K2 / 2;
                if constexpr (IN == IN_BF16) {
                    // the map's raw bf16 pairs are A_hi as they are
                    uint32_t p[K2 / 2];
                    const long long m0 = static_cast<long long>(tile - a.seg.tile0[sg]) * a.tile_maps + st * 128 + gt;
                    if (from_global) {
                        const long long e0 = m0 * a.NN, total = a.seg.total_elems[sg];
                        const uint16_t* xs = static_cast<const uint16_t*>(a.seg.x[sg]);
#pragma unroll
                        for (int i = 0; i < K2 / 2; ++i) {
                            const uint32_t x0 = (2 * i < a.NN && e0 + 2 * i < total) ? xs[e0 + 2 * i] : 0u;
                            const uint32_t x1 = (2 * i + 1 < a.NN && e0 + 2 * i + 1 < total) ? xs[e0 + 2 * i + 1] : 0u;
                            p[i] = x0 | (x1 << 16);
                        }
                    } else if constexpr (EVEN) {
                        const uint4* row = reinterpret_cast<const uint4*>(stg + s * S::STG_STRIDE) + static_cast<uint32_t>(st * 128 + gt) * (a.row_elems >> 3);
#pragma unroll
                        for (int i = 0; i < K2 / 8; ++i) {
                            const uint4 q4 = 8 * i < a.NN ? row[i] : make_uint4(0u, 0u, 0u, 0u);
                            p[4 * i] = q4.x; p[4 * i + 1] = q4.y; p[4 * i + 2] = q4.z; p[4 * i + 3] = q4.w;
                        }
                    } else {
                        const uint16_t* row = reinterpret_cast<const uint16_t*>(stg + s * S::STG_STRIDE) + static_cast<uint32_t>(st * 128 + gt) * a.NN;
#pragma unroll
                        for (int i = 0; i < K2 / 2; ++i)
                            p[i] = (2 * i < a.NN ? static_cast<uint32_t>(row[2 * i]) : 0u) | ((2 * i + 1 < a.NN ? static_cast<uint32_t>(row[2 * i + 1]) : 0u) << 16);
                    }
#pragma unroll
                    for (int c = 0; c < K2 / 2; c += 16) {
                        uint32_t h[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) h[i] = c + i < K2 / 2 ? p[c + i] : 0u;
                        if (c + 16 <= K2 / 2) tmem_st16(ahi + c, h);
                        else tmem_st8(ahi + c, h);
                    }
                    tmem_st_wait();
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(a_full + sl);
                    continue;
                }
                float v[K2];
                if constexpr (IN == IN_F16) {                            // widened in registers, split as fp32
                    if (from_global) {
                        const long long e0 = (static_cast<long long>(tile - a.seg.tile0[sg]) * a.tile_maps + st * 128 + gt) * a.NN;
                        const long long total = a.seg.total_elems[sg];
                        const uint16_t* xs = static_cast<const uint16_t*>(a.seg.x[sg]);
#pragma unroll
                        for (int i = 0; i < K2; ++i) v[i] = (i < a.NN && e0 + i < total) ? in16_to_float<IN_F16>(xs, e0 + i) : 0.f;
                    } else if constexpr (EVEN) {
                        const uint4* row = reinterpret_cast<const uint4*>(stg + s * S::STG_STRIDE) + static_cast<uint32_t>(st * 128 + gt) * (a.row_elems >> 3);
#pragma unroll
                        for (int i = 0; i < K2 / 8; ++i) {
                            const uint4 q4 = 8 * i < a.NN ? row[i] : make_uint4(0u, 0u, 0u, 0u);
                            const uint32_t w[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const float2 f = f16x2_to_float2(w[k]);
                                v[8 * i + 2 * k] = f.x; v[8 * i + 2 * k + 1] = f.y;
                            }
                        }
                    } else {
                        const uint16_t* row = reinterpret_cast<const uint16_t*>(stg + s * S::STG_STRIDE) + static_cast<uint32_t>(st * 128 + gt) * a.NN;
#pragma unroll
                        for (int i = 0; i < K2; ++i) v[i] = i < a.NN ? in16_to_float<IN_F16>(row, i) : 0.f;
                    }
                } else if (from_global) {
                    const long long e0 = (static_cast<long long>(tile - a.seg.tile0[sg]) * a.tile_maps + st * 128 + gt) * a.NN;
                    const long long total = a.seg.total_elems[sg];
                    const float* xs = static_cast<const float*>(a.seg.x[sg]);
#pragma unroll
                    for (int i = 0; i < K2; ++i) v[i] = (i < a.NN && e0 + i < total) ? xs[e0 + i] : 0.f;
                } else if constexpr (EVEN) {
                    const float4* row = reinterpret_cast<const float4*>(stg + s * S::STG_STRIDE) + static_cast<uint32_t>(st * 128 + gt) * (a.row_elems >> 2);
#pragma unroll
                    for (int i = 0; i < K2 / 4; ++i) {
                        const float4 q4 = 4 * i < a.NN ? row[i] : make_float4(0.f, 0.f, 0.f, 0.f);
                        v[4 * i] = q4.x; v[4 * i + 1] = q4.y; v[4 * i + 2] = q4.z; v[4 * i + 3] = q4.w;
                    }
                } else {
                    const float* row = reinterpret_cast<const float*>(stg + s * S::STG_STRIDE) + static_cast<uint32_t>(st * 128 + gt) * a.NN;
#pragma unroll
                    for (int i = 0; i < K2; ++i) v[i] = i < a.NN ? row[i] : 0.f;
                }
#pragma unroll
                for (int c = 0; c < K2 / 2; c += 16) {                   // 16 packed columns (32 contraction values) per store
                    uint32_t h[16], l[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        if (c + i < K2 / 2) split2(v[2 * (c + i)], v[2 * (c + i) + 1], h[i], l[i]);
                        else { h[i] = 0u; l[i] = 0u; }
                    }
                    if (c + 16 <= K2 / 2) { tmem_st16(ahi + c, h); tmem_st16(alo + c, l); }
                    else { tmem_st8(ahi + c, h); tmem_st8(alo + c, l); }
                }
                tmem_st_wait();
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(a_full + sl);
            }
            if (!from_global) {
                __syncwarp();
                if (lane == 0) mbar_arrive(stg_free + s);
                ++it;
            }
        }
    } else if (warp < 16) {
        // ================================================================ epilogue: thread = map, energy of its own row of D
        const uint32_t grp = (warp >> 2) & 1u, et = tid & 127u;
        const uint32_t lane_bits = ((warp & 3u) * 32u) << 16;
        uint32_t j = 0;
        int sg = 0;
        for (int tile = first; tile < a.num_tiles && !dead; tile += stride) {
            seg_of(tile, sg);
            const uint32_t C = static_cast<uint32_t>(a.seg.c_count[sg]), seg_maps = static_cast<uint32_t>(a.seg.n_maps[sg]);
            double* const accum = a.seg.accum[sg];
            for (int st = 0; st < a.sub_tiles; ++st, ++j) {
                if ((j & 1u) != grp) continue;
                const uint32_t sl = j & 3u;
                KRON_WAIT(d_full + sl, (j >> 2) & 1u);
                tc_fence_after_sync();
                const uint32_t m = static_cast<uint32_t>(tile - a.seg.tile0[sg]) * a.tile_maps + st * 128 + et;   // map within its segment
                // the lane's K2 coefficients in ONE TMEM round trip; D is handed back as soon as they have landed
                uint32_t z[K2];
#pragma unroll
                for (int c = 0; c < K2; c += 16) tmem_ld16(tmem + TM_D + sl * 64 + lane_bits + c, reinterpret_cast<uint32_t (&)[16]>(z[c]));
                tmem_ld_wait();
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(d_free + sl);
                float e0 = 0.f, e1 = 0.f, e2 = 0.f, e3 = 0.f;
#pragma unroll
                for (int c = 0; c < K2; c += 4) {
                    e0 = fmaf(__uint_as_float(z[c]), __uint_as_float(z[c]), e0);
                    e1 = fmaf(__uint_as_float(z[c + 1]), __uint_as_float(z[c + 1]), e1);
                    e2 = fmaf(__uint_as_float(z[c + 2]), __uint_as_float(z[c + 2]), e2);
                    e3 = fmaf(__uint_as_float(z[c + 3]), __uint_as_float(z[c + 3]), e3);
                }
                if (a.dump != nullptr && m < seg_maps)
#pragma unroll
                    for (int i = 0; i < K2; ++i)
                        if (i < a.NN) a.dump[static_cast<long long>(m) * a.NN + i] = __uint_as_float(z[i]);
                if (m < seg_maps) {
                    const float e = (e0 + e1) + (e2 + e3);
                    atomicAdd(accum + (m % C), static_cast<double>(e));
                    if (a.energy_out) a.energy_out[m] = e;
                }
            }
        }
    }
#undef KRON_WAIT
    if (dead) {
        atomicExch(a.status, DCTP_DEV_MMA_TIMEOUT);
        for (int sgi = 0; sgi < a.seg.n_seg; ++sgi)
            for (int c = lane; c < a.seg.c_count[sgi]; c += 32) a.seg.accum[sgi][c] = __longlong_as_double(0x7FF8000000000000ll);
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == KRON_W_MMA) tmem_dealloc<512>(tmem);
}

}  // namespace dctp
