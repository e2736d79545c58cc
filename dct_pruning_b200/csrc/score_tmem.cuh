// Fused DCT-score hook kernel, TMEM-operand formulation (dense tensors, even map side 10..64).
//
// Same contract as score_umma.cuh (/root/reference/utils/common.py:262-277: per-(image,channel)
// orthonormal 2-D DCT-II energy, summed per channel), re-arranged because ncu shows the K-major/MN-major
// formulation bound by SHARED-MEMORY bandwidth (tensor-core operand reads + thread stores = 85 % of the
// L1/shared data pipe at 2.7 TB/s).  Here the only shared-memory operand traffic is the raw data once
// and the small resident basis:
//
//   tile      G = 128 / Ms maps (Ms = N rounded up to 8), map g owns TMEM lanes [g*Ms, g*Ms + N)
//   stage 1   D1[(g,v), h] = sum_{(g',w)} A'[(g,v),(g',w)] * Bx[h,(g',w)]
//             A' = I_G (x) C_N  (block diagonal, bf16 hi/lo) lives in TMEM for the whole kernel  -> no smem reads
//             Bx[h, g*N + w] = X_g[h, w]  is the data, K-major in shared memory, N-side operand (N1 rows)
//             -> D1 = (C X^T) per map: the intermediate comes out TRANSPOSED, lanes (g,v), columns h
//   epi   1   tcgen05.ld D1 -> bf16 hi/lo -> tcgen05.st A2 (packed pairs): stays in TMEM, no smem round trip
//   stage 2   D2[(g,v), u] = sum_h A2[(g,v),h] * C[u,h]      A from TMEM, B = C_N resident in shared memory
//   epi   2   tcgen05.ld D2 -> sum of squares per lane -> fixed-order tree over the map's lanes -> fp64 atomicAdd
//
// Three bf16 MMAs per product (hi*hi + hi*lo + lo*hi, fp32 accumulate).  Shared-memory wavefronts per 25 KB
// of input: ~300 data stores + 336 + 192 basis/data operand reads, against ~2070 for the smem-operand kernel.
// The price: the block-diagonal A' wastes a factor G of stage-1 tensor work (1056 tensor cycles per 25 KB at
// 56x56 vs 768), still below the HBM time (1080 cycles at the measured 6.55 TB/s).
//
// TMEM: [0,128) A' (hi | lo, written once), then per tile slot 2*N1MAX columns: D (N1MAX, D2 re-uses D1) |
// A2 hi (N1MAX/2) | A2 lo (N1MAX/2).  One CTA runs NSLOT independent tile slots, one warpgroup (4 warps = 128
// TMEM lanes) each, sharing A' and C: 3 slots for maps up to 64 wide, 6 for maps up to 32 or 16 wide (the
// per-tile dependency chain is what bounds this kernel, so smaller tiles get more slots).
#pragma once
#include "score_common.cuh"
#include "umma.cuh"

namespace dctp {

namespace detail {
// three passes x KS k-steps of D (+)= A[tmem] * B[smem]^T, fully unrolled.  Pass p reads the TMEM operand at
// column a_p + 8*ks and the K-major shared-memory operand whose descriptor low word is b_p (+ k-step offset;
// KB16 = distance between 64-element K blocks in 16-byte units).
template <int KS, int KB16>
__device__ __forceinline__ void issue_ts3(uint32_t d, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t b0, uint32_t b1, uint32_t b2,
                                          uint64_t desc, uint32_t idesc) {
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
        const uint32_t ac = pass == 0 ? a0 : pass == 1 ? a1 : a2;
        const uint32_t bl = pass == 0 ? b0 : pass == 1 ? b1 : b2;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks)
            umma::mma_bf16_ts(d, ac + 8 * ks, umma::desc_with_lo(desc, bl + (ks >> 2) * KB16 + (ks & 3) * 2), idesc,
                              (pass | ks) != 0);
    }
}
}  // namespace detail

struct TScoreArgs {
    const float* x_dense;           // first scored element; all scored maps back to back, 16-B aligned
    long long total_elems;          // n_maps * NN
    int n_maps, c_count;
    int N, NN, Ms, G;
    int J, MT;                      // maps side by side along the D columns (1, 2 for Ms = 16, 4 for Ms = 8) and maps per tile = G * J
    int j_shift, ms_shift;          // log2(J), log2(Ms) (used when J > 1)
    int NQ;                         // J > 1: 16-column groups stage 2 runs over (N1 / 16); with Ms = 8 a group holds two maps
    int tile_vec;                   // float4 vectors per full tile = MT*NN/4
    int num_tiles;
    int K1S;                        // stage-1 k-steps = ceil(G*N / 16)
    int N1;                         // MMA N of stage 1 = D columns in use: N rounded up to 16 (J = 1) or J * Ms (J = 2)
    int TPM, tpm_shift;             // threads per map in the final reduction (power of two), its log2
    int chan_step;                  // (tiles between a slot's consecutive tiles * G) mod c_count
    uint32_t idesc;                 // M = 128, N = N1, bf16 x bf16 -> f32, K-major B
    uint32_t idesc_g;               // J > 1: stage 2 runs per 16-column group, N = 16
    const uint16_t* scatter;        // [tile_vec][VPE] byte offsets of each float4's pieces in the K-major data operand
    uint32_t scatter_bytes;
    const uint32_t* a_hi;           // [128][64] packed bf16 pairs of A' = I_G (x) C_N (row (g,v), column pair (g',w)/2)
    const uint32_t* a_lo;
    const uint16_t* c_hi;           // [64][64] bf16 C_N zero padded (row u, column h); Ms = 8: I_2 (x) C_N in the top-left 16 x 16
    const uint16_t* c_lo;
    double* accum;
    float* energy_out;
    float* dump;
    int* status;
    long long* trace;               // bring-up aid: clock64 at phase boundaries of CTA 0 / slot 0 (8 stamps per tile, 32 tiles)
    FastDiv div_ms;
};

template <int N1MAX, int NPROD = 0>
struct TScoreSmem {
    static constexpr uint32_t BX_HALF = 2 * N1MAX * 128;           // data operand (hi or lo): 2 K-blocks x N1MAX rows x 128 B
    static constexpr uint32_t SLOT_BYTES = 2 * BX_HALF;
    static constexpr uint32_t C_HALF = 64 * 128;                   // stage-2 basis (hi or lo)
    // the 6-slot variants (768 threads, 80 registers each) cannot hold the next tile in registers without spilling it,
    // which makes every load wait for its own spill store; they stage it in shared memory with cp.async instead
    static constexpr bool STAGED = N1MAX < 64;
    static constexpr uint32_t PF = N1MAX == 64 ? 16 : 8;                       // float4 of a tile per thread
    static constexpr uint32_t STAGE_BYTES = STAGED ? PF * 128 * 16 : 0;        // per slot: fp32 tile, thread-private vectors
    // producer variant (NPROD extra warpgroups convert for all slots): per producer two fp32 tiles in flight, 13 float4 per thread each
    static constexpr uint32_t PPF = 13, PSTAGE_BYTES = PPF * 128 * 16;
    __host__ __device__ static constexpr uint32_t off_stage(int nslot) { return nslot * SLOT_BYTES; }
    __host__ __device__ static constexpr uint32_t off_c(int nslot) {
        return nslot * (SLOT_BYTES + STAGE_BYTES) + NPROD * 2 * PSTAGE_BYTES;
    }
    __host__ __device__ static constexpr uint32_t off_ctrl(int nslot) { return off_c(nslot) + 2 * C_HALF; }
    __host__ __device__ static constexpr uint32_t off_red(int nslot) { return off_ctrl(nslot) + 128; }
    __host__ __device__ static constexpr uint32_t off_table(int nslot) { return off_red(nslot) + nslot * 2048; }   // 4 x 128 floats per slot
    __host__ __device__ static constexpr uint32_t total(int nslot, uint32_t table_bytes) {
        return off_table(nslot) + ((table_bytes + 15u) & ~15u);
    }
};

// N1MAX: widest accumulator a slot holds (64 / 32 columns); NSLOT tile slots per CTA (one warpgroup each);
// VPE: scatter pieces per float4 (1: N % 4 == 0, one 8-byte store; 2: N even, two 4-byte stores; 4: N odd, four 2-byte stores)
// NPROD: 0 = every slot's warpgroup loads and converts its own tiles; 2 = two extra producer warpgroups load (cp.async, two tiles
// each in flight) and convert for all slots, so a slot's chain is only MMA / epilogue / MMA / epilogue (tiles of <= 1664 float4)
template <int N1MAX, int NSLOT, int VPE, int NPROD = 0>
__global__ void __launch_bounds__(128 * (NSLOT + NPROD), 1) score_t_kernel(const TScoreArgs a) {
    using S = TScoreSmem<N1MAX, NPROD>;
    using namespace umma;
    constexpr int WPS = 4, TPS = 128;                              // one warpgroup (= all 128 TMEM lanes) per slot
    constexpr int NT = TPS * (NSLOT + NPROD);
    constexpr int TSCORE_PF = S::PF;                               // float4 per thread: a full tile
    constexpr bool STAGED = S::STAGED;
    static_assert(NPROD == 0 || !STAGED, "the producer variant is for the 3-slot kernel");
    constexpr uint32_t SLOT_COLS = 2 * N1MAX;
    constexpr uint32_t TMEM_COLS = 512;
    static_assert(128 + NSLOT * SLOT_COLS <= TMEM_COLS, "TMEM budget");
    constexpr int KB16 = N1MAX * 8;                                // 64-element K block of the data operand, in 16-byte units
    using Entry = typename detail::Scatter<VPE>::Entry;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // (shuffle: the compiler then knows it is warp-uniform)
    const uint32_t wg = warp / WPS, wtid = tid - wg * TPS;         // tile slot of this warp set, thread within it
    const uint32_t swarp = warp - wg * WPS;                        // warp within the slot: lane quarter swarp & 3, column half swarp >> 2
    uint8_t* bx_hi = smem + wg * S::SLOT_BYTES;
    uint8_t* bx_lo = bx_hi + S::BX_HALF;
    uint8_t* c_hi = smem + S::off_c(NSLOT);
    uint8_t* c_lo = c_hi + S::C_HALF;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::off_ctrl(NSLOT));
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::off_ctrl(NSLOT) + 112);
    [[maybe_unused]] uint64_t* full = bars + NSLOT;                // (NPROD) a slot's data operand has been written
    [[maybe_unused]] uint64_t* bxfree = bars + 2 * NSLOT;          // (NPROD) [slot][producer]: the MMAs that read it are done, signalled
                                                                   //         to the producer that writes the slot next (each barrier has one waiter
                                                                   //         that sees every phase: a waiter skipping phases would mis-read parity)
    float* red = reinterpret_cast<float*>(smem + S::off_red(NSLOT)) + (wg < NSLOT ? wg : 0) * 512;      // [map column j][lane]
    const Entry* scat = reinterpret_cast<const Entry*>(smem + S::off_table(NSLOT));
    uint64_t* bar = bars + (wg < NSLOT ? wg : 0);

    if ((smem_u32(smem) & 1023u) != 0) {
        if (tid == 0) atomicExch(a.status, DCTP_DEV_SMEM_ALIGN);
        return;
    }

    // tiles of this slot: tile = first + i * stride
    const int first = blockIdx.x * NSLOT + (int)wg, stride = gridDim.x * NSLOT;

    // ---- register prefetch of a tile
    [[maybe_unused]] float4 pf[(STAGED || NPROD > 0) ? 1 : TSCORE_PF];
    uint32_t pf_full = 0;
    float4* stage = reinterpret_cast<float4*>(smem + S::off_stage(NSLOT) + wg * S::STAGE_BYTES) + wtid;   // (STAGED)
    auto prefetch = [&](int tile) {
        const long long elem0 = static_cast<long long>(tile) * a.MT * a.NN;
        pf_full = static_cast<uint32_t>(min(static_cast<long long>(a.tile_vec), (a.total_elems - elem0) >> 2));
        const float4* src = reinterpret_cast<const float4*>(a.x_dense + elem0) + wtid;
        if constexpr (STAGED) {
            const uint32_t dst = smem_u32(stage);
#pragma unroll
            for (int u = 0; u < TSCORE_PF; ++u)
                if (wtid + u * TPS < pf_full) cp_async16(dst + u * TPS * 16, src + u * TPS);
            cp_async_commit();
        } else if constexpr (NPROD == 0) {
#pragma unroll
            for (int u = 0; u < TSCORE_PF; ++u)
                if (wtid + u * TPS < pf_full) pf[u] = detail::ldg_stream(src + u * TPS);
        }
    };
    // ---- one-time setup (independent of the activation: overlaps the preceding kernel's tail under a dependent launch): zero the data operands, stage C and the scatter table, barriers, TMEM, A' into TMEM
    for (uint32_t off = tid * 16; off < S::off_stage(NSLOT); off += NT * 16)
        *reinterpret_cast<uint4*>(smem + off) = make_uint4(0, 0, 0, 0);
    for (uint32_t i = tid; i < 64 * 8; i += NT) {
        const uint32_t n = i >> 3, c8 = i & 7;
        const uint32_t off = detail::kmajor_off(n, c8 * 8, 64);
        *reinterpret_cast<uint4*>(c_hi + off) = *reinterpret_cast<const uint4*>(a.c_hi + n * 64 + c8 * 8);
        *reinterpret_cast<uint4*>(c_lo + off) = *reinterpret_cast<const uint4*>(a.c_lo + n * 64 + c8 * 8);
    }
    {
        const uint4* src = reinterpret_cast<const uint4*>(a.scatter);
        uint4* dst = reinterpret_cast<uint4*>(smem + S::off_table(NSLOT));
        for (uint32_t i = tid; i < (a.scatter_bytes + 15) / 16; i += NT) dst[i] = src[i];
    }
    if (warp == 0) tmem_alloc<TMEM_COLS>(tmem_slot);
    if (tid == 0) {
        for (int s = 0; s < NSLOT; ++s) mbar_init(bars + s, 1);
        if constexpr (NPROD > 0) {
            for (int s = 0; s < NSLOT; ++s) mbar_init(full + s, TPS);
            for (int s = 0; s < NSLOT * NPROD; ++s) mbar_init(bxfree + s, 1);
        }
        mbar_init_fence();
    }
    fence_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t lane_bits = ((swarp & 3) * 32u) << 16;          // this warp's TMEM lane quarter
    if (warp < 4) {                                                // A' = I_G (x) C_N, hi at columns [0,64), lo at [64,128)
#pragma unroll 1
        for (int part = 0; part < 8; ++part) {
            const uint32_t* src = (part < 4 ? a.a_hi : a.a_lo) + tid * 64 + (part & 3) * 16;
            uint32_t v[16];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint4 q = *reinterpret_cast<const uint4*>(src + 4 * i);
                v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
            }
            tmem_st16(tmem + ((warp * 32u) << 16) + part * 16, v);
        }
        tmem_st_wait();
    }
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();

    launch_dependents();                                           // only now: this CTA holds its TMEM columns (see score_umma.cuh)
    grid_dependency_wait();                                        // the activation (written by the preceding kernel) is complete
    bool alive = true;
    if constexpr (NPROD > 0) {
        if (wg >= (uint32_t)NSLOT) {
            // ===================================================== producer warpgroup: load + convert for every slot of the CTA
            // The CTA's tiles in the order q = 0, 1, 2, ...: slot q % NSLOT, tile (blockIdx.x * NSLOT + slot) + (q / NSLOT) * stride;
            // producer pw takes q = pw, pw + NPROD, ...  Two tiles per producer are in flight as cp.async copies (thread-private
            // staging: each thread later converts exactly the vectors it requested, so no barrier guards the staging buffers).
            const uint32_t pw = wg - NSLOT;
            float4* pst = reinterpret_cast<float4*>(smem + S::off_stage(NSLOT) + pw * 2 * S::PSTAGE_BYTES) + wtid;
            auto tile_of = [&](uint32_t q) { return (int)(blockIdx.x * NSLOT + q % NSLOT) + (int)(q / NSLOT) * stride; };
            auto vectors_of = [&](int tile) {
                const long long elem0 = static_cast<long long>(tile) * a.MT * a.NN;
                return static_cast<uint32_t>(min(static_cast<long long>(a.tile_vec), (a.total_elems - elem0) >> 2));
            };
            auto request = [&](uint32_t q, uint32_t buf) {
                const int tile = tile_of(q);
                if (tile < a.num_tiles) {
                    const uint32_t n = vectors_of(tile);
                    const float4* src = reinterpret_cast<const float4*>(a.x_dense + static_cast<long long>(tile) * a.MT * a.NN) + wtid;
                    const uint32_t dst = smem_u32(pst) + buf * S::PSTAGE_BYTES;
#pragma unroll
                    for (uint32_t u = 0; u < S::PPF; ++u)
                        if (wtid + u * TPS < n) cp_async16(dst + u * TPS * 16, src + u * TPS);
                }
                cp_async_commit();
            };
            uint32_t q = pw, seen = 0;                             // seen: parity of the next bxfree phase to wait for, one bit per slot
            request(q, 0);
            request(q + NPROD, 1);
            for (uint32_t k = 0;; ++k, q += NPROD) {
                const int tile = tile_of(q);
                if (tile >= a.num_tiles) break;
                cp_async_wait_but_one();
                const uint32_t slot = q % NSLOT, fill = q / NSLOT;
                if (fill >= 1) {                                   // stage-1 MMAs of the slot's previous tile are done
                    if (alive && !mbar_wait(bxfree + slot * NPROD + pw, (seen >> slot) & 1u)) alive = false;
                    seen ^= 1u << slot;
                }
                uint8_t* hi = smem + slot * S::SLOT_BYTES;
                uint8_t* lo = hi + S::BX_HALF;
                const uint32_t n = vectors_of(tile);
                const float4* stg = pst + (k & 1u) * (S::PSTAGE_BYTES / 16);
#pragma unroll
                for (uint32_t u = 0; u < S::PPF; ++u)
                    if (wtid + u * TPS < n) detail::Scatter<VPE>::st(hi, lo, scat[wtid + u * TPS], stg[u * TPS]);
                fence_async_smem();
                mbar_arrive(full + slot);
                request(q + 2 * NPROD, k & 1u);
            }
            if (!alive && wtid == 0) atomicExch(a.status, DCTP_DEV_MMA_TIMEOUT);
        }
    } else {
        if (first < a.num_tiles) prefetch(first);
    }

    const uint32_t slot_col = tmem + 128 + SLOT_COLS * wg;         // this slot's TMEM columns
    const uint32_t d_col = slot_col, a2_hi_col = slot_col + N1MAX, a2_lo_col = slot_col + N1MAX + N1MAX / 2;
    const uint32_t tmem_lane = lane_bits;                          // added to column addresses for ld/st

    const uint64_t desc_k = make_smem_desc(0, 16, 1024, SWIZZLE_128B);
    const uint32_t k_lo = static_cast<uint32_t>(desc_k);
    const uint32_t lo_bx_hi = smem_u32(bx_hi) >> 4, lo_bx_lo = smem_u32(bx_lo) >> 4;
    const uint32_t lo_c_hi = smem_u32(c_hi) >> 4, lo_c_lo = smem_u32(c_lo) >> 4;

    uint32_t fill = 0;                                             // (NPROD) how many tiles this slot has consumed
    // MMA issue is straight-line code (step counts are template parameters): a runtime loop costs ~100 cycles of
    // dependent uniform-datapath work per MMA, three times the 32 cycles the tensor core needs for it.
    auto issue_stage1 = [&]() {                                    // D1 = A' * Bx^T : A'hi*Bxhi + A'hi*Bxlo + A'lo*Bxhi
        tc_fence_after_sync();
        const uint32_t b_hi_lo = k_lo + lo_bx_hi, b_lo_lo = k_lo + lo_bx_lo;
        switch (a.K1S) {
            case 5: detail::issue_ts3<5, KB16>(d_col, tmem, tmem, tmem + 64, b_hi_lo, b_lo_lo, b_hi_lo, desc_k, a.idesc); break;
            case 6: detail::issue_ts3<6, KB16>(d_col, tmem, tmem, tmem + 64, b_hi_lo, b_lo_lo, b_hi_lo, desc_k, a.idesc); break;
            case 7: detail::issue_ts3<7, KB16>(d_col, tmem, tmem, tmem + 64, b_hi_lo, b_lo_lo, b_hi_lo, desc_k, a.idesc); break;
            default: detail::issue_ts3<8, KB16>(d_col, tmem, tmem, tmem + 64, b_hi_lo, b_lo_lo, b_hi_lo, desc_k, a.idesc); break;
        }
        mma_commit(bar);
        if constexpr (NPROD > 0)                                   // the data operand may be overwritten once these have read it:
            mma_commit(bxfree + wg * NPROD + ((fill + 1) * NSLOT + wg) % NPROD);   // tell the producer of the slot's next tile
    };
    auto issue_stage2 = [&]() {                                    // D2 = A2 * C^T : A2hi*Chi + A2lo*Chi + A2hi*Clo
        tc_fence_after_sync();
        const uint32_t c_hi_lo = k_lo + lo_c_hi, c_lo_lo = k_lo + lo_c_lo;
        if (a.J > 1) {                                             // per 16-column group: D2[:, (j,u)] = A2[:, (j,h)] * C[u,h]^T
            for (int j = 0; j < a.NQ; ++j)
                detail::issue_ts3<1, 0>(d_col + 16 * j, a2_hi_col + 8 * j, a2_lo_col + 8 * j, a2_hi_col + 8 * j, c_hi_lo, c_hi_lo,
                                        c_lo_lo, desc_k, a.idesc_g);
            mma_commit(bar);
            return;
        }
        switch (a.N1 >> 4) {
            case 1: detail::issue_ts3<1, 0>(d_col, a2_hi_col, a2_lo_col, a2_hi_col, c_hi_lo, c_hi_lo, c_lo_lo, desc_k, a.idesc); break;
            case 2: if constexpr (N1MAX >= 32) detail::issue_ts3<2, 0>(d_col, a2_hi_col, a2_lo_col, a2_hi_col, c_hi_lo, c_hi_lo, c_lo_lo, desc_k, a.idesc); break;
            case 3: if constexpr (N1MAX >= 64) detail::issue_ts3<3, 0>(d_col, a2_hi_col, a2_lo_col, a2_hi_col, c_hi_lo, c_hi_lo, c_lo_lo, desc_k, a.idesc); break;
            default: if constexpr (N1MAX >= 64) detail::issue_ts3<4, 0>(d_col, a2_hi_col, a2_lo_col, a2_hi_col, c_hi_lo, c_hi_lo, c_lo_lo, desc_k, a.idesc); break;
        }
        mma_commit(bar);
    };

    const uint32_t my_lane = (swarp & 3) * 32 + (tid & 31);        // TMEM lane of this thread
    const uint32_t my_g = a.div_ms.div(my_lane);
    const uint32_t my_v = my_lane - my_g * a.Ms;
    constexpr int PARTS = N1MAX >= 64 ? 2 : 1;                     // 32-column parts of an accumulator row
    const int part0 = 0;
    const bool lane_in_map = my_g < (uint32_t)a.G && my_v < (uint32_t)a.N;
    const uint32_t bar_id = 1 + wg;
    uint32_t phase = 0;

    // final reduction roles, fixed for the whole kernel
    const uint32_t tpm = a.TPM;
    const uint32_t red_t = wtid >> a.tpm_shift, red_sub = wtid & (tpm - 1);          // map t of the tile = (g, j), t = g * J + j
    const uint32_t red_tc = min(red_t, (uint32_t)a.MT - 1);
    const uint32_t red_g = red_tc >> a.j_shift, red_j = red_tc & ((uint32_t)a.J - 1u);
    const float* red_row = red + red_j * 128 + red_g * a.Ms;
    uint32_t chan = (uint32_t)((static_cast<long long>(first) * a.MT + red_t) % a.c_count);

    int trace_i = 0;
    auto stamp = [&](int k) {
        if (a.trace != nullptr && blockIdx.x == 0 && wtid == 0 && wg == 0 && trace_i < 32) a.trace[trace_i * 8 + k] = clock64();
    };
    for (int tile = (NPROD > 0 && wg >= (uint32_t)NSLOT) ? a.num_tiles : first; tile < a.num_tiles; tile += stride) {
        stamp(0);
        const int map0 = tile * a.MT;
        const int maps_here = min(a.MT, a.n_maps - map0);

        // ---- stage 0: registers (prefetched) -> bf16 hi/lo -> data operand in shared memory
        if constexpr (STAGED) {
            cp_async_wait_all();
#pragma unroll
            for (int u = 0; u < TSCORE_PF; ++u)
                if (wtid + u * TPS < pf_full) detail::Scatter<VPE>::st(bx_hi, bx_lo, scat[wtid + u * TPS], stage[u * TPS]);
        } else if constexpr (NPROD == 0) {
#pragma unroll
            for (int u = 0; u < TSCORE_PF; ++u)
                if (wtid + u * TPS < pf_full) detail::Scatter<VPE>::st(bx_hi, bx_lo, scat[wtid + u * TPS], pf[u]);
        }
        stamp(1);
        fence_async_smem();
        tc_fence_before_sync();                                    // this warp's tcgen05.ld of the previous tile are done
        named_bar_sync(bar_id, TPS);
        stamp(2);
        if (swarp == 0) {
            if (elect_one()) {
                if constexpr (NPROD > 0) {                         // a producer has written this tile's data operand
                    if (alive && !mbar_wait(full + wg, fill & 1u)) alive = false;
                }
                issue_stage1();
            }
            __syncwarp();
        }
        ++fill;
        if constexpr (NPROD == 0) {
            if (tile + stride < a.num_tiles) prefetch(tile + stride);  // lands while the tensor core and the epilogues work
        }
        stamp(3);
        if (!mbar_wait(bar, phase)) { alive = false; break; }
        phase ^= 1;
        tc_fence_after_sync();
        stamp(4);

        // ---- epilogue 1: D1 row (g,v) -> bf16 hi/lo pairs -> A2 in TMEM (columns h/2)
#pragma unroll
        for (int pi = 0; pi < PARTS; ++pi) {
            const int part = part0 + pi;
            if (part * 32 < a.N1) {
                uint32_t r[2][16];
                tmem_ld16(d_col + tmem_lane + part * 32, r[0]);
                if (N1MAX >= 32 && part * 32 + 16 < a.N1) tmem_ld16(d_col + tmem_lane + part * 32 + 16, r[1]);
                else {
#pragma unroll
                    for (int i = 0; i < 16; ++i) r[1][i] = 0u;
                }
                tmem_ld_wait();
                uint32_t hi[16], lo[16];
#pragma unroll
                for (int p = 0; p < (N1MAX >= 32 ? 16 : 8); ++p)
                    split2(__uint_as_float(r[p >> 3][(p & 7) * 2]), __uint_as_float(r[p >> 3][(p & 7) * 2 + 1]), hi[p], lo[p]);
                if constexpr (N1MAX >= 32) {
                    tmem_st16(a2_hi_col + tmem_lane + part * 16, hi);
                    tmem_st16(a2_lo_col + tmem_lane + part * 16, lo);
                } else {
                    tmem_st8(a2_hi_col + tmem_lane, hi);
                    tmem_st8(a2_lo_col + tmem_lane, lo);
                }
            }
        }
        tmem_st_wait();
        tc_fence_before_sync();
        named_bar_sync(bar_id, TPS);
        stamp(5);
        if (swarp == 0) {
            if (elect_one()) issue_stage2();
            __syncwarp();
        }
        if (!mbar_wait(bar, phase)) { alive = false; break; }
        phase ^= 1;
        tc_fence_after_sync();
        stamp(6);

        // ---- epilogue 2: coefficients -> energy.  Lane = (g, v), column = u.
        float e0 = 0.f, e1 = 0.f, f0 = 0.f, f1 = 0.f;              // columns [0,8) / [16,24) and [8,16) / [24,32) of a part
#pragma unroll
        for (int pi = 0; pi < PARTS; ++pi) {
            const int part = part0 + pi;
            if (part * 32 < a.N1) {
                uint32_t r[2][16];
                tmem_ld16(d_col + tmem_lane + part * 32, r[0]);
                if (N1MAX >= 32 && part * 32 + 16 < a.N1) tmem_ld16(d_col + tmem_lane + part * 32 + 16, r[1]);
                else {
#pragma unroll
                    for (int i = 0; i < 16; ++i) r[1][i] = 0u;
                }
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float z0 = __uint_as_float(r[0][i]), z1 = __uint_as_float(r[1][i]);
                    const float y0 = __uint_as_float(r[0][8 + i]), y1 = __uint_as_float(r[1][8 + i]);
                    e0 = fmaf(z0, z0, e0);
                    e1 = fmaf(z1, z1, e1);
                    f0 = fmaf(y0, y0, f0);
                    f1 = fmaf(y1, y1, f1);
                }
                if (a.dump != nullptr && lane_in_map) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const uint32_t col = part * 32 + i;
                        const uint32_t j = a.J > 1 ? col >> a.ms_shift : 0u, u = a.J > 1 ? col & ((uint32_t)a.Ms - 1u) : col;   // map column, coefficient row
                        const int t = (int)(my_g * a.J + j);
                        if (u < (uint32_t)a.N && j < (uint32_t)a.J && t < maps_here)
                            a.dump[(long long)(map0 + t) * a.NN + u * a.N + my_v] = __uint_as_float(r[i >> 4][i & 15]);
                    }
                }
            }
        }
        if (a.J == 4) {                                            // (N1MAX = 32, Ms = 8: one map per 8 columns)
            red[wtid] = e0;
            red[128 + wtid] = f0;
            red[256 + wtid] = e1;
            red[384 + wtid] = f1;
        } else if (a.J == 2) {                                     // (Ms = 16: r[0] was map column 0, r[1] map column 1)
            red[wtid] = e0 + f0;
            red[128 + wtid] = e1 + f1;
        } else {
            red[wtid] = (e0 + f0) + (e1 + f1);
        }
        named_bar_sync(bar_id, TPS);
        {
            // TPM threads per map, fixed summation order -> bit-reproducible per-map energy
            float s = 0.f;
#pragma unroll
            for (uint32_t k = 0; k < 4; ++k)                       // N <= 4 * TPM for every shape routed here
                if (red_sub + k * tpm < (uint32_t)a.N) s += red_row[red_sub + k * tpm];
#pragma unroll
            for (uint32_t o = 16; o > 0; o >>= 1)
                if (o < tpm) s += __shfl_xor_sync(0xffffffffu, s, o);
            if ((int)red_t < maps_here && red_sub == 0) {
                double e = s;
                if (!isfinite(s)) {                                // a non-finite map in the tile (rare: see map_energy64)
                    e = detail::map_energy64(a.x_dense + static_cast<long long>(map0 + (int)red_t) * a.NN, a.N);
                    s = static_cast<float>(e);
                }
                atomicAdd(a.accum + chan, e);
                if (a.energy_out) a.energy_out[map0 + (int)red_t] = s;
            }
            chan += a.chan_step;                                   // (map0 + red_t) mod c_count, without the division
            if (chan >= (uint32_t)a.c_count) chan -= a.c_count;
        }
        stamp(7);
        ++trace_i;
        // (`red` is rewritten only after two more barriers of this slot)
    }

    if (!alive && wtid == 0) {                                      // a hand-over never came: flag it and poison the result
        atomicExch(a.status, DCTP_DEV_MMA_TIMEOUT);
        for (int c = 0; c < a.c_count; ++c) a.accum[c] = __longlong_as_double(0x7FF8000000000000ll);
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc<TMEM_COLS>(tmem);
}

}  // namespace dctp
