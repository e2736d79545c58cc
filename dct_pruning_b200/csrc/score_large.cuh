// DCT-score hook kernel for LARGE square maps (128 < N <= 320, N % 16 == 0: U^2-Netp's 144 / 160 / 288 / 320 stages).
//
// Same contract as score_umma.cuh (/root/reference/utils/common.py:262-277 and, for the side inputs,
// :296-309: per-(image,channel) orthonormal 2-D DCT-II energy, summed per channel).  A map no longer fits on
// chip (320 x 320 fp32 = 400 KB; the bf16 hi/lo basis is another 400 KB), so the separable contraction is tiled:
//
//   work item   (map, v-chunk): 128 rows v of Y^T = C X^T, i.e. 128 columns of the coefficient matrix Z
//   for each h-tile (128 rows of the map):
//     stage 1   D1[v, h] = sum_w C[v,w] X[h,w]      K-loop over 64-wide w blocks; A = C[v-chunk, w-block] slab, B = X slab
//               (fp32 -> bf16 hi/lo, K-major), both in shared memory; accumulates in TMEM columns [0,128): the
//               intermediate comes out TRANSPOSED (lanes v, columns h), which is what stage 2 contracts over
//     epi   1   D1 row v -> bf16 hi/lo pairs -> A2, written IN PLACE over D1 (hi pairs in columns [0,64), lo pairs in
//               [64,128)): it never leaves TMEM
//     stage 2   D2[v, u] += sum_{h in tile} A2[v,h] C[u,h]   for u-chunks of <= 128; A from TMEM, B = C[u-chunk, h-block]
//               slab; D2 (NU * NUC columns) stays in TMEM columns [128, ...) across all h-tiles: the K-split over h
//   epi   2   D2 -> sum of squares per lane -> block reduction -> one fp64 atomicAdd per (map, v-chunk)
//
// Every product is three bf16 MMAs (hi*hi + lo*hi + hi*lo, fp32 accumulate), like the small-map kernels.
// The kernel is tensor-bound by design (2*N^3 flops per stage and map); the map is re-read once per v-chunk out
// of L2 and the basis slabs come from L2.  Measured on B200: an MMA with both operands in shared memory and N <= 128
// is bound by operand delivery (~118 cycles per M128 N128 K16 MMA against 64 cycles of math: 8 KB of operands each),
// with the A operand in TMEM it runs at the math rate - hence stage 2 reads A2 from TMEM.
// Warp-specialised pipeline, operand slabs ring-buffered in shared memory:
//   basis producer (one elected thread) basis slabs by 1-D bulk copy into a ring of three buffers (the basis image in
//                                       global memory is already in the swizzled operand layout: a slab is one blob)
//   MMA issuer (one elected thread)     issues the MMAs of a step once its slabs are full and does nothing else: the
//                                       tensor pipe's queue is shallow, every cycle this thread spends elsewhere is idle
//                                       tensor time; tcgen05.commit frees the buffers
//   map producer (one elected thread)   one cp.async.bulk.tensor.2d per map slab: the activation is a 2-D tensor [n_maps * N rows, N floats],
//                                       a slab is the box {64 floats, 128 rows} at (w0, map * N + h0), landing row-major in a ring of two
//                                       staging buffers; columns past N arrive as zeros (partial w blocks need no special path)
//   16 converter / epilogue warps       staged fp32 slab -> bf16 hi/lo -> K-major operand slab; the two epilogues.
//                                       No block-wide barrier inside the pipeline, only mbarriers.
// One resident CTA of 19 warps per SM (226 KB of shared memory, 512 TMEM columns).
#pragma once
#include "score_common.cuh"
#include "umma.cuh"

namespace dctp {

struct LargeScoreArgs {
    ScoreSegments seg;              // the activations of the launch; a tile of the table is a work item (map, v-chunk)
    int n_maps;                     // all segments together
    int N, NPR;                     // map side; rows per column block of the basis image (>= N and >= NU * NUC, zero padded)
    int NVC;                        // v-chunks per map = ceil(N / 128)
    int NU, NUC;                    // u-chunk width (multiple of 16, <= 128) and count: NU * NUC >= N
    int n_items;                    // n_maps * NVC
    const uint8_t* c_hi;            // basis image, bf16: [column blocks of 64][NPR rows][128 B], 16-B chunks XOR-swizzled by
    const uint8_t* c_lo;            //   (row & 7): any (8-aligned row range, column block) is one contiguous operand slab
    float* energy_out;              // (unused by the kernel: the host sums energy_parts into it)
    float* energy_parts;            // optional (single-segment launches only) [n_maps][NVC]: each work item's share of its map's energy; summed in a fixed order by
                                    // sum_parts_kernel, so per-map energies are bit-reproducible like the other kernels'
    float* dump;                    // optional (single-segment launches only) [n_maps][N][N] coefficients Z[u][v]
    int* status;
    long long* trace;               // bring-up aid: cycles the control thread of CTA 0 spent in each kind of wait
};

struct LargeSmem {
    static constexpr uint32_t A1_HALF = 128 * 128;                 // X slab: 128 rows x 64 k (hi or lo)
    static constexpr uint32_t A1_BUF = 2 * A1_HALF;                // hi | lo
    static constexpr uint32_t B_HALF = 128 * 128;                  // basis slab: up to 128 rows x 64 k
    static constexpr uint32_t B_BUF = 2 * B_HALF;                  // hi | lo
    static constexpr uint32_t NXB = 2, NBB = 3;                    // map slab ring (the converters run up to three steps ahead of the
                                                                   // tensor core), basis slab ring (a bulk copy takes about one step)
    static constexpr uint32_t OFF_A1 = 0;
    static constexpr uint32_t OFF_B = NXB * A1_BUF;
    static constexpr uint32_t STAGE_BUF = 128 * 64 * 4;            // one fp32 map slab as the TMA delivers it: 128 rows x 64 floats
    static constexpr uint32_t OFF_STAGE = OFF_B + NBB * B_BUF;     // two of them
    static constexpr uint32_t OFF_CTRL = OFF_STAGE + 2 * STAGE_BUF;   // 21 mbarriers, TMEM slot
    static constexpr uint32_t OFF_RED = OFF_CTRL + 192;
    static constexpr uint32_t TOTAL = OFF_RED + 512 * 4;
    static_assert(OFF_B % 1024 == 0 && B_BUF % 1024 == 0, "swizzle atoms are 1024-byte aligned");
    static_assert(TOTAL <= 227 * 1024, "shared memory budget");
};

constexpr int LARGE_CONV = 512;        // 16 converter / epilogue warps: warp w owns TMEM lane quarter w % 4 and every 4th
                                       // 16-column block (w / 4) of an epilogue
constexpr int LARGE_NT = LARGE_CONV + 96;   // + the MMA issuer, basis producer and map producer warps (one elected thread each)

// TRACE: the cycle accounting of DCTP_L_TRACE and the coefficient dump; the production instantiation carries neither
template <bool TRACE>
__global__ void __launch_bounds__(LARGE_NT, 1) score_large_kernel(const __grid_constant__ ScoreTensorMaps xmap, const LargeScoreArgs a) {
    constexpr int NC = LARGE_CONV;
    constexpr int XV = 2048 / NC;                                  // float4 per thread and map slab
    using S = LargeSmem;
    using namespace umma;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* a1_base = smem + S::OFF_A1;                           // buffer p at + p * A1_BUF: hi, then lo
    uint8_t* b_base = smem + S::OFF_B;                             // buffer p at + p * B_BUF: hi, then lo
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_CTRL);
    uint64_t* x_full = bars;            // [4] map slab stored (16 warp arrivals)
    uint64_t* x_empty = bars + 4;       // [4] MMAs that read it are done (tcgen05.commit)
    uint64_t* b_full = bars + 8;        // [3] basis slab landed (bulk-copy bytes)
    uint64_t* b_empty = bars + 11;      // [3] MMAs that read it are done
    uint64_t* acc_ready = bars + 14;    // D1 of an h-tile complete / D2 of an item complete
    uint64_t* a2_full = bars + 15;      // epilogue 1 wrote A2 into TMEM (16 warp arrivals)
    uint64_t* d2_free = bars + 16;      // epilogue 2 has read D2 (16 warp arrivals)
    uint64_t* stg_full = bars + 17;     // [2] staged fp32 slab landed (TMA bytes)
    uint64_t* stg_free = bars + 19;     // [2] the converters have read it (16 warp arrivals)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::OFF_CTRL + 176);
    float* red = reinterpret_cast<float*>(smem + S::OFF_RED);
    const uint32_t tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);      // (a shuffle: the compiler then knows it is warp-uniform)
    if ((smem_u32(smem) & 1023u) != 0) {
        if (tid == 0) atomicExch(a.status, DCTP_DEV_SMEM_ALIGN);
        return;
    }
    for (uint32_t off = tid * 16; off < S::OFF_STAGE; off += LARGE_NT * 16) *reinterpret_cast<uint4*>(smem + off) = make_uint4(0, 0, 0, 0);
    if (warp == 0) tmem_alloc<512>(tmem_slot);
    if (tid == 0) {
        for (uint32_t i = 0; i < S::NXB; ++i) {
            mbar_init(x_full + i, NC / 32);
            mbar_init(x_empty + i, 1);
        }
        for (uint32_t i = 0; i < S::NBB; ++i) {
            mbar_init(b_full + i, 1);
            mbar_init(b_empty + i, 1);
        }
        for (uint32_t i = 0; i < 2; ++i) {
            mbar_init(stg_full + i, 1);
            mbar_init(stg_free + i, NC / 32);
        }
        mbar_init(acc_ready, 1);
        mbar_init(a2_full, NC / 32);
        mbar_init(d2_free, NC / 32);
        mbar_init_fence();
    }
    fence_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    launch_dependents();                                           // only now: this CTA holds its TMEM columns (see score_umma.cuh)
    grid_dependency_wait();                                        // the activation (written by the preceding kernel) is complete
    const uint32_t d1_col = 0, d2_col = 128;
    const int N = a.N, NN = N * N;

    // a timed-out wait (pipeline bug) is recorded once; afterwards this thread stops waiting so the kernel still ends
    bool dead = false;
    auto wait = [&](uint64_t* bar, uint32_t parity) {
        if (!dead && !mbar_wait(bar, parity)) {
            dead = true;
            atomicExch(a.status, DCTP_DEV_MMA_TIMEOUT);
        }
    };

    // The steps of the kernel in issue order: per item (map, v-chunk), per h-tile: one stage-1 step per 64-wide w block,
    // then one stage-2 step per (u-chunk, 64-wide h block).  The issuer and the basis producer walk the same loop nest;
    // a lone thread retires an instruction every few cycles, so both loops are kept to the bare minimum.
    if (warp == NC / 32) {
        // =========================================================== MMA issuer: one elected thread
        if (elect_one()) {
            const uint64_t desc_k = make_smem_desc(0, 16, 1024, SWIZZLE_128B);
            const uint32_t k_lo = static_cast<uint32_t>(desc_k);
            const uint32_t x_lo0 = k_lo + (smem_u32(a1_base) >> 4), b_lo0 = k_lo + (smem_u32(b_base) >> 4);
            const uint32_t idesc2 = make_idesc_bf16(128, a.NU, false, false);
            uint32_t bp = 0, bpar = 0;                              // basis ring: buffer of the next step, its parity
            uint32_t xp = 0, xpar = 0;                              // map slab ring
            uint32_t tile_par = 0, item_par = 0;
            bool first_item = true;
            long long tr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            const bool tracing = TRACE && a.trace != nullptr && blockIdx.x == 0;
            auto twait = [&](int slot, uint64_t* bar, uint32_t parity) {
                if (tracing) {
                    const long long t0 = clock64();
                    wait(bar, parity);
                    tr[slot] += clock64() - t0;
                } else {
                    wait(bar, parity);
                }
            };
            const long long t_begin = clock64();
            long long n_steps = 0;
            for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
                for (int h0 = 0; h0 < N; h0 += 128) {
                    const int MH = min(128, N - h0);
                    const uint32_t idesc1 = make_idesc_bf16(128, (MH + 15) & ~15, false, false);
                    // ---- stage 1: D1[v, h] (+)= C[v-chunk, w-block] X[h-tile, w-block]^T
                    for (int w0 = 0; w0 < N; w0 += 64) {
                        const int ks = min(64, N - w0) >> 4;
                        twait(1, x_full + xp, xpar);
                        twait(4, b_full + bp, bpar);
                        tc_fence_after_sync();
                        const uint32_t bh = b_lo0 + bp * (S::B_BUF >> 4), bl = bh + (S::B_HALF >> 4);
                        const uint32_t xh = x_lo0 + xp * (S::A1_BUF >> 4), xl = xh + (S::A1_HALF >> 4);
                        const uint32_t d = tmem + d1_col;
                        if (ks == 4) {
                            detail::issue_ss_pass<4, false>(d, bh, xh, desc_k, desc_k, idesc1, w0 != 0);     // C_hi X_hi^T
                            detail::issue_ss_pass<4, false>(d, bl, xh, desc_k, desc_k, idesc1, true);        // C_lo X_hi^T
                            detail::issue_ss_pass<4, false>(d, bh, xl, desc_k, desc_k, idesc1, true);        // C_hi X_lo^T
                        } else {
                            detail::issue_ss_pass_n<false>(ks, d, bh, xh, desc_k, desc_k, idesc1, w0 != 0);
                            detail::issue_ss_pass_n<false>(ks, d, bl, xh, desc_k, desc_k, idesc1, true);
                            detail::issue_ss_pass_n<false>(ks, d, bh, xl, desc_k, desc_k, idesc1, true);
                        }
                        mma_commit(x_empty + xp);
                        mma_commit(b_empty + bp);
                        if (w0 + 64 >= N) mma_commit(acc_ready);    // D1 of this tile is complete
                        if (++xp == S::NXB) { xp = 0; xpar ^= 1u; }
                        if (++bp == S::NBB) { bp = 0; bpar ^= 1u; }
                        ++n_steps;
                    }
                    // ---- stage 2: D2[v, u-chunk] (+)= A2[v, h-block] C[u-chunk, h-block]^T, A2 from TMEM
                    twait(2, a2_full, tile_par);
                    tile_par ^= 1u;
                    if (h0 == 0 && !first_item) {                   // the first MMAs of an item overwrite D2
                        twait(3, d2_free, item_par);
                        item_par ^= 1u;
                    }
                    const int nkb = (MH + 63) >> 6;
                    for (int uc = 0; uc < a.NUC; ++uc) {
                        const uint32_t d = tmem + d2_col + uc * a.NU;
                        for (int kb = 0; kb < nkb; ++kb) {
                            const int ks = min(64, MH - kb * 64) >> 4;
                            twait(5, b_full + bp, bpar);
                            tc_fence_after_sync();
                            const uint32_t bh = b_lo0 + bp * (S::B_BUF >> 4), bl = bh + (S::B_HALF >> 4);
                            const uint32_t a2h = tmem + d1_col + kb * 32, a2l = a2h + 64;
                            const bool acc0 = !(h0 == 0 && kb == 0);
                            if (ks == 4) {
                                detail::issue_ts_pass<4>(d, a2h, bh, desc_k, idesc2, acc0);                  // A2_hi C_hi^T
                                detail::issue_ts_pass<4>(d, a2l, bh, desc_k, idesc2, true);                  // A2_lo C_hi^T
                                detail::issue_ts_pass<4>(d, a2h, bl, desc_k, idesc2, true);                  // A2_hi C_lo^T
                            } else {
                                detail::issue_ts_pass_n(ks, d, a2h, bh, desc_k, idesc2, acc0);
                                detail::issue_ts_pass_n(ks, d, a2l, bh, desc_k, idesc2, true);
                                detail::issue_ts_pass_n(ks, d, a2h, bl, desc_k, idesc2, true);
                            }
                            mma_commit(b_empty + bp);
                            if (++bp == S::NBB) { bp = 0; bpar ^= 1u; }
                            ++n_steps;
                        }
                    }
                }
                mma_commit(acc_ready);                              // D2 of this item is complete
                first_item = false;
            }
            if (tracing) {
                tr[6] = clock64() - t_begin;
                tr[7] = n_steps;
                for (int i = 0; i < 8; ++i) a.trace[i] = tr[i];
            }
        }
        __syncwarp();
    } else if (warp == NC / 32 + 1) {
        // =========================================================== basis producer: one elected thread
        if (elect_one()) {
            uint32_t bp = 0, round = 0;                             // buffer of this step, how often the ring wrapped
            auto fetch = [&](uint32_t cb, uint32_t row0, uint32_t rows) {           // slab (rows row0.., column block cb) -> buffer bp
                if (round >= 1) wait(b_empty + bp, (round - 1) & 1u);               // the MMAs that last read this buffer are done
                const uint32_t bytes = rows * 128u, off = (cb * (uint32_t)a.NPR + row0) * 128u;
                mbar_arrive_expect_tx(b_full + bp, 2 * bytes);
                bulk_g2s(b_base + bp * S::B_BUF, a.c_hi + off, bytes, b_full + bp);
                bulk_g2s(b_base + bp * S::B_BUF + S::B_HALF, a.c_lo + off, bytes, b_full + bp);
                if (++bp == S::NBB) { bp = 0; ++round; }
            };
            for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
                const int v0 = (item % a.NVC) * 128;
                const uint32_t mv16 = (uint32_t)((min(128, N - v0) + 15) & ~15);
                for (int h0 = 0; h0 < N; h0 += 128) {
                    const int nkb = (min(128, N - h0) + 63) >> 6;
                    for (int w0 = 0; w0 < N; w0 += 64) fetch(w0 >> 6, v0, mv16);
                    for (int uc = 0; uc < a.NUC; ++uc)
                        for (int kb = 0; kb < nkb; ++kb) fetch((h0 >> 6) + kb, uc * a.NU, a.NU);
                }
            }
        }
        __syncwarp();
    } else if (warp == NC / 32 + 2) {
        // =========================================================== map producer: one elected thread, one TMA per map slab,
        //     in the order the converters consume them: (item, h-tile, 64-wide w block)
        if (elect_one()) {
            tma_prefetch_desc(&xmap.m[0]);
            uint32_t k = 0;
            int sg = 0;
            for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
                advance_segment(a.seg, item, sg);
                const int row0 = ((item - a.seg.tile0[sg]) / a.NVC) * N;
                for (int h0 = 0; h0 < N; h0 += 128)
                    for (int w0 = 0; w0 < N; w0 += 64, ++k) {
                        const uint32_t set = k & 1u;
                        if (k >= 2) wait(stg_free + set, ((k >> 1) - 1u) & 1u);
                        mbar_arrive_expect_tx(stg_full + set, S::STAGE_BUF);
                        tma_load_2d(smem + S::OFF_STAGE + set * S::STAGE_BUF, &xmap.m[sg], w0, row0 + h0, stg_full + set);
                    }
            }
        }
        __syncwarp();
    } else {
        // =========================================================== converter / epilogue warps
        const uint32_t lane = tid & 31;
        const uint32_t lane_idx = (warp & 3) * 32 + lane;          // this thread's TMEM lane
        const uint32_t col_blk = warp >> 2;                        // which 16-column blocks of an epilogue it handles
        const uint32_t tmem_lane = tmem + (((warp & 3) * 32u) << 16);
        uint32_t xp = 0, xround = 0, acc_cnt = 0;                  // map slab ring position / wraps, accumulator hand-overs consumed

        // The staged slab is row-major [128 rows][64 floats]; thread t converts vectors t, t + 512, ...: row (i >> 4), float4 (i & 15),
        // so a warp reads 512 contiguous bytes and the operand offset of a thread's vector is fixed up to + 32 rows per step.
        uint8_t* stage = smem + S::OFF_STAGE;
        uint32_t xk = 0;                                           // map slabs consumed so far (staging buffer xk & 1)
        const uint32_t xoff16 = detail::kmajor_off(tid >> 4, (tid & 15) * 4, 128);    // full-width block: + j * 4096 B per 32 rows
        auto store_x = [&](uint32_t set, uint32_t p) {
            uint8_t* hi = a1_base + p * S::A1_BUF;
            uint8_t* lo = hi + S::A1_HALF;
            const float4* src = reinterpret_cast<const float4*>(stage + set * S::STAGE_BUF) + tid;
            float4 v[XV];
#pragma unroll
            for (int j = 0; j < XV; ++j) v[j] = src[j * NC];
#pragma unroll
            for (int j = 0; j < XV; ++j)
                detail::Scatter<1>::st(hi + j * (NC / 16) * 128, lo + j * (NC / 16) * 128, static_cast<uint16_t>(xoff16), v[j]);
        };
        long long ctr[5] = {0, 0, 0, 0, 0};
        // one stage-1 step of this thread: wait for the operand buffer and the staged slab, convert + store, hand both over
        auto x_step = [&]() {
            const bool tr = TRACE && a.trace != nullptr && blockIdx.x == 0 && tid == 0;
            const uint32_t set = xk & 1u;
            const long long t0 = tr ? clock64() : 0;
            if (xround >= 1) wait(x_empty + xp, (xround - 1) & 1u);       // the MMAs that last read this buffer are done
            const long long t1 = tr ? clock64() : 0;
            wait(stg_full + set, (xk >> 1) & 1u);
            const long long t2 = tr ? clock64() : 0;
            store_x(set, xp);
            __syncwarp();
            if (lane == 0) mbar_arrive(stg_free + set);                   // (the slab is in registers / stored: the TMA may refill it)
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(x_full + xp);
            if (tr) {
                ctr[0] += t1 - t0; ctr[3] += t2 - t1; ctr[1] += clock64() - t2; ctr[4] += 1;
            }
            ++xk;
            if (++xp == S::NXB) { xp = 0; ++xround; }
        };

        int item = blockIdx.x;
        const int NB = (N + 63) >> 6;                              // 64-wide w blocks per tile
        const int PS = min((int)S::NXB, NB);                       // slabs of the following tile stored ahead of time
        int first_block = 0;                                       // this tile's slabs [0, first_block) are already stored
        int sg = 0;
        for (; item < a.n_items; item += gridDim.x) {
            advance_segment(a.seg, item, sg);
            const int map = (item - a.seg.tile0[sg]) / a.NVC, vc = item % a.NVC;       // map within its segment, v-chunk
            const int v0 = vc * 128, MV = min(128, N - v0);
            const int nitem = item + (int)gridDim.x;               // what this CTA works on next

            for (int h0 = 0; h0 < N; h0 += 128) {
                const int MH = min(128, N - h0);
                // ---- stage 1 operands: X slab rows h0.., one step per 64-wide w block
                for (int b = first_block; b < NB; ++b) x_step();
                const bool more = h0 + 128 < N || nitem < a.n_items;   // is there a tile after this one (next h-tile, or the next item's first)
                // ---- epilogue 1: D1 row v (lane), columns h -> bf16 hi/lo pairs -> A2 over the same TMEM columns
                wait(acc_ready, acc_cnt & 1u);                     // all stage-1 MMAs of the tile (and everything before) are complete
                ++acc_cnt;
                tc_fence_after_sync();
                {
                    const int MH16 = (MH + 15) & ~15;
                    uint32_t r0[16], r1[16];
                    const int c0 = col_blk * 16, c1 = c0 + 64;     // this warp's 16-column blocks
                    if (c0 < MH16) tmem_ld16(tmem_lane + d1_col + c0, r0);
                    if (c1 < MH16) tmem_ld16(tmem_lane + d1_col + c1, r1);
                    tmem_ld_wait();
                    tc_fence_before_sync();
                    named_bar_sync(2, NC);                         // every warp has read its columns: they may be overwritten now
                    tc_fence_after_sync();
                    uint32_t hi[16], lo[16];
                    if (c0 < MH16) {
#pragma unroll
                        for (int p = 0; p < 8; ++p) split2(__uint_as_float(r0[2 * p]), __uint_as_float(r0[2 * p + 1]), hi[p], lo[p]);
                        tmem_st8(tmem_lane + d1_col + (c0 >> 1), hi);
                        tmem_st8(tmem_lane + d1_col + 64 + (c0 >> 1), lo);
                    }
                    if (c1 < MH16) {
#pragma unroll
                        for (int p = 0; p < 8; ++p) split2(__uint_as_float(r1[2 * p]), __uint_as_float(r1[2 * p + 1]), hi[p], lo[p]);
                        tmem_st8(tmem_lane + d1_col + (c1 >> 1), hi);
                        tmem_st8(tmem_lane + d1_col + 64 + (c1 >> 1), lo);
                    }
                    tmem_st_wait();
                }
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(a2_full);
                // ---- the X ring is idle during stage 2: fill it with the next tile's first slabs now (the loads of the
                //      third and fourth have the whole of stage 2 to arrive), so its stage 1 never waits for operands
                first_block = 0;
                if (more) {
                    for (int b = 0; b < PS; ++b) x_step();
                    first_block = PS;
                }
            }

            // ---- epilogue 2: lane v < MV holds Z[:, v]; energy of the v-chunk = sum over lanes and all N columns
            wait(acc_ready, acc_cnt & 1u);
            ++acc_cnt;
            tc_fence_after_sync();
            float e = 0.f;
#pragma unroll 1
            for (int c0 = col_blk * 16; c0 < a.NU * a.NUC; c0 += 64) {
                uint32_t r[16];
                tmem_ld16(tmem_lane + d2_col + c0, r);
                tmem_ld_wait();
                if ((int)lane_idx < MV) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const int u = c0 + i;
                        const float z = u < N ? __uint_as_float(r[i]) : 0.f;
                        e = fmaf(z, z, e);
                        if (TRACE && a.dump != nullptr && u < N) a.dump[(size_t)map * NN + (size_t)u * N + v0 + lane_idx] = z;
                    }
                }
            }
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(d2_free);
            red[tid] = (int)lane_idx < MV ? e : 0.f;
            named_bar_sync(1, NC);
            if (tid < 32) {
                float s = 0.f;
#pragma unroll
                for (int j = 0; j < NC / 32; ++j) s += red[tid + 32 * j];          // fixed order
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if (tid == 0) {
                    atomicAdd(a.seg.accum[sg] + (map % a.seg.c_count[sg]), (double)s);
                    if (a.energy_parts) a.energy_parts[(size_t)map * a.NVC + vc] = s;
                }
            }
            named_bar_sync(1, NC);
        }
        if (TRACE && a.trace != nullptr && blockIdx.x == 0 && tid == 0)
            for (int i = 0; i < 5; ++i) a.trace[8 + i] = ctr[i];
    }
    if (dead && (tid & 31u) == 0)                                  // a hand-over never came (status word set): poison the result
        for (int sgi = 0; sgi < a.seg.n_seg; ++sgi)
            for (int c = 0; c < a.seg.c_count[sgi]; ++c) a.seg.accum[sgi][c] = __longlong_as_double(0x7FF8000000000000ll);
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem);
}

// energy_out[m] = parts[m][0] + parts[m][1] + ... (fixed order)
__global__ void sum_parts_kernel(const float* parts, int nvc, float* out, int n) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m < n) {
        float s = 0.f;
        for (int j = 0; j < nvc; ++j) s += parts[(size_t)m * nvc + j];
        out[m] = s;
    }
}

}  // namespace dctp
