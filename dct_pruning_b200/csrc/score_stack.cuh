// Fused DCT-score hook kernel, "stacked basis" formulation (dense tensors, even map side 10..64).
//
// Same contract as score_umma.cuh / score_tmem.cuh (/root/reference/utils/common.py:262-277: per-(image, channel)
// orthonormal 2-D DCT-II energy, summed per channel).  What changes is how the first contraction is laid on the
// tensor core.  score_tmem.cuh gets its transposed intermediate from a block-diagonal TMEM operand I_G (x) C_N and
// pays a factor G of wasted MMA work plus three passes; here the TMEM operand is the basis itself with its bf16
// hi and lo parts STACKED along M (the 128 accumulator lanes), and the maps of a tile are concatenated along the
// MMA's N dimension:
//
//   lanes     lane = 32q + 16p + r :  p = 0 rows of C_hi, p = 1 rows of C_lo, basis row v = v(q, r)
//             J = 64 / KP map "sets" share the 128 lanes (KP = N rounded up to 16):
//               KP 48/64: J = 1, v = 16q + r     KP 32: J = 2, set = q / 2, v = 16 (q % 2) + r     KP 16: J = 4, set = q, v = r
//   stage 1   D1[(q,p,r), (g,h)] = sum_{(set',w)} A[(q,p,r), (set',w)] * Bx[(g,h), (set',w)]         2 passes: Bx_hi, Bx_lo
//             A  = the stacked basis, block structured over the sets, resident in TMEM for the whole kernel
//             Bx[(g,h), (set,w)] = X_{g,set}[h,w]: the raw rows of the maps, K-major in shared memory (N-side operand)
//             -> lanes p = 0 hold C_hi (X_hi + X_lo)^T, lanes p = 1 hold C_lo (X_hi + X_lo)^T: all four split-precision
//                terms in two passes, no block-diagonal waste (the maps sit side by side along N, not along K)
//   epi   1   tcgen05.ld 16x256b fragments of both lane halves -> y = za + zb (fp32) -> bf16 hi/lo pairs ->
//             tcgen05.st 16x128b: A2[(q,s,r), h] for map g = 2t + s of the warp's set; never leaves TMEM
//   stage 2   per A2 tile t:  D2[(q,s,r), u] = sum_h A2[(q,s,r), h] * C[u,h]       3 passes (hi*hi + lo*hi + hi*lo)
//             B = C_N resident in shared memory; every lane of a tile is a live row (two maps per warp)
//             KP >= 32 folded (stack_folded): epilogue 1 writes the row sums and differences of D1 (y + y', y - y' of rows h, N-1-h),
//             and each pass is two chains of half the K and N, even u against the sums and odd u against the differences
//   epi   2   tcgen05.ld 32x32b -> sum of squares per lane -> 16-lane shuffle tree -> fixed-order sum over the
//             warps of a map -> one fp64 atomicAdd per map
//
// Tensor-core time per 25 KB of input: 448 + 192 cycles at 56x56 (unfolded stage 2 384; score_tmem.cuh: 672 + 384), 512 + 96 at 28x28
// (unfolded 192), 512 + 96 at 14x14 (not folded), against 940-1113 cycles of HBM time at the measured 6.55 TB/s (the SM clock under this
// load is 1.65-1.7 GHz, not the 1.965 GHz nvidia-smi shows).  The fold also halves the shared-memory reads of the stage-2 basis, 192 -> 96
// wavefronts per tile at 56x56 and 28x28.
//
// The kernel is warp specialised (one CTA per SM), every hand-over is an mbarrier.  Roles, in warp order:
//   converters  NCONV warps (12 in production) in NCG = 2 groups that alternate tiles: fp32 tile -> bf16 hi/lo -> Bx (two buffers),
//               offsets from a host-built table
//   epilogue 1  NE1G groups of 8 warps (one in production; warp = lane quarter q x row slot s); group g takes the CTA's tiles g, g + NE1G, ...
//   epilogue 2  NE2G groups of 4 warps (two in production) that alternate tiles
//   producer    1 warp (one thread): one cp.async.bulk.tensor.2d per tile (tensor map over the dense fp32 stream viewed as
//               [rows, 32 floats]; a tile is a box of tile_rows rows; rows past the end arrive as zeros) into a ring of 3
//   issuers     2 warps (one thread each): stage 1 and stage 2 have their own issuing thread, so that neither the waits nor
//               the ~25 cycles it takes to issue an MMA of one stage hold up the other
// TMEM (512 columns): A 32 | D1 2 x 128 | A2 2 x 64 | D2 NB2 x 64 (NB2 = 1: 480 columns in use).
//
// 16-bit input (IN = IN_BF16 / IN_F16, an autocast forward's activations): the tensor map views the stream as [rows, 32 elements]
// (64-byte rows: tile_rows and the tail rule stay those of fp32 - a tile of 2 x 22 x 22 or 8 x 18 x 18 maps is not a whole number of
// 128-byte rows of 16-bit elements), and a converter thread reads 4 elements (8 bytes) per table entry, so the offset table and the
// Bx layout are the fp32 ones.  A bf16 value is its own bf16 hi part: the converters store it into Bx_hi unchanged and stage 1 issues
// the Bx_hi pass only (the Bx_lo pass would add exact zeros).  fp16 (11 significant bits) splits exactly into a bf16 hi / lo pair: it
// is widened in registers and runs the fp32 split.
#pragma once
#include <type_traits>
#include "score_common.cuh"
#include "umma.cuh"

namespace dctp {

struct StackArgs {
    ScoreSegments seg;
    int N, NN, Np;                  // map side, N*N, rows a map takes in Bx (= D1 columns per map): N rounded up to 8
    int G, MT;                      // maps per set and per tile (MT = G * J)
    int ncols;                      // G * Np = MMA N of stage 1
    int tile_elems, tile_rows, tile_vec, num_tiles;
    uint32_t idesc1, idesc2;
    uint32_t lbo1;                  // Bx: byte distance between consecutive 8-element k-chunks (2048 + 16 u, u chosen per side for conflict-free stores)
    const uint32_t* a_img;          // [128][32] packed bf16 pairs: the stacked basis as it sits in TMEM
    const uint8_t* c2_hi;           // stage-2 basis as a shared-memory operand image (hi, lo): OperandImage64::BYTES each
    const uint8_t* c2_lo;
    const uint16_t* table;          // [tile_vec] (VEC 4) / [2 * tile_vec] (VEC 2) byte offsets of a float4's pieces in Bx
    uint32_t table_bytes;
    float* energy_out;              // optional, single-segment launches only: [n_maps] per-map energies
    float* dump;                    // optional, single-segment launches only: coefficients
    int* status;
    long long* trace;               // bring-up aid (DCTP_S_TRACE): per role of CTA 0, cycles spent waiting / working
};

struct StackSmem {
    static constexpr uint32_t NSTG = 3, STG_STRIDE = 32768;              // TMA ring: fp32 tiles of at most 32 KB
    static constexpr uint32_t LBO1_MAX = 128 * 16 + 16 * 7;              // Bx: k-chunk c of row n at c * lbo1 + n * 16; lbo1 = 2048 + 16 u spreads the banks
    static constexpr uint32_t BX_HALF = 8 * LBO1_MAX;                    // 17280
    static constexpr uint32_t OFF_BX = NSTG * STG_STRIDE;
    static constexpr uint32_t NBX = 3;                                   // room for three Bx buffers (hi | lo each); how many a kernel uses: see NBXK
    static constexpr uint32_t OFF_C2 = OFF_BX + 2 * NBX * BX_HALF;
    static constexpr uint32_t OFF_TABLE = OFF_C2 + 2 * OperandImage64::BYTES;   // stage-2 basis (hi | lo)
    static constexpr uint32_t TABLE_MAX = 8192;
    static constexpr uint32_t OFF_RED = OFF_TABLE + TABLE_MAX;
    static constexpr uint32_t OFF_BARS = OFF_RED + 256;
    static constexpr uint32_t OFF_SLOT = OFF_BARS + 256;
    static constexpr uint32_t TOTAL = OFF_SLOT + 128;
};

// Role groups: converters in NCG groups (group g converts the CTA's tiles g, g + NCG, ...), NE1G epilogue-1 groups and NE2G
// epilogue-2 groups (group g takes the CTA's tiles g, g + NE1G / NE2G, ...).
constexpr int STACK_NCG = 2, STACK_NE1G = 1, STACK_NE2G = 2;
// warps of a CTA with NCONV converter warps: converters, epilogue 1 (8 per group), epilogue 2 (4 per group), producer, two issuers
constexpr int stack_warps(int nconv) { return nconv + 8 * STACK_NE1G + 4 * STACK_NE2G + 3; }

// Folded stage 2 (KP >= 32; at KP = 16 one chain is already K = 16, the minimum).  The DCT-II basis has C[u][N-1-h] = (-1)^u C[u][h],
// so  D2[., u] = sum_{h < N/2} C[u][h] (Y[., h] + (-1)^u Y[., N-1-h]):  two chains of K = N = stack_fold_k(KP) each - even u against
// the row sums of Y = D1, odd u against the row differences - do the work of one chain of K = N = KP, with half the MMA work and half
// the basis reads.  The converters' table puts row N-1-h of a map at D1 column fold_d + h (fold_d = 8 * (Np / 16)), so that each
// thread of epilogue 1 holds both rows of a pair; with Np / 8 odd (N = 18..24, 36, 40, 52, 56 - whole 8-column halves would not fit
// in Np) only rows h < fold_d are paired, and the middle rows [fold_d, N - fold_d) sit unpaired in the 8 columns from 2 * fold_d on,
// in both chains (the basis holds C[u][h] there for every u).  A2 and D2 of a map: even chain at [0, K), odd chain at [K, 2K).
__host__ __device__ constexpr bool stack_folded(int kp) { return kp >= 32; }
__host__ __device__ constexpr int stack_fold_k(int kp) { return kp == 32 ? 16 : 32; }

// KP: contraction length per map (N rounded up to 16); VEC: granularity of a row in the fp32 stream (4: N % 4 == 0, 2: N even)
// NCONV: converter warps (8 or 12).
// Every warp polls the mbarriers it depends on itself.  (Measured and dropped: one polling warp per role releasing its siblings
// through a named barrier - the polls cost issue slots, the sleep behind mbarrier.try_wait being woken by any barrier event of
// the CTA, but the extra hop costs more: 56x56 3.17 against 3.49 TB/s.)
// NP8: Np / 8 as a compile-time constant - epilogue 1's column loops lose their branches.
// TRACE: the debug instantiation - the cycle accounting of DCTP_S_TRACE, the per-map energies (energy_out) and the coefficient dump
// (coeff_out); the production instantiations carry none of that code (the host routes launches that ask for any of it here).
// IN: element type of the activation (IN_F32, IN_BF16, IN_F16; see the head of this file).
template <int KP, int VEC, int NCONV, int NP8, bool TRACE, int IN = IN_F32>
__global__ void __launch_bounds__(stack_warps(NCONV) * 32, 1) score_stack_kernel(const __grid_constant__ ScoreTensorMaps tmaps, const __grid_constant__ StackArgs a) {
    using S = StackSmem;
    using namespace umma;
    constexpr int NCG = STACK_NCG, NE1G = STACK_NE1G, NE2G = STACK_NE2G;
    constexpr int J = KP <= 32 ? 64 / KP : 1;
    constexpr int K1S = J * KP / 16;
    constexpr int G = KP == 16 ? 8 : KP == 32 ? 4 : 2, T2 = G / 2;
    // stage 2: NC2 chains (two when folded) of K = N = W2; a map's A2 (hi part, in bf16 elements) and D2 take KF = NC2 * W2 columns
    constexpr bool FOLD = stack_folded(KP);
    constexpr int W2 = FOLD ? stack_fold_k(KP) : KP, NC2 = FOLD ? 2 : 1, KF = NC2 * W2, K2S = W2 / 16;
    static_assert(T2 * KF <= 64, "A2 and D2 buffers are 64 columns");
    constexpr uint32_t W_E1 = NCONV, W_E2 = NCONV + 8 * NE1G, W_PROD = W_E2 + 4 * NE2G, W_MMA = W_PROD + 1, W_MMA2 = W_PROD + 2, NT = (W_MMA2 + 1) * 32;
    constexpr uint32_t NCT = NCONV * 32 / NCG;                            // threads that convert one tile
    // Bx buffers in use: with three the converters run a tile further ahead of stage 1 (same box: 56x56 4.25 -> 4.59 TB/s, 64-channel launches
    // 3.74 -> 4.1, 14x14 3.55 -> 3.6; at KP = 32 it loses, 28x28 3.95 -> 3.60, so those instantiations keep two)
    constexpr uint32_t NBXK = KP == 32 ? 2u : 3u;
    constexpr uint32_t TM_A = 0, TM_D1 = 32;                              // TMEM columns: A | D1 x 2 | A2 x 2 (64 each) | D2 x NB2 (64 each)
    const uint32_t d1_stride = a.ncols <= 112 ? 112u : 128u;
    const uint32_t TM_A2 = TM_D1 + 2 * d1_stride, TM_D2 = TM_A2 + 128;
    const uint32_t nb2 = TM_D2 + 128 <= 512 ? 2u : 1u;                    // a second D2 buffer when D1 is at most 112 columns wide
    const uint32_t STEP1 = (2 * a.lbo1) >> 4;                             // one k-step (two 8-element chunks) in descriptor units
    constexpr uint32_t STEP2 = (2 * OperandImage64::LBO) >> 4;

    extern __shared__ __align__(1024) uint8_t smem[];
    // (the warp index comes out of a shuffle so that the compiler knows it is warp-uniform: role addresses stay in uniform registers)
    const uint32_t tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    uint8_t* stg = smem;
    uint8_t* bx = smem + S::OFF_BX;                                       // [buffer][hi | lo]
    uint8_t* c2 = smem + S::OFF_C2;
    const uint8_t* tab = smem + S::OFF_TABLE;
    float* red = reinterpret_cast<float*>(smem + S::OFF_RED);             // [parity][q][8]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BARS);
    uint64_t* stg_full = bars;                                            // [3] TMA landed (tx bytes)
    uint64_t* stg_free = bars + 3;                                        // [3] NCONV converter warps
    uint64_t* bx_full = bars + 6;                                         // [3] the converter warps of the tile's group
    uint64_t* bx_free = bars + 9;                                         // [3] stage-1 MMAs of the buffer have completed
    uint64_t* d1_full = bars + 12;                                        // [2] ... and D1 is complete
    uint64_t* d1_free = bars + 14;                                        // [2] 8 epilogue-1 warps have read it
    uint64_t* a2_full = bars + 16;                                        // [2] 8 epilogue-1 warps have written A2
    uint64_t* a2_free = bars + 18;                                        // [2] stage-2 MMAs have read it
    uint64_t* d2_full = bars + 20;                                        // [2]
    uint64_t* d2_free = bars + 22;                                        // [2] 4 epilogue-2 warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::OFF_SLOT);

    long long tr_entry = 0;                                               // (debug instantiation) wall-clock stamps of the launch's phases
    if (TRACE && a.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_entry));
    // ---- prologue (independent of the activation).  Barriers and TMEM first: once they exist the producer warp goes ahead and has
    //      the first three tiles on their way from HBM while the other warps stage the bases and zero the operand buffers.
    if (warp == W_MMA) tmem_alloc<512>(tmem_slot);
    if (tid == 0) {
        for (int s = 0; s < 3; ++s) { mbar_init(stg_full + s, 1); mbar_init(stg_free + s, NCONV / NCG); }
        for (int b = 0; b < (int)S::NBX; ++b) { mbar_init(bx_full + b, NCONV / NCG); mbar_init(bx_free + b, 1); }
        for (int b = 0; b < 2; ++b) {
            mbar_init(d1_full + b, 1); mbar_init(d1_free + b, 8);
            mbar_init(a2_full + b, 8); mbar_init(a2_free + b, 1);
            mbar_init(d2_full + b, 1); mbar_init(d2_free + b, 4);              // (4 warps of ONE epilogue-2 group read a tile)
        }
        mbar_init_fence();
    }
    if (warp == W_PROD && lane == 0) tma_prefetch_desc(&tmaps.m[0]);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    launch_dependents();                                                  // this CTA holds its TMEM columns (see score_umma.cuh)
    if (TRACE && a.trace != nullptr && blockIdx.x == 0 && tid == 0) { long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); a.trace[52] = t_ - tr_entry; }
    if (warp != W_PROD) {
        const uint32_t ptid = tid < W_PROD * 32 ? tid : tid - 32;          // thread index among the NT - 32 staging threads
        constexpr uint32_t PNT = NT - 32;
        // Every global load of the prologue is issued before the first store (the stores are to shared memory / TMEM, which the compiler
        // will not move loads across): one exposed L2 / HBM latency instead of four - 3.4 -> ~1.5 us of the ~10 us a launch costs beyond
        // its bytes, which is what the 6-50 MB launches of the small layers are made of.
        static_assert(2 * PNT * 16 >= OperandImage64::BYTES && PNT * 16 >= S::TABLE_MAX, "prologue loads are unrolled for these sizes");
        uint4 c2h[2], c2l[2], tb = make_uint4(0, 0, 0, 0), ai[8];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const uint32_t off = (ptid + i * PNT) * 16;
            if (off < OperandImage64::BYTES) {
                c2h[i] = *reinterpret_cast<const uint4*>(a.c2_hi + off);
                c2l[i] = *reinterpret_cast<const uint4*>(a.c2_lo + off);
            }
        }
        if (ptid * 16 < a.table_bytes) tb = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(a.table) + ptid * 16);
        if (warp < 4) {
#pragma unroll
            for (int i = 0; i < 8; ++i) ai[i] = reinterpret_cast<const uint4*>(a.a_img + tid * 32)[i];
        }
        for (uint32_t off = ptid * 16; off < 2 * S::NBX * S::BX_HALF; off += PNT * 16) *reinterpret_cast<uint4*>(bx + off) = make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const uint32_t off = (ptid + i * PNT) * 16;
            if (off < OperandImage64::BYTES) {
                *reinterpret_cast<uint4*>(c2 + off) = c2h[i];
                *reinterpret_cast<uint4*>(c2 + OperandImage64::BYTES + off) = c2l[i];
            }
        }
        if (ptid * 16 < a.table_bytes) *reinterpret_cast<uint4*>(smem + S::OFF_TABLE + ptid * 16) = tb;
        if (warp < 4) {                                                   // the stacked basis -> TMEM columns [0,32)
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                uint32_t v[16];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint4 q4 = ai[4 * part + i];
                    v[4 * i] = q4.x; v[4 * i + 1] = q4.y; v[4 * i + 2] = q4.z; v[4 * i + 3] = q4.w;
                }
                tmem_st16(tmem + ((warp * 32u) << 16) + TM_A + part * 16, v);
            }
            tmem_st_wait();
        } else if (warp < 8) {                                            // A2 (both buffers): columns a tile never writes stay zero
            uint32_t z[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) z[i] = 0u;
#pragma unroll
            for (int part = 0; part < 8; ++part) tmem_st16(tmem + (((warp & 3u) * 32u) << 16) + TM_A2 + part * 16, z);
            tmem_st_wait();
        }
        fence_async_smem();
        tc_fence_before_sync();
        named_bar_sync(6, NT - 32);                                       // every warp but the producer
        tc_fence_after_sync();
    }
    grid_dependency_wait();                                               // the activation is complete

    long long tr_c0 = 0, tr_g0 = 0;
    if (TRACE && a.trace != nullptr && blockIdx.x == 0 && tid == 0) {
        tr_c0 = clock64();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_g0));
        a.trace[53] = tr_g0 - tr_entry;                                   // TMEM + barriers + bases staged + the preceding kernel complete
    }
    const int first = blockIdx.x, stride = gridDim.x;
    const uint32_t tile_bytes = static_cast<uint32_t>(a.tile_rows) * (32u * in_bytes(IN));      // rows of 32 elements
    bool dead = false;
    // segment of a tile: the roles walk the tiles in increasing order, so each keeps a cursor.  A segment whose stream does not end
    // on a 32-element row (128 bytes in fp32, 64 in 16-bit) has its last tile converted from global memory (that row is not in the tensor map).
    auto is_tail = [&](int tile, int sg) {
        return tile == a.seg.tile0[sg + 1] - 1 && (a.seg.total_elems[sg] & 31) != 0;
    };
    // bring-up trace: one thread per role accumulates cycles in registers and writes them when its loop ends
    const bool tr_on = TRACE && a.trace != nullptr && blockIdx.x == 0;
    bool tr_me = false;
    long long tr_mark = 0, tr0 = 0, tr1 = 0, tr2 = 0, tr3 = 0, tr4 = 0, tr5 = 0;
#define TR_START() do { if (tr_me) tr_mark = clock64(); } while (0)
#define TR_ADD(acc) do { if (tr_me) { const long long now_ = clock64(); (acc) += now_ - tr_mark; tr_mark = now_; } } while (0)
#define TR_FLUSH(base) do { if (tr_me) { a.trace[(base)] = tr0; a.trace[(base) + 1] = tr1; a.trace[(base) + 2] = tr2; a.trace[(base) + 3] = tr3; \
                                         a.trace[(base) + 4] = tr4; a.trace[(base) + 5] = tr5; } } while (0)
    if (warp == W_PROD) {
        // ================================================================ TMA producer
        if (elect_one()) {
            tr_me = tr_on;
            uint32_t it = 0;
            int sg = 0;
            for (int tile = first; tile < a.num_tiles; tile += stride) {
                advance_segment(a.seg, tile, sg);
                if (is_tail(tile, sg)) continue;
                const uint32_t s = it % S::NSTG;
                TR_START();
                if (it >= S::NSTG && !mbar_wait(stg_free + s, ((it / S::NSTG) - 1u) & 1u)) { dead = true; break; }
                TR_ADD(tr0);
                mbar_arrive_expect_tx(stg_full + s, tile_bytes);
                tma_load_2d(stg + s * S::STG_STRIDE, &tmaps.m[sg], 0, (tile - a.seg.tile0[sg]) * a.tile_rows, stg_full + s);
                ++it;
            }
            TR_FLUSH(0);
        }
        __syncwarp();
    } else if (warp == W_MMA) {
        // ================================================================ MMA issuer, stage 1: D1 = A * Bx^T (Bx_hi, then Bx_lo)
        constexpr int P1 = IN == IN_BF16 ? 1 : 2;                          // bf16 input: X_lo = 0, the Bx_lo pass is not issued
        if (elect_one()) {
            tr_me = tr_on;
            const uint64_t desc = make_smem_desc(0, a.lbo1, 128, SWIZZLE_NONE);
            uint32_t n = 0;
            for (int tile = first; tile < a.num_tiles; tile += stride, ++n) {
                const uint32_t b = n & 1u, bb = n % NBXK;                  // D1 buffer, Bx buffer
                TR_START();
                if (!mbar_wait(bx_full + bb, (n / NBXK) & 1u)) { dead = true; break; }
                TR_ADD(tr0);
                if (n >= 2 && !mbar_wait(d1_free + b, ((n >> 1) - 1u) & 1u)) { dead = true; break; }
                TR_ADD(tr1);
                tc_fence_after_sync();
                const uint32_t d1 = tmem + TM_D1 + b * d1_stride;
                const uint32_t lo_hi = static_cast<uint32_t>(desc) + (smem_u32(bx + bb * 2 * S::BX_HALF) >> 4);
                const uint32_t lo_lo = lo_hi + (S::BX_HALF >> 4);
#pragma unroll
                for (int pass = 0; pass < P1; ++pass)
#pragma unroll
                    for (int ks = 0; ks < K1S; ++ks)
                        mma_bf16_ts(d1, tmem + TM_A + 8 * ks, desc_with_lo(desc, (pass ? lo_lo : lo_hi) + ks * STEP1), a.idesc1,
                                    (pass | ks) != 0);
                mma_commit(d1_full + b);
                mma_commit(bx_free + bb);
                TR_ADD(tr2);
            }
            TR_FLUSH(8);
            if (TRACE && tr_me) a.trace[14] = n;
        }
        __syncwarp();
    } else if (warp == W_MMA2) {
        // ================================================================ MMA issuer, stage 2: D2 = A2 * C^T (hi*hi + lo*hi + hi*lo)
        if (elect_one()) {
            tr_me = tr_on;
            const uint64_t desc2 = make_smem_desc(0, OperandImage64::LBO, 128, SWIZZLE_NONE);
            const uint32_t lo_c2_hi = static_cast<uint32_t>(desc2) + (smem_u32(c2) >> 4);
            const uint32_t lo_c2_lo = lo_c2_hi + (OperandImage64::BYTES >> 4);
            uint32_t m = 0;
            for (int tile = first; tile < a.num_tiles; tile += stride, ++m) {
                const uint32_t b = m & 1u;
                TR_START();
                if (!mbar_wait(a2_full + b, (m >> 1) & 1u)) { dead = true; break; }
                TR_ADD(tr0);
                // D2 barriers go by tile parity (each epilogue-2 group, or the one group alternately, sees every phase of its own
                // barrier); the buffer is b with two buffers, 0 with one - then the previous tile's reader must have let go of it
                const uint32_t b2 = nb2 == 2 ? b : 0u;
                if (nb2 == 2 ? (m >= 2 && !mbar_wait(d2_free + b, ((m >> 1) - 1u) & 1u))
                             : (m >= 1 && !mbar_wait(d2_free + ((m - 1u) & 1u), ((m - 1u) >> 1) & 1u))) { dead = true; break; }
                TR_ADD(tr1);
                tc_fence_after_sync();
#pragma unroll
                for (int t = 0; t < T2; ++t)
#pragma unroll
                    for (int c = 0; c < NC2; ++c) {                        // chain c: columns [c W2, (c + 1) W2) of the map, basis rows too
                        const uint32_t d = tmem + TM_D2 + b2 * 64 + t * KF + c * W2;
                        const uint32_t ahi = tmem + TM_A2 + b * 64 + t * KF + c * (W2 / 2), alo = ahi + KF / 2;
#pragma unroll
                        for (int pass = 0; pass < 3; ++pass)
#pragma unroll
                            for (int ks = 0; ks < K2S; ++ks)
                                mma_bf16_ts(d, (pass == 1 ? alo : ahi) + 8 * ks,
                                            desc_with_lo(desc2, (pass == 2 ? lo_c2_lo : lo_c2_hi) + c * W2 + ks * STEP2), a.idesc2,
                                            (pass | ks) != 0);
                    }
                mma_commit(d2_full + b);
                mma_commit(a2_free + b);
                TR_ADD(tr2);
            }
            TR_FLUSH(40);
        }
        __syncwarp();
    } else if (warp < W_E1) {
        // ================================================================ converters: fp32 tile -> bf16 hi/lo -> Bx
        const uint32_t cg = warp / (NCONV / NCG), ctid = tid - cg * NCT;     // converter group, thread within it
        uint32_t n = 0, it = 0;                                            // the CTA's tile number / its TMA sequence number
        int sg = 0;
        tr_me = tr_on && tid == 0;
        for (int tile = first; tile < a.num_tiles; tile += stride, ++n) {
            advance_segment(a.seg, tile, sg);
            const bool tail = is_tail(tile, sg);
            if (n % NCG != cg) {                                           // the other group's tile: only keep the TMA count in step
                if (!tail) ++it;
                continue;
            }
            const uint32_t b = n % NBXK, s = it % S::NSTG;
            TR_START();
            {
                bool ok = true;
                if (n >= NBXK) ok = mbar_wait(bx_free + b, ((n / NBXK) - 1u) & 1u);
                TR_ADD(tr0);
                if (ok && !tail) ok = mbar_wait(stg_full + s, (it / S::NSTG) & 1u);
                TR_ADD(tr1);
                if (!ok) { dead = true; break; }
            }
            uint8_t* hi = bx + b * 2 * S::BX_HALF;
            uint8_t* lo = hi + S::BX_HALF;
            auto emit = [&](uint32_t o, const float4 v) {                  // o: table entry of the vector
                uint32_t h0, l0, h1, l1;
                split2_packed(pack2(__float_as_uint(v.x), __float_as_uint(v.y)), h0, l0);
                split2_packed(pack2(__float_as_uint(v.z), __float_as_uint(v.w)), h1, l1);
                if constexpr (VEC == 4) {
                    *reinterpret_cast<uint2*>(hi + o) = make_uint2(h0, h1);
                    *reinterpret_cast<uint2*>(lo + o) = make_uint2(l0, l1);
                } else {
                    const uint32_t o0 = o & 0xFFFFu, o1 = o >> 16;
                    *reinterpret_cast<uint32_t*>(hi + o0) = h0;
                    *reinterpret_cast<uint32_t*>(lo + o0) = l0;
                    *reinterpret_cast<uint32_t*>(hi + o1) = h1;
                    *reinterpret_cast<uint32_t*>(lo + o1) = l1;
                }
            };
            // 16-bit input, 4 elements (8 bytes) per table entry: bf16 goes into Bx_hi as it is, fp16 is widened and split as fp32
            auto emit16 = [&](uint32_t o, const uint2 r) {
                if constexpr (IN == IN_BF16) {
                    if constexpr (VEC == 4) {
                        *reinterpret_cast<uint2*>(hi + o) = r;
                    } else {
                        *reinterpret_cast<uint32_t*>(hi + (o & 0xFFFFu)) = r.x;
                        *reinterpret_cast<uint32_t*>(hi + (o >> 16)) = r.y;
                    }
                } else {
                    const float2 p = f16x2_to_float2(r.x), q = f16x2_to_float2(r.y);
                    emit(o, make_float4(p.x, p.y, q.x, q.y));
                }
            };
            using Vec = std::conditional_t<IN == IN_F32, float4, uint2>;
            auto put = [&](uint32_t o, const Vec& v) {
                if constexpr (IN == IN_F32) emit(o, v);
                else emit16(o, v);
            };
            auto entry = [&](int f) {
                return VEC == 4 ? static_cast<uint32_t>(reinterpret_cast<const uint16_t*>(tab)[f]) : reinterpret_cast<const uint32_t*>(tab)[f];
            };
            if (!tail) {
                const Vec* src = reinterpret_cast<const Vec*>(stg + s * S::STG_STRIDE);
                // CB vectors (and their table entries) are loaded before the first store: the stores go to shared memory
                // too, so the compiler cannot hoist a later iteration's loads above them by itself
                // (full rounds run without predicates in one basic block, so that the compiler interleaves the three vectors)
                constexpr int CB = 3;
                int f0 = ctid;
                for (; f0 + (int)NCT * (CB - 1) < a.tile_vec - (a.tile_vec % (int)NCT) ; f0 += NCT * CB) {
                    Vec v[CB];
                    uint32_t o[CB];
#pragma unroll
                    for (int i = 0; i < CB; ++i) { v[i] = src[f0 + (int)NCT * i]; o[i] = entry(f0 + (int)NCT * i); }
#pragma unroll
                    for (int i = 0; i < CB; ++i) put(o[i], v[i]);
                }
                {
                    Vec v[CB];
                    uint32_t o[CB];
#pragma unroll
                    for (int i = 0; i < CB; ++i) {
                        const int f = f0 + (int)NCT * i;
                        if (f < a.tile_vec) { v[i] = src[f]; o[i] = entry(f); }
                    }
#pragma unroll
                    for (int i = 0; i < CB; ++i)
                        if (f0 + (int)NCT * i < a.tile_vec) put(o[i], v[i]);
                }
                TR_ADD(tr2);
                __syncwarp();
                if (lane == 0) mbar_arrive(stg_free + s);
                ++it;
            } else {                                                      // the stream's last, partial 32-element row is not in the tensor map
                const long long e0 = static_cast<long long>(tile - a.seg.tile0[sg]) * a.tile_elems, total = a.seg.total_elems[sg];
                if constexpr (IN == IN_F32) {
                    const float* xs = static_cast<const float*>(a.seg.x[sg]);
                    for (int f = ctid; f < a.tile_vec; f += NCT) {
                        const long long e = e0 + 4ll * f;
                        float4 v;
                        v.x = e + 0 < total ? xs[e + 0] : 0.f;
                        v.y = e + 1 < total ? xs[e + 1] : 0.f;
                        v.z = e + 2 < total ? xs[e + 2] : 0.f;
                        v.w = e + 3 < total ? xs[e + 3] : 0.f;
                        emit(entry(f), v);
                    }
                } else {
                    const uint16_t* xs = static_cast<const uint16_t*>(a.seg.x[sg]);
                    for (int f = ctid; f < a.tile_vec; f += NCT) {
                        const long long e = e0 + 4ll * f;
                        uint32_t p[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) p[k] = e + k < total ? xs[e + k] : 0u;        // (0x0000 is +0 in bf16 and fp16)
                        emit16(entry(f), make_uint2(p[0] | (p[1] << 16), p[2] | (p[3] << 16)));
                    }
                }
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bx_full + b);
            TR_ADD(tr3);
        }
        TR_FLUSH(16);
    } else if (warp < W_E2) {
        // ================================================================ epilogue 1: D1 -> y = za + zb -> bf16 hi/lo -> A2
        const uint32_t q = warp & 3u, s = ((warp - W_E1) >> 2) & 1u, eg = (warp - W_E1) >> 3;
        const uint32_t lane_q = (q * 32u) << 16, lane_s = (q * 32u + s * 16u) << 16;
        constexpr int np8 = NP8;
        tr_me = tr_on && warp == W_E1 && lane == 0;
        auto convert16 = [&](const uint32_t (&za)[8], const uint32_t (&zb)[8], uint32_t dst_hi, uint32_t dst_lo) {
            uint32_t h[4], l[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
                split2_packed(add2_packed(pack2(za[2 * i], za[2 * i + 1]), pack2(zb[2 * i], zb[2 * i + 1])), h[i], l[i]);
            tmem_st_frag8(dst_hi, h);
            tmem_st_frag8(dst_lo, l);
        };
        uint32_t n = eg;                                                   // this CTA's tile number
        for (int tile = first + (int)eg * stride; tile < a.num_tiles; tile += NE1G * stride, n += NE1G) {
            const uint32_t b = n & 1u;
            const uint32_t d1 = tmem + TM_D1 + b * d1_stride;
            TR_START();
            {
                bool ok = true;
                ok = mbar_wait(d1_full + b, (n >> 1) & 1u);
                TR_ADD(tr0);
                if (ok && n >= 2) ok = mbar_wait(a2_free + b, ((n >> 1) - 1u) & 1u);
                TR_ADD(tr1);
                if (!ok) { dead = true; break; }
            }
            tc_fence_after_sync();
            // The warp's share of D1 is T2 maps x (KP / 16) chunks of 16 columns (both lane halves: 8 + 8 registers a chunk).  Two chunks
            // are requested per TMEM round trip (a load takes hundreds of cycles while the tensor core and the other warps use the same
            // memory), whichever maps they belong to: two round trips a tile for every KP (one per map would be four at KP = 16).
            // (folded stage 2: the loop after this one)
            constexpr int CPT = KP / 16, NCH = FOLD ? 0 : T2 * CPT;        // chunks per map, chunks per tile
#pragma unroll
            for (int ch0 = 0; ch0 < NCH; ch0 += 2) {
                uint32_t za[16], zb[16];
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int ch = ch0 + k;
                    if (ch < NCH) {
                        const int t = ch / CPT, c8 = 2 * (ch % CPT);
                        const uint32_t src_a = d1 + lane_q + (2 * t + s) * a.Np + c8 * 8, src_b = src_a + (16u << 16);
                        if (c8 + 2 <= np8) {
                            tmem_ld_frag16(src_a, reinterpret_cast<uint32_t (&)[8]>(za[8 * k]));
                            tmem_ld_frag16(src_b, reinterpret_cast<uint32_t (&)[8]>(zb[8 * k]));
                        } else if (c8 < np8) {
                            tmem_ld_frag8(src_a, reinterpret_cast<uint32_t (&)[4]>(za[8 * k]));
                            tmem_ld_frag8(src_b, reinterpret_cast<uint32_t (&)[4]>(zb[8 * k]));
                        }
                    }
                }
                tmem_ld_wait();
                if (ch0 + 2 >= NCH) {                                     // every column of D1 this warp needs is in registers
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(d1_free + b);
                }
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int ch = ch0 + k;
                    if (ch < NCH) {
                        const int t = ch / CPT, c8 = 2 * (ch % CPT);
                        const uint32_t dst_hi = tmem + TM_A2 + b * 64 + t * KP + lane_s + c8 * 4, dst_lo = dst_hi + KP / 2;
                        if (c8 + 2 <= np8) {
                            convert16(reinterpret_cast<const uint32_t (&)[8]>(za[8 * k]), reinterpret_cast<const uint32_t (&)[8]>(zb[8 * k]), dst_hi, dst_lo);
                        } else if (c8 < np8) {
                            uint32_t h[2], l[2];
#pragma unroll
                            for (int i = 0; i < 2; ++i)
                                split2_packed(add2_packed(pack2(za[8 * k + 2 * i], za[8 * k + 2 * i + 1]), pack2(zb[8 * k + 2 * i], zb[8 * k + 2 * i + 1])),
                                              h[i], l[i]);
                            tmem_st_frag4(dst_hi, h[0], h[1]);
                            tmem_st_frag4(dst_lo, l[0], l[1]);
                        }
                    }
                }
            }
            // Folded stage 2 (stack_folded): a unit is either the 8 D1 columns of rows h with the 8 columns of their partners N-1-h
            // fold_d further on (a fold unit: y + y' to the even chain's A2 columns at the unit's position, y - y' to the odd chain's),
            // or the 8 columns of the unpaired middle rows (to both chains).  Two units per TMEM round trip (two fold units, a fold unit
            // and the middle rows, or the middle rows alone): two round trips a tile, as above.
            constexpr int D8 = NP8 / 2, MID = NP8 & 1, RT = (D8 + MID + 1) / 2, NRT = FOLD ? T2 * RT : 0;   // round trips per map, per tile
#pragma unroll
            for (int rt = 0; rt < NRT; ++rt) {
                const int t = rt / RT, k0 = 2 * (rt % RT);                // the warp's map t, units k0 and k0 + 1
                const int nf = k0 + 1 < D8 ? 2 : k0 < D8 ? 1 : 0;          // fold units of the round
                const bool mid = MID && k0 + 1 >= D8;                      // ... and the middle rows (unit D8)
                const uint32_t src = d1 + lane_q + (2 * t + s) * a.Np, hb = 16u << 16;    // (+ hb: the lanes of C_lo)
                uint32_t za[16], zb[16];                                   // [0, 8): rows (fold units; or a fold unit | the middle rows), [8, 16): partners
                if (nf == 2) {
                    tmem_ld_frag16(src + 8 * k0, reinterpret_cast<uint32_t (&)[8]>(za[0]));
                    tmem_ld_frag16(src + hb + 8 * k0, reinterpret_cast<uint32_t (&)[8]>(zb[0]));
                    tmem_ld_frag16(src + 8 * (k0 + D8), reinterpret_cast<uint32_t (&)[8]>(za[8]));
                    tmem_ld_frag16(src + hb + 8 * (k0 + D8), reinterpret_cast<uint32_t (&)[8]>(zb[8]));
                } else {
                    if (nf == 1) {
                        tmem_ld_frag8(src + 8 * k0, reinterpret_cast<uint32_t (&)[4]>(za[0]));
                        tmem_ld_frag8(src + hb + 8 * k0, reinterpret_cast<uint32_t (&)[4]>(zb[0]));
                        tmem_ld_frag8(src + 8 * (k0 + D8), reinterpret_cast<uint32_t (&)[4]>(za[8]));
                        tmem_ld_frag8(src + hb + 8 * (k0 + D8), reinterpret_cast<uint32_t (&)[4]>(zb[8]));
                    }
                    if (mid) {
                        tmem_ld_frag8(src + 16 * D8, reinterpret_cast<uint32_t (&)[4]>(za[4]));
                        tmem_ld_frag8(src + hb + 16 * D8, reinterpret_cast<uint32_t (&)[4]>(zb[4]));
                    }
                }
                tmem_ld_wait();
                if (rt + 1 == NRT) {                                       // every column of D1 this warp needs is in registers
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(d1_free + b);
                }
                uint32_t sh[4], sl[4], dh[4], dl[4];
#pragma unroll
                for (int i = 0; i < 2 * nf; ++i) {
                    const uint64_t y = add2_packed(pack2(za[2 * i], za[2 * i + 1]), pack2(zb[2 * i], zb[2 * i + 1]));
                    const uint64_t yp = add2_packed(pack2(za[8 + 2 * i], za[9 + 2 * i]), pack2(zb[8 + 2 * i], zb[9 + 2 * i]));
                    split2_packed(add2_packed(y, yp), sh[i], sl[i]);
                    split2_packed(sub2_packed(y, yp), dh[i], dl[i]);
                }
                const uint32_t even = tmem + TM_A2 + b * 64 + t * KF + lane_s, odd = even + W2 / 2;      // hi parts; lo: + KF / 2
                if (nf == 2) {
                    tmem_st_frag8(even + 4 * k0, sh);
                    tmem_st_frag8(even + KF / 2 + 4 * k0, sl);
                    tmem_st_frag8(odd + 4 * k0, dh);
                    tmem_st_frag8(odd + KF / 2 + 4 * k0, dl);
                } else if (nf == 1) {
                    tmem_st_frag4(even + 4 * k0, sh[0], sh[1]);
                    tmem_st_frag4(even + KF / 2 + 4 * k0, sl[0], sl[1]);
                    tmem_st_frag4(odd + 4 * k0, dh[0], dh[1]);
                    tmem_st_frag4(odd + KF / 2 + 4 * k0, dl[0], dl[1]);
                }
                if (mid) {
                    uint32_t h[2], l[2];
#pragma unroll
                    for (int i = 0; i < 2; ++i)
                        split2_packed(add2_packed(pack2(za[4 + 2 * i], za[5 + 2 * i]), pack2(zb[4 + 2 * i], zb[5 + 2 * i])), h[i], l[i]);
                    tmem_st_frag4(even + 4 * D8, h[0], h[1]);
                    tmem_st_frag4(even + KF / 2 + 4 * D8, l[0], l[1]);
                    tmem_st_frag4(odd + 4 * D8, h[0], h[1]);
                    tmem_st_frag4(odd + KF / 2 + 4 * D8, l[0], l[1]);
                }
            }
            tmem_st_wait();
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(a2_full + b);
            TR_ADD(tr2);
        }
        TR_FLUSH(24);
    } else if (warp < W_PROD) {
        // ================================================================ epilogue 2: D2 -> energies
        const uint32_t q = warp & 3u, eg2 = (warp - W_E2) >> 2, et = tid - (W_E2 + 4 * eg2) * 32;      // group, thread within it
        const uint32_t lane_q = (q * 32u) << 16;
        const uint32_t s = lane >> 4, r = lane & 15u;
        const uint32_t my_set = J == 4 ? q : J == 2 ? (q >> 1) : 0u;
        const uint32_t my_v = J == 4 ? r : J == 2 ? 16u * (q & 1u) + r : 16u * q + r;
        const uint32_t my_v0 = my_v - r;                                  // the warp's share of a map: basis rows [my_v0, my_v0 + 16)
        uint32_t n = eg2;
        int sg = 0, chan_sg = -1;
        uint32_t chan0 = 0, chan_step = 0;
        tr_me = tr_on && warp == W_E2 && lane == 0;
        for (int tile = first + (int)eg2 * stride; tile < a.num_tiles; tile += NE2G * stride, n += NE2G) {
            advance_segment(a.seg, tile, sg);
            const uint32_t C = static_cast<uint32_t>(a.seg.c_count[sg]), seg_maps = static_cast<uint32_t>(a.seg.n_maps[sg]);
            double* const accum = a.seg.accum[sg];
            const uint32_t pb = n & 1u, b2 = nb2 == 2 ? pb : 0u;           // barrier pair by tile parity, buffer
            TR_START();
            if (!mbar_wait(d2_full + pb, (n >> 1) & 1u)) { dead = true; break; }
            TR_ADD(tr0);
            tc_fence_after_sync();
            const uint32_t d2 = tmem + TM_D2 + b2 * 64 + lane_q;
            const uint32_t m0 = static_cast<uint32_t>(tile - a.seg.tile0[sg]) * a.MT;      // first map of the tile within its segment
            // channel of the tile's first map: m0 mod C, kept up incrementally (one division per segment, not per tile)
            if (sg != chan_sg) {
                chan_sg = sg;
                chan0 = m0 % C;                                            // (n_maps < 2^30: 32-bit arithmetic)
                chan_step = (static_cast<uint32_t>(NE2G * stride) * static_cast<uint32_t>(a.MT)) % C;
            } else {
                chan0 += chan_step;
                if (chan0 >= C) chan0 -= C;
            }
            float e[T2];
            // the lane's T2 * KF (64) coefficients in two round trips of 32 registers; D2 is handed back as soon as the second one has
            // landed
            constexpr int TOT = T2 * KF, HALF = TOT >= 32 ? 32 : TOT;
            float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int c0 = 0; c0 < TOT; c0 += HALF) {
                uint32_t z[HALF];
#pragma unroll
                for (int c = 0; c < HALF; c += 16)
                    if (c0 + c < TOT) tmem_ld16(d2 + c0 + c, reinterpret_cast<uint32_t (&)[16]>(z[c]));
                tmem_ld_wait();
                if (c0 + HALF >= TOT) {
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(d2_free + pb);
                    TR_ADD(tr2);
                }
#pragma unroll
                for (int c = 0; c < HALF; c += 16) {
                    if (c0 + c < TOT) {
                        const int t = (c0 + c) / KF;                        // A2 tile these 16 columns belong to (KF is a multiple of 16)
                        float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            p0 = fmaf(__uint_as_float(z[c + i]), __uint_as_float(z[c + i]), p0);
                            p1 = fmaf(__uint_as_float(z[c + 4 + i]), __uint_as_float(z[c + 4 + i]), p1);
                            p2 = fmaf(__uint_as_float(z[c + 8 + i]), __uint_as_float(z[c + 8 + i]), p2);
                            p3 = fmaf(__uint_as_float(z[c + 12 + i]), __uint_as_float(z[c + 12 + i]), p3);
                        }
                        const float p = (p0 + p1) + (p2 + p3);
                        if (T2 == 4) part[t] += p;
                        else if (T2 == 2) part[t] += p;
                        else part[0] += p;
                        if (TRACE && a.dump != nullptr) {
                            const uint32_t m = m0 + (2 * t + s) * J + my_set;
                            const int col = (c0 + c) - t * KF;                // of the map: u = col, folded 2 (col % W2) + chain col / W2
                            if (m < seg_maps && my_v < (uint32_t)a.N)
#pragma unroll
                                for (int i = 0; i < 16; ++i) {
                                    const int u = FOLD ? 2 * (col % W2 + i) + col / W2 : col + i;
                                    if (u < a.N) a.dump[static_cast<long long>(m) * a.NN + u * a.N + my_v] = __uint_as_float(z[c + i]);
                                }
                        }
                    }
                }
            }
#pragma unroll
            for (int t = 0; t < T2; ++t) {
                float v = part[t];
                v += __shfl_xor_sync(0xffffffffu, v, 8);
                v += __shfl_xor_sync(0xffffffffu, v, 4);
                v += __shfl_xor_sync(0xffffffffu, v, 2);
                v += __shfl_xor_sync(0xffffffffu, v, 1);
                e[t] = v;                                                  // lanes of one half: the warp's share of map (2t + s, my_set)
            }
            TR_ADD(tr3);
            if (!TRACE || a.energy_out == nullptr) {
                // production: each warp adds its fp64 share of a map straight into the channel sum (J = 1: four shares per map).
                // The warp's 2 * T2 shares are gathered into its first lanes so that they leave in ONE atomic instruction
                // (lane l: A2 tile t = l / 2, row slot s = l % 2; the share sits in lane 16 s).
                float mine = 0.f;
#pragma unroll
                for (int t = 0; t < T2; ++t) {
                    const float got = __shfl_sync(0xffffffffu, e[t], (lane & 1u) * 16u);
                    if ((lane >> 1) == (uint32_t)t) mine = got;
                }
                if (lane < 2u * T2) {
                    const uint32_t ml = lane * J + my_set;                 // map (g = 2t + s = lane, my_set) of the tile
                    if (m0 + ml < seg_maps) {
                        uint32_t ch = chan0 + ml;
                        while (ch >= C) ch -= C;
                        // With J > 1 a non-finite map in the tile (rare: see map_energy64) makes every share of the maps of its lanes
                        // non-finite: the share of rows from 0 then carries the map's whole fp64 energy (NaN for that map itself), the
                        // others 0.  (With J = 1 the maps of a tile never meet in one contraction.)
                        double share = mine;
                        if (J > 1 && !isfinite(mine))
                            share = my_v0 == 0 ? map_energy64_in<IN>(a.seg.x[sg], static_cast<long long>(m0 + ml), a.NN, a.N) : 0.0;
                        atomicAdd(accum + ch, share);
                    }
                }
            } else {
                // per-map energies asked for: the shares of a map are summed in a fixed order (bit-reproducible fp32 energy)
                float* red_w = red + eg2 * 32;                             // (each epilogue-2 group its own)
                if (r == 0)
#pragma unroll
                    for (int t = 0; t < T2; ++t) red_w[q * 8 + 2 * t + s] = e[t];
                named_bar_sync(1 + eg2, 128);
                if (et < (uint32_t)a.MT) {
                    const uint32_t g = et / J, set = et % J;
                    float en;
                    if (J == 4) en = red_w[set * 8 + g];
                    else if (J == 2) en = red_w[(2 * set) * 8 + g] + red_w[(2 * set + 1) * 8 + g];
                    else en = (red_w[g] + red_w[8 + g]) + (red_w[16 + g] + red_w[24 + g]);
                    const uint32_t m = m0 + et;
                    if (m < seg_maps) {
                        uint32_t ch = chan0 + et;
                        while (ch >= C) ch -= C;
                        double e = en;
                        if (!isfinite(en)) {                       // a non-finite map in the tile (rare: see map_energy64)
                            e = map_energy64_in<IN>(a.seg.x[sg], static_cast<long long>(m), a.NN, a.N);
                            en = static_cast<float>(e);
                        }
                        atomicAdd(accum + ch, e);
                        a.energy_out[m] = en;
                    }
                }
            }
            TR_ADD(tr1);
        }
        TR_FLUSH(32);
    }
#undef TR_START
#undef TR_ADD
#undef TR_FLUSH
    if (dead) {                                                           // a hand-over never came: flag it and poison the result
        atomicExch(a.status, DCTP_DEV_MMA_TIMEOUT);
        for (int sgi = 0; sgi < a.seg.n_seg; ++sgi)
            for (int c = lane; c < a.seg.c_count[sgi]; c += 32) a.seg.accum[sgi][c] = __longlong_as_double(0x7FF8000000000000ll);
    }
    tc_fence_before_sync();
    __syncthreads();
    if (TRACE && a.trace != nullptr && blockIdx.x == 0 && tid == 0) {    // tile loop of CTA 0 in SM cycles and in nanoseconds: the clock it ran at
        long long g1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
        a.trace[50] = clock64() - tr_c0;
        a.trace[51] = g1 - tr_g0;
    }
    if (warp == W_MMA) tmem_dealloc<512>(tmem);
}

}  // namespace dctp
