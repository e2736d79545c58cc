// libdctp.so - C ABI (include/dctp.h) over the sm_100a DCT importance-score kernels.
// Host side only: argument checks, cosine-basis cache, kernel selection and launch geometry.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "../../include/dctp.h"
#include "score_simt.cuh"
#include "score_large.cuh"
#include "score_tmem.cuh"
#include "score_stack.cuh"
#include "score_kron.cuh"
#include "score_umma.cuh"
#include "topk.cuh"
#include "gather.cuh"
#include "score_alt.cuh"
#include "widen.cuh"

namespace {

using namespace dctp;

thread_local char g_err[512] = "";
std::mutex g_mu;

void note_kernel(const char* fmt, ...);

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_TRY(expr)                                                                                  \
    do {                                                                                                \
        cudaError_t e_ = (expr);                                                                        \
        if (e_ != cudaSuccess) return fail(DCTP_E_CUDA, "%s: %s", #expr, cudaGetErrorString(e_));       \
    } while (0)

struct UmmaBasis {                                                       // per (N, KP)
    uint16_t *hi = nullptr, *lo = nullptr;                               // [KP x KP] block-diagonal I_J (x) C_N
    uint16_t* scatter = nullptr;                                         // [tile_vec][vpe] operand offsets of a dense tile (or null)
    int vpe = 0, tile_vec = 0;
};
struct TBasis {                                                          // per N: operands of the TMEM-operand kernel
    uint32_t *a_hi = nullptr, *a_lo = nullptr;                           // [128][64] packed bf16 pairs of I_G (x) C_N
    uint16_t *c_hi = nullptr, *c_lo = nullptr;                           // [64][64] C_N zero padded
    uint16_t* scatter = nullptr;                                         // [tile_vec][vpe]
    int tile_vec = 0, vpe = 1;
};
struct StackBasis {                                                      // per N: operands of the stacked-basis kernel
    uint32_t* a_img = nullptr;                                           // [128][32] packed bf16 pairs, the TMEM image of the stacked basis
    uint8_t *c2_hi = nullptr, *c2_lo = nullptr;                          // stage-2 basis operand images
    uint16_t* table = nullptr;                                           // Bx offsets of a tile's float4 pieces
    int kp = 0, vec = 0, tile_vec = 0;
    uint32_t table_bytes = 0, lbo1 = 0;
};
struct KronBasis { uint8_t *hi = nullptr, *lo = nullptr; };             // per N <= 8: C_N (x) C_N as a shared-memory operand image
struct LargeBasis { uint16_t *hi = nullptr, *lo = nullptr; int NP = 0, NPR = 0; };   // operand image of C_N: [NP/64][NPR][64], see get_large_basis
struct SimtBasis { float* t = nullptr; };                               // [N x N], t[n*N + k] = C_N[k][n]

struct State {
    bool ready = false;
    int device = -1, sm_count = 0;
    size_t smem_per_sm = 0;
    int* status = nullptr;
    long long launches = 0;
    char last_kernel[160] = "";                       // instantiation the most recent score launch ran (dctp_last_kernel)
    std::map<std::pair<int, int>, UmmaBasis> umma;     // (N, KP)
    std::map<int, SimtBasis> simt;                     // N
    std::map<int, TBasis> tmem;                        // N
    std::map<int, LargeBasis> large;                   // N
    std::map<int, StackBasis> stack;                   // N
    std::map<int, KronBasis> kron;                     // N
    std::vector<void*> bases;                          // every device allocation of the basis caches above (dctp_shutdown frees them)
    long long* trace = nullptr;                        // cycle stamps of a traced launch (DCTP_S/L/T_TRACE), TRACE_LEN entries
    void* encode_tiled = nullptr;                      // cuTensorMapEncodeTiled, resolved through the runtime (no libcuda link dependency)
    bool pdl = true;                                   // programmatic dependent launch of the score kernels (DCTP_PDL=0 disables)
    int regs[2][6][2] = {};                            // registers/thread per (KP, load mode, prefetch) instantiation
    // scratch of dctp_score_host (grow-only)
    float* hx = nullptr; size_t hx_bytes = 0;
    double* hacc = nullptr; float* hout = nullptr; size_t hc = 0;
} g;

void note_kernel(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g.last_kernel, sizeof g.last_kernel, fmt, ap);
    va_end(ap);
}

// the end of every launch: count it, report a launch error
int launched() {
    ++g.launches;
    CUDA_TRY(cudaGetLastError());
    return DCTP_OK;
}

constexpr int TRACE_LEN = 256;                        // entries of the trace buffer: the longest trace (DCTP_T_TRACE) has 32 tiles x 8 stamps
// trace = the zeroed trace buffer when the environment variable `var` asks for a traced launch, else null
int trace_for(const char* var, long long*& trace) {
    trace = nullptr;
    if (!std::getenv(var)) return DCTP_OK;
    if (!g.trace) CUDA_TRY(cudaMalloc(&g.trace, TRACE_LEN * sizeof(long long)));
    CUDA_TRY(cudaMemset(g.trace, 0, TRACE_LEN * sizeof(long long)));
    trace = g.trace;
    return DCTP_OK;
}
// the trace the preceding launch wrote
int read_trace(long long (&h)[TRACE_LEN]) {
    CUDA_TRY(cudaMemcpy(h, g.trace, sizeof h, cudaMemcpyDeviceToHost));
    return DCTP_OK;
}

// ------------------------------------------------------------------ cosine bases
inline double dct_coef(int k, int n, int N) {          // orthonormal DCT-II: C_N[k][n]
    // cos(pi (2n + 1) k / 2N) is exactly 0 where (2n + 1) k = N mod 2N (sides with an odd factor).  std::cos returns rounding noise
    // there (1e-17 .. 1e-15, and 1e-33 for products of two in C_N (x) C_N), whose split lo parts go down to 2^-117: multiplied by a
    // map of small values they underflow, and the coefficients they make stop scaling with the map.
    if (((2 * n + 1) * k) % (2 * N) == N) return 0.0;
    const double s = k == 0 ? std::sqrt(1.0 / N) : std::sqrt(2.0 / N);
    return s * std::cos(M_PI * (2.0 * n + 1.0) * k / (2.0 * N));
}
inline uint16_t bf16_rn(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return static_cast<uint16_t>(u >> 16);
}
inline float bf16_to_f(uint16_t b) {
    uint32_t u = static_cast<uint32_t>(b) << 16;
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}
inline void split_bf16(double c, uint16_t& hi, uint16_t& lo) {
    hi = bf16_rn(static_cast<float>(c));
    lo = bf16_rn(static_cast<float>(c - static_cast<double>(bf16_to_f(hi))));
}

// device copy of a host-built basis table; the allocation is recorded before anything can fail, so dctp_shutdown frees it
template <typename T>
int upload(const std::vector<T>& host, T*& dev) {
    void* p = nullptr;
    CUDA_TRY(cudaMalloc(&p, host.size() * sizeof(T)));
    g.bases.push_back(p);
    dev = static_cast<T*>(p);
    CUDA_TRY(cudaMemcpy(p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
    return DCTP_OK;
}

// out = cache[key], built by build(B&) and inserted on first use (a failed build inserts nothing)
template <class Map, class Key, class B, class Build>
int cached(Map& cache, const Key& key, B& out, Build build) {
    auto it = cache.find(key);
    if (it != cache.end()) { out = it->second; return DCTP_OK; }
    B b;
    if (int rc = build(b)) return rc;
    cache[key] = b;
    out = b;
    return DCTP_OK;
}

int get_umma_basis(int N, int KP, UmmaBasis& out) {
    return cached(g.umma, std::make_pair(N, KP), out, [&](UmmaBasis& b) {
        const int Ms = (N + 7) / 8 * 8, J = KP / Ms;
        std::vector<uint16_t> hi(static_cast<size_t>(KP) * KP, 0), lo(hi.size(), 0);
        for (int j = 0; j < J; ++j)
            for (int v = 0; v < N; ++v)
                for (int w = 0; w < N; ++w)
                    split_bf16(dct_coef(v, w, N), hi[(size_t)(j * Ms + v) * KP + j * Ms + w], lo[(size_t)(j * Ms + v) * KP + j * Ms + w]);
        int rc;
        if ((rc = upload(hi, b.hi)) || (rc = upload(lo, b.lo))) return rc;
        // scatter table of the dense load path: where element e of a full tile (maps back to back) lands in A1
        const int G = 128 / Ms, MT = G * J, NN = N * N;
        if ((MT * NN) % 4 == 0) {
            b.vpe = (N % 4 == 0) ? 1 : (N % 2 == 0) ? 2 : 4;
            b.tile_vec = MT * NN / 4;
            const int step = 4 / b.vpe;
            std::vector<uint16_t> tab(static_cast<size_t>(b.tile_vec) * b.vpe + 8, 0);
            for (int v = 0; v < b.tile_vec; ++v)
                for (int s = 0; s < b.vpe; ++s) {
                    const int e = 4 * v + s * step, t = e / NN, r = e % NN;
                    tab[(size_t)v * b.vpe + s] =
                        static_cast<uint16_t>(detail::kmajor_off((t / J) * Ms + r / N, (t % J) * Ms + r % N, 128));
                }
            if ((rc = upload(tab, b.scatter))) return rc;
        }
        return DCTP_OK;
    });
}

// D columns per tile slot of the TMEM-operand kernel; maps of side <= 16 sit two side by side (J = 2) in a 32-column slot
inline int t_n1max(int N) { return N <= 32 ? 32 : 64; }
inline int t_groups(int N) { return N <= 8 ? 4 : N <= 16 ? 2 : 1; }

int get_t_basis(int N, TBasis& out) {
    return cached(g.tmem, N, out, [&](TBasis& b) {
        const int Ms = (N + 7) / 8 * 8, G = 128 / Ms, NN = N * N, rows = t_n1max(N), J = t_groups(N);
        std::vector<uint32_t> ahi(128 * 64, 0), alo(128 * 64, 0);
        std::vector<uint16_t> chi(64 * 64, 0), clo(64 * 64, 0);
        for (int gI = 0; gI < G; ++gI)
            for (int v = 0; v < N; ++v)
                for (int w = 0; w < N; ++w) {
                    uint16_t h, l;
                    split_bf16(dct_coef(v, w, N), h, l);
                    const int row = gI * Ms + v, k = gI * N + w;          // element k of the row sits in half (k & 1) of packed column k / 2
                    ahi[row * 64 + k / 2] |= static_cast<uint32_t>(h) << (16 * (k & 1));
                    alo[row * 64 + k / 2] |= static_cast<uint32_t>(l) << (16 * (k & 1));
                }
        for (int rep = 0; rep < (Ms == 8 ? 2 : 1); ++rep)           // Ms = 8: two maps share a 16-column stage-2 group -> I_2 (x) C_N
            for (int u = 0; u < N; ++u)
                for (int h = 0; h < N; ++h) split_bf16(dct_coef(u, h, N), chi[(rep * 8 + u) * 64 + rep * 8 + h], clo[(rep * 8 + u) * 64 + rep * 8 + h]);
        b.vpe = (N % 4 == 0) ? 1 : (N % 2 == 0) ? 2 : 4;
        b.tile_vec = G * J * NN / 4;
        const int step = 4 / b.vpe;
        std::vector<uint16_t> tab(static_cast<size_t>(b.tile_vec) * b.vpe + 8, 0);
        for (int v = 0; v < b.tile_vec; ++v)
            for (int sI = 0; sI < b.vpe; ++sI) {               // map t = (g, j) of the tile: operand row (j, h), contraction column (g, w)
                const int e = 4 * v + sI * step, t = e / NN, r = e % NN, gI = t / J, j = t % J;
                tab[(size_t)v * b.vpe + sI] = static_cast<uint16_t>(detail::kmajor_off(j * Ms + r / N, gI * N + r % N, rows));
            }
        int rc;
        if ((rc = upload(ahi, b.a_hi)) || (rc = upload(alo, b.a_lo)) || (rc = upload(chi, b.c_hi)) || (rc = upload(clo, b.c_lo)) ||
            (rc = upload(tab, b.scatter)))
            return rc;
        return DCTP_OK;
    });
}

// ------------------------------------------------------------------ stacked-basis kernel (score_stack.cuh)
inline int stack_kp(int N) { return (N + 15) / 16 * 16; }
inline int stack_sets(int kp) { return kp <= 32 ? 64 / kp : 1; }
inline int stack_g(int kp) { return kp == 16 ? 8 : kp == 32 ? 4 : 2; }
// dense square maps, even side 10..64; above 32 a tile is two maps, and 2*N*N must be a whole number of 128-byte rows
bool stack_shape_supported(int N) { return N >= 10 && N <= 64 && (N % 2) == 0 && (N <= 32 || (N % 4) == 0); }

int get_stack_basis(int N, StackBasis& out) {
    return cached(g.stack, N, out, [&](StackBasis& b) {
        const int KP = stack_kp(N), J = stack_sets(KP), G = stack_g(KP), NN = N * N, Np = (N + 7) / 8 * 8, MT = G * J;
        std::vector<uint32_t> img(128 * 32, 0);
        for (int lane = 0; lane < 128; ++lane) {
            const int q = lane >> 5, part = (lane >> 4) & 1, r = lane & 15;
            const int set = J == 4 ? q : J == 2 ? q >> 1 : 0;
            const int v = J == 4 ? r : J == 2 ? 16 * (q & 1) + r : 16 * q + r;
            if (v >= N) continue;
            for (int w = 0; w < N; ++w) {
                uint16_t h, l;
                split_bf16(dct_coef(v, w, N), h, l);
                const int k = set * KP + w;
                img[lane * 32 + k / 2] |= static_cast<uint32_t>(part ? l : h) << (16 * (k & 1));
            }
        }
        // folded stage 2 (stack_folded): rows h < fd of a map are paired with rows N-1-h, the middle rows [fd, N - fd) (Np / 8 odd) are not
        const bool folded = stack_folded(KP);
        const int fd = 8 * (Np / 16), fold = std::min(N / 2, fd);
        // stage-2 basis: C_N[u][h] unfolded; folded, chain c (u = 2 u' + c) in rows [c W2, (c + 1) W2): C_N[2 u' + c][k] at contraction
        // column k < N - fold (the paired rows' h, then the middle rows' h)
        std::vector<uint8_t> chi(OperandImage64::BYTES, 0), clo(OperandImage64::BYTES, 0);
        for (int u = 0; u < N; ++u)
            for (int h = 0; h < (folded ? N - fold : N); ++h) {
                uint16_t hh, ll;
                split_bf16(dct_coef(u, h, N), hh, ll);
                const int row = folded ? (u & 1) * stack_fold_k(KP) + u / 2 : u;
                const size_t off = static_cast<size_t>(h / 8) * OperandImage64::LBO + row * 16 + (h % 8) * 2;
                std::memcpy(&chi[off], &hh, 2);
                std::memcpy(&clo[off], &ll, 2);
            }
        // Bx row (= D1 column) of row h of a map: h unfolded; folded, row N-1-h' (h' < fold) at fd + h', so that each thread of epilogue 1
        // holds both rows of a pair, and the middle rows from 2 fd on
        auto bx_row = [&](int h) { return !folded || h < fold ? h : h >= N - fold ? fd + (N - 1 - h) : 2 * fd + (h - fold); };
        b.kp = KP;
        b.vec = (N % 4) == 0 ? 4 : 2;
        b.tile_vec = MT * NN / 4;
        const int pieces = b.vec == 4 ? 1 : 2;
        std::vector<uint16_t> tab(static_cast<size_t>(b.tile_vec) * pieces + 8, 0);
        auto fill = [&](uint32_t lbo) {
            for (int f = 0; f < b.tile_vec; ++f)
                for (int pc = 0; pc < pieces; ++pc) {
                    const int e = 4 * f + 2 * pc, m = e / NN, rem = e % NN, h = rem / N, w = rem % N, gI = m / J, set = m % J;
                    const int n = gI * Np + bx_row(h), k = set * KP + w;
                    tab[static_cast<size_t>(f) * pieces + pc] = static_cast<uint16_t>((k / 8) * lbo + n * 16 + (k % 8) * 2);
                }
        };
        // shared-memory wavefronts of the converters' stores (thread t of a warp stores the pieces of vector f0 + t: 8-byte stores
        // are served per half-warp, 4-byte stores per warp) for a given chunk distance: pick the bank spread with the fewest
        auto store_wavefronts = [&]() {
            long long total = 0;
            const int width = b.vec == 4 ? 2 : 1, lanes = b.vec == 4 ? 16 : 32;      // banks per store, threads per phase
            for (int f0 = 0; f0 < b.tile_vec; f0 += lanes)
                for (int pc = 0; pc < pieces; ++pc) {
                    int cnt[32] = {0}, worst = 0;
                    for (int t = 0; t < lanes && f0 + t < b.tile_vec; ++t)
                        for (int w = 0; w < width; ++w) {
                            const int bank = (tab[static_cast<size_t>(f0 + t) * pieces + pc] / 4 + w) % 32;
                            if (++cnt[bank] > worst) worst = cnt[bank];
                        }
                    total += worst;
                }
            return total;
        };
        long long best = -1;
        for (uint32_t u = 0; u < 8; ++u) {
            fill(2048u + 16u * u);
            const long long wf = store_wavefronts();
            if (best < 0 || wf < best) { best = wf; b.lbo1 = 2048u + 16u * u; }
        }
        fill(b.lbo1);
        b.table_bytes = static_cast<uint32_t>((static_cast<size_t>(b.tile_vec) * pieces * 2 + 15) / 16 * 16);
        if (b.table_bytes > StackSmem::TABLE_MAX) return fail(DCTP_E_UNSUPPORTED, "stacked-basis kernel: offset table of side %d does not fit", N);
        int rc;
        if ((rc = upload(img, b.a_img)) || (rc = upload(chi, b.c2_hi)) || (rc = upload(clo, b.c2_lo)) || (rc = upload(tab, b.table))) return rc;
        return DCTP_OK;
    });
}

// instantiations: variant v = (KP, VEC, Np / 8) - (16,4,2) (16,2,2) (32,4,3) (32,4,4) (32,2,3) (32,2,4) (48,4,5) (48,4,6) (64,4,7) (64,4,8);
// role layout (one epilogue-1 group of 8 warps, two epilogue-2 groups of 4, producer, two issuers), named in dctp_last_kernel():
//   cfg7: production, 12 converter warps (two groups of 6), 31 warps
//   cfg6: debug, 8 converter warps (two groups of 4), 27 warps, with the debug outputs compiled in (DCTP_S_TRACE cycle accounting,
//         per-map energies, coefficient dump); the host routes launches that ask for any of them here, production launches never
// 12 converter warps won over 8 (the retired cfg 4): 56x56 4.14 against 4.06 TB/s, 14x14 3.55 against 3.45, 28x28 equal.
// Layouts measured and retired in round 2 (same box, 56x56 / 28x28 / 14x14 TB/s, before the instruction diet): one epilogue-2 group
// 3.73 / 3.47 / 3.19 (two: 3.73 / 3.62 / 3.25), two epilogue-1 groups 3.78 / 3.57 / 3.12, 4 converter warps 3.59 / 3.31 / 2.89;
// after it: 16 converter warps with one epilogue-2 group 4.08 / 3.55 / 3.38 and two epilogue-1 groups with one epilogue-2 group 4.05 / 3.66 /
// 3.40 (cfg 7: 4.14 / 3.99 / 3.55); register rebalancing (setmaxnreg: converters 56, epilogue 1 104 registers and ONE TMEM round trip per tile) 3.36 against
// 3.61 at 56x56; converters reading global memory directly behind an L2 bulk prefetch instead of the TMA-staged copy 3.46 against 4.07.
constexpr int STACK_VARIANTS = 10;
typedef void (*StackKernel)(const ScoreTensorMaps, const StackArgs);
template <bool TRACE, int NCONV, int IN>
StackKernel stack_kernel_of(int v) {
    switch (v) {
        case 0: return score_stack_kernel<16, 4, NCONV, 2, TRACE, IN>;
        case 1: return score_stack_kernel<16, 2, NCONV, 2, TRACE, IN>;
        case 2: return score_stack_kernel<32, 4, NCONV, 3, TRACE, IN>;
        case 3: return score_stack_kernel<32, 4, NCONV, 4, TRACE, IN>;
        case 4: return score_stack_kernel<32, 2, NCONV, 3, TRACE, IN>;
        case 5: return score_stack_kernel<32, 2, NCONV, 4, TRACE, IN>;
        case 6: return score_stack_kernel<48, 4, NCONV, 5, TRACE, IN>;
        case 7: return score_stack_kernel<48, 4, NCONV, 6, TRACE, IN>;
        case 8: return score_stack_kernel<64, 4, NCONV, 7, TRACE, IN>;
        default: return score_stack_kernel<64, 4, NCONV, 8, TRACE, IN>;
    }
}
constexpr int STACK_NCONV = 12, STACK_NCONV_DEBUG = 8;
template <int IN>
StackKernel stack_kernel_in(bool debug, int v) {
    return debug ? stack_kernel_of<true, STACK_NCONV_DEBUG, IN>(v) : stack_kernel_of<false, STACK_NCONV, IN>(v);
}
StackKernel stack_kernel_fn(bool debug, int v, int in) {
    return in == IN_BF16 ? stack_kernel_in<IN_BF16>(debug, v) : in == IN_F16 ? stack_kernel_in<IN_F16>(debug, v) : stack_kernel_in<IN_F32>(debug, v);
}
const char* in_name(int in) { return in == IN_BF16 ? "bf16" : in == IN_F16 ? "f16" : "f32"; }
// what a 16-bit instantiation adds to its template arguments in dctp_last_kernel()
const char* in_suffix(int in) { return in == IN_BF16 ? ",IN=bf16" : in == IN_F16 ? ",IN=f16" : ""; }
int stack_variant(int KP, int vec, int np8) {
    if (KP == 16) return vec == 4 ? 0 : 1;
    if (KP == 32) return (vec == 4 ? 2 : 4) + (np8 == 4 ? 1 : 0);
    if (KP == 48) return np8 == 6 ? 7 : 6;
    return np8 == 8 ? 9 : 8;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D tensor map: `rows` rows of `inner` elements (fp32 unless `in` says otherwise), `pitch` bytes apart; box = `box_inner`
// elements x `box_rows` rows
int encode_2d(CUtensorMap& map, const void* base, long long inner, long long rows, long long pitch, int box_inner, int box_rows,
              CUtensorMapL2promotion l2, int in = IN_F32) {
    std::memset(&map, 0, sizeof map);
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(inner), static_cast<cuuint64_t>(rows)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(pitch)};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(box_inner), static_cast<cuuint32_t>(box_rows)}, estr[2] = {1, 1};
    const CUresult r = reinterpret_cast<EncodeTiledFn>(g.encode_tiled)(
        &map, in == IN_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : in == IN_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
        const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_NONE, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(DCTP_E_CUDA, "cuTensorMapEncodeTiled failed (%d) for %lld rows of %lld %s elements, box %d x %d", (int)r, rows, inner,
                    in_name(in), box_inner, box_rows);
    return DCTP_OK;
}

// a dense stream viewed as [rows, 32 elements] (whole rows only: 128 bytes of fp32, 64 of 16-bit input), box = `box_rows` rows
int encode_flat_map(CUtensorMap& map, const void* first, long long total_elems, int box_rows, int in = IN_F32) {
    const long long rows = total_elems / 32;
    if (rows <= 0) {                                         // (never dereferenced: the only tile is converted from global memory)
        std::memset(&map, 0, sizeof map);
        return DCTP_OK;
    }
    return encode_2d(map, first, 32, rows, 32 * in_bytes(in), 32, box_rows, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, in);
}

// Score kernels are launched with programmatic stream serialization: their prologue (shared-memory fill, basis staging,
// TMEM allocation) may run while the preceding kernel drains; each kernel waits for that kernel's completion
// (griddepcontrol.wait) before it touches the activation.  DCTP_PDL=0 turns it off.
template <typename... Params, typename... Args>
cudaError_t launch_pdl(void (*kern)(Params...), int grid, int block, size_t smem, cudaStream_t stream, const Args&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(static_cast<unsigned>(block));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g.pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

struct SiteDesc { const void* first; int B; int c_count; double* accum; };      // one dense activation: B * c_count maps back to back

// fills seg (tile ranges, per-site sizes); returns the launch's tile count.  A map is items_per_map work items (score_large.cuh:
// its v-chunks), and a tile holds up to `per_tile` of them.
int fill_segments(ScoreSegments& seg, const SiteDesc* sites, int n, int NN, int items_per_map, int per_tile) {
    seg.n_seg = n;
    int tiles = 0;
    for (int i = 0; i < n; ++i) {
        seg.tile0[i] = tiles;
        seg.n_maps[i] = sites[i].B * sites[i].c_count;
        seg.c_count[i] = sites[i].c_count;
        seg.total_elems[i] = static_cast<long long>(seg.n_maps[i]) * NN;
        seg.x[i] = sites[i].first;
        seg.accum[i] = sites[i].accum;
        tiles += (seg.n_maps[i] * items_per_map + per_tile - 1) / per_tile;
    }
    for (int i = n; i <= SCORE_MAX_SEG; ++i) seg.tile0[i] = tiles;
    return tiles;
}

// the tensor maps of a multi-site launch: encode(i, map) for each of the n sites, the unused entries copies of the first
template <class Encode>
int fill_maps(ScoreTensorMaps& maps, int n, Encode encode) {
    for (int i = 0; i < n; ++i)
        if (int rc = encode(i, maps.m[i])) return rc;
    for (int i = n; i < SCORE_MAX_SEG; ++i) maps.m[i] = maps.m[0];
    return DCTP_OK;
}

// up to SCORE_MAX_SEG dense activations of side N in ONE launch (energy_out / coeff_out: single-site launches only)
int launch_stack(const SiteDesc* sites, int n, int N, float* energy_out, float* coeff_out, int in, cudaStream_t stream) {
    StackBasis basis;
    int rc = get_stack_basis(N, basis);
    if (rc) return rc;
    StackArgs a;
    std::memset(&a, 0, sizeof a);
    const int KP = basis.kp, J = stack_sets(KP);
    a.N = N; a.NN = N * N; a.Np = (N + 7) / 8 * 8; a.G = stack_g(KP); a.MT = a.G * J;
    a.ncols = a.G * a.Np;
    a.tile_elems = a.MT * a.NN; a.tile_rows = a.tile_elems / 32; a.tile_vec = basis.tile_vec;
    a.num_tiles = fill_segments(a.seg, sites, n, a.NN, 1, a.MT);
    a.idesc1 = umma::make_idesc_bf16(128, a.ncols, false, false);
    a.idesc2 = umma::make_idesc_bf16(128, stack_folded(KP) ? stack_fold_k(KP) : KP, false, false);
    a.lbo1 = basis.lbo1;
    a.a_img = basis.a_img; a.c2_hi = basis.c2_hi; a.c2_lo = basis.c2_lo; a.table = basis.table; a.table_bytes = basis.table_bytes;
    a.energy_out = n == 1 ? energy_out : nullptr; a.dump = n == 1 ? coeff_out : nullptr; a.status = g.status;
    ScoreTensorMaps maps;
    if ((rc = fill_maps(maps, n, [&](int i, CUtensorMap& m) { return encode_flat_map(m, sites[i].first, a.seg.total_elems[i], a.tile_rows, in); })))
        return rc;
    int grid = g.sm_count < a.num_tiles ? g.sm_count : a.num_tiles;
    const size_t smem = StackSmem::TOTAL;
    if ((rc = trace_for("DCTP_S_TRACE", a.trace))) return rc;
    const int variant = stack_variant(KP, basis.vec, a.Np / 8);
    // per-map energies, coefficients and the cycle trace live in the debug instantiation (cfg6) only
    const bool debug = a.energy_out || a.dump || a.trace;
    CUDA_TRY(launch_pdl(stack_kernel_fn(debug, variant, in), grid, 32 * stack_warps(debug ? STACK_NCONV_DEBUG : STACK_NCONV), smem, stream,
                        maps, a));
    note_kernel("score_stack_kernel<KP=%d,VEC=%d,cfg%d%s> (tcgen05, stacked hi/lo basis in TMEM, TMA tile ring, warp specialised)", KP, basis.vec,
                debug ? 6 : 7, in_suffix(in));
    if (a.trace) {
        long long h[TRACE_LEN];
        if ((rc = read_trace(h))) return rc;
        const double nt = h[14] > 0 ? double(h[14]) : 1.0;
        fprintf(stderr, "[dctp trace] stack N=%d, CTA 0, %lld tiles, cycles per tile | producer: wait slot %.0f | converter: wait Bx free %.0f, "
                        "wait TMA %.0f, convert %.0f, fence+arrive %.0f | issuer 1: wait Bx %.0f, wait D1 free %.0f, issue %.0f | issuer 2: wait A2 %.0f, "
                        "wait D2 free %.0f, issue %.0f | epi1 (first group, per tile of the CTA): wait D1 %.0f, wait A2 free %.0f, work %.0f | "
                        "epi2: wait D2 %.0f, TMEM loads %.0f, sums+shuffles %.0f, atomics %.0f\n",
                N, h[14], h[0] / nt, h[16] / nt, h[17] / nt, h[18] / nt, h[19] / nt, h[8] / nt, h[9] / nt, h[10] / nt, h[40] / nt,
                h[41] / nt, h[42] / nt, h[24] / nt, h[25] / nt, h[26] / nt, h[32] / nt, h[34] / nt, h[35] / nt, h[33] / nt);
        fprintf(stderr, "[dctp trace] CTA 0, ns since kernel entry: TMEM + barriers ready %lld, bases staged and dependency wait over %lld, tile loop %lld\n", h[52], h[53], h[51]);
        fprintf(stderr, "[dctp trace] tile loop of CTA 0: %lld SM cycles in %lld ns = %.0f MHz, %.0f cycles per tile\n", h[50], h[51],
                h[51] > 0 ? 1e3 * double(h[50]) / double(h[51]) : 0.0, double(h[50]) / nt);
    }
    return launched();
}

// ------------------------------------------------------------------ Kronecker kernel (score_kron.cuh), sides 1..8
int get_kron_basis(int N, KronBasis& out) {
    return cached(g.kron, N, out, [&](KronBasis& b) {
        std::vector<uint8_t> hi(OperandImage64::BYTES, 0), lo(OperandImage64::BYTES, 0);
        for (int u = 0; u < N; ++u)
            for (int v = 0; v < N; ++v)
                for (int h = 0; h < N; ++h)
                    for (int w = 0; w < N; ++w) {
                        uint16_t hh, ll;
                        split_bf16(dct_coef(u, h, N) * dct_coef(v, w, N), hh, ll);
                        const int n = u * N + v, k = h * N + w;
                        const size_t off = static_cast<size_t>(k / 8) * OperandImage64::LBO + n * 16 + (k % 8) * 2;
                        std::memcpy(&hi[off], &hh, 2);
                        std::memcpy(&lo[off], &ll, 2);
                    }
        int rc;
        if ((rc = upload(hi, b.hi)) || (rc = upload(lo, b.lo))) return rc;
        return DCTP_OK;
    });
}

typedef void (*KronKernel)(const ScoreTensorMaps, const KronArgs);
// the instantiations a (K2, layout, input type) runs on; 16-bit maps take the row layout at sides 4 and 8 only (K2 16 and 64), so
// 16-bit row-layout kernels of K2 32 and 48 are not built (kron_kernel_built)
bool kron_kernel_built(int K2, bool even, int in) { return !even || in == IN_F32 || K2 == 16 || K2 == 64; }
template <int IN>
KronKernel kron_kernel_in(int K2, bool even) {
    switch (K2) {
        case 16: return even ? score_kron_kernel<16, true, IN> : score_kron_kernel<16, false, IN>;
        case 32:
            if constexpr (IN == IN_F32)
                if (even) return score_kron_kernel<32, true, IN>;
            return score_kron_kernel<32, false, IN>;
        case 48:
            if constexpr (IN == IN_F32)
                if (even) return score_kron_kernel<48, true, IN>;
            return score_kron_kernel<48, false, IN>;
        default: return even ? score_kron_kernel<64, true, IN> : score_kron_kernel<64, false, IN>;
    }
}
KronKernel kron_kernel_fn(int K2, bool even, int in) {
    return in == IN_BF16 ? kron_kernel_in<IN_BF16>(K2, even) : in == IN_F16 ? kron_kernel_in<IN_F16>(K2, even) : kron_kernel_in<IN_F32>(K2, even);
}

int launch_kron(const SiteDesc* sites, int n, int N, float* energy_out, float* coeff_out, int in, cudaStream_t stream) {
    KronBasis basis;
    int rc = get_kron_basis(N, basis);
    if (rc) return rc;
    KronArgs a;
    std::memset(&a, 0, sizeof a);
    const int NN = N * N, K2 = (NN + 15) / 16 * 16, eb = in_bytes(in);
    // the row layout needs a row pitch of whole 16-byte units: every even side in fp32, sides 4 and 8 in 16-bit
    const bool even = (N % 2) == 0 && (NN * eb) % 16 == 0;
    a.N = N; a.NN = NN;
    a.idesc = umma::make_idesc_bf16(128, K2, false, false);
    a.k_hi = basis.hi; a.k_lo = basis.lo;
    a.energy_out = n == 1 ? energy_out : nullptr; a.dump = n == 1 ? coeff_out : nullptr; a.status = g.status;
    if (even) {
        a.sub_tiles = N == 8 ? 1 : 2;
        const int unit = 16 / eb;                                       // elements per 16-byte unit
        a.row_elems = NN + (((NN / unit) % 2) == 0 ? unit : 0);         // an odd number of 16-byte units per row: conflict-free 128-bit reads
        a.tile_maps = 128 * a.sub_tiles;
        a.box_rows = a.tile_maps;
        a.tile_bytes = static_cast<uint32_t>(a.tile_maps) * a.row_elems * eb;
    } else {
        // (16-bit 6x6 and 2x2 maps take this layout too; one sub-tile of 6x6 is already 144 rows, and a box holds at most 256)
        a.sub_tiles = N == 7 || N == 6 ? 1 : N == 5 || N == 2 ? 2 : 4;
        a.row_elems = NN;
        a.tile_maps = 128 * a.sub_tiles;
        a.box_rows = a.tile_maps * NN / 32;
        a.tile_bytes = static_cast<uint32_t>(a.box_rows) * 32u * eb;
    }
    a.num_tiles = fill_segments(a.seg, sites, n, NN, 1, a.tile_maps);
    ScoreTensorMaps maps;
    // even sides: one map per row of the box, padded to row_elems; odd sides: the flat stream
    rc = fill_maps(maps, n, [&](int i, CUtensorMap& m) {
        return even ? encode_2d(m, sites[i].first, NN, a.seg.n_maps[i], static_cast<long long>(eb) * NN, a.row_elems, a.tile_maps,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, in)
                    : encode_flat_map(m, sites[i].first, a.seg.total_elems[i], a.box_rows, in);
    });
    if (rc) return rc;
    const int grid = g.sm_count < a.num_tiles ? g.sm_count : a.num_tiles;
    const size_t smem = KronSmem::TOTAL;
    CUDA_TRY(launch_pdl(kron_kernel_fn(K2, even, in), grid, KRON_NT, smem, stream, maps, a));
    note_kernel("score_kron_kernel<K2=%d,%s%s> (tcgen05, single-stage Kronecker, TMA tile ring, warp specialised)", K2, even ? "even" : "odd",
                in_suffix(in));
    return launched();
}

// stage-2 output chunks of the large-map kernel: NUC chunks of NU columns (multiple of 16, at most 128: one basis slab)
void large_u_chunks(int N, int& nu, int& nuc) {
    nuc = (N + 127) / 128;
    nu = ((N + nuc - 1) / nuc + 15) / 16 * 16;
}

int get_large_basis(int N, LargeBasis& out) {
    return cached(g.large, N, out, [&](LargeBasis& b) {
        b.NP = (N + 63) / 64 * 64;
        // operand image: [column block cb][row k][64 columns], the eight 16-byte chunks of a row XOR-swizzled by (k & 7);
        // rows padded so that every u-chunk slab of the kernel stays inside its column block
        int nu, nuc;
        large_u_chunks(N, nu, nuc);
        b.NPR = b.NP > nu * nuc ? b.NP : nu * nuc;
        std::vector<uint16_t> hi(static_cast<size_t>(b.NP / 64) * b.NPR * 64, 0), lo(hi.size(), 0);
        for (int k = 0; k < N; ++k)
            for (int n = 0; n < N; ++n) {
                const size_t at = (static_cast<size_t>(n >> 6) * b.NPR + k) * 64 + ((((n & 63) >> 3) ^ (k & 7)) << 3) + (n & 7);
                split_bf16(dct_coef(k, n, N), hi[at], lo[at]);
            }
        int rc;
        if ((rc = upload(hi, b.hi)) || (rc = upload(lo, b.lo))) return rc;
        return DCTP_OK;
    });
}

int get_simt_basis(int N, SimtBasis& out) {
    return cached(g.simt, N, out, [&](SimtBasis& b) {
        std::vector<float> t(static_cast<size_t>(N) * N);
        for (int n = 0; n < N; ++n)
            for (int k = 0; k < N; ++k) t[(size_t)n * N + k] = static_cast<float>(dct_coef(k, n, N));
        return upload(t, b.t);
    });
}

// ------------------------------------------------------------------ init
// fn may use `bytes` of dynamic shared memory, and prefers the largest shared-memory carveout
template <class F>
int allow_smem(F* fn, int bytes) {
    CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    return DCTP_OK;
}

template <int KP, int MODE, bool PF>
int setup_umma(int& regs) {
    auto* fn = score_umma_kernel<KP, MODE, PF>;
    if (int rc = allow_smem(fn, KP == 64 ? 100 * 1024 : 200 * 1024)) return rc;
    cudaFuncAttributes fa;
    CUDA_TRY(cudaFuncGetAttributes(&fa, fn));
    regs = fa.numRegs;
    return DCTP_OK;
}

// Resident CTAs per SM from the kernel's own resources.  (cudaOccupancyMaxActiveBlocksPerMultiprocessor
// answered 1 for this kernel on B200 / CUDA 12.9 although shared memory allows 4 and registers 5 - ncu's
// launch__occupancy_limit_* agree with the arithmetic below - so the grid is sized from first principles.)
int umma_occupancy(int kp, int mode, bool pf, size_t smem_bytes) {
    const int regs = g.regs[kp == 64 ? 0 : 1][mode][pf ? 1 : 0];
    const int by_smem = static_cast<int>(g.smem_per_sm / (smem_bytes + 1024));       // + driver-reserved KB per CTA
    const int regs_per_cta = ((regs + 7) / 8 * 8) * 128;
    const int by_regs = regs_per_cta > 0 ? 65536 / regs_per_cta : 1;
    const int by_tmem = 512 / (2 * kp);                                              // TMEM columns are a per-SM resource too
    int occ = by_smem < by_regs ? by_smem : by_regs;
    if (occ > by_tmem) occ = by_tmem;
    if (occ > 16) occ = 16;
    return occ < 1 ? 1 : occ;
}

template <int KP>
int setup_umma_all(int (*regs)[2]) {
    int rc;
    if ((rc = setup_umma<KP, LOAD_DENSE1, false>(regs[LOAD_DENSE1][0]))) return rc;
    if ((rc = setup_umma<KP, LOAD_DENSE2, false>(regs[LOAD_DENSE2][0]))) return rc;
    if ((rc = setup_umma<KP, LOAD_DENSE1, true>(regs[LOAD_DENSE1][1]))) return rc;
    if ((rc = setup_umma<KP, LOAD_DENSE2, true>(regs[LOAD_DENSE2][1]))) return rc;
    if constexpr (KP == 64) {                        // (KP = 128: see umma_dense_mode)
        if ((rc = setup_umma<KP, LOAD_DENSE4, false>(regs[LOAD_DENSE4][0]))) return rc;
        if ((rc = setup_umma<KP, LOAD_DENSE4, true>(regs[LOAD_DENSE4][1]))) return rc;
    }
    if ((rc = setup_umma<KP, LOAD_GEN4, false>(regs[LOAD_GEN4][0]))) return rc;
    if ((rc = setup_umma<KP, LOAD_GEN2, false>(regs[LOAD_GEN2][0]))) return rc;
    return setup_umma<KP, LOAD_GEN1, false>(regs[LOAD_GEN1][0]);
}

int ensure_init() {
    if (g.ready) {                                       // bases, status word and kernel attributes belong to the device of the first call
        int cur = -1;
        CUDA_TRY(cudaGetDevice(&cur));
        if (cur != g.device)
            return fail(DCTP_E_INVALID, "libdctp was initialised on device %d; the current device is %d (one device per process: launch one "
                                        "process per GPU, or dctp_shutdown() before switching)", g.device, cur);
        return DCTP_OK;
    }
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10)
        return fail(DCTP_E_UNSUPPORTED, "libdctp is built for sm_100a only; device %d is sm_%d%d", dev, prop.major, prop.minor);
    g.device = dev;
    g.sm_count = prop.multiProcessorCount;
    g.smem_per_sm = prop.sharedMemPerMultiprocessor;
    int rc;
    if ((rc = setup_umma_all<64>(g.regs[0]))) return rc;
    if ((rc = setup_umma_all<128>(g.regs[1]))) return rc;
    {
        const void* fns[] = {reinterpret_cast<const void*>(score_t_kernel<64, 3, 1>), reinterpret_cast<const void*>(score_t_kernel<64, 3, 2>),
                             reinterpret_cast<const void*>(score_t_kernel<32, 6, 1>), reinterpret_cast<const void*>(score_t_kernel<32, 6, 2>),
                             reinterpret_cast<const void*>(score_t_kernel<32, 6, 4>), reinterpret_cast<const void*>(score_t_kernel<64, 3, 1, 2>)};
        for (const void* fn : fns)
            if ((rc = allow_smem(fn, 227 * 1024))) return rc;
    }
    {
        for (const int in : {IN_F32, IN_BF16, IN_F16}) {
            for (const bool debug : {false, true})
                for (int v = 0; v < STACK_VARIANTS; ++v)
                    if ((rc = allow_smem(stack_kernel_fn(debug, v, in), static_cast<int>(StackSmem::TOTAL)))) return rc;
            for (const int k2 : {16, 32, 48, 64})
                for (const bool even : {true, false})
                    if (kron_kernel_built(k2, even, in) && (rc = allow_smem(kron_kernel_fn(k2, even, in), static_cast<int>(KronSmem::TOTAL))))
                        return rc;
        }
        cudaDriverEntryPointQueryResult qres;
        CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &g.encode_tiled, cudaEnableDefault, &qres));
        if (!g.encode_tiled) return fail(DCTP_E_CUDA, "the driver does not export cuTensorMapEncodeTiled");
    }
    if (const char* e = std::getenv("DCTP_PDL")) g.pdl = std::atoi(e) != 0;
    CUDA_TRY(cudaFuncSetAttribute(score_large_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LargeSmem::TOTAL));
    CUDA_TRY(cudaFuncSetAttribute(score_large_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LargeSmem::TOTAL));
    CUDA_TRY(cudaFuncSetAttribute(score_simt_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SIMT_SMALL_SMEM));
    CUDA_TRY(cudaFuncSetAttribute(score_simt_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CUDA_TRY(cudaFuncSetAttribute(rank_jacobi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RANK_SMEM_MAX));
    CUDA_TRY(cudaMalloc(&g.status, sizeof(int)));
    CUDA_TRY(cudaMemset(g.status, 0, sizeof(int)));
    g.ready = true;
    return DCTP_OK;
}

inline int pow2_floor(int v) {
    int p = 1;
    while (p * 2 <= v) p *= 2;
    return p;
}

bool umma_shape_ok(int H, int W, long long stride_h) { return H == W && H >= 1 && H <= 128 && stride_h == W; }

int pick_vec(const float* x, long long stride_b, long long stride_c, int N) {
    auto aligned = [&](int v) {
        return (N % v) == 0 && (reinterpret_cast<uintptr_t>(x) % (4 * v)) == 0 && (stride_b % v) == 0 && (stride_c % v) == 0;
    };
    if (aligned(4)) return 4;
    if (aligned(2)) return 2;
    return 1;
}

// the tiled large-map kernel takes square maps of side 80..320 (multiples of 16), and AUTO gives it all of them: measured against
// the smem-operand kernel, [12,64,N,N]: 80 0.92 vs 0.67 TB/s (a tie in round 1, before the large kernel lost a fifth of its
// instructions), 96 1.22 vs 0.73
bool large_shape_supported(int H, int W, long long stride_h) { return H == W && H >= 80 && H <= 320 && (H % 16) == 0 && stride_h == W; }

// up to SCORE_MAX_SEG dense activations of side N in ONE launch (energy_out / coeff_out: single-site launches only)
int launch_large(const SiteDesc* sites, int n, int N, float* energy_out, float* coeff_out, cudaStream_t stream) {
    LargeBasis basis;
    int rc = get_large_basis(N, basis);
    if (rc) return rc;
    LargeScoreArgs a;
    std::memset(&a, 0, sizeof a);
    a.N = N; a.NPR = basis.NPR; a.NVC = (N + 127) / 128;
    large_u_chunks(N, a.NU, a.NUC);
    long long items = 0;
    for (int i = 0; i < n; ++i) {
        const long long maps = static_cast<long long>(sites[i].B) * sites[i].c_count;
        if (maps * N >= (1ll << 31) || items + maps * a.NVC >= (1ll << 31))
            return fail(DCTP_E_INVALID, "too many maps of side %d in one launch (tensor-map row coordinates and work-item numbers are 32-bit)", N);
        a.n_maps += static_cast<int>(maps);
        items += maps * a.NVC;
    }
    a.n_items = fill_segments(a.seg, sites, n, N * N, a.NVC, 1);
    a.c_hi = reinterpret_cast<const uint8_t*>(basis.hi); a.c_lo = reinterpret_cast<const uint8_t*>(basis.lo);
    a.energy_out = n == 1 ? energy_out : nullptr; a.dump = n == 1 ? coeff_out : nullptr; a.status = g.status;
    energy_out = a.energy_out;
    if (energy_out) CUDA_TRY(cudaMallocAsync(&a.energy_parts, sizeof(float) * a.n_maps * a.NVC, stream));   // (debug / parity output only)
    int grid = g.sm_count < a.n_items ? g.sm_count : a.n_items;
    if ((rc = trace_for("DCTP_L_TRACE", a.trace))) return rc;
    // every activation as a 2-D tensor [n_maps * N rows, N floats]; a map slab is the box {64 floats, 128 rows}, out-of-range parts zero
    ScoreTensorMaps xmap;
    if ((rc = fill_maps(xmap, n, [&](int i, CUtensorMap& m) {
             return encode_2d(m, sites[i].first, N, static_cast<long long>(a.seg.n_maps[i]) * N, 4ll * N, 64, 128, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
         })))
        return rc;
    CUDA_TRY(launch_pdl((a.trace || a.dump) ? score_large_kernel<true> : score_large_kernel<false>, grid, LARGE_NT, LargeSmem::TOTAL, stream,
                        xmap, a));
    if (energy_out) {
        sum_parts_kernel<<<(a.n_maps + 255) / 256, 256, 0, stream>>>(a.energy_parts, a.NVC, energy_out, a.n_maps);
        CUDA_TRY(cudaFreeAsync(a.energy_parts, stream));
    }
    note_kernel("score_large_kernel (tcgen05, tiled two-stage, TMA-staged map slabs, 19 warps)");
    if (a.trace) {
        long long h[TRACE_LEN];
        if ((rc = read_trace(h))) return rc;
        const double n = h[7] > 0 ? double(h[7]) : 1.0;
        fprintf(stderr, "[dctp trace] large N=%d steps=%lld, issuer thread cycles/step: total %.0f | waiting for: map slab %.0f, "
                        "basis slab %.0f (+%.0f look-ahead), A2 %.0f, D2 free %.0f\n",
                N, h[7], h[6] / n, h[1] / n, h[4] / n, h[5] / n, h[2] / n, h[3] / n);
        const double m = h[12] > 0 ? double(h[12]) : 1.0;
        fprintf(stderr, "[dctp trace] converter thread 0, cycles per map slab (%lld slabs): operand buffer wait %.0f, staged slab wait %.0f, "
                        "convert + store + hand-over %.0f\n", h[12], h[8] / m, h[11] / m, h[9] / m);
    }
    return launched();
}

// which maps the TMEM-operand kernel takes at all (dense; side 5..64, odd sides up to 13 and only when the whole stream is a
// multiple of four floats), and which ones AUTO gives it
bool t_shape_supported(int N) { return N >= 5 && N <= 64 && ((N % 2) == 0 || N <= 13); }   // (odd sides: 8-byte scatter entries must fit in shared memory)
// measured A/B on one B200 (tools/prof_one.py, [256,C,N,N], TB/s, this kernel vs the smem-operand kernel):
// 56x56 3.16 vs 2.65, 64x64 3.43 vs 2.94 (3 slots); 28x28 3.28 vs 2.68, 32x32 2.93 vs 2.41 (6 slots, cp.async staging);
// 14x14 2.87 vs 2.18, 16x16 3.10 vs 2.58 (6 slots, two maps side by side per slot); 34..50 not better
constexpr int T_AUTO_LO = 52, T_AUTO_SMALL_HI = 32;
bool t_shape_ok(int N) { return t_shape_supported(N) && (N >= T_AUTO_LO || N <= T_AUTO_SMALL_HI); }
// ... and how much work a launch must carry before AUTO prefers it below T_AUTO_LO: the 6-slot variant's prologue (768 threads,
// A' into TMEM, 96 KB of operand slots) costs a few microseconds more than the smem-operand kernel's, which decides launches of a
// few MB (ResNet-56 [256,16,32,32] = 17 MB: 0.655 vs 0.754 ms per batch over its 55 hooks with / without this rule)
// (sides <= 8, four maps side by side per slot, are supported but not routed: back to back on one shape this kernel shows
//  [256,2048,7,7] at 2.09 vs 1.48 TB/s because its longer prologue hides behind the previous launch, but inside ResNet-50's
//  step the launch takes 69 us with either kernel and the step is not faster)
constexpr int T_AUTO_SMALL_LO = 10;
constexpr long long T_AUTO_MIN_BYTES = 32ll << 20;
bool t_launch_ok(int N, long long bytes) {
    return t_shape_ok(N) && (N >= T_AUTO_LO || (N >= T_AUTO_SMALL_LO && bytes >= T_AUTO_MIN_BYTES));
}
// odd sides: a float4 of the stream may straddle maps, the stream itself must not end inside one
bool t_stream_ok(int N, long long n_maps) { return (N % 2) == 0 || (n_maps * N * N) % 4 == 0; }

int launch_t(const float* first, int B, int N, int c_count, double* accum, float* energy_out, float* coeff_out, cudaStream_t stream) {
    TBasis basis;
    int rc = get_t_basis(N, basis);
    if (rc) return rc;
    TScoreArgs a;
    std::memset(&a, 0, sizeof a);
    a.x_dense = first; a.n_maps = B * c_count; a.c_count = c_count;
    a.N = N; a.NN = N * N; a.Ms = (N + 7) / 8 * 8; a.G = 128 / a.Ms;
    a.total_elems = static_cast<long long>(a.n_maps) * a.NN;
    a.tile_vec = basis.tile_vec;
    a.J = t_groups(N); a.MT = a.G * a.J;
    a.num_tiles = (a.n_maps + a.MT - 1) / a.MT;
    a.K1S = (a.G * N + 15) / 16; a.N1 = a.J > 1 ? a.J * a.Ms : (N + 15) / 16 * 16;
    a.TPM = pow2_floor(128 / a.MT < 32 ? 128 / a.MT : 32);
    a.idesc_g = umma::make_idesc_bf16(128, 16, false, false);
    a.NQ = a.N1 / 16;
    a.j_shift = a.J == 4 ? 2 : a.J == 2 ? 1 : 0;
    a.ms_shift = a.Ms == 8 ? 3 : 4;
    a.tpm_shift = 0;
    while ((1 << a.tpm_shift) < a.TPM) ++a.tpm_shift;
    a.idesc = umma::make_idesc_bf16(128, a.N1, false, false);
    a.scatter = basis.scatter; a.scatter_bytes = static_cast<uint32_t>(basis.tile_vec) * basis.vpe * 2u;
    a.a_hi = basis.a_hi; a.a_lo = basis.a_lo; a.c_hi = basis.c_hi; a.c_lo = basis.c_lo;
    a.accum = accum; a.energy_out = energy_out; a.dump = coeff_out; a.status = g.status;
    if ((rc = trace_for("DCTP_T_TRACE", a.trace))) return rc;
    a.div_ms.set(a.Ms);
    const int n1max = t_n1max(N), ns = n1max == 64 ? 3 : 6;
    const size_t smem = n1max == 64 ? TScoreSmem<64>::total(ns, a.scatter_bytes) : TScoreSmem<32>::total(ns, a.scatter_bytes);
    int grid = g.sm_count;
    const int need = (a.num_tiles + ns - 1) / ns;
    if (grid > need) grid = need;
    a.chan_step = static_cast<int>((static_cast<long long>(grid) * ns * a.MT) % c_count);
    const bool v2 = basis.vpe == 2;
    // two producer warpgroups (ResNet-50 step 3.30 -> 3.15 ms) where a tile is at most 13 float4 per thread and the scatter table
    // has one entry per float4 (52x52, 56x56: it fits in shared memory)
    const bool producers = n1max == 64 && basis.tile_vec <= 13 * 128 && basis.vpe == 1;
    if (producers) {
        CUDA_TRY(launch_pdl(score_t_kernel<64, 3, 1, 2>, grid, 640, TScoreSmem<64, 2>::total(ns, a.scatter_bytes), stream, a));
    } else if (n1max == 64) {
        if (v2) CUDA_TRY(launch_pdl(score_t_kernel<64, 3, 2>, grid, 384, smem, stream, a));
        else CUDA_TRY(launch_pdl(score_t_kernel<64, 3, 1>, grid, 384, smem, stream, a));
    } else {
        if (basis.vpe == 4) CUDA_TRY(launch_pdl(score_t_kernel<32, 6, 4>, grid, 768, smem, stream, a));
        else if (v2) CUDA_TRY(launch_pdl(score_t_kernel<32, 6, 2>, grid, 768, smem, stream, a));
        else CUDA_TRY(launch_pdl(score_t_kernel<32, 6, 1>, grid, 768, smem, stream, a));
    }
    note_kernel("score_t_kernel<%d,%d,VPE=%d%s> (tcgen05, block-diagonal basis in TMEM)", n1max, ns, basis.vpe,
                producers ? ",2 producer warpgroups" : "");
    if (a.trace) {
        long long h[TRACE_LEN];
        if ((rc = read_trace(h))) return rc;
        const char* names[7] = {"convert", "fence+bar", "issue1+prefetch", "wait1", "epi1+bar", "issue2+wait2", "epi2+reduce"};
        double sum[7] = {0}; int n = 0; double gap = 0;
        for (int t = 2; t < 32 && h[t * 8 + 7]; ++t, ++n) {
            for (int k = 0; k < 7; ++k) sum[k] += double(h[t * 8 + k + 1] - h[t * 8 + k]);
            gap += double(h[t * 8] - h[(t - 1) * 8 + 7]);
        }
        if (n) {
            fprintf(stderr, "[dctp trace] N=%d tiles=%d cycles/tile:", N, n);
            double tot = 0;
            for (int k = 0; k < 7; ++k) { fprintf(stderr, " %s %.0f", names[k], sum[k] / n); tot += sum[k] / n; }
            fprintf(stderr, " loop-gap %.0f total %.0f\n", gap / n, tot + gap / n);
        }
    }
    return launched();
}

struct Call {                                            // the arguments of one dctp_score_accum_ex call
    const void* x;
    int B, H, W;
    long long stride_b, stride_c, stride_h;
    int c_begin, c_count;
    double* accum;
    float *energy_out, *coeff_out;
    const void* first;                                   // dense_first()
    int in;                                              // element type of x (IN_*: DCTP_DTYPE_*)
    long long maps() const { return static_cast<long long>(B) * c_count; }
    const float* xf() const { return static_cast<const float*>(x); }          // (fp32 calls only)
};

// The first scored map when the call's maps are one contiguous, 16-byte-aligned stream (packed rows and channels, and
// images back to back unless there is one), null otherwise.  The TMA-fed kernels read only such streams.
const void* dense_first(const Call& c) {
    const long long hw = static_cast<long long>(c.H) * c.W;
    const void* first = static_cast<const char*>(c.x) + static_cast<long long>(c.c_begin) * c.stride_c * in_bytes(c.in);
    const bool dense = c.stride_h == c.W && c.stride_c == hw && (c.B == 1 || c.stride_b == c.c_count * hw) &&
                       (reinterpret_cast<uintptr_t>(first) % 16) == 0;
    return dense ? first : nullptr;
}

template <int KP>
int launch_umma(const Call& c, cudaStream_t stream) {
    const int N = c.H;
    UmmaBasis basis;
    int rc = get_umma_basis(N, KP, basis);
    if (rc) return rc;
    UmmaScoreArgs a;
    std::memset(&a, 0, sizeof a);
    a.x = c.xf(); a.stride_b = c.stride_b; a.stride_c = c.stride_c; a.c_begin = c.c_begin; a.c_count = c.c_count;
    a.n_maps = c.B * c.c_count;
    a.N = N; a.NN = N * N;
    a.Ms = (N + 7) / 8 * 8; a.G = 128 / a.Ms; a.J = KP / a.Ms; a.MT = a.G * a.J;
    a.num_tiles = (a.n_maps + a.MT - 1) / a.MT;
    a.K1 = (a.J * a.Ms + 15) / 16; a.N1 = 16 * a.K1;
    if (a.Ms == 8) { a.NQ = a.J / 2; a.K2S = 1; a.N2 = 16; }
    else { a.NQ = a.J; a.K2S = (a.Ms + 15) / 16; a.N2 = 16 * a.K2S; }
    a.a2_lbo = static_cast<uint32_t>(a.K2S) * 2048u; a.a2_group_bytes = 2u * a.a2_lbo;
    a.TPM = pow2_floor(128 / a.MT < 32 ? 128 / a.MT : 32);
    a.tpm_shift = 0;
    while ((1 << a.tpm_shift) < a.TPM) ++a.tpm_shift;
    a.idesc1 = umma::make_idesc_bf16(128, a.N1, false, false);
    a.idesc2 = umma::make_idesc_bf16(128, a.N2, true, false);
    a.basis_hi = basis.hi; a.basis_lo = basis.lo;
    a.accum = c.accum; a.energy_out = c.energy_out; a.dump = c.coeff_out; a.status = g.status;
    a.div_n.set(N); a.div_ms.set(a.Ms); a.div_j.set(a.J);
    // the dense load modes read the stream through a table of where each float4 of a full tile lands, which exists when a tile is a
    // whole number of float4.  (KP = 128 serves sides 65..128, one map per tile: only even sides have a table, and its entries are
    // never 2-byte (LOAD_DENSE4), so that instantiation is not compiled.)
    const bool dense = c.first && basis.scatter;
    int mode;
    if (dense) {
        mode = basis.vpe == 1 ? LOAD_DENSE1 : basis.vpe == 2 ? LOAD_DENSE2 : LOAD_DENSE4;
        a.x_dense = static_cast<const float*>(c.first); a.total_elems = static_cast<long long>(a.n_maps) * a.NN;
        a.tile_vec = basis.tile_vec; a.scatter = basis.scatter;
        a.var_bytes = static_cast<uint32_t>(basis.tile_vec) * basis.vpe * 2u;
        a.div_vpm.set(1);
    } else {
        const int vec = pick_vec(c.xf(), c.stride_b, c.stride_c, N);
        mode = vec == 4 ? LOAD_GEN4 : vec == 2 ? LOAD_GEN2 : LOAD_GEN1;
        a.var_bytes = 128 * sizeof(void*);
        a.div_vpm.set(a.NN / vec);
    }
    a.red_bytes = (a.Ms == 8 ? 8u : static_cast<uint32_t>(a.NQ * (a.N2 / 16))) * 512u;
    const bool pf = dense && basis.tile_vec <= UMMA_PF_SLOTS * 128;
    const size_t smem = UmmaScoreSmem<KP>::total(a.red_bytes, a.var_bytes);
    int grid = g.sm_count * umma_occupancy(KP, mode, pf, smem);
    if (grid > a.num_tiles) grid = a.num_tiles;
    a.chan_step = static_cast<int>((static_cast<long long>(grid) * a.MT) % c.c_count);
    switch (mode) {
        case LOAD_DENSE1:
            if (pf) CUDA_TRY(launch_pdl(score_umma_kernel<KP, LOAD_DENSE1, true>, grid, 128, smem, stream, a));
            else CUDA_TRY(launch_pdl(score_umma_kernel<KP, LOAD_DENSE1, false>, grid, 128, smem, stream, a));
            break;
        case LOAD_DENSE2:
            if (pf) CUDA_TRY(launch_pdl(score_umma_kernel<KP, LOAD_DENSE2, true>, grid, 128, smem, stream, a));
            else CUDA_TRY(launch_pdl(score_umma_kernel<KP, LOAD_DENSE2, false>, grid, 128, smem, stream, a));
            break;
        case LOAD_DENSE4:
            if constexpr (KP != 64) return fail(DCTP_E_UNSUPPORTED, "no <%d, LOAD_DENSE4> instantiation (side %d)", KP, N);
            else if (pf) CUDA_TRY(launch_pdl(score_umma_kernel<KP, LOAD_DENSE4, true>, grid, 128, smem, stream, a));
            else CUDA_TRY(launch_pdl(score_umma_kernel<KP, LOAD_DENSE4, false>, grid, 128, smem, stream, a));
            break;
        case LOAD_GEN4: CUDA_TRY(launch_pdl(score_umma_kernel<KP, LOAD_GEN4, false>, grid, 128, smem, stream, a)); break;
        case LOAD_GEN2: CUDA_TRY(launch_pdl(score_umma_kernel<KP, LOAD_GEN2, false>, grid, 128, smem, stream, a)); break;
        default: CUDA_TRY(launch_pdl(score_umma_kernel<KP, LOAD_GEN1, false>, grid, 128, smem, stream, a)); break;
    }
    note_kernel("score_umma_kernel<%d,%d,%d> (tcgen05 bf16x3, operands in shared memory)", KP, mode, pf ? 1 : 0);
    return launched();
}

int launch_simt(const Call& c, cudaStream_t stream) {
    const int H = c.H, W = c.W;
    SimtBasis bh, bw;
    int rc = get_simt_basis(H, bh);
    if (rc) return rc;
    if ((rc = get_simt_basis(W, bw))) return rc;
    SimtScoreArgs a;
    std::memset(&a, 0, sizeof a);
    a.x = c.xf(); a.stride_b = c.stride_b; a.stride_c = c.stride_c; a.stride_h = c.stride_h;
    a.c_begin = c.c_begin; a.c_count = c.c_count; a.n_maps = c.B * c.c_count; a.H = H; a.W = W;
    a.basis_h_t = bh.t; a.basis_w_t = bw.t; a.accum = c.accum; a.energy_out = c.energy_out; a.dump = c.coeff_out;
    if (H <= SIMT_T && W <= SIMT_T) {
        const int G = SIMT_T / H, tiles = (a.n_maps + G - 1) / G;
        int grid = g.sm_count * 2;
        if (grid > tiles) grid = tiles;
        score_simt_small_kernel<<<grid, 256, SIMT_SMALL_SMEM, stream>>>(a);
        note_kernel("score_simt_small_kernel (fp32 CUDA cores)");
    } else {
        const int Hpad = (H + SIMT_T - 1) / SIMT_T * SIMT_T;
        const size_t smem = static_cast<size_t>(Hpad + 2 * SIMT_T) * SIMT_LD * sizeof(float);
        if (smem > 200 * 1024) return fail(DCTP_E_UNSUPPORTED, "map height %d needs %zu B of shared memory", H, smem);
        if (c.energy_out) CUDA_TRY(cudaMemsetAsync(c.energy_out, 0, sizeof(float) * a.n_maps, stream));
        const unsigned grid = static_cast<unsigned>((W + SIMT_T - 1) / SIMT_T) * static_cast<unsigned>(a.n_maps);
        score_simt_large_kernel<<<grid, 256, smem, stream>>>(a);
        note_kernel("score_simt_large_kernel (fp32 CUDA cores)");
    }
    return launched();
}

// ------------------------------------------------------------------ routing
// The kernels a score call can run on.  takes() says whether a kernel takes a call; AUTO's choice and every forced
// DCTP_PATH_* value go through it.
enum Route { R_KRON, R_STACK, R_TMEM, R_UMMA64, R_UMMA128, R_LARGE, R_SIMT };

bool takes(Route r, const Call& c) {
    const bool square = c.H == c.W, dense = c.first != nullptr;
    switch (r) {
        case R_KRON: return square && c.H <= 8 && dense;
        case R_STACK: return square && stack_shape_supported(c.H) && dense;
        case R_TMEM: return square && t_shape_supported(c.H) && dense && t_stream_ok(c.H, c.maps());
        case R_UMMA64: return umma_shape_ok(c.H, c.W, c.stride_h) && c.H <= 64;
        case R_UMMA128: return umma_shape_ok(c.H, c.W, c.stride_h) && c.H > 64;
        case R_LARGE: return large_shape_supported(c.H, c.W, c.stride_h) && dense;
        default: return true;
    }
}

Route auto_route(const Call& c) {
    if (takes(R_LARGE, c)) return R_LARGE;
    if (takes(R_UMMA128, c)) return R_UMMA128;                  // (windows and strided batches of large maps too)
    if (!takes(R_UMMA64, c)) return R_SIMT;
    if (takes(R_KRON, c)) return R_KRON;
    if (takes(R_STACK, c)) return R_STACK;
    if (takes(R_TMEM, c) && t_launch_ok(c.H, 4 * c.maps() * c.H * c.W)) return R_TMEM;
    return R_UMMA64;
}

// a call on one map at a 16-byte-aligned address: what AUTO and the forced paths do with dense maps of this shape
Call dense_call(int H, int W, long long stride_h) {
    alignas(16) static const float base[4] = {};
    Call c = {base, 1, H, W, 0, static_cast<long long>(H) * W, stride_h, 0, 1, nullptr, nullptr, nullptr, nullptr, IN_F32};
    c.first = dense_first(c);
    return c;
}

// the kernels that score up to SCORE_MAX_SEG activations in one launch
bool multi_site(Route r) { return r == R_KRON || r == R_STACK || r == R_LARGE; }
// the kernels that read 16-bit input themselves; every other route scores a widened fp32 copy of the window (score_accum)
bool reads_16bit(Route r) { return r == R_KRON || r == R_STACK; }
int launch_sites(Route r, const SiteDesc* sites, int n, int N, float* energy_out, float* coeff_out, int in, cudaStream_t s) {
    if (r == R_KRON) return launch_kron(sites, n, N, energy_out, coeff_out, in, s);
    if (r == R_STACK) return launch_stack(sites, n, N, energy_out, coeff_out, in, s);
    return launch_large(sites, n, N, energy_out, coeff_out, s);
}

int launch(Route r, const Call& c, cudaStream_t s) {
    switch (r) {
        case R_TMEM: return launch_t(static_cast<const float*>(c.first), c.B, c.H, c.c_count, c.accum, c.energy_out, c.coeff_out, s);
        case R_UMMA64: return launch_umma<64>(c, s);
        case R_UMMA128: return launch_umma<128>(c, s);
        case R_SIMT: return launch_simt(c, s);
        default: {
            const SiteDesc one = {c.first, c.B, c.c_count, c.accum};
            return launch_sites(r, &one, 1, c.H, c.energy_out, c.coeff_out, c.in, s);
        }
    }
}

}  // namespace

// ====================================================================== C ABI
extern "C" {

int dctp_version(void) { return DCTP_VERSION; }
const char* dctp_last_error(void) { return g_err; }

int dctp_init(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    return ensure_init();
}

int dctp_shutdown(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g.ready) return DCTP_OK;
    for (void* p : g.bases) cudaFree(p);
    cudaFree(g.status); cudaFree(g.trace); cudaFree(g.hx); cudaFree(g.hacc); cudaFree(g.hout);
    g = State();
    return DCTP_OK;
}

int dctp_sm_count(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    int rc = ensure_init();
    return rc ? rc : g.sm_count;
}
long long dctp_launch_count(void) { return g.launches; }
const char* dctp_last_kernel(void) { return g.last_kernel; }

int dctp_path_for(int H, int W, long long stride_h) {
    const Route r = auto_route(dense_call(H, W, stride_h));
    return r == R_LARGE ? DCTP_PATH_LARGE : r == R_SIMT ? DCTP_PATH_SIMT : DCTP_PATH_UMMA;
}

int dctp_occupancy(int kp, int mode) {
    std::lock_guard<std::mutex> lk(g_mu);
    int rc = ensure_init();
    if (rc) return rc;
    if ((kp != 64 && kp != 128) || mode < 0 || mode > 5) return fail(DCTP_E_INVALID, "dctp_occupancy(%d, %d)", kp, mode);
    if (kp == 128 && mode == LOAD_DENSE4) return fail(DCTP_E_UNSUPPORTED, "dctp_occupancy: no <128, LOAD_DENSE4> instantiation");
    const size_t smem = kp == 64 ? UmmaScoreSmem<64>::total(2048, 3136) : UmmaScoreSmem<128>::total(2560, 3200);
    return umma_occupancy(kp, mode, mode <= LOAD_DENSE4, smem);
}

int dctp_prepare(int H, int W) {
    std::lock_guard<std::mutex> lk(g_mu);
    int rc = ensure_init();
    if (rc) return rc;
    if (H < 1 || W < 1) return fail(DCTP_E_INVALID, "dctp_prepare: H=%d W=%d", H, W);
    // the bases of the kernels dense maps of this shape can run on (the TMEM-operand kernel: the sides AUTO may give it)
    const Call c = dense_call(H, W, W);
    LargeBasis lb;
    if (takes(R_LARGE, c) && (rc = get_large_basis(H, lb))) return rc;
    if (!takes(R_UMMA64, c) && !takes(R_UMMA128, c)) {
        SimtBasis b;
        if ((rc = get_simt_basis(H, b))) return rc;
        return get_simt_basis(W, b);
    }
    KronBasis kb;
    StackBasis sb;
    TBasis tb;
    UmmaBasis ub;
    if (takes(R_KRON, c) && (rc = get_kron_basis(H, kb))) return rc;
    if (takes(R_STACK, c) && (rc = get_stack_basis(H, sb))) return rc;
    if (t_shape_ok(H) && (rc = get_t_basis(H, tb))) return rc;
    return get_umma_basis(H, H <= 64 ? 64 : 128, ub);
}

}  // extern "C"

namespace {

// one score call; the caller holds g_mu
int score_accum(const void* x, int dtype, int B, int H, int W, long long stride_b, long long stride_c, long long stride_h, int c_begin,
                int c_count, double* accum, float* energy_out, float* coeff_out, int path, cudaStream_t s) {
    int rc = ensure_init();
    if (rc) return rc;
    if (B < 0 || H < 1 || W < 1 || c_begin < 0 || c_count < 0 || stride_h < W)
        return fail(DCTP_E_INVALID, "dctp_score_accum: B=%d H=%d W=%d c_begin=%d c_count=%d stride_h=%lld", B, H, W, c_begin,
                    c_count, stride_h);
    if (path < DCTP_PATH_AUTO || path > DCTP_PATH_KRON) return fail(DCTP_E_INVALID, "unknown path %d", path);
    if (dtype != DCTP_DTYPE_F32 && dtype != DCTP_DTYPE_BF16 && dtype != DCTP_DTYPE_F16) return fail(DCTP_E_INVALID, "unknown dtype %d", dtype);
    if (B == 0 || c_count == 0) return DCTP_OK;                     // empty batch / empty window: nothing to add
    if (!x || !accum) return fail(DCTP_E_INVALID, "dctp_score_accum: null pointer");
    if (static_cast<long long>(B) * c_count > (1ll << 30)) return fail(DCTP_E_INVALID, "too many maps in one call");
    Call c = {x, B, H, W, stride_b, stride_c, stride_h, c_begin, c_count, accum, energy_out, coeff_out, nullptr, dtype};
    c.first = dense_first(c);
    Route r = R_SIMT;
    const char* needs = "";
    switch (path) {
        case DCTP_PATH_AUTO: r = auto_route(c); break;
        case DCTP_PATH_UMMA: r = H <= 64 ? R_UMMA64 : R_UMMA128; needs = "UMMA path takes contiguous square maps of side <= 128"; break;
        case DCTP_PATH_TMEM:
            r = R_TMEM;
            needs = "TMEM-operand path takes dense 16-B aligned square maps of side 5..64 (odd sides: up to 13, and a whole number of float4 in the call)";
            break;
        case DCTP_PATH_KRON: r = R_KRON; needs = "Kronecker path takes dense 16-B aligned square maps of side <= 8"; break;
        case DCTP_PATH_STACK:
            r = R_STACK;
            needs = "stacked-basis path takes dense 16-B aligned square maps of even side 10..64 (above 32: multiples of 4)";
            break;
        case DCTP_PATH_LARGE: r = R_LARGE; needs = "large-map path takes dense 16-B aligned square maps, side 80..320 multiple of 16"; break;
    }
    if (!takes(r, c)) return fail(DCTP_E_UNSUPPORTED, "%s (got %dx%d, stride_h %lld)", needs, H, W, stride_h);
    if (dtype == DCTP_DTYPE_F32 || reads_16bit(r)) return launch(r, c, s);
    // 16-bit input on a kernel that reads fp32 only: the scored window is widened into a dense fp32 copy, allocated and freed on the
    // caller's stream (calls on different streams never share it; a call captured into a graph allocates inside the graph), and scored
    // as the fp32 entry scores that copy with the same path
    const long long rows = c.maps() * H;
    void* buf = nullptr;
    CUDA_TRY(cudaMallocAsync(&buf, sizeof(float) * rows * W, s));
    WidenArgs wa = {static_cast<const uint16_t*>(x), stride_b, stride_c, stride_h, c_begin, c_count, H, W, rows, static_cast<float*>(buf)};
    long long blocks = (rows + 7) / 8;
    if (blocks > 16ll * g.sm_count) blocks = 16ll * g.sm_count;
    if (dtype == DCTP_DTYPE_BF16) widen_window_kernel<IN_BF16><<<static_cast<unsigned>(blocks), 256, 0, s>>>(wa);
    else widen_window_kernel<IN_F16><<<static_cast<unsigned>(blocks), 256, 0, s>>>(wa);
    ++g.launches;
    const cudaError_t launched = cudaGetLastError();
    rc = launched != cudaSuccess ? fail(DCTP_E_CUDA, "widen_window_kernel: %s", cudaGetErrorString(launched)) : DCTP_OK;
    if (!rc) {
        Call w = {buf, B, H, W, static_cast<long long>(c_count) * H * W, static_cast<long long>(H) * W, W, 0, c_count, accum, energy_out, coeff_out,
                  nullptr, IN_F32};
        w.first = dense_first(w);
        rc = launch(path == DCTP_PATH_AUTO ? auto_route(w) : r, w, s);
    }
    const cudaError_t freed = cudaFreeAsync(buf, s);
    if (rc) return rc;
    CUDA_TRY(freed);
    return DCTP_OK;
}

}  // namespace

extern "C" {

int dctp_score_accum_ex(const void* x, int dtype, int B, int H, int W, long long stride_b, long long stride_c, long long stride_h,
                        int c_begin, int c_count, double* accum, float* energy_out, float* coeff_out, int path, void* stream) {
    std::lock_guard<std::mutex> lk(g_mu);
    return score_accum(x, dtype, B, H, W, stride_b, stride_c, stride_h, c_begin, c_count, accum, energy_out, coeff_out, path,
                       static_cast<cudaStream_t>(stream));
}

int dctp_score_accum(const float* x, int B, int H, int W, long long stride_b, long long stride_c, long long stride_h,
                     int c_begin, int c_count, double* accum, float* energy_out, float* coeff_out, int path,
                     void* stream) {
    return dctp_score_accum_ex(x, DCTP_DTYPE_F32, B, H, W, stride_b, stride_c, stride_h, c_begin, c_count, accum, energy_out, coeff_out, path,
                               stream);
}

int dctp_score_accum_multi_ex(const dctp_site* sites, int n_sites, int H, int W, int dtype, void* stream) {
    std::vector<int> single;                                 // sites left to the single-site entry
    {
        std::lock_guard<std::mutex> lk(g_mu);
        int rc = ensure_init();
        if (rc) return rc;
        if (n_sites < 0 || H < 1 || W < 1 || (n_sites > 0 && !sites)) return fail(DCTP_E_INVALID, "dctp_score_accum_multi: n_sites=%d H=%d W=%d", n_sites, H, W);
        if (dtype != DCTP_DTYPE_F32 && dtype != DCTP_DTYPE_BF16 && dtype != DCTP_DTYPE_F16) return fail(DCTP_E_INVALID, "unknown dtype %d", dtype);
        for (int i = 0; i < n_sites; ++i) {
            if (sites[i].B < 0 || sites[i].c_count < 0 || ((sites[i].B > 0 && sites[i].c_count > 0) && (!sites[i].x || !sites[i].accum)))
                return fail(DCTP_E_INVALID, "dctp_score_accum_multi: site %d: B=%d c_count=%d or a null pointer", i, sites[i].B, sites[i].c_count);
            if (static_cast<long long>(sites[i].B) * sites[i].c_count > (1ll << 30)) return fail(DCTP_E_INVALID, "too many maps in site %d", i);
        }
        cudaStream_t s = static_cast<cudaStream_t>(stream);
        // sites AUTO gives to a multi-site kernel that reads their dtype: one launch per SCORE_MAX_SEG of them; the others go through
        // the single-site entry below
        SiteDesc batch[SCORE_MAX_SEG];
        int nb = 0;
        Route batched = R_SIMT;
        for (int i = 0; i < n_sites; ++i) {
            const dctp_site& site = sites[i];
            if (site.B == 0 || site.c_count == 0) continue;
            Call c = {site.x, site.B, H, W, static_cast<long long>(site.c_count) * H * W, static_cast<long long>(H) * W, W, 0, site.c_count,
                      site.accum, nullptr, nullptr, nullptr, dtype};
            c.first = dense_first(c);
            const Route r = auto_route(c);
            if (!multi_site(r) || (dtype != DCTP_DTYPE_F32 && !reads_16bit(r))) { single.push_back(i); continue; }
            batched = r;                                     // (the same for every dense site of the shape)
            batch[nb++] = SiteDesc{c.first, site.B, site.c_count, site.accum};
            if (nb == SCORE_MAX_SEG) {
                if ((rc = launch_sites(r, batch, nb, H, nullptr, nullptr, dtype, s))) return rc;
                nb = 0;
            }
        }
        if (nb > 0 && (rc = launch_sites(batched, batch, nb, H, nullptr, nullptr, dtype, s))) return rc;
    }
    for (int i : single) {
        const int rc = dctp_score_accum_ex(sites[i].x, dtype, sites[i].B, H, W, static_cast<long long>(sites[i].c_count) * H * W,
                                           static_cast<long long>(H) * W, W, 0, sites[i].c_count, sites[i].accum, nullptr, nullptr, DCTP_PATH_AUTO,
                                           stream);
        if (rc) return rc;
    }
    return DCTP_OK;
}

int dctp_score_accum_multi(const dctp_site* sites, int n_sites, int H, int W, void* stream) {
    return dctp_score_accum_multi_ex(sites, n_sites, H, W, DCTP_DTYPE_F32, stream);
}

// ------------------------------------------------------------------ alternative scoring ops (SURVEY §8f-3)
// DCTP_OP_DCT3 with caller-owned scratch: per-channel sums part [c_count], and per-(image, channel) energies [B * c_count] when
// values_out is wanted
static int dct3_energy(const float* x, int B, int H, int W, long long stride_b, long long stride_c, long long stride_h, int c_begin,
                       int c_count, double* accum, float* values_out, double* part, float* energy, cudaStream_t s) {
    CUDA_TRY(cudaMemsetAsync(part, 0, sizeof(double) * c_count, s));
    int rc = dctp_score_accum(x, B, H, W, stride_b, stride_c, stride_h, c_begin, c_count, part, energy, nullptr, DCTP_PATH_AUTO, s);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(g_mu);
    if (values_out) dct3_reduce_kernel<<<B, 256, 0, s>>>(energy, c_count, values_out, accum);
    else sum_to_one_kernel<<<1, 256, 0, s>>>(part, c_count, accum);
    return launched();
}

int dctp_score_op(int op, const float* x, int B, int H, int W, long long stride_b, long long stride_c, long long stride_h,
                  int c_begin, int c_count, double* accum, float* values_out, void* stream) {
    if (op == DCTP_OP_DCT2)
        return dctp_score_accum(x, B, H, W, stride_b, stride_c, stride_h, c_begin, c_count, accum, values_out, nullptr, DCTP_PATH_AUTO, stream);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (op == DCTP_OP_RANK || op == DCTP_OP_RANK_SQ) {
        std::lock_guard<std::mutex> lk(g_mu);
        int rc = ensure_init();
        if (rc) return rc;
        if (B < 0 || H < 1 || W < 1 || c_begin < 0 || c_count < 0 || stride_h < W)
            return fail(DCTP_E_INVALID, "dctp_score_op: B=%d H=%d W=%d c_begin=%d c_count=%d stride_h=%lld", B, H, W, c_begin, c_count, stride_h);
        if (B == 0 || c_count == 0) return DCTP_OK;
        if (!x || !accum) return fail(DCTP_E_INVALID, "dctp_score_op: null pointer");
        RankArgs a;
        a.x = x; a.stride_b = stride_b; a.stride_c = stride_c; a.stride_h = stride_h;
        a.H = H; a.W = W; a.c_begin = c_begin; a.c_count = c_count;
        a.n_maps = static_cast<long long>(B) * c_count;
        a.accum = accum; a.out = values_out; a.squared = op == DCTP_OP_RANK_SQ;
        a.by_cols = H > W;
        a.n = H > W ? W : H; a.m = H > W ? H : W; a.ld = a.m | 1;
        const size_t per_map = (static_cast<size_t>(a.n) * a.ld + a.n + 1) * sizeof(float);
        if (a.m > RANK_MAX_LEN || per_map > static_cast<size_t>(RANK_SMEM_MAX))
            return fail(DCTP_E_UNSUPPORTED, "the rank op holds a map in shared memory: longer side <= %d and %zu bytes <= %d (got %dx%d)",
                        RANK_MAX_LEN, per_map, RANK_SMEM_MAX, H, W);
        a.log2L = 0;
        while ((RANK_EPT << a.log2L) < a.m) ++a.log2L;                  // lanes per pair: 8 elements each
        const int L = 1 << a.log2L, np = (a.n + 1) / 2;
        int threads = a.m <= 64 ? 256 : a.m <= 128 ? 512 : 1024;
        const int workers = threads / L;
        a.wpm = np < workers ? np : workers;
        a.G = workers / a.wpm;
        const int g_smem = static_cast<int>(static_cast<size_t>(64 * 1024) / per_map);       // keep several CTAs resident per SM
        if (a.G > g_smem) a.G = g_smem < 1 ? 1 : g_smem;
        if (a.G < 1) a.G = 1;
        if (a.G > a.n_maps) a.G = static_cast<int>(a.n_maps);
        threads = ((a.G * a.wpm * L + 31) / 32) * 32;
        const size_t smem = per_map * a.G;
        long long blocks = (a.n_maps + a.G - 1) / a.G;
        const long long cap = static_cast<long long>(g.sm_count) * 32;
        if (blocks > cap) blocks = cap;
        rank_jacobi_kernel<<<static_cast<unsigned>(blocks), threads, smem, s>>>(a);
        note_kernel("rank_jacobi_kernel (fp32 one-sided Jacobi SVD in shared memory, %d lanes per pair, %d maps per CTA)", L, a.G);
        return launched();
    }
    if (op != DCTP_OP_DCT3) return fail(DCTP_E_INVALID, "dctp_score_op: unknown op %d", op);
    // dct_3d energy of x[b, window] = sum over the window's channels of the 2-D energies (the channel-axis DCT is orthonormal)
    if (B < 0 || c_count < 0) return fail(DCTP_E_INVALID, "dctp_score_op: B=%d c_count=%d", B, c_count);
    if (B == 0 || c_count == 0) return DCTP_OK;
    if (!accum) return fail(DCTP_E_INVALID, "dctp_score_op: null pointer");
    {
        std::lock_guard<std::mutex> lk(g_mu);
        int rc = ensure_init();
        if (rc) return rc;
    }
    // the scratch is allocated and freed on the caller's stream: calls on different streams never share it, and a call captured
    // into a graph allocates inside the graph
    const size_t part_bytes = sizeof(double) * ((c_count + 1) & ~1);   // the energies start 16-byte aligned
    void* scratch = nullptr;
    CUDA_TRY(cudaMallocAsync(&scratch, part_bytes + (values_out ? sizeof(float) * B * c_count : 0), s));
    double* part = static_cast<double*>(scratch);
    float* energy = values_out ? reinterpret_cast<float*>(static_cast<char*>(scratch) + part_bytes) : nullptr;
    const int rc = dct3_energy(x, B, H, W, stride_b, stride_c, stride_h, c_begin, c_count, accum, values_out, part, energy, s);
    const cudaError_t freed = cudaFreeAsync(scratch, s);
    if (rc) return rc;
    CUDA_TRY(freed);
    return DCTP_OK;
}

int dctp_finalize(const double* accum, double n_images, float* out, int n, void* stream) {
    std::lock_guard<std::mutex> lk(g_mu);
    int rc = ensure_init();
    if (rc) return rc;
    if (n < 0 || (n > 0 && (!accum || !out)) || !(n_images > 0)) return fail(DCTP_E_INVALID, "dctp_finalize: n=%d n_images=%g", n, n_images);
    if (n == 0) return DCTP_OK;
    finalize_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(accum, n_images, out, n);
    return launched();
}

int dctp_topk_segmented(const float* scores, const int* seg_offsets, const int* seg_k, int n_seg, long long* out_idx,
                        const int* out_offsets, void* stream) {
    std::lock_guard<std::mutex> lk(g_mu);
    int rc = ensure_init();
    if (rc) return rc;
    if (n_seg < 0 || (n_seg > 0 && (!scores || !seg_offsets || !seg_k || !out_idx || !out_offsets)))
        return fail(DCTP_E_INVALID, "dctp_topk_segmented: null pointer or n_seg=%d", n_seg);
    if (n_seg == 0) return DCTP_OK;
    topk_segmented_kernel<<<n_seg, TOPK_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(scores, seg_offsets, seg_k, out_idx,
                                                                                         out_offsets);
    return launched();
}

int dctp_gather_weight(const float* w, int c_out, int c_in, int inner, const long long* sel_out, int k_out,
                       const long long* sel_in, int k_in, float* out, void* stream) {
    std::lock_guard<std::mutex> lk(g_mu);
    int rc = ensure_init();
    if (rc) return rc;
    if (c_out < 0 || c_in < 0 || inner < 0 || k_out < 0 || k_in < 0)
        return fail(DCTP_E_INVALID, "dctp_gather_weight: negative size (c_out=%d c_in=%d inner=%d k_out=%d k_in=%d)", c_out, c_in,
                    inner, k_out, k_in);
    if ((!sel_out && k_out != c_out) || (!sel_in && k_in != c_in))
        return fail(DCTP_E_INVALID, "dctp_gather_weight: a NULL selection means all channels (k_out=%d c_out=%d k_in=%d c_in=%d)",
                    k_out, c_out, k_in, c_in);
    GatherArgs a;
    a.w = w; a.out = out; a.sel_out = sel_out; a.sel_in = sel_in;
    a.c_out = c_out; a.c_in = c_in; a.inner = inner; a.k_out = k_out; a.k_in = k_in;
    a.total = static_cast<long long>(k_out) * k_in * inner;
    a.status = g.status;
    if (a.total == 0) return DCTP_OK;
    if (!w || !out) return fail(DCTP_E_INVALID, "dctp_gather_weight: null pointer");
    long long blocks = (a.total + GATHER_THREADS - 1) / GATHER_THREADS;
    const long long cap = static_cast<long long>(g.sm_count) * 16;
    if (blocks > cap) blocks = cap;
    gather_weight_kernel<<<static_cast<unsigned>(blocks), GATHER_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(a);
    return launched();
}

int dctp_check(void* stream) {
    std::lock_guard<std::mutex> lk(g_mu);
    int rc = ensure_init();
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    int st = 0;
    CUDA_TRY(cudaMemcpy(&st, g.status, sizeof st, cudaMemcpyDeviceToHost));
    if (st != 0) {
        cudaMemset(g.status, 0, sizeof(int));
        return fail(DCTP_E_DEVICE, st == DCTP_DEV_BAD_INDEX ? "device status %d: a channel index passed to dctp_gather_weight is out of range"
                                                            : "device status %d: a tensor-core completion wait timed out", st);
    }
    return DCTP_OK;
}

int dctp_score_host(const float* x_host, int B, int C, int H, int W, int c_begin, int c_count, float* scores_host, int path) {
    {
        std::lock_guard<std::mutex> lk(g_mu);
        int rc = ensure_init();
        if (rc) return rc;
        if (!x_host || !scores_host || B < 1 || C < 1 || H < 1 || W < 1 || c_begin < 0 || c_count < 1 || c_begin + c_count > C)
            return fail(DCTP_E_INVALID, "dctp_score_host: B=%d C=%d H=%d W=%d window [%d,+%d)", B, C, H, W, c_begin, c_count);
        const size_t bytes = sizeof(float) * B * C * H * W;
        if (bytes > g.hx_bytes) {
            cudaFree(g.hx);
            g.hx = nullptr; g.hx_bytes = 0;
            CUDA_TRY(cudaMalloc(&g.hx, bytes));
            g.hx_bytes = bytes;
        }
        if (static_cast<size_t>(c_count) > g.hc) {
            cudaFree(g.hacc); cudaFree(g.hout);
            g.hacc = nullptr; g.hout = nullptr; g.hc = 0;
            CUDA_TRY(cudaMalloc(&g.hacc, sizeof(double) * c_count));
            CUDA_TRY(cudaMalloc(&g.hout, sizeof(float) * c_count));
            g.hc = c_count;
        }
        CUDA_TRY(cudaMemcpyAsync(g.hx, x_host, bytes, cudaMemcpyHostToDevice, 0));
        CUDA_TRY(cudaMemsetAsync(g.hacc, 0, sizeof(double) * c_count, 0));
    }
    int rc = dctp_score_accum(g.hx, B, H, W, static_cast<long long>(C) * H * W, static_cast<long long>(H) * W, W, c_begin, c_count,
                              g.hacc, nullptr, nullptr, path, nullptr);
    if (rc) return rc;
    if ((rc = dctp_finalize(g.hacc, static_cast<double>(B), g.hout, c_count, nullptr))) return rc;
    CUDA_TRY(cudaMemcpyAsync(scores_host, g.hout, sizeof(float) * c_count, cudaMemcpyDeviceToHost, 0));
    return dctp_check(nullptr);
}

}  // extern "C"
