// score_alt.cuh - the alternative per-slice scoring ops the reference keeps beside the DCT (SURVEY §8f-3):
//
//   /root/reference/utils/common.py:268   c = torch.tensor([torch.matrix_rank(output[i,j,:,:]).item() ...])      (HRank)
//   /root/reference/utils/common.py:269   c = [dct.dct_3d(output[i,:,:,:], norm='ortho') for i in range(a)]
//
// Both go through the same capture / accumulate / top-k plumbing as the DCT energy; only the per-slice reduction differs.
//
// rank_jacobi_kernel: numerical rank of every (image, channel) map with torch.matrix_rank's rule - singular values of the
// fp32 map, rank = #{sigma > sigma_max * max(H, W) * eps_fp32} - by a one-sided (Hestenes) Jacobi SVD held in shared memory.
// The min(H,W) vectors of a map (rows, or columns when the map is taller than wide) are orthogonalised pairwise; a sweep
// visits every pair once in round-robin order (all pairs of a step are disjoint, so a step is one parallel phase); when a
// sweep rotates nothing the vector norms are the singular values.  A pair is worked by L lanes (8 elements each, kept in
// registers between the three dot products and the rotation); small maps share a CTA.  This is CUDA-core work by nature
// (data-dependent plane rotations, ~N^3 flops per sweep on a 12 KB matrix): there is nothing for the tensor cores here.
//
// sum_to_one_kernel / dct3_reduce_kernel: dct_3d over [C, H, W] followed by cnt_score is ONE number per image, the energy
// of the 3-D coefficient cube.  The 3-D transform is the 2-D transform of every channel followed by an orthonormal DCT along
// the channel axis, which leaves the sum of squares unchanged, so the energy is the sum over the channels of the 2-D energies
// the tensor-core kernels already produce; only that sum is added here.
#pragma once
#include <cfloat>
#include <cstdint>
#include <cuda_runtime.h>

namespace dctp {

constexpr int RANK_EPT = 8;            // elements of a vector per lane (registers)
constexpr int RANK_MAX_SWEEPS = 30;    // LAPACK's xGESVJ bound; fp32 maps converge in 5-9
constexpr int RANK_MAX_LEN = 256;      // longest vector: 32 lanes x 8 elements
constexpr float RANK_NEGLIGIBLE = 1.4e-20f;   // (1e-3 * eps_fp32)^2, on squared norms
constexpr int RANK_SMEM_MAX = 200 * 1024;   // a map (n vectors, odd leading dimension) has to fit: side <= 225, 256 x 198

struct RankArgs {
    const float* x;
    long long stride_b, stride_c, stride_h;
    int H, W, c_begin, c_count;
    long long n_maps;
    double* accum;        // [c_count] += rank (or rank^2)
    float* out;           // optional [B * c_count]
    int squared;          // 1: add rank^2 (what cnt_score makes of the rank tensor, common.py:249-255 applied to :268)
    int n, m, ld;         // n vectors of length m, leading dimension ld (odd)
    int by_cols;          // vectors are the map's columns (H > W)
    int log2L, wpm, G;    // lanes per pair worker, pair workers per map, maps per CTA
};

__global__ void __launch_bounds__(1024) rank_jacobi_kernel(const RankArgs a) {
    extern __shared__ float rk_smem[];
    const int t = threadIdx.x;
    const int L = 1 << a.log2L;
    const int tpm = a.wpm << a.log2L;                       // threads per map
    const int g = t / tpm, r = t - g * tpm;
    const int wk = r >> a.log2L, l = r & (L - 1);
    const bool active = g < a.G;
    float* v = rk_smem + static_cast<size_t>(active ? g : 0) * a.n * a.ld;
    float* sig = rk_smem + static_cast<size_t>(a.G) * a.n * a.ld + (active ? g : 0) * a.n;
    unsigned* mx = reinterpret_cast<unsigned*>(rk_smem + static_cast<size_t>(a.G) * a.n * (a.ld + 1)) + (active ? g : 0);
    const int np = (a.n + 1) >> 1, ring = 2 * np - 1;      // circle method over 2*np players, the last one fixed
    const float tol = FLT_EPSILON * sqrtf(static_cast<float>(a.m));

    for (long long grp = blockIdx.x; grp * a.G < a.n_maps; grp += gridDim.x) {
        const long long mi = grp * a.G + g;
        const bool live = active && mi < a.n_maps;
        __syncthreads();                                    // the previous group's readers are done with v / sig
        if (live && r == 0) *mx = 0u;
        __syncthreads();
        const int HW = a.H * a.W;
        if (live) {
            const long long b = mi / a.c_count;
            const int c = static_cast<int>(mi - b * a.c_count);
            const float* src = a.x + b * a.stride_b + static_cast<long long>(a.c_begin + c) * a.stride_c;
            float big = 0.f;
            for (int e = r; e < HW; e += tpm) {
                const int h = e / a.W, w = e - h * a.W;
                const float val = src[static_cast<long long>(h) * a.stride_h + w];
                big = fmaxf(big, fabsf(val));
                if (a.by_cols) v[w * a.ld + h] = val; else v[h * a.ld + w] = val;
            }
            atomicMax(mx, __float_as_uint(big));            // bit patterns of non-negative floats order like the floats
        }
        __syncthreads();
        if (live) {
            // bring the largest entry into [1, 2) with an exact power of two: the rank rule is scale-free, the skip test below
            // and the squared norms then cannot under- or overflow for any finite input
            const float top = __uint_as_float(*mx);
            if (top > 0.f && top < INFINITY) {
                const int ex = ilogbf(top);
                if (ex != 0) {
                    for (int e = r; e < HW; e += tpm) {
                        const int h = e / a.W, w = e - h * a.W;
                        float* cell = a.by_cols ? v + w * a.ld + h : v + h * a.ld + w;
                        *cell = scalbnf(*cell, -ex);
                    }
                }
            }
        }
        __syncthreads();

        for (int sweep = 0; sweep < RANK_MAX_SWEEPS; ++sweep) {
            int rotated = 0;
            for (int s = 0; s < ring; ++s) {
                for (int k0 = 0; k0 < np; k0 += a.wpm) {
                    const int k = k0 + wk;
                    int p, q;
                    if (k == 0) { p = ring; q = s; }
                    else { p = s + k; if (p >= ring) p -= ring; q = s - k; if (q < 0) q += ring; }
                    const bool ok = live && k < np && p < a.n && q < a.n;       // p == n: the dummy player of an odd n
                    float xa[RANK_EPT], xb[RANK_EPT];
                    float al = 0.f, be = 0.f, ga = 0.f;
                    const float* vp = v + p * a.ld;
                    const float* vq = v + q * a.ld;
#pragma unroll
                    for (int e = 0; e < RANK_EPT; ++e) {
                        const int i = l + (e << a.log2L);
                        const bool in = ok && i < a.m;
                        xa[e] = in ? vp[i] : 0.f;
                        xb[e] = in ? vq[i] : 0.f;
                        al = fmaf(xa[e], xa[e], al);
                        be = fmaf(xb[e], xb[e], be);
                        ga = fmaf(xa[e], xb[e], ga);
                    }
                    for (int o = L >> 1; o > 0; o >>= 1) {                      // butterfly: every lane of the worker gets the same bits
                        al += __shfl_xor_sync(0xffffffffu, al, o);
                        be += __shfl_xor_sync(0xffffffffu, be, o);
                        ga += __shfl_xor_sync(0xffffffffu, ga, o);
                    }
                    // a vector below 1e-3 * eps of its partner cannot reach the rank cut (sigma_max * max(H,W) * eps) whatever is done
                    // to it, and cannot move the partner: leave the pair (this is also what ends the sweeps on rank-deficient ReLU
                    // maps, whose null vectors are rounding noise that no rotation makes more orthogonal)
                    if (ok && al > RANK_NEGLIGIBLE * be && be > RANK_NEGLIGIBLE * al && fabsf(ga) > tol * (sqrtf(al) * sqrtf(be))) {
                        const float zeta = (be - al) / (2.f * ga);
                        float tn = copysignf(1.f, zeta) / (fabsf(zeta) + sqrtf(fmaf(zeta, zeta, 1.f)));
                        if (fabsf(zeta) > 1e15f) tn = 0.5f / zeta;
                        const float cs = 1.f / sqrtf(fmaf(tn, tn, 1.f)), sn = cs * tn;
                        float* wp = v + p * a.ld;
                        float* wq = v + q * a.ld;
#pragma unroll
                        for (int e = 0; e < RANK_EPT; ++e) {
                            const int i = l + (e << a.log2L);
                            if (i < a.m) {
                                wp[i] = fmaf(cs, xa[e], -sn * xb[e]);
                                wq[i] = fmaf(sn, xa[e], cs * xb[e]);
                            }
                        }
                        rotated = 1;
                    }
                }
                __syncthreads();
            }
            if (!__syncthreads_or(rotated)) break;
        }

        for (int j0 = 0; j0 < a.n; j0 += a.wpm) {           // singular values = norms of the orthogonalised vectors
            const int j = j0 + wk;
            const bool ok = live && j < a.n;
            float nn = 0.f;
            const float* vj = v + (ok ? j : 0) * a.ld;
#pragma unroll
            for (int e = 0; e < RANK_EPT; ++e) {
                const int i = l + (e << a.log2L);
                const float val = (ok && i < a.m) ? vj[i] : 0.f;
                nn = fmaf(val, val, nn);
            }
            for (int o = L >> 1; o > 0; o >>= 1) nn += __shfl_xor_sync(0xffffffffu, nn, o);
            if (ok && l == 0) sig[j] = sqrtf(nn);
        }
        __syncthreads();
        if (live && r == 0) {
            float smax = 0.f;
            for (int j = 0; j < a.n; ++j) smax = fmaxf(smax, sig[j]);
            const float cut = smax * static_cast<float>(a.H > a.W ? a.H : a.W) * FLT_EPSILON;   // torch.matrix_rank's default tol
            int rank = 0;
            for (int j = 0; j < a.n; ++j) rank += sig[j] > cut;
            const long long b = mi / a.c_count;
            const int c = static_cast<int>(mi - b * a.c_count);
            const double val = a.squared ? static_cast<double>(rank) * rank : static_cast<double>(rank);
            atomicAdd(a.accum + c, val);
            if (a.out) a.out[mi] = static_cast<float>(val);
        }
    }
}

// accum[0] += sum_j part[j]   (one CTA; the order is fixed, the result bit-reproducible)
__global__ void __launch_bounds__(256) sum_to_one_kernel(const double* __restrict__ part, int n, double* accum) {
    __shared__ double red[256];
    double s = 0.0;
    for (int j = threadIdx.x; j < n; j += 256) s += part[j];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *accum += red[0];
}

// per image: out[b] = sum_c energy[b, c]; accum[0] += sum_b out[b]   (one CTA per image)
__global__ void __launch_bounds__(256) dct3_reduce_kernel(const float* __restrict__ energy, int c_count, float* out, double* accum) {
    __shared__ double red[256];
    const float* e = energy + static_cast<long long>(blockIdx.x) * c_count;
    double s = 0.0;
    for (int j = threadIdx.x; j < c_count; j += 256) s += static_cast<double>(e[j]);
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[blockIdx.x] = static_cast<float>(red[0]);
        atomicAdd(accum, red[0]);
    }
}

}  // namespace dctp
