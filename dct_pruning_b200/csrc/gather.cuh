// Pruned-weight gather: the step right after top-k (SURVEY 8f-1).
//
// The reference copies kept filters into the pruned model one (out, in) pair at a time in Python:
//   for index_i, i in enumerate(select_index):
//       for index_j, j in enumerate(last_select_index):
//           state_dict[name][index_i][index_j] = oristate_dict[name][i][j]
// (/root/reference/utils/load_models.py:43-51 vgg, :106-114 resnet_56/110, :482-500 and :526-542 resnet_50 incl. the
// BatchNorm vectors, :633-639 u2netp ...), O(k_out * k_in) tensor assignments per convolution.  Here it is one launch:
//   out[i][j][r] = w[ sel_out ? sel_out[i] : i ][ sel_in ? sel_in[j] : j ][r],   r < inner (kH*kW, or 1 for vectors)
// Pure data movement: 4 * k_out * k_in * inner bytes written, the same amount read (gathered in runs of `inner`).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace dctp {

constexpr int GATHER_THREADS = 256;
enum : int { DCTP_DEV_BAD_INDEX = 3 };         // (continues DCTP_DEV_* of score_common.cuh)

struct GatherArgs {
    const float* w;                 // [c_out][c_in][inner]
    float* out;                     // [k_out][k_in][inner]
    const long long* sel_out;       // kept output channels (ascending ids) or nullptr = identity
    const long long* sel_in;        // kept input channels or nullptr = identity
    int c_out, c_in, inner, k_out, k_in;
    long long total;                // k_out * k_in * inner
    int* status;
};

__global__ void __launch_bounds__(GATHER_THREADS) gather_weight_kernel(const GatherArgs a) {
    const long long stride = static_cast<long long>(gridDim.x) * GATHER_THREADS;
    const int row = a.k_in * a.inner;           // elements per output filter
    for (long long e = static_cast<long long>(blockIdx.x) * GATHER_THREADS + threadIdx.x; e < a.total; e += stride) {
        const int i = static_cast<int>(e / row);
        const int rem = static_cast<int>(e - static_cast<long long>(i) * row);
        const int j = rem / a.inner, r = rem - j * a.inner;
        const long long si = a.sel_out ? a.sel_out[i] : i;
        const long long sj = a.sel_in ? a.sel_in[j] : j;
        if (si < 0 || si >= a.c_out || sj < 0 || sj >= a.c_in) {
            atomicExch(a.status, DCTP_DEV_BAD_INDEX);
            continue;
        }
        a.out[e] = __ldg(a.w + (si * a.c_in + sj) * a.inner + r);
    }
}

}  // namespace dctp
