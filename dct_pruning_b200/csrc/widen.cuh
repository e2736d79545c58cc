// 16-bit activations on the kernels without a 16-bit variant: the scored window of a bf16 / fp16 activation is widened into a dense
// fp32 copy (scratch on the caller's stream), and the fp32 kernels score that copy.  Only the stacked-basis and Kronecker kernels read
// 16-bit input themselves (score_stack.cuh, score_kron.cuh).
#pragma once
#include "score_stack.cuh"

namespace dctp {

struct WidenArgs {
    const uint16_t* x;                       // element (b, c, h, w) at x[b*stride_b + c*stride_c + h*stride_h + w]
    long long stride_b, stride_c, stride_h;
    int c_begin, c_count, H, W;
    long long rows;                          // B * c_count * H
    float* out;                              // dense [B, c_count, H, W]
};

// one warp per map row (the row's index is divided once, its elements are read with unit stride)
template <int IN>
__global__ void __launch_bounds__(256) widen_window_kernel(const WidenArgs a) {
    const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    for (long long r = static_cast<long long>(blockIdx.x) * warps + (threadIdx.x >> 5); r < a.rows; r += static_cast<long long>(gridDim.x) * warps) {
        const long long bc = r / a.H, b = bc / a.c_count;
        const int h = static_cast<int>(r - bc * a.H), j = static_cast<int>(bc - b * a.c_count);
        const uint16_t* src = a.x + b * a.stride_b + (a.c_begin + j) * a.stride_c + h * a.stride_h;
        float* dst = a.out + r * a.W;
        for (int w = lane; w < a.W; w += 32) dst[w] = in16_to_float<IN>(src, w);
    }
}

}  // namespace dctp
