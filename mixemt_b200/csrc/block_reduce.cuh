// Warp- and block-wide reductions of doubles in a fixed order (deterministic), shared by the
// EM kernels (em_kernels.cuh) and the log-likelihood kernel (loglik.cu).
#pragma once

namespace mxb {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}

// Block-wide deterministic reductions (every thread gets the result).
template <int kThreads>
__device__ __forceinline__ double block_sum(double v, double *scratch /*[kThreads/32]*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();  // scratch free
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < kThreads / 32; ++i) t += scratch[i];
    return t;
}
template <int kThreads>
__device__ __forceinline__ double block_max(double v, double *scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_max(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    double t = scratch[0];
#pragma unroll
    for (int i = 1; i < kThreads / 32; ++i) t = fmax(t, scratch[i]);
    return t;
}

}  // namespace mxb
