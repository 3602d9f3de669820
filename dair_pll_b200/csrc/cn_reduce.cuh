// Fixed-order reductions shared by the loss kernels of the box (cn_kernels.cu) and of the two-body tree (cn_elbow_wf.cu).
#pragma once

#include <cuda_runtime.h>
#include <cstdint>

namespace {

template <typename T> __device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Fixed-order reduction of the per-block partials: warp w owns accumulator w.
// NACC accumulators per block: [0, NPARAM) parameter gradients, slot NPARAM = loss sum.
template <typename T, typename IO, int NACC, int NPARAM>
__global__ void reduce_partials_kernel(const T* __restrict__ partials, int nblocks, IO* __restrict__ grad,
                                       IO* __restrict__ loss_sum, const int32_t* __restrict__ skip_flag) {
  if (skip_flag && *skip_flag) return;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (w >= NACC) return;
  T s = T(0);
  for (int b = lane; b < nblocks; b += 32) s += partials[(int64_t)b * NACC + w];
  s = warp_sum(s);
  if (lane == 0) {
    if (w < NPARAM) { if (grad) grad[w] = IO(s); }
    else if (w == NPARAM) { if (loss_sum) *loss_sum = IO(s); }
  }
}

}  // namespace
