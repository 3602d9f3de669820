// Translation unit for the forward-mode (dual-number) backward of the generic chain rollout (see cn_tangent.cu).
#include <cuda_runtime.h>

#include "../../include/dair_pll_b200.h"
#include "cn_chain_tangent.cuh"
#include "cn_launch.cuh"

namespace {

// one (toss, direction) pair per thread; gparams (B, 14 N), gx0 (B, NX)
template <typename T, int N>
__global__ void __launch_bounds__(64)
chain_rollout_grad_kernel(const T* __restrict__ x0, const T* __restrict__ inertia, const T* __restrict__ mu,
                          const T* __restrict__ half, const T* __restrict__ kin, T dt, T eps, int64_t B, int steps,
                          const T* __restrict__ xbar, T* __restrict__ gparams, T* __restrict__ gx0) {
  constexpr int NX = 13 + 2 * (N - 1), NP = 14 * N, NTAN = NP + NX;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * NTAN) return;
  const int64_t b = t / NTAN;
  const int dir = (int)(t % NTAN);
  const T g = cn::chain_rollout_tangent<T, N>(inertia, mu, half, kin, dt, eps, x0 + b * NX, steps,
                                              xbar + b * (int64_t)steps * NX, dir);
  if (dir < NP) gparams[b * NP + dir] = g;
  else gx0[b * NX + (dir - NP)] = g;
}

}  // namespace

extern "C" {

int dpll_chain_rollout_grad_f64(int32_t n_links, const double* x0, const double* inertia, const double* mu_pair,
                                const double* half, const double* kin, double dt, double eps, int64_t B, int32_t steps,
                                const double* xbar, double* gparams, double* gx0, void* stream) {
  if (B < 0 || steps < 0 || !inertia || !mu_pair || !half || !kin) return DPLL_EINVAL;
  if (B > 0 && (!x0 || !xbar || !gparams || !gx0)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  return cn::with_links(n_links, [&](auto N) {
    constexpr int NTAN = 14 * N + 13 + 2 * (N - 1);       // (toss, direction) pairs per toss
    chain_rollout_grad_kernel<double, N><<<cn::grid_for(B * NTAN, 64), 64, 0, static_cast<cudaStream_t>(stream)>>>(
        x0, inertia, mu_pair, half, kin, dt, eps, B, steps, xbar, gparams, gx0);
    return cn::launch_status();
  });
}

}  // extern "C"
