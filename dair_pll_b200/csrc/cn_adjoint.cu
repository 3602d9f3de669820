// Reverse-mode backward of the cube rollout (cn_cube_adjoint.cuh): one toss per thread walks its trajectory
// backwards, one 6x6 SPD solve per step.  Separate translation unit (compiled in parallel with the others).
#include <cuda_runtime.h>

#include "../../include/dair_pll_b200.h"
#include "cn_cube_adjoint.cuh"
#include "cn_launch.cuh"

namespace {

template <typename T>
__global__ void __launch_bounds__(64)
cube_rollout_backward_kernel(const T* __restrict__ traj, const T* __restrict__ usol, const T* __restrict__ inertia,
                             const T* __restrict__ mu, const T* __restrict__ half, T dt, T eps, int64_t B, int steps,
                             const T* __restrict__ xbar, T* __restrict__ gparams, T* __restrict__ gx0) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  T in[10], m[1], h[3];
  for (int i = 0; i < 10; ++i) in[i] = inertia[i];
  m[0] = mu[0];
  for (int i = 0; i < 3; ++i) h[i] = half[i];
  cn::CubeParams<T> P;
  cn::cube_params_init(P, in, m, h, dt, eps);
  T gp[cn::CUBE_NPARAM], g0[13];
  cn::cube_rollout_backward_sample<T>(P, traj + b * (int64_t)(steps + 1) * 13, usol + b * (int64_t)steps * 6,
                                      xbar + b * (int64_t)steps * 13, steps, gp, g0);
  for (int i = 0; i < cn::CUBE_NPARAM; ++i) gparams[b * cn::CUBE_NPARAM + i] = gp[i];
  for (int i = 0; i < 13; ++i) gx0[b * 13 + i] = g0[i];
}

}  // namespace

extern "C" {

int dpll_cube_rollout_backward_f64(const double* traj, const double* usol, const double* inertia, const double* mu_pair,
                                   const double* half, double dt, double eps, int64_t B, int32_t steps, const double* xbar,
                                   double* gparams, double* gx0, void* stream) {
  if (B < 0 || steps < 0 || !inertia || !mu_pair || !half) return DPLL_EINVAL;
  if (B > 0 && (!traj || !gparams || !gx0 || (steps > 0 && (!usol || !xbar)))) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  // a toss is one sequential chain: spread the tosses over as many warps as there are (2 per warp at 4,096 tosses)
  cube_rollout_backward_kernel<double><<<cn::grid_for(B, 64), 64, 0, static_cast<cudaStream_t>(stream)>>>(
      traj, usol, inertia, mu_pair, half, dt, eps, B, steps, xbar, gparams, gx0);
  return cn::launch_status();
}

}  // extern "C"
