// Separate translation unit for the forward-mode (dual-number) backward of the cube rollout: the dual
// instantiation of the step code is large and compiles slowly, so it is built in parallel with
// cn_kernels.cu and linked into the same library.
#include <cuda_runtime.h>

#include "../../include/dair_pll_b200.h"
#include "cn_cube_tangent.cuh"
#include "cn_launch.cuh"

namespace {

// Backward of the cube rollout: forward-mode tangents (cn_cube_tangent.cuh), one (toss, direction) pair
// per thread.  Used for the prediction-loss path where batches are small (experiment.py:230-248).
template <typename T>
__global__ void __launch_bounds__(128)
cube_rollout_grad_kernel(const T* __restrict__ x0, const T* __restrict__ inertia, const T* __restrict__ mu,
                         const T* __restrict__ half, T dt, T eps, int64_t B, int steps, const T* __restrict__ xbar,
                         T* __restrict__ gparams, T* __restrict__ gx0) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * cn::CUBE_NTAN) return;
  const int64_t b = t / cn::CUBE_NTAN;
  const int dir = (int)(t % cn::CUBE_NTAN);
  T in[10], m[1], h[3], xs[13];
  for (int i = 0; i < 10; ++i) in[i] = inertia[i];
  m[0] = mu[0];
  for (int i = 0; i < 3; ++i) h[i] = half[i];
  for (int i = 0; i < 13; ++i) xs[i] = x0[b * 13 + i];
  const T g = cn::cube_rollout_tangent<T>(in, m, h, dt, eps, xs, steps, xbar + b * (int64_t)steps * 13, dir);
  if (dir < 14) gparams[b * 14 + dir] = g;
  else gx0[b * 13 + (dir - 14)] = g;
}

template <typename T>
int launch_cube_rollout_grad(const T* x0, const T* inertia, const T* mu, const T* half, T dt, T eps, int64_t B,
                             int32_t steps, const T* xbar, T* gparams, T* gx0, void* stream) {
  if (B < 0 || steps < 0 || !inertia || !mu || !half) return DPLL_EINVAL;
  if (B > 0 && (!x0 || !xbar || !gparams || !gx0)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  cube_rollout_grad_kernel<T><<<cn::grid_for(B * cn::CUBE_NTAN, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(x0, inertia, mu, half, dt, eps, B, steps,
                                                                                  xbar, gparams, gx0);
  return cn::launch_status();
}

// backward of one witness-point step: one (sample, direction) pair per thread; gparams (B, 11), gpts (B, 12), gx (B, 13)
template <typename T>
__global__ void __launch_bounds__(128)
body_step_pts_grad_kernel(const T* __restrict__ x, const T* __restrict__ inertia, const T* __restrict__ mu,
                          const T* __restrict__ pts, int n_c, T dt, T eps, int64_t B, const T* __restrict__ xbar,
                          T* __restrict__ gparams, T* __restrict__ gpts, T* __restrict__ gx) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * cn::BODY_PTS_NTAN) return;
  const int64_t b = t / cn::BODY_PTS_NTAN;
  const int dir = (int)(t % cn::BODY_PTS_NTAN);
  T in[10], m[1], xs[13], p[12], xb[13];
  for (int i = 0; i < 10; ++i) in[i] = inertia[i];
  m[0] = mu[0];
  for (int i = 0; i < 13; ++i) { xs[i] = x[b * 13 + i]; xb[i] = xbar[b * 13 + i]; }
  for (int i = 0; i < 12; ++i) p[i] = pts[b * 12 + i];
  const T g = cn::body_step_pts_tangent<T>(in, m, dt, eps, xs, p, n_c, xb, dir);
  if (dir < 11) gparams[b * 11 + dir] = g;
  else if (dir < 23) gpts[b * 12 + (dir - 11)] = g;
  else gx[b * 13 + (dir - 23)] = g;
}

}  // namespace

extern "C" {

int dpll_body_step_pts_grad_f64(const double* x, const double* inertia, const double* mu_pair, const double* pts,
                                int32_t n_contacts, double dt, double eps, int64_t B, const double* xbar,
                                double* gparams, double* gpts, double* gx, void* stream) {
  if (B < 0 || !inertia || !mu_pair || n_contacts < 0 || n_contacts > 4) return DPLL_EINVAL;
  if (B > 0 && (!x || !pts || !xbar || !gparams || !gpts || !gx)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  body_step_pts_grad_kernel<double><<<cn::grid_for(B * cn::BODY_PTS_NTAN, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      x, inertia, mu_pair, pts, n_contacts, dt, eps, B, xbar, gparams, gpts, gx);
  return cn::launch_status();
}

int dpll_cube_rollout_grad_f64(const double* x0, const double* inertia, const double* mu_pair, const double* half,
                               double dt, double eps, int64_t B, int32_t steps, const double* xbar, double* gparams,
                               double* gx0, void* stream) {
  return launch_cube_rollout_grad<double>(x0, inertia, mu_pair, half, dt, eps, B, steps, xbar, gparams, gx0,
                                                  stream);
}

}  // extern "C"
