// Translation unit for the forward-mode (dual-number) backward of the elbow rollout (see cn_tangent.cu).
#include <cuda_runtime.h>

#include "../../include/dair_pll_b200.h"
#include "cn_elbow_tangent.cuh"
#include "cn_launch.cuh"

namespace {

template <typename T>
__global__ void __launch_bounds__(128)
elbow_rollout_grad_kernel(const T* __restrict__ x0, const T* __restrict__ inertia, const T* __restrict__ mu,
                          const T* __restrict__ half, const T* __restrict__ kin, T dt, T eps, int64_t B, int steps,
                          const T* __restrict__ xbar, T* __restrict__ gparams, T* __restrict__ gx0,
                          const T* __restrict__ usol) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * cn::ELBOW_NTAN) return;
  const int64_t b = t / cn::ELBOW_NTAN;
  const int dir = (int)(t % cn::ELBOW_NTAN);
  T in[20], m[2], h[6], k[12], xs[15];
  for (int i = 0; i < 20; ++i) in[i] = inertia[i];
  for (int i = 0; i < 2; ++i) m[i] = mu[i];
  for (int i = 0; i < 6; ++i) h[i] = half[i];
  for (int i = 0; i < 12; ++i) k[i] = kin[i];
  for (int i = 0; i < 15; ++i) xs[i] = x0[b * 15 + i];
  const T g = cn::elbow_rollout_tangent<T>(in, m, h, k, dt, eps, xs, steps, xbar + b * (int64_t)steps * 15, dir,
                                           usol ? usol + b * (int64_t)steps * 7 : (const T*)nullptr);
  if (dir < cn::ELBOW_NPARAM_TAN) gparams[b * cn::ELBOW_NPARAM_TAN + dir] = g;
  else gx0[b * 15 + (dir - cn::ELBOW_NPARAM_TAN)] = g;
}

// one (sample, direction) per thread; gparams (B, 22), gpts (B, 24), gx (B, 15)
template <typename T>
__global__ void __launch_bounds__(128)
elbow_step_pts_grad_kernel(const T* __restrict__ x, const T* __restrict__ inertia, const T* __restrict__ mu,
                           const T* __restrict__ kin, const T* __restrict__ pts, T dt, T eps, int64_t B,
                           const T* __restrict__ xbar, T* __restrict__ gparams, T* __restrict__ gpts, T* __restrict__ gx,
                           const T* __restrict__ usol) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * cn::ELBOW_PTS_NTAN) return;
  const int64_t b = t / cn::ELBOW_PTS_NTAN;
  const int dir = (int)(t % cn::ELBOW_PTS_NTAN);
  T in[20], m[2], k[12], xs[15], p[24], xb[15];
  for (int i = 0; i < 20; ++i) in[i] = inertia[i];
  for (int i = 0; i < 2; ++i) m[i] = mu[i];
  for (int i = 0; i < 12; ++i) k[i] = kin[i];
  for (int i = 0; i < 15; ++i) { xs[i] = x[b * 15 + i]; xb[i] = xbar[b * 15 + i]; }
  for (int i = 0; i < 24; ++i) p[i] = pts[b * 24 + i];
  const T g = cn::elbow_step_pts_tangent<T>(in, m, k, dt, eps, xs, p, xb, dir, usol ? usol + b * 7 : (const T*)nullptr);
  if (dir < cn::ELBOW_PTS_NPARAM) gparams[b * cn::ELBOW_PTS_NPARAM + dir] = g;
  else if (dir < cn::ELBOW_PTS_NPARAM + 24) gpts[b * 24 + (dir - cn::ELBOW_PTS_NPARAM)] = g;
  else gx[b * 15 + (dir - cn::ELBOW_PTS_NPARAM - 24)] = g;
}

}  // namespace

extern "C" {

int dpll_elbow_step_pts_grad_f64(const double* x, const double* inertia, const double* mu_pair, const double* kin,
                                 const double* pts, const double* usol, double dt, double eps, int64_t B,
                                 const double* xbar, double* gparams, double* gpts, double* gx, void* stream) {
  if (B < 0 || !inertia || !mu_pair || !kin) return DPLL_EINVAL;
  if (B > 0 && (!x || !pts || !xbar || !gparams || !gpts || !gx)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  elbow_step_pts_grad_kernel<double><<<cn::grid_for(B * cn::ELBOW_PTS_NTAN, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      x, inertia, mu_pair, kin, pts, dt, eps, B, xbar, gparams, gpts, gx, usol);
  return cn::launch_status();
}


int dpll_elbow_rollout_grad_saved_f64(const double* x0, const double* inertia, const double* mu_pair, const double* half,
                                      const double* kin, const double* usol, double dt, double eps, int64_t B,
                                      int32_t steps, const double* xbar, double* gparams, double* gx0, void* stream) {
  if (B < 0 || steps < 0 || !inertia || !mu_pair || !half || !kin) return DPLL_EINVAL;
  if (B > 0 && (!x0 || !xbar || !gparams || !gx0)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  elbow_rollout_grad_kernel<double><<<cn::grid_for(B * cn::ELBOW_NTAN, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      x0, inertia, mu_pair, half, kin, dt, eps, B, steps, xbar, gparams, gx0, usol);
  return cn::launch_status();
}

}  // extern "C"
