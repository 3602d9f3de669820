// Parameter preparation of ANY system as two tiny launches (forward, chain rule) instead of ~100 PyTorch glue kernels:
//   theta (n_bodies, 10)      -> [m, c, I_cm / m] per body   (inertia.py:205-234, 304-331, 376-382; multibody_terms.py:230-231)
//   friction_params (n_geoms) -> |.| -> 2 mu_a mu_b / (mu_a + mu_b) per collision pair   (multibody_terms.py:321-324, 466-471)
//   length_params (n_len)     -> |.|                                                      (geometry.py:394-397)
// The single floating box has this fused into its training entry point (cube_prep_kernel / reduce_partials_leaf_kernel,
// cn_kernels.cu); the two-body tree and the generic chains go through these two kernels (dair_pll_b200/ops.py:LeafPrepare),
// which is what took their CUDA-graph-replayed step from "kernel + 0.4 ms of glue" to "kernel + two launches".
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/dair_pll_b200.h"
#include "cn_params.cuh"
#include "cn_launch.cuh"

namespace {

__device__ __forceinline__ double sign0(double v) { return v > 0 ? 1.0 : (v < 0 ? -1.0 : 0.0); }   // d|v|/dv, 0 at 0 (as torch)

__global__ void leaf_prepare_kernel(const double* __restrict__ theta, int n_bodies, const double* __restrict__ friction,
                                    const int32_t* __restrict__ pair_a, const int32_t* __restrict__ pair_b, int n_pairs,
                                    const double* __restrict__ length, int n_len, double* __restrict__ inertia,
                                    double* __restrict__ mu, double* __restrict__ half) {
  const int t = threadIdx.x;
  for (int b = t; b < n_bodies; b += blockDim.x) {
    double th[10], out[10];
    for (int i = 0; i < 10; ++i) th[i] = theta[10 * b + i];
    cn::theta_to_inertia_vector<double>(th, out);
    for (int i = 0; i < 10; ++i) inertia[10 * b + i] = out[i];
  }
  for (int p = t; p < n_pairs; p += blockDim.x) {
    const double a = fabs(friction[pair_a[p]]), b = fabs(friction[pair_b[p]]);
    mu[p] = 2.0 * a * b / (a + b);
  }
  for (int i = t; i < n_len; i += blockDim.x) half[i] = fabs(length[i]);
}

__global__ void leaf_backward_kernel(const double* __restrict__ theta, int n_bodies, const double* __restrict__ friction,
                                     int n_geoms, const int32_t* __restrict__ pair_a, const int32_t* __restrict__ pair_b,
                                     int n_pairs, const double* __restrict__ length, int n_len,
                                     const double* __restrict__ g_inertia, const double* __restrict__ g_mu,
                                     const double* __restrict__ g_half, double* __restrict__ g_theta,
                                     double* __restrict__ g_friction, double* __restrict__ g_length) {
  const int t = threadIdx.x;
  // one (body, theta component) per thread: a dual number through the same templated map (10 x 10 Jacobian)
  for (int idx = t; idx < 10 * n_bodies; idx += blockDim.x) {
    const int b = idx / 10, i = idx % 10;
    cn::Dual<double> th[10], out[10];
    for (int j = 0; j < 10; ++j) th[j] = cn::Dual<double>(theta[10 * b + j], j == i ? 1.0 : 0.0);
    cn::theta_to_inertia_vector<cn::Dual<double>>(th, out);
    double s = 0;
    for (int o = 0; o < 10; ++o) s += (g_inertia ? g_inertia[10 * b + o] : 0.0) * out[o].d;
    g_theta[idx] = s;
  }
  for (int g = t; g < n_geoms; g += blockDim.x) {
    double acc = 0;
    for (int p = 0; p < n_pairs && g_mu; ++p) {
      const double a = fabs(friction[pair_a[p]]), b = fabs(friction[pair_b[p]]);
      const double inv = 1.0 / ((a + b) * (a + b));
      if (pair_a[p] == g) acc += g_mu[p] * 2.0 * b * b * inv;
      if (pair_b[p] == g) acc += g_mu[p] * 2.0 * a * a * inv;
    }
    g_friction[g] = acc * sign0(friction[g]);
  }
  for (int i = t; i < n_len; i += blockDim.x) g_length[i] = (g_half ? g_half[i] : 0.0) * sign0(length[i]);
}

}  // namespace

extern "C" {

int dpll_leaf_prepare_f64(const double* theta, int32_t n_bodies, const double* friction, const int32_t* pair_a,
                          const int32_t* pair_b, int32_t n_pairs, const double* length, int32_t n_len, double* inertia,
                          double* mu, double* half, void* stream) {
  if (n_bodies < 0 || n_pairs < 0 || n_len < 0) return DPLL_EINVAL;
  if ((n_bodies && (!theta || !inertia)) || (n_pairs && (!friction || !pair_a || !pair_b || !mu)) || (n_len && (!length || !half)))
    return DPLL_EINVAL;
  leaf_prepare_kernel<<<1, 64, 0, static_cast<cudaStream_t>(stream)>>>(theta, n_bodies, friction, pair_a, pair_b, n_pairs,
                                                                     length, n_len, inertia, mu, half);
  return cn::launch_status();
}

int dpll_leaf_backward_f64(const double* theta, int32_t n_bodies, const double* friction, int32_t n_geoms,
                           const int32_t* pair_a, const int32_t* pair_b, int32_t n_pairs, const double* length, int32_t n_len,
                           const double* g_inertia, const double* g_mu, const double* g_half, double* g_theta,
                           double* g_friction, double* g_length, void* stream) {
  if (n_bodies < 0 || n_geoms < 0 || n_pairs < 0 || n_len < 0) return DPLL_EINVAL;
  if ((n_bodies && (!theta || !g_theta)) || (n_geoms && (!friction || !g_friction)) || (n_pairs && (!pair_a || !pair_b)) ||
      (n_len && (!length || !g_length)))
    return DPLL_EINVAL;
  leaf_backward_kernel<<<1, 64, 0, static_cast<cudaStream_t>(stream)>>>(theta, n_bodies, friction, n_geoms, pair_a, pair_b,
                                                                      n_pairs, length, n_len, g_inertia, g_mu, g_half,
                                                                      g_theta, g_friction, g_length);
  return cn::launch_status();
}

}  // extern "C"
