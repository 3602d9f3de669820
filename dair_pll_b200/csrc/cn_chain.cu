// Kernels of the generic floating-base serial chain (cn_chain.cuh; SURVEY.md section 8(f) N2, first slice): one sample
// per thread, N = 2 .. 4 links.  The general path for models the specialised kernels do not cover.
#include <cuda_runtime.h>

#include "../../include/dair_pll_b200.h"
#include "cn_chain.cuh"
#include "cn_launch.cuh"

namespace {

constexpr int kChThreads = 64;
constexpr int kChNAcc = 96;                 // 14 N parameter gradients + loss sum (N <= 6: 85)
constexpr int kChMaxBlocks = 148 * 5;
static_assert((size_t)kChMaxBlocks * kChNAcc * sizeof(double) <= cn::kWsPartialsBytes, "chain partials exceed the workspace");

template <typename T> __device__ __forceinline__ T ch_warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T, int N>
__global__ void __launch_bounds__(kChThreads)
chain_loss_kernel(const T* __restrict__ x, const T* __restrict__ xp, const T* __restrict__ weight,
                  const T* __restrict__ inertia, const T* __restrict__ mu, const T* __restrict__ half,
                  const T* __restrict__ kin, T dt, T eps, int64_t B, T* __restrict__ loss, T* __restrict__ force,
                  int32_t* __restrict__ iters, T* __restrict__ partials, int want_grad,
                  const T* __restrict__ pts = nullptr, unsigned npts = 0u, T* __restrict__ grad_pts = nullptr) {
  // pts (nullable, (B, N, 4, 3)): witness points per box slot instead of box corners (half is then unused and may be
  // null); grad_pts (nullable, same shape): w_b d loss_b / d pts_b
  constexpr int NX = 13 + 2 * (N - 1), NP = 14 * N, NF = 12 * N;
  cn::ChainParams<T, N> P;
  cn::chain_params_init<T, N>(P, inertia, mu, half, kin, dt, eps);
  const cn::SolverCfg<T> cfg = cn::default_cfg<T>();
  T acc[NP + 1];
  for (int i = 0; i <= NP; ++i) acc[i] = T(0);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += stride) {
    T xs[NX], xps[NX], gs[NP], fo[NF];
    for (int i = 0; i < NX; ++i) { xs[i] = x[b * NX + i]; xps[i] = xp[b * NX + i]; }
    for (int i = 0; i < NP; ++i) gs[i] = T(0);
    int it;
    T ps[12 * N], gps[12 * N];
    if (pts) for (int i = 0; i < 12 * N; ++i) ps[i] = pts[b * 12 * N + i];
    const T l = cn::chain_loss_sample<T, N>(P, cfg, xs, xps, (want_grad || grad_pts) ? gs : (T*)nullptr, force ? fo : (T*)nullptr, &it,
                                            pts ? ps : (const T*)nullptr, npts, grad_pts ? gps : (T*)nullptr);
    if (force) for (int i = 0; i < NF; ++i) force[b * NF + i] = fo[i];
    const T w = weight ? weight[b] : T(1);
    if (grad_pts) for (int i = 0; i < 12 * N; ++i) grad_pts[b * 12 * N + i] = w * gps[i];
    for (int i = 0; i < NP; ++i) acc[i] += w * gs[i];
    if (loss) loss[b] = l;
    acc[NP] += l;
    if (iters) iters[b] = it;
  }
  if (!partials) return;
  __shared__ T red[kChThreads / 32][kChNAcc];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = 0; i <= NP; ++i) {
    const T s = ch_warp_sum(acc[i]);
    if (lane == 0) red[warp][i] = s;
  }
  __syncthreads();
  for (int i = threadIdx.x; i <= NP; i += kChThreads) {
    T s = T(0);
    for (int w = 0; w < kChThreads / 32; ++w) s += red[w][i];
    partials[(int64_t)blockIdx.x * kChNAcc + i] = s;
  }
}

template <typename T>
__global__ void chain_reduce_kernel(const T* __restrict__ partials, int nblocks, int nparam, T* __restrict__ grad,
                                    T* __restrict__ loss_sum) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int a = w; a <= nparam; a += blockDim.x >> 5) {
    T s = T(0);
    for (int b = lane; b < nblocks; b += 32) s += partials[(int64_t)b * kChNAcc + a];
    s = ch_warp_sum(s);
    if (lane == 0) {
      if (a < nparam) { if (grad) grad[a] = s; }
      else if (loss_sum) *loss_sum = s;
    }
  }
}

template <typename T, int N>
__global__ void __launch_bounds__(kChThreads)
chain_rollout_kernel(const T* __restrict__ x0, const T* __restrict__ inertia, const T* __restrict__ mu,
                     const T* __restrict__ half, const T* __restrict__ kin, T dt, T eps, int64_t B, int steps,
                     T* __restrict__ traj) {
  constexpr int NX = 13 + 2 * (N - 1);
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  cn::ChainParams<T, N> P;
  cn::chain_params_init<T, N>(P, inertia, mu, half, kin, dt, eps);
  const cn::SolverCfg<T> cfg = cn::default_cfg<T>();
  T xc[NX], xn[NX];
  T* out = traj + b * (int64_t)(steps + 1) * NX;
  for (int i = 0; i < NX; ++i) { xc[i] = x0[b * NX + i]; out[i] = xc[i]; }
  for (int s = 0; s < steps; ++s) {
    cn::chain_step_sample<T, N>(P, cfg, xc, xn);
    for (int i = 0; i < NX; ++i) { xc[i] = xn[i]; out[(int64_t)(s + 1) * NX + i] = xn[i]; }
  }
}

template <int N>
int launch_chain_loss(const double* x, const double* xp, const double* weight, const double* inertia, const double* mu,
                      const double* half, const double* kin, double dt, double eps, int64_t B, double* loss, double* force,
                      int32_t* iters, double* grad, double* loss_sum, void* workspace, size_t workspace_bytes,
                      cudaStream_t st, const double* pts = nullptr, unsigned npts = 0u, double* grad_pts = nullptr) {
  const bool want_red = grad || loss_sum;
  if (want_red && !cn::workspace_ok(workspace, workspace_bytes)) return DPLL_EWORKSPACE;
  int64_t need = (B + kChThreads - 1) / kChThreads;
  int blocks = (int)(need < kChMaxBlocks ? need : kChMaxBlocks);
  if (blocks < 1) blocks = 1;
  double* partials = want_red ? static_cast<double*>(workspace) : nullptr;
  chain_loss_kernel<double, N><<<blocks, kChThreads, 0, st>>>(x, xp, weight, inertia, mu, half, kin, dt, eps, B, loss, force,
                                                             iters, partials, grad ? 1 : 0, pts, npts, grad_pts);
  if (int rc = cn::launch_status()) return rc;
  if (!want_red) return DPLL_OK;
  chain_reduce_kernel<double><<<1, 512, 0, st>>>(partials, blocks, 14 * N, grad, loss_sum);
  return cn::launch_status();
}

// Dense terms export (MultibodyTerms.forward, multibody_terms.py:584-609) for a tree; one sample per thread.
template <typename T, int N>
__global__ void __launch_bounds__(kChThreads)
chain_terms_kernel(const T* __restrict__ q, const T* __restrict__ v, const T* __restrict__ inertia, const T* __restrict__ mu,
                   const T* __restrict__ half, const T* __restrict__ kin, int n_boxes, int64_t B, T* __restrict__ M,
                   T* __restrict__ J, T* __restrict__ phi, T* __restrict__ acc, T* __restrict__ D) {
  constexpr int NV = 6 + N - 1, NQ = 7 + N - 1;
  cn::ChainParams<T, N> P;
  cn::chain_params_init<T, N>(P, inertia, mu, half, kin, T(1), T(1));
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int nc = 4 * n_boxes, kk = 3 * nc;
  T qs[NQ], vs[NV];
  for (int i = 0; i < NQ; ++i) qs[i] = q[b * NQ + i];
  for (int i = 0; i < NV; ++i) vs[i] = v[b * NV + i];
  // outputs are assembled in place (global memory): M, J and D are this sample's own rows
  cn::chain_terms_sample<T, N>(P, qs, vs, n_boxes, M + b * NV * NV, J + b * kk * NV, phi + b * nc, acc + b * NV,
                               D ? D + b * kk * kk : (T*)nullptr);
}

}  // namespace

extern "C" {

int dpll_chain_loss_f64(int32_t n_links, const double* x, const double* x_plus, const double* weight, const double* inertia,
                        const double* mu_pair, const double* half, const double* kin, double dt, double eps, int64_t B,
                        double* loss, double* force, int32_t* iters, double* grad, double* loss_sum, void* workspace,
                        size_t workspace_bytes, void* stream) {
  if (B < 0 || !inertia || !mu_pair || !half || !kin) return DPLL_EINVAL;
  if (B > 0 && (!x || !x_plus)) return DPLL_EINVAL;
  return cn::with_links(n_links, [&](auto N) {
    return launch_chain_loss<N>(x, x_plus, weight, inertia, mu_pair, half, kin, dt, eps, B, loss, force, iters, grad,
                                loss_sum, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
  });
}

int dpll_chain_rollout_f64(int32_t n_links, const double* x0, const double* inertia, const double* mu_pair,
                           const double* half, const double* kin, double dt, double eps, int64_t B, int32_t steps,
                           double* traj, void* stream) {
  if (B < 0 || steps < 0 || !inertia || !mu_pair || !half || !kin) return DPLL_EINVAL;
  if (B > 0 && (!x0 || !traj)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  return cn::with_links(n_links, [&](auto N) {
    chain_rollout_kernel<double, N><<<cn::grid_for(B, kChThreads), kChThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        x0, inertia, mu_pair, half, kin, dt, eps, B, steps, traj);
    return cn::launch_status();
  });
}

int dpll_chain_terms_f64(int32_t n_links, int32_t n_boxes, const double* q, const double* v, const double* inertia,
                         const double* mu_pair, const double* half, const double* kin, int64_t B, double* M, double* J,
                         double* phi, double* acc, double* delassus, void* stream) {
  if (B < 0 || n_boxes < 1 || n_boxes > n_links || !inertia || !mu_pair || !half || !kin) return DPLL_EINVAL;
  if (B > 0 && (!q || !v || !M || !J || !phi || !acc)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  return cn::with_links(n_links, [&](auto N) {
    chain_terms_kernel<double, N><<<cn::grid_for(B, kChThreads), kChThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        q, v, inertia, mu_pair, half, kin, n_boxes, B, M, J, phi, acc, delassus);
    return cn::launch_status();
  });
}

int dpll_chain_loss_pts_f64(int32_t n_links, const double* x, const double* x_plus, const double* weight, const double* inertia,
                            const double* mu_pair, const double* kin, const double* pts, uint32_t n_pts_packed, double dt,
                            double eps, int64_t B, double* loss, double* grad_pts, double* grad, double* loss_sum,
                            void* workspace, size_t workspace_bytes, void* stream) {
  if (B < 0 || !inertia || !mu_pair || !kin) return DPLL_EINVAL;
  if (B > 0 && (!x || !x_plus || !pts)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  return cn::with_links(n_links, [&](auto N) {
    return launch_chain_loss<N>(x, x_plus, weight, inertia, mu_pair, nullptr, kin, dt, eps, B, loss, nullptr, nullptr, grad,
                                loss_sum, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), pts, n_pts_packed,
                                grad_pts);
  });
}

}  // extern "C"
