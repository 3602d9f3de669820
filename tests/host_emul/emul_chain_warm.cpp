// Host build of the warm-started tree loss (dair_pll_b200/csrc/cn_chain.cuh: chain_loss_sample with a start point u0 and
// the optimum u_opt), per sample as the warm instance of chain_loss_kernel runs it.
// TEST INFRASTRUCTURE ONLY: nothing in the package loads this; tests/test_chain_warm_host.py builds it.
#include "../../dair_pll_b200/csrc/cn_chain.cuh"
#include <cstdint>
using namespace cn;

template <int N>
static int chain_warm(const double* x, const double* xp, const double* inertia, const double* mu, const double* half,
                      const double* kin, const double* pts, unsigned npts, double dt, double eps, int64_t B,
                      const double* u_init, double* u_out, double* loss, double* grad, double* grad_pts, int32_t* iters) {
  constexpr int NX = 13 + 2 * (N - 1), NV = 5 + N;
  ChainParams<double, N> P;
  chain_params_init<double, N>(P, inertia, mu, half, kin, dt, eps);
  const SolverCfg<double> cfg = default_cfg<double>();
  for (int i = 0; i < 14 * N; ++i) grad[i] = 0;
  for (int64_t b = 0; b < B; ++b) {
    int it;
    double u0[NV], uo[NV];
    if (u_init) for (int i = 0; i < NV; ++i) u0[i] = u_init[NV * b + i];
    loss[b] = chain_loss_sample<double, N>(P, cfg, x + NX * b, xp + NX * b, grad, nullptr, &it,
                                           pts ? pts + 12 * N * b : nullptr, npts, pts ? grad_pts + 12 * N * b : nullptr,
                                           u_init ? u0 : nullptr, u_out ? uo : nullptr);
    if (u_out) for (int i = 0; i < NV; ++i) u_out[NV * b + i] = uo[i];
    if (iters) iters[b] = it;
  }
  return 0;
}

extern "C" {
// loss (B), grad (14 n, summed), grad_pts (B, n, 4, 3; with pts), iters (B, nullable), u_out (B, 5 + n, nullable; may
// equal u_init)
int emul_chain_loss_warm_f64(int n, const double* x, const double* xp, const double* inertia, const double* mu,
                             const double* half, const double* kin, const double* pts, unsigned npts, double dt, double eps,
                             int64_t B, const double* u_init, double* u_out, double* loss, double* grad, double* grad_pts,
                             int32_t* iters) {
  if (n == 3) return chain_warm<3>(x, xp, inertia, mu, half, kin, pts, npts, dt, eps, B, u_init, u_out, loss, grad, grad_pts, iters);
  if (n == 4) return chain_warm<4>(x, xp, inertia, mu, half, kin, pts, npts, dt, eps, B, u_init, u_out, loss, grad, grad_pts, iters);
  return -1;
}
}
