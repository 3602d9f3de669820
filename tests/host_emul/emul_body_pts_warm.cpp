// Host build of the warm-started witness-point loss of the single body (dair_pll_b200/csrc/cn_cube.cuh:
// body_loss_{free_flight,prologue,epilogue}_pts), composed per sample as body_loss_pts_warm_kernel runs it: free-flight
// triage (optimum 0), prologue, start point from u_init (or the feasible-segment point when u_init is NULL), Newton
// visits, epilogue, optimum to u_out.
// TEST INFRASTRUCTURE ONLY: nothing in the package loads this; tests/test_body_warm_host.py builds it.
#include "../../dair_pll_b200/csrc/cn_cube.cuh"
#include <cstdint>
using namespace cn;

extern "C" {
// loss (B), grad11 (d/d [inertia 10 | mu], summed), grad_pts (B, 4, 3), iters (B, nullable), u_out (B, 6, nullable; may
// equal u_init)
int emul_body_loss_pts_warm_f64(const double* x, const double* xp, const double* inertia, const double* mu,
                                const double* pts, int n_c, double dt, double eps, int64_t B, const double* u_init,
                                double* u_out, double* loss, double* grad11, double* grad_pts, int32_t* iters) {
  CubeParams<double> P;
  double h[3] = {0, 0, 0};
  cube_params_init(P, inertia, mu, h, dt, eps);
  const SolverCfg<double> cfg = default_cfg<double>();
  for (int i = 0; i < 11; ++i) grad11[i] = 0;
  for (int64_t b = 0; b < B; ++b) {
    const double* xs = x + 13 * b;
    const double* xps = xp + 13 * b;
    double l = 0;
    if (body_loss_free_flight_pts<double>(P, xs, xps, pts + 12 * b, n_c, 1.0, grad11, grad_pts + 12 * b, &l)) {
      loss[b] = l;
      if (iters) iters[b] = 0;
      if (u_out) for (int i = 0; i < 6; ++i) u_out[6 * b + i] = 0;
      continue;
    }
    double store[CUBE_PROB_FIELDS];
    const CubeProb<double> S{store, 1};
    CubeLossAux<double> A;
    body_loss_prologue_pts<double, 1>(P, xs, xps, pts + 12 * b, n_c, S, A);
    double u[6];
    if (u_init) for (int i = 0; i < 6; ++i) u[i] = u_init[6 * b + i];
    else cube_loss_start<double>(A, CN_LOSS_START_FACTOR, u);
    double d[6], d0 = 0, best = -1;
    CubeTrial<double> tr{1.0, 0.0, 1.0};
    int it = 0;
    while (cube_newton_visit<double, 1>(P, S, cfg, u, d, d0, best, tr, it) != NEWTON_DONE) {}
    if (iters) iters[b] = it & 0xff;
    loss[b] = body_loss_epilogue_pts<double, 1, true>(P, S, A, u, n_c, 1.0, grad11, grad_pts + 12 * b, (double*)nullptr);
    if (u_out) for (int i = 0; i < 6; ++i) u_out[6 * b + i] = u[i];
  }
  return 0;
}
}
