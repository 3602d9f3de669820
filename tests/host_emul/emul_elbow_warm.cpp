// Host build of the two-body (elbow) loss pieces of the wavefront kernel (dair_pll_b200/csrc/cn_elbow_wf.cuh), composed per
// sample as the warm instance of elbow_loss_wf_kernel runs them: free-flight triage (optimum 0), prologue, start point from
// u_init (or the feasible-segment point when u_init is NULL), Newton visits, epilogue, optimum to u_out.
// TEST INFRASTRUCTURE ONLY: nothing in the package loads this; tests/test_elbow_warm_host.py builds it.
#include "../../dair_pll_b200/csrc/cn_elbow_wf.cuh"
#include <cstdint>
using namespace cn;

extern "C" {
// loss (B), grad28 (d/d [inertia 20 | mu_pair 2 | half 6], summed), iters (B, nullable), u_out (B, 7, nullable; may equal
// u_init)
int emul_elbow_loss_warm_f64(const double* x, const double* xp, const double* inertia, const double* mu, const double* half,
                             const double* kin, const double* pts, double dt, double eps, int64_t B, const double* u_init,
                             double* u_out, double* loss, double* grad28, int32_t* iters) {
  const double h0[6] = {0, 0, 0, 0, 0, 0};
  ElbowParams<double> P;
  elbow_params_init(P, inertia, mu, half ? half : h0, kin, dt, eps);
  const SolverCfg<double> cfg = default_cfg<double>();
  for (int i = 0; i < 28; ++i) grad28[i] = 0;
  for (int64_t b = 0; b < B; ++b) {
    const double* xs = x + 15 * b;
    const double* xps = xp + 15 * b;
    const double* pb = pts ? pts + 24 * b : nullptr;
    double l = 0;
    if (elbow_loss_free_flight<double, double>(P, xs, xps, pb, grad28, nullptr, 1.0, &l)) {
      loss[b] = l;
      if (iters) iters[b] = 0;
      if (u_out) for (int i = 0; i < 7; ++i) u_out[7 * b + i] = 0;
      continue;
    }
    double store[EW_REC];
    const ElbowRec<double> S{store, 1};
    ElbowSetup<double> E;
    ElbowLossCore<double> A;
    elbow_loss_prologue_wf<double, double>(P, xs, xps, pb, S, E, A);
    double u[7];
    for (int i = 0; i < 7; ++i) u[i] = u_init ? u_init[7 * b + i] : (1.0 - A.a_start) * A.dv[i];
    int it = 0;
    double d[7], d0 = 0, best = -1;
    CubeTrial<double> tr{1.0, 0.0, 1.0};
    while (elbow_newton_visit<double>(P, S, cfg, u, d, d0, best, tr, it) != NEWTON_DONE) {}
    if (iters) iters[b] = it & 0xff;
    loss[b] = elbow_loss_epilogue_wf<double, double>(P, S, E, A, u, grad28, nullptr, nullptr, 1.0);
    if (u_out) for (int i = 0; i < 7; ++i) u_out[7 * b + i] = u[i];
  }
  return 0;
}
}
