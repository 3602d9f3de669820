// Host build of the witness-point pieces of the wavefront loss kernel (dair_pll_b200/csrc/cn_cube.cuh:
// body_loss_{free_flight,prologue,epilogue}_pts), composed per sample as the kernel's PTS instance runs them.
// TEST INFRASTRUCTURE ONLY: nothing in the package loads this; tests/test_cube_mesh_host.py builds it.
#include "../../dair_pll_b200/csrc/cn_cube.cuh"
#include <cstdint>
using namespace cn;

extern "C" {
// loss, grad11 (d/d [inertia 10 | mu], summed) and grad_pts (B, 4, 3); flags[b] = 1 (nullable) where the free-flight
// triage finalised the sample
int emul_body_loss_pts_wf_f64(const double* x, const double* xp, const double* inertia, const double* mu, const double* pts,
                              int n_c, double dt, double eps, int64_t B, double* loss, double* grad11, double* grad_pts,
                              int32_t* flags) {
  CubeParams<double> P;
  double h[3] = {0, 0, 0};
  cube_params_init(P, inertia, mu, h, dt, eps);
  SolverCfg<double> cfg = default_cfg<double>();
  for (int i = 0; i < 11; ++i) grad11[i] = 0;
  for (int64_t b = 0; b < B; ++b) {
    int it;
    loss[b] = body_loss_sample_pts_wf<double>(P, cfg, x + 13 * b, xp + 13 * b, pts + 12 * b, n_c, grad11, grad_pts + 12 * b,
                                              &it);
    if (flags) {
      double l = 0, g[11] = {0};
      flags[b] = body_loss_free_flight_pts<double>(P, x + 13 * b, xp + 13 * b, pts + 12 * b, n_c, 1.0, g, nullptr, &l) ? 1 : 0;
    }
  }
  return 0;
}
}
