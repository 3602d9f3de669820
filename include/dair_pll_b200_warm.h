/*
 * dair_pll_b200 -- warm-started ContactNets loss of the two-body (elbow) system.
 *
 * Conventions, return codes and the workspace are those of dair_pll_b200.h, which this header extends; the ABI version
 * is its DPLL_VERSION.
 *
 * A training loop revisits the same (x, x_plus) pairs every epoch while the parameters move slowly.  The cone QP of a
 * pair has a unique optimum, so starting its Newton solve from last epoch's optimum changes only the number of Newton
 * directions, not the results (to the solver's tolerance).
 */
#ifndef DAIR_PLL_B200_WARM_H_
#define DAIR_PLL_B200_WARM_H_

#include "dair_pll_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/*
 * dpll_elbow_loss_{f64,f32} with warm starts.  The arguments before `u_init` and after `u_out` are those of
 * dpll_elbow_loss_*, with the same meaning, checks and return codes (box or witness-point geometry, `flags`,
 * `skip_flag`, `weight`, `iters`).
 *
 * u_init: (B, 7) row-major, nullable: start point of sample b's solve (world twist of link 1 | hinge rate; v+ = v- + u),
 *         e.g. the optimum recorded for the same pair in the previous epoch.  NULL: the feasible-segment start of the
 *         cold solve.
 * u_out:  (B, 7) row-major, nullable: receives sample b's optimum; zero for the free-flight samples, whose optimum
 *         that is.
 * u_init may equal u_out: a sample reads its row before it writes it (training loops keep one buffer per batch).
 * With both NULL the call launches exactly what dpll_elbow_loss_* launches.  With either given and B == 0, a call that
 * asks for no gradient and no loss sum launches nothing and returns DPLL_OK.
 */
int dpll_elbow_loss_warm_f64(const double* x, const double* x_plus, const double* weight, const double* inertia,
                             const double* mu_pair, const double* half, const double* kin, const double* pts, double dt,
                             double eps, int64_t B, int32_t flags, double* loss, double* force, double* grad_pts,
                             int32_t* iters, double* grad, double* loss_sum, const int32_t* skip_flag,
                             const double* u_init, double* u_out, void* workspace, size_t workspace_bytes, void* stream);
int dpll_elbow_loss_warm_f32(const float* x, const float* x_plus, const float* weight, const float* inertia,
                             const float* mu_pair, const float* half, const float* kin, const float* pts, float dt,
                             float eps, int64_t B, int32_t flags, float* loss, float* force, float* grad_pts,
                             int32_t* iters, float* grad, float* loss_sum, const int32_t* skip_flag,
                             const float* u_init, float* u_out, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif

#endif  /* DAIR_PLL_B200_WARM_H_ */
