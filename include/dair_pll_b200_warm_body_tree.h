/*
 * dair_pll_b200 -- warm-started ContactNets losses of the single floating body with witness points and of the generic
 * kinematic trees.
 *
 * Conventions, return codes and the workspace are those of dair_pll_b200.h, which this header extends; the ABI version
 * is its DPLL_VERSION.  As for dpll_elbow_loss_warm_* (dair_pll_b200_warm.h): a training loop revisits the same
 * (x, x_plus) pairs every epoch while the parameters move slowly, and the cone QP of a pair has a unique optimum, so
 * starting its Newton solve from last epoch's optimum changes only the number of Newton directions, not the results
 * (to the solver's tolerance).
 */
#ifndef DAIR_PLL_B200_WARM_BODY_TREE_H_
#define DAIR_PLL_B200_WARM_BODY_TREE_H_

#include "dair_pll_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/*
 * dpll_body_loss_pts_f64 with warm starts.  The arguments before `u_init` and after `u_out` are its own, with the same
 * meaning, checks and return codes (`flags`, `skip_flag`, `weight`, `iters`, `force`, `grad_pts`).
 * u_init: (B, 6) row-major, nullable: start point of sample b's solve (world twist of the body; v+ = v- + u), e.g. the
 *         optimum recorded for the same pair in the previous epoch.  NULL: the feasible-segment start of the cold solve.
 * u_out:  (B, 6) row-major, nullable: receives sample b's optimum; zero for the free-flight samples, whose optimum that is.
 * u_init may equal u_out: a sample reads its row before it writes it.  With both NULL the call launches exactly what
 * dpll_body_loss_pts_f64 launches.  With either given and B == 0, a call that asks for no gradient and no loss sum launches
 * nothing and returns DPLL_OK.
 */
int dpll_body_loss_pts_warm_f64(const double* x, const double* x_plus, const double* weight, const double* inertia,
                                const double* mu_pair, const double* pts, int32_t n_contacts, double dt, double eps,
                                int64_t B, int32_t flags, double* loss, double* force, double* grad_pts, int32_t* iters,
                                double* grad, double* loss_sum, const int32_t* skip_flag, const double* u_init,
                                double* u_out, void* workspace, size_t workspace_bytes, void* stream);

/*
 * dpll_chain_loss_f64 (boxes) and dpll_chain_loss_pts_f64 (witness points) with warm starts.  The arguments before
 * `u_init` are theirs, with the same meaning, checks and return codes.  W = 5 + n_links: [world angular velocity |
 * world linear velocity of link 0 | joint rates] (v+ = v- + u).
 *
 * u_init: (B, W) row-major, nullable: start point of sample b's solve, e.g. the optimum recorded for the same pair in
 *         the previous epoch.  NULL: u = 0, the start of the cold solve.  Ignored where every contact is already in the
 *         polar cone (free flight), whose exact optimum is 0.
 * u_out:  (B, W) row-major, nullable: receives sample b's optimum; 0 in free flight, and 0 for a sample whose forces
 *         are clipped (any |f| > 1e3: loss 0 and no gradient, as in the cold call), so that its next solve starts cold.
 * iters:  (B, nullable) Newton directions of sample b's solve (dpll_chain_loss_warm_f64 has it among its cold arguments).
 * u_init may equal u_out: a sample reads its row before it writes it (training loops keep one buffer per batch).  With
 * both NULL the call launches exactly what its cold counterpart launches.  dpll_chain_loss_warm_f64 with either given
 * and B == 0, asking for no gradient and no loss sum, launches nothing and returns DPLL_OK; dpll_chain_loss_pts_warm_f64
 * returns DPLL_OK at B == 0, as dpll_chain_loss_pts_f64 does.
 */
int dpll_chain_loss_warm_f64(int32_t n_links, const double* x, const double* x_plus, const double* weight,
                             const double* inertia, const double* mu_pair, const double* half, const double* kin,
                             double dt, double eps, int64_t B, double* loss, double* force, int32_t* iters, double* grad,
                             double* loss_sum, const double* u_init, double* u_out, void* workspace,
                             size_t workspace_bytes, void* stream);
int dpll_chain_loss_pts_warm_f64(int32_t n_links, const double* x, const double* x_plus, const double* weight,
                                 const double* inertia, const double* mu_pair, const double* kin, const double* pts,
                                 uint32_t n_pts_packed, double dt, double eps, int64_t B, double* loss, double* grad_pts,
                                 double* grad, double* loss_sum, const double* u_init, double* u_out, int32_t* iters,
                                 void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif

#endif  /* DAIR_PLL_B200_WARM_BODY_TREE_H_ */
