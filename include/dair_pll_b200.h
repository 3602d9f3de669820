/*
 * dair_pll_b200 -- C ABI of the B200 (sm_100a) ContactNets hot path.
 *
 * The reference (DAIRLab/dair_pll) is pure Python: the seam this library sits behind
 * is the torch.nn.Module API of MultibodyLearnableSystem, not an FFI.  These entry
 * points are what the reference-side binding (dair_pll_b200/ops.py, a ctypes stub; see
 * INTEGRATION.md) calls from torch.autograd.Function objects.  Each one replaces a
 * span of reference Python, cited per function.
 *
 * Conventions
 *  - All pointers are DEVICE pointers owned by the caller (torch tensors); contiguous,
 *    row-major.  The library never allocates or frees; scratch is passed in
 *    (`workspace`, at least dpll_workspace_bytes() bytes, 16-byte aligned).
 *  - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it and
 *    performs no host synchronisation.  Compute calls are re-entrant.  Mutable library state: the
 *    cube loss-kernel selector dpll_set_loss_variant (process-wide, measurement only) and the
 *    communicator objects of the data-parallel exchange (dpll_comm_*, one stream at a time each).
 *  - Return value: 0 on success, a positive cudaError_t value if a launch failed, a
 *    negative DPLL_E* value for argument errors.  Numerical failure of a sample's QP
 *    is NOT an error: as in the reference (multibody_learnable_system.py:186-192) that
 *    sample's force and loss are set to 0.
 *  - State layout (state_space.py:400-486): cube x = [qw qx qy qz | px py pz |
 *    w_body(3) | v_world(3)] (13); elbow adds the hinge angle after the position and the
 *    hinge rate after the velocities (15).
 *  - Parameter layout for the cube: inertia[10] = [m, cx, cy, cz, Ixx, Iyy, Izz, Ixy,
 *    Ixz, Iyz] exactly as the reference's generated callables receive it
 *    (multibody_terms.py:230-234; inertia.py:376-382), mu_pair[1] = combined friction
 *    2 mu_a mu_b / (mu_a + mu_b) (multibody_terms.py:466-471), half[3] =
 *    |length_params| (geometry.py:394-397).  Gradients come back in the same layout,
 *    concatenated: grad[14] = [d/d inertia (10) | d/d mu_pair | d/d half (3)].
 */
#ifndef DAIR_PLL_B200_H_
#define DAIR_PLL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPLL_OK 0
#define DPLL_EINVAL (-1)     /* null pointer / negative size */
#define DPLL_EWORKSPACE (-2) /* workspace too small */
#define DPLL_ECOMM (-3)      /* a peer did not arrive within the exchange's timeout */

#define DPLL_VERSION 214     /* bumped with every change of a signature below; the binding checks it */

#define DPLL_CUBE_NX 13
#define DPLL_CUBE_NC 4
#define DPLL_CUBE_NPARAM 14
#define DPLL_ELBOW_NX 15
#define DPLL_ELBOW_NC 8
#define DPLL_ELBOW_NPARAM 28
#define DPLL_ELBOW_NKIN 12

/* Library/ABI version (major*100 + minor). */
int dpll_version(void);

/* Selects the cube loss-kernel implementation, for A/B measurement only: 0 = warp-level wavefront
 * scheduler with static sample ranges (default; gradient sums bitwise reproducible), 1 = one sample
 * per thread, 2 = wavefront scheduler whose warps draw 32-sample chunks from a global counter (as
 * DPLL_LOSS_DYNAMIC below).  All three produce bitwise-identical PER-SAMPLE losses and forces; the
 * summed gradient of variant 2 depends on the chunk-to-warp assignment and is reproducible to
 * rounding only.  Process-wide setting.  The elbow loss always runs its wavefront kernel. */
int dpll_set_loss_variant(int variant);

/* Bytes of device scratch any entry point below may need. */
size_t dpll_workspace_bytes(void);

/*
 * ContactNets loss and its fused envelope-theorem backward for the cube.
 * Replaces MultibodyLearnableSystem.contactnets_loss
 * (dair_pll/multibody_learnable_system.py:104-197) together with everything it calls
 * per sample -- MultibodyTerms.forward (multibody_terms.py:584-609), ContactTerms.forward
 * (:428-521), GeometryCollider.collide_plane_convex (geometry.py:553-582), the top-4 corner
 * selection (geometry.py:162-202), SAPSolver.apply (sappy, un-vendored) -- and the autograd
 * backward of `loss.sum()` w.r.t. the callable-level parameters.
 *
 *   x, x_plus : (B, 13)   states (only the velocity part of x is read, :127)
 *   weight    : (B)       nullable; per-sample upstream gradient w_b.  NULL means w_b = 1.
 *   loss      : (B)       nullable; per-sample loss (:194-197)
 *   force     : (B, 12)   nullable; solved contact impulses in the reference's ordering
 *                         [n_1..n_4, t_1x, t_1y, ..., t_4x, t_4y] (tensor_utils.py:460-497),
 *                         contacts ordered by ascending box-vertex index
 *   iters     : (B)       nullable; Newton iterations used
 *   grad      : (14)      nullable; OVERWRITTEN with d(sum_b w_b loss_b)/d params
 *   loss_sum  : (1)       nullable; OVERWRITTEN with sum_b loss_b
 *   skip_flag : (1) int32 nullable DEVICE flag; if non-null and non-zero when the kernels start,
 *                         the whole call is a no-op on the device (outputs untouched).  Lets a
 *                         caller make the launch conditional on a device-side predicate without
 *                         a host synchronisation (used by the autograd backward).
 * Deterministic: fixed sample->thread mapping and fixed-order reductions (bitwise
 * reproducible for a given B).
 */
int dpll_cube_loss_f64(const double* x, const double* x_plus, const double* weight,
                       const double* inertia, const double* mu_pair, const double* half,
                       double dt, double eps, int64_t B, double* loss, double* force,
                       int32_t* iters, double* grad, double* loss_sum, const int32_t* skip_flag,
                       void* workspace, size_t workspace_bytes, void* stream);
int dpll_cube_loss_f32(const float* x, const float* x_plus, const float* weight,
                       const float* inertia, const float* mu_pair, const float* half, float dt,
                       float eps, int64_t B, float* loss, float* force, int32_t* iters,
                       float* grad, float* loss_sum, const int32_t* skip_flag, void* workspace,
                       size_t workspace_bytes, void* stream);

/*
 * Same computation driven by the LEARNABLE LEAVES instead of the callable-level parameters, so a
 * training step needs no PyTorch glue: the preparation
 *   theta (1,10) -> [m, c, I_cm/m]   (inertia.py:205-234, 304-331, 376-382; multibody_terms.py:230-231)
 *   friction_params (2) [box, ground] -> |.| -> 2 mu_a mu_b/(mu_a+mu_b)   (multibody_terms.py:321-324, 466-471)
 *   length_params (1,3) -> |.|       (geometry.py:394-397)
 * runs in a one-thread kernel, and the reduction kernel applies its chain rule:
 *   grad_leaf : (15) = [d/d theta (10) | d/d friction_params (2) | d/d length_params (3)] of sum_b w_b loss_b.
 * Three launches per call (prepare, loss+backward, reduce+chain).  Other arguments as above.
 */
int dpll_cube_loss_leaf_f64(const double* x, const double* x_plus, const double* weight,
                            const double* theta, const double* friction, const double* length,
                            double dt, double eps, int64_t B, double* loss, double* force,
                            int32_t* iters, double* grad_leaf, double* loss_sum,
                            const int32_t* skip_flag, void* workspace, size_t workspace_bytes,
                            void* stream);
int dpll_cube_loss_leaf_f32(const float* x, const float* x_plus, const float* weight,
                            const float* theta, const float* friction, const float* length, float dt,
                            float eps, int64_t B, float* loss, float* force, int32_t* iters,
                            float* grad_leaf, float* loss_sum, const int32_t* skip_flag,
                            void* workspace, size_t workspace_bytes, void* stream);

/*
 * The data-parallel / training-loop form of dpll_cube_loss_leaf_*: what one rank of the sharded step
 * (SURVEY.md section 8(e); the reference has no distributed code) calls on its B samples.
 *   x_row_stride, xp_row_stride : distance in ELEMENTS between consecutive rows of x / x_plus (>= 13), so the
 *       training loop's views x_past[..., -1, :] / x_future[..., 0, :] (drake_experiment.py:217-218) are read in
 *       place instead of being copied first
 *   flags : DPLL_LOSS_DYNAMIC -- warps draw their 32-sample chunks from a global counter instead of a static
 *       range.  Chunks are handed out in batch order, so a batch ordered by decreasing expected Newton count
 *       (last epoch's `iters`, dataset_management.DeviceTrajectorySliceDataset) starts its longest solves first
 *       and ends with the cheap samples: no serial tail.  Per-sample outputs are unaffected; the summed
 *       gradient is reproducible to rounding only.
 *       DPLL_LOSS_RACE (with DPLL_LOSS_DYNAMIC, cold solves, 4,096 <= B <= 300,000) -- the batch is cost-ordered, so its
 *       first B/64 (<= 2,048) samples are the expensive ones: they go to racing warps in the first blocks of the same
 *       launch (four start points per sample in four slots, a vote after every Newton visit, first to converge wins;
 *       the optimum is unique) while the other blocks take the rest.  A small launch lasts as long as its longest
 *       Newton chain; racing shortens the worst chain from ~47 to ~28 visits.  Per-sample outputs as without the
 *       flag, up to the solver tolerance.
 *   comm  : nullable communicator (dpll_comm_create).  When given, the reduction kernel exchanges
 *       [grad_leaf 15 | loss sum | B] with every peer over NVLink itself and the outputs are the sums over
 *       ranks, bitwise identical on every rank; every rank of the communicator must make the call.
 *   u_init, u_out : (B, 6) nullable; start point of every sample's Newton solve / its optimum u* (world-frame twist of
 *       the impulse, M u* = J^T f).  The QP's optimum is unique, so the start changes only the number of Newton
 *       visits: a training loop that keeps u* per pair (DeviceTrajectorySliceDataset.update_solutions) and hands it
 *       back next epoch solves in a few visits instead of ~11.  u_out of a free-flight sample is 0.
 *   sums  : (17) nullable; [d(sum_b loss_b)/d leaves (15) | sum_b loss_b | number of samples summed]
 *   means : (16) nullable; sums[0..15] / sums[16]: loss.mean() (drake_experiment.py:222-223) and its gradient
 *   local : (16) nullable; this rank's own [grad_leaf 15 | loss sum] (before the exchange)
 * No `weight`, `force` or `skip_flag`: this is the loss.mean()/loss.sum() training path.
 */
#define DPLL_LOSS_DYNAMIC 1
#define DPLL_LOSS_RACE 2
int dpll_cube_loss_leaf_dp_f64(const double* x, int64_t x_row_stride, const double* x_plus, int64_t xp_row_stride,
                               const double* theta, const double* friction, const double* length, double dt,
                               double eps, int64_t B, int32_t flags, void* comm, const double* u_init, double* u_out,
                               double* loss, int32_t* iters, double* sums, double* means, double* local,
                               void* workspace, size_t workspace_bytes, void* stream);
int dpll_cube_loss_leaf_dp_f32(const float* x, int64_t x_row_stride, const float* x_plus, int64_t xp_row_stride,
                               const float* theta, const float* friction, const float* length, float dt, float eps,
                               int64_t B, int32_t flags, void* comm, const float* u_init, float* u_out, float* loss,
                               int32_t* iters, float* sums, float* means, float* local, void* workspace,
                               size_t workspace_bytes, void* stream);

/*
 * Data-parallel exchange over peer memory.  One communicator per rank (= per process and GPU); `create`
 * allocates the rank's exchange buffer (the only allocation this library ever makes) and returns its CUDA IPC
 * handle (dpll_comm_handle_bytes() bytes, HOST memory); the caller gathers all ranks' handles by any means
 * (torch.distributed.all_gather_object in dair_pll_b200/parallel.py) and passes them, in rank order, to
 * `connect`, which maps the peers' buffers (NVLink / NVSwitch P2P).  The kernels then all-reduce up to 32
 * doubles by direct peer stores + flags (csrc/cn_comm.cuh): no NCCL launch on the step's critical path.  A
 * peer that never arrives is reported by dpll_comm_error (DPLL_ECOMM) after a 4 s device-side timeout
 * instead of hanging the GPU.  dpll_comm_allreduce_f64: the stand-alone form, buf[i] <- scale * sum over ranks.
 */
size_t dpll_comm_handle_bytes(void);
int dpll_comm_create(int32_t rank, int32_t world, void** comm_out, void* handle_out);
int dpll_comm_connect(void* comm, const void* handles);
int dpll_comm_destroy(void* comm);
void* dpll_comm_device_state(void* comm);
int dpll_comm_error(void* comm);
int dpll_comm_allreduce_f64(void* comm, double* buf, int32_t n, double scale, void* stream);

/*
 * Learnable time stepping for the cube: `steps` applications of
 * VelocityIntegrator.step (dair_pll/integrator.py:153-162) around
 * MultibodyLearnableSystem.sim_step / forward_dynamics
 * (multibody_learnable_system.py:199-313) and FloatingBaseSpace.exponential
 * (state_space.py:466-486; quaternion.py:89-104, 276-309); the time loop is
 * Integrator.simulate (integrator.py:75-99).
 *
 *   x0    : (B, 13)              initial states
 *   traj  : (B, steps+1, 13)     traj[:,0] = x0, traj[:,t+1] = step(traj[:,t])
 *   force : (B, steps, 12)       nullable; impulses of every step (reference ordering)
 *   iters : (B)                  nullable; total Newton iterations over the rollout
 * eps is the QP regulariser (the reference hard-codes 1e-4, :283,298).
 */
int dpll_cube_rollout_f64(const double* x0, const double* inertia, const double* mu_pair,
                          const double* half, double dt, double eps, int64_t B, int32_t steps,
                          double* traj, double* force, int32_t* iters, void* stream);
int dpll_cube_rollout_f32(const float* x0, const float* inertia, const float* mu_pair,
                          const float* half, float dt, float eps, int64_t B, int32_t steps,
                          float* traj, float* force, int32_t* iters, void* stream);

/*
 * Support-function network of learned geometries (HomogeneousICNN.forward, dair_pll/deep_support_function.py:238-266,
 * called from DeepSupportConvex.get_vertices, dair_pll/geometry.py:309-325): the memory-bound layers around the
 * three (D x W) x (W x W) products, which the caller runs as FP64 library GEMMs.  D direction rows, width W,
 * LeakyReLU slope `slope`; row-major arrays; weights Wd0, Wd1 (3, W).
 *   dpll_icnn_input_f64     h0aug (D, W+8) = [lrelu(d Wd0) | d | 0]      (so that z1 = h0aug [|Wh| ; Wd1 ; 0])
 *   dpll_icnn_mask_f64      z (n) -> slope mask of z, in place            (m1 from z1)
 *   dpll_icnn_output_f64    T (D, W) = m1 (|wout| * |Wh|^T) -> a0 = T o m0 in place;  p (D, 3) = m1 V1^T + a0 Wd0^T,
 *                           V1 = |wout| * Wd1 (3, W): the support points
 *   dpll_icnn_backward_f64  cotangent gp (D, 3): t (D, W) = (gp Wd0) o m0 and per-block partial sums
 *                           part (dpll_icnn_backward_blocks(D), 6, W) of gp^T m1 (rows 0-2) and gp^T a0 (rows 3-5)
 */
int dpll_icnn_input_f64(const double* d, const double* Wd0, int64_t D, int32_t W, double slope, double* h0aug,
                        void* stream);
int dpll_icnn_mask_f64(double* z, int64_t n, double slope, void* stream);
int dpll_icnn_output_f64(double* T, const double* h0aug, const double* m1, const double* Wd0, const double* V1, int64_t D,
                         int32_t W, double slope, double* p, void* stream);
int dpll_icnn_backward_blocks(int64_t D);
int dpll_icnn_backward_f64(const double* gp, const double* h0aug, const double* m1, const double* a0, const double* Wd0,
                           int64_t D, int32_t W, double slope, double* t, double* part, void* stream);

/*
 * Support directions of the two elbow links against the ground -- minus the third row of each link's world rotation
 * (GeometryCollider.collide_plane_convex, geometry.py:560-567) -- and their n_query perturbed, normalised copies
 * (DeepSupportConvex.get_vertices, geometry.py:309-325): q rows of 8 configuration values at stride q_stride, axis (3),
 * pert0 / pert1 (n_query, 3) the two geometries' fixed perturbations; dirs0 / dirs1 (B, n_query, 3).
 */
int dpll_elbow_support_directions_f64(const double* q, int64_t q_stride, const double* axis, const double* pert0,
                                      const double* pert1, int32_t n_query, int64_t B, double* dirs0, double* dirs1,
                                      void* stream);

/*
 * The same for a single floating body whose learned geometry sits in the link frame: q rows of >= 4 values (the
 * quaternion first) at stride q_stride, pert (n_query, 3) the geometry's fixed perturbations; dirs (B, n_query, 3).
 */
int dpll_body_support_directions_f64(const double* q, int64_t q_stride, const double* pert, int32_t n_query, int64_t B,
                                     double* dirs, void* stream);

/*
 * Support points on the tensor cores (csrc/cn_icnn_tc.cu; width W = 256 only): HomogeneousICNN.forward
 * (deep_support_function.py:238-266) for all D direction rows in one kernel.  The layer Jacobian d z1 / d d is a
 * (binary mask) x (constant matrix) product, evaluated exactly as int8 digit-plane products by tcgen05.mma with int32
 * accumulators in tensor memory and rebuilt in fp64 per row (42-bit fixed point per weight column; rows whose
 * pre-activation is within 1e-9 of zero are re-evaluated in plain fp64 before the mask is taken).  No (D x W) array
 * exists in HBM.  dpll_icnn_tc_prepare_f64 turns the four weights into the digit-plane image (dpll_icnn_tc_image_bytes())
 * and the epilogue constants (dpll_icnn_tc_const_bytes()); run it whenever the weights change.
 */
size_t dpll_icnn_tc_image_bytes(void);
size_t dpll_icnn_tc_const_bytes(void);
int dpll_icnn_tc_prepare_f64(const double* Wd0, const double* Wd1, const double* Wh, const double* wout, int32_t W,
                             double slope, void* image, double* consts, void* stream);
int dpll_icnn_tc_support_f64(const double* d, int64_t D, const void* image, const double* consts, const double* Wh,
                             int32_t W, double slope, double* p, void* stream);

/*
 * Backward of the support-function network on the tensor cores (csrc/cn_icnn_tc_bwd.cu, W = 256), for the rows of a
 * batch whose cotangent is non-zero, WITHOUT a host read: the caller compacts those rows (e.g. torch.nonzero_static) into
 * the first *n_rows of `capacity` gathered rows and passes the count as a device scalar; every grid is fixed.
 *   dpll_icnn_tc_record_f64   first pass over the gathered directions d (capacity, 3): the two layers' slope-mask bits as
 *                             transposed byte matrices m0t[j][row] in {0x00, 0xFF}, m1t[i][row] in {0, 1}, row stride ldk
 *                             (a multiple of 128, >= capacity); same kernel as dpll_icnn_tc_support_f64
 *   dpll_icnn_tc_bwd_f64      gathered cotangent gp (capacity, 3), amax (3) = max |gp_k| -> C (3, W, W),
 *                             C_k[j,i] = sum_r gp_k[r] m0[r,j] m1[r,i] (m = slope + (1 - slope) bit), and
 *                             sums (6 W + 3) = [R0_k[j] = sum_r gp_k[r] b0[r,j] | R1_k[i] = sum_r gp_k[r] b1[r,i] | S_k = sum_r gp_k[r]].
 *                             The (rows x W x W) contraction runs as exact int8 digit-plane products of the cotangent
 *                             (56-bit fixed point per coordinate) against the mask bytes: tcgen05.mma M 128 N 256.
 *                             Scratch: planes (dpll_icnn_tc_bwd_planes() * ldk bytes), partial (dpll_icnn_tc_bwd_partial_bytes()).
 * All weight gradients then follow from C and sums by (W x W)-sized arithmetic (dair_pll_b200/deep_support_function.py).
 */
size_t dpll_icnn_tc_bwd_partial_bytes(void);
int32_t dpll_icnn_tc_bwd_planes(void);
int dpll_icnn_tc_record_f64(const double* d, int64_t capacity, const int64_t* n_rows, const void* image, const double* consts,
                            const double* Wh, int32_t W, double slope, uint8_t* m0t, uint8_t* m1t, int64_t ldk, void* stream);
int dpll_icnn_tc_bwd_f64(const double* gp, const int64_t* n_rows, const double* amax, const uint8_t* m0t, const uint8_t* m1t,
                         int64_t ldk, double slope, int8_t* planes, int32_t* partial, double* sums, double* C, void* stream);

/*
 * A single floating body whose collision geometry is ANY convex shape against the ground plane
 * (GeometryCollider.collide_plane_convex, dair_pll/geometry.py:553-582): the caller passes the shape's support
 * points in the direction -R^T e_z -- Sphere: 1 point d r (geometry.py:415-456); Polygon: the top-n_query vertices
 * (geometry.py:220-252, 162-202); Box / DeepSupportConvex likewise -- as pts (B, 4, 3) in the geometry frame, of
 * which the first n_contacts (1..4) rows are used, and gets the loss, the gradient w.r.t. [inertia 10 | mu_pair]
 * (grad, 11) and grad_pts (B, 4, 3) = w_b d loss_b / d pts[b] back (rows >= n_contacts zero).  The box's wavefront
 * kernel runs it (its witness-point instance: free-flight triage, Newton visits over shared-memory slots), so per-sample
 * losses, forces, grad_pts and iteration counts do not depend on `flags`:
 *   flags     : DPLL_LOSS_DYNAMIC as for dpll_cube_loss_leaf_dp_f64 (32-sample chunks in batch order, for cost-ordered
 *               batches; the gradient sums are then rounded in a timing-dependent order); other bits are ignored.
 *   skip_flag : (nullable, device) when *skip_flag != 0 every launch returns at once and writes nothing -- the weighted
 *               backward pass of a uniform upstream gradient, decided on the device so that the step can be captured
 *               into a CUDA graph.
 * dpll_body_step_pts_f64: one learnable time step x -> x_next with the same contact set.
 */
int dpll_body_loss_pts_f64(const double* x, const double* x_plus, const double* weight, const double* inertia,
                           const double* mu_pair, const double* pts, int32_t n_contacts, double dt, double eps,
                           int64_t B, int32_t flags, double* loss, double* force, double* grad_pts, int32_t* iters,
                           double* grad, double* loss_sum, const int32_t* skip_flag, void* workspace,
                           size_t workspace_bytes, void* stream);
int dpll_body_step_pts_f64(const double* x, const double* inertia, const double* mu_pair, const double* pts,
                           int32_t n_contacts, double dt, double eps, int64_t B, double* x_next, double* force,
                           void* stream);

/*
 * Backward of ONE witness-point step (the prediction-loss path for Sphere / Polygon geometries, whose support points
 * depend on the state, so that rollout runs step by step): given xbar (B, 13) w.r.t. the next state, gparams (B, 11) =
 * [d/d inertia (10) | d/d mu_pair], gpts (B, 12) and gx (B, 13) w.r.t. the current state at fixed points.  Forward-mode
 * tangents through the step code, 36 directions per sample.
 */
int dpll_body_step_pts_grad_f64(const double* x, const double* inertia, const double* mu_pair, const double* pts,
                                int32_t n_contacts, double dt, double eps, int64_t B, const double* xbar,
                                double* gparams, double* gpts, double* gx, void* stream);

/*
 * Dense dynamics terms of the cube in the reference's coordinates and ordering, for callers of
 * MultibodyTerms.forward (dair_pll/multibody_terms.py:584-609; LagrangianTerms.forward :214-237,
 * ContactTerms.forward :428-521): q (B,7), v (B,6) -> M (B,6,6), J (B,12,6) = [J_n ; mu J_t interleaved]
 * (:401-426), phi (B,4), contact-free acceleration (B,6), delassus (B,12,12) (nullable).  Contacts by
 * ascending box-vertex index.  (The loss / step kernels never form these matrices.)
 */
int dpll_cube_terms_f64(const double* q, const double* v, const double* inertia, const double* mu_pair,
                        const double* half, int64_t B, double* M, double* J, double* phi, double* acc,
                        double* delassus, void* stream);

/*
 * The same export for the two-body (elbow) system with box geometries: q (B,8), v (B,7) -> M (B,7,7), J (B,24,7),
 * phi (B,8), contact-free acceleration (B,7), delassus (B,24,24) (nullable).  Contacts of box 1 then box 2, each by
 * ascending vertex index; J rows [normals (8) ; mu (x, y) interleaved per contact (16)].
 */
int dpll_elbow_terms_f64(const double* q, const double* v, const double* inertia, const double* mu_pair,
                         const double* half, const double* kin, int64_t B, double* M, double* J, double* phi,
                         double* acc, double* delassus, void* stream);

/*
 * Backward of dpll_cube_rollout_f64 (the gradient the reference obtains by autograd through
 * forward_dynamics and sappy's backward, multibody_learnable_system.py:293-304; used by the
 * prediction loss, experiment.py:230-248, 292-320): given the upstream gradient xbar (B, steps, 13)
 * w.r.t. traj[:, 1:], returns PER-SAMPLE gradients
 *   gparams (B, 14) w.r.t. [inertia 10 | mu_pair 1 | half 3]   and   gx0 (B, 13) w.r.t. x0
 * (sum gparams over B for the parameter gradient; add xbar of traj[:, 0] to gx0 yourself).
 * Implemented by forward-mode differentiation of the step code (27 tangent directions); exact
 * implicit differentiation of the QP at the converged solution.
 */
int dpll_cube_rollout_grad_f64(const double* x0, const double* inertia, const double* mu_pair,
                               const double* half, double dt, double eps, int64_t B, int32_t steps,
                               const double* xbar, double* gparams, double* gx0, void* stream);

/*
 * Reverse-mode form of the same backward (SURVEY.md K7: "adjoint solve n_v x n_v"): the forward rollout keeps every
 * step's QP optimum,
 *   dpll_cube_rollout_saved_f64   as dpll_cube_rollout_f64, plus usol (B, steps, 6): the optimum u* of every step's
 *                                 cone QP (world-frame twist; v+ = v- + u*)
 * and the backward walks each trajectory once, last step first: per step one evaluation of the Newton Hessian at
 * u*, ONE 6x6 SPD (Cholesky) solve -- implicit differentiation of the QP -- and the hand-derived adjoints of the
 * step's remaining lines (csrc/cn_cube_adjoint.cuh).
 *   dpll_cube_rollout_backward_f64   traj (B, steps+1, 13), usol (B, steps, 6), xbar (B, steps, 13) w.r.t. traj[:, 1:]
 *                                    -> gparams (B, 14), gx0 (B, 13), exactly as dpll_cube_rollout_grad_f64
 * About the arithmetic of three Newton visits per step instead of 27 dual-number rollouts; agrees with the
 * forward-mode entry point to 1e-10 (tests), which is kept as the independent check.
 */
int dpll_cube_rollout_saved_f64(const double* x0, const double* inertia, const double* mu_pair, const double* half,
                                double dt, double eps, int64_t B, int32_t steps, double* traj, double* usol,
                                void* stream);
int dpll_cube_rollout_backward_f64(const double* traj, const double* usol, const double* inertia,
                                   const double* mu_pair, const double* half, double dt, double eps, int64_t B,
                                   int32_t steps, const double* xbar, double* gparams, double* gx0, void* stream);

/*
 * Backward of ONE learnable step of the two-body system with caller-supplied witness points pts (B, 8, 3) -- the learned
 * (support-function) geometry, whose points depend on the state through the caller's networks, so the time loop of that
 * rollout runs step by step (forward_dynamics multibody_learnable_system.py:199-304 with geometry.py:309-325): given
 * xbar (B, 15) w.r.t. the next state, gparams (B, 22) = [d/d inertia (20) | d/d mu_pair (2)], gpts (B, 24) and
 * gx (B, 15) w.r.t. the current state at fixed points.  Forward-mode tangents through the step code, 61 directions per
 * sample, implicit derivative of the QP by the polishing Newton step.
 */
int dpll_elbow_step_pts_grad_f64(const double* x, const double* inertia, const double* mu_pair, const double* kin,
                                 const double* pts, const double* usol, double dt, double eps, int64_t B,
                                 const double* xbar, double* gparams, double* gpts, double* gx, void* stream);

/*
 * The two-body rollout keeping every step's QP optimum, usol (B, steps, 7) (world twist of the first link + hinge rate;
 * v+ = v- + u*), and the forward-mode backward that uses it, for box geometries: gparams (B, 28) = [d/d inertia (20) |
 * d/d mu_pair (2) | d/d half (6)], gx0 (B, 15), 43 tangent directions per toss.  With the optimum known, a dual-number
 * step is ONE evaluation and one 7x7 Cholesky solve at u* (whose tangent is the implicit-function derivative) instead of
 * a whole dual-number Newton solve.  usol nullable in the two *_grad entry points (then every step is solved again in
 * dual arithmetic).  pts as in dpll_elbow_rollout_f64 (steps <= 1 when given).
 */
int dpll_elbow_rollout_saved_f64(const double* x0, const double* inertia, const double* mu_pair, const double* half,
                                 const double* kin, const double* pts, double dt, double eps, int64_t B, int32_t steps,
                                 double* traj, double* usol, void* stream);
int dpll_elbow_rollout_grad_saved_f64(const double* x0, const double* inertia, const double* mu_pair, const double* half,
                                      const double* kin, const double* usol, double dt, double eps, int64_t B,
                                      int32_t steps, const double* xbar, double* gparams, double* gx0, void* stream);

/*
 * The same two operations for the elbow (assets/contactnets_elbow.urdf: floating base + one
 * revolute child, two boxes, 2 x 4 contacts): states (B, 15) = [quat | pos | hinge angle | w_body |
 * v_world | hinge rate]; parameters inertia[20] (two bodies' 10-vectors), mu_pair[2] (ground-box1,
 * ground-box2), half[6]; kin[12] = URDF constants [joint origin (3) in link 1 | joint axis (3) | box-1
 * offset (3) | box-2 offset (3)] (not learnable).  force: (B, 24) = [n_1..n_8, t_1x, t_1y, ...], contacts
 * of box 1 then box 2, each by ascending vertex index.  grad[28] = [d/d inertia (20) | d/d mu_pair (2) |
 * d/d half (6)].  Same reference spans as the cube entry points; the articulated M(q), F(q,v) and
 * geometry Jacobians are the closed forms of what multibody_terms.py:114-157, 267-319 derive
 * symbolically.  The loss runs in a warp-level wavefront kernel like the cube's (csrc/cn_elbow_wf.cu: mass matrix
 * as a composite body + hinge column, 96-double shared-memory records, one Newton visit per scheduling step).
 *
 * Learned (mesh) geometry: `pts` (B, 8, 3), nullable.  When given, the 4 + 4 witness points of the two
 * geometries (geometry frames) are taken from it instead of the box corners -- they are the outputs of
 * DeepSupportConvex.get_vertices (geometry.py:309-325; the ICNN of deep_support_function.py:238-266 is
 * evaluated by the caller) -- `half` may then be NULL, and `grad_pts` (B, 8, 3), nullable, receives
 * w_b * d loss_b / d pts[b] for the caller's network backward (grad[22..27] stay zero).  The rollout
 * accepts `pts` only for steps <= 1 (witness points depend on the state).
 *
 * `flags` of the loss: DPLL_LOSS_DYNAMIC hands 32-sample chunks to the warps in batch order, for cost-ordered
 * batches (see dpll_cube_loss_leaf_dp_*); 0 keeps static sample ranges.
 */
int dpll_elbow_loss_f64(const double* x, const double* x_plus, const double* weight, const double* inertia,
                        const double* mu_pair, const double* half, const double* kin, const double* pts,
                        double dt, double eps, int64_t B, int32_t flags, double* loss, double* force,
                        double* grad_pts, int32_t* iters, double* grad, double* loss_sum,
                        const int32_t* skip_flag, void* workspace, size_t workspace_bytes, void* stream);
int dpll_elbow_loss_f32(const float* x, const float* x_plus, const float* weight, const float* inertia,
                        const float* mu_pair, const float* half, const float* kin, const float* pts, float dt,
                        float eps, int64_t B, int32_t flags, float* loss, float* force, float* grad_pts,
                        int32_t* iters, float* grad, float* loss_sum, const int32_t* skip_flag,
                        void* workspace, size_t workspace_bytes, void* stream);
int dpll_elbow_rollout_f64(const double* x0, const double* inertia, const double* mu_pair,
                           const double* half, const double* kin, const double* pts, double dt,
                           double eps, int64_t B, int32_t steps, double* traj, double* force,
                           int32_t* iters, void* stream);
int dpll_elbow_rollout_f32(const float* x0, const float* inertia, const float* mu_pair,
                           const float* half, const float* kin, const float* pts, float dt, float eps,
                           int64_t B, int32_t steps, float* traj, float* force, int32_t* iters,
                           void* stream);

/*
 * Generic floating-base kinematic tree (SURVEY.md section 8(f) N2): n_links = 2..6 rigid links joined by revolute
 * or prismatic joints -- a serial chain or a branching tree, link b > 0 hanging off any link parent(b) < b -- one box per link
 * against the ground: what the reference derives symbolically for any plant
 * (multibody_terms.py:114-157, 267-319) evaluated by recursion over the links (csrc/cn_chain.cuh), for models the
 * specialised cube / elbow kernels do not cover.  States (B, 13 + 2 (n-1)) = [quat | pos | joint angles | w_body |
 * v_world | joint rates] (joint b - 1 is the one whose child is link b); inertia (n, 10), mu_pair (n) (ground-link i),
 * half (n, 3); kin (n, 31): row b carries LINK b's joint -- [joint origin in the parent link (0:3) | fixed rotation parent
 * -> joint frame, row-major (3:12) | joint axis (12:15) | index of the parent link, as a number (18) | joint type: 0
 * revolute / continuous, 1 prismatic (28)] -- and BOX SLOT b -- [box offset in its link (15:18) | rotation link frame <-
 * collision (box) frame, row-major (19:28) | index of the link the box sits on (29) | 1 if the slot holds a box, 0 if it is
 * empty (30)]: there are as many box slots as links and a slot may sit on ANY link, so up to n boxes can be spread over the
 * links in any way; mu_pair, half and the gradient entries are per slot (empty slots: ignored / zero).  Row 0 has no joint;
 * a parent index outside [0, b - 1] and a box link outside [0, n - 1] are clamped.  grad (14 n) = [d/d inertia (10 n) | d/d mu_pair (n) |
 * d/d half (3 n)] of sum_b w_b loss_b; force (B, 12 n) = [normals (4 n) ; (tx, ty) (4 n)], links in order, contacts by
 * ascending vertex index.  One sample per thread.  dpll_chain_rollout_f64: traj (B, steps+1, n_x).
 */
int dpll_chain_loss_f64(int32_t n_links, const double* x, const double* x_plus, const double* weight,
                        const double* inertia, const double* mu_pair, const double* half, const double* kin,
                        double dt, double eps, int64_t B, double* loss, double* force, int32_t* iters, double* grad,
                        double* loss_sum, void* workspace, size_t workspace_bytes, void* stream);
int dpll_chain_rollout_f64(int32_t n_links, const double* x0, const double* inertia, const double* mu_pair,
                           const double* half, const double* kin, double dt, double eps, int64_t B, int32_t steps,
                           double* traj, void* stream);
/* Backward of the chain rollout (prediction loss): xbar (B, steps, n_x) w.r.t. traj[:, 1:] -> gparams (B, 14 n) =
 * [d/d inertia (10 n) | d/d mu_pair (n) | d/d half (3 n)] and gx0 (B, n_x), by forward-mode tangents through the step code
 * (14 n + n_x directions per toss), as dpll_elbow_rollout_grad_saved_f64 without usol. */
int dpll_chain_rollout_grad_f64(int32_t n_links, const double* x0, const double* inertia, const double* mu_pair,
                                const double* half, const double* kin, double dt, double eps, int64_t B, int32_t steps,
                                const double* xbar, double* gparams, double* gx0, void* stream);

/*
 * The tree LOSS kernel with WITNESS POINTS instead of box corners (as dpll_body_loss_pts_f64 / the elbow's `pts` for the
 * specialised systems): any plane-convex shape on any link -- GeometryCollider.collide_plane_convex, geometry.py:553-582,
 * is "the shape's support points in the direction -R_WG^T e_z", whatever the shape (Sphere :415-456, Polygon :220-252,
 * DeepSupportConvex :255-325, a Box in any collision frame).  pts (B, n, 4, 3): per box SLOT up to four points in the frame
 * of the slot's LINK (the caller evaluates and places them); n_pts_packed: the number of points of slot b in bits
 * 3 b .. 3 b + 2; kin as for dpll_chain_loss_f64 with the slots' own offset / rotation unused (the points are already in
 * link coordinates).  grad_pts (B, n, 4, 3) nullable: w_b d loss_b / d pts_b; grad (14 n) nullable: [d/d inertia (10 n) |
 * d/d mu_pair (n) | zeros (3 n)] of sum_b w_b loss_b.  (The time step with witness points exists in the device math,
 * chain_step_sample, and is checked against the reference on the host emulation; it has no entry point yet.)
 */
int dpll_chain_loss_pts_f64(int32_t n_links, const double* x, const double* x_plus, const double* weight,
                            const double* inertia, const double* mu_pair, const double* kin, const double* pts,
                            uint32_t n_pts_packed, double dt, double eps, int64_t B, double* loss, double* grad_pts,
                            double* grad, double* loss_sum, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Dense terms export of MultibodyTerms.forward (multibody_terms.py:584-609) for a tree (same tables as dpll_chain_loss_f64):
 * q (B, 7 + n - 1), v (B, n_v = 6 + n - 1) -> M (B, n_v, n_v), J (B, 12 n_boxes, n_v) = [normals (4 n_boxes) ; mu (x, y)
 * interleaved per contact (8 n_boxes)], phi (B, 4 n_boxes), contact-free acceleration (B, n_v), delassus (B, 12 n_boxes,
 * 12 n_boxes) (nullable) -- the contacts of the first n_boxes box slots (1 <= n_boxes <= n_links), each box by ascending
 * vertex index; state coordinates as the reference's (body-frame angular velocity of link 0).
 */
int dpll_chain_terms_f64(int32_t n_links, int32_t n_boxes, const double* q, const double* v, const double* inertia,
                         const double* mu_pair, const double* half, const double* kin, int64_t B, double* M, double* J,
                         double* phi, double* acc, double* delassus, void* stream);

/*
 * Parameter preparation of any system and its chain rule, one launch each (csrc/cn_leaf.cu): theta (n_bodies, 10)
 * -> inertia (n_bodies, 10) = [m, c, I_cm / m] (inertia.py:205-234, 304-331, 376-382 as LagrangianTerms.forward applies
 * them, multibody_terms.py:230-231); friction_params (n_geoms) -> mu_pair (n_pairs) = 2 |a| |b| / (|a| + |b|) for the
 * pair's two geometry indices pair_a[p], pair_b[p] (multibody_terms.py:321-324, 466-471); length_params (n_len doubles)
 * -> half = |length| (geometry.py:394-397).  dpll_leaf_backward_f64 maps the cotangents of (inertia, mu_pair, half)
 * (any of them NULL = zero) to those of (theta, friction_params, length_params); d|v|/dv = 0 at v = 0.  The single
 * floating box has the same maps fused into dpll_cube_loss_leaf_*.
 */
int dpll_leaf_prepare_f64(const double* theta, int32_t n_bodies, const double* friction, const int32_t* pair_a,
                          const int32_t* pair_b, int32_t n_pairs, const double* length, int32_t n_len, double* inertia,
                          double* mu_pair, double* half, void* stream);
int dpll_leaf_backward_f64(const double* theta, int32_t n_bodies, const double* friction, int32_t n_geoms,
                           const int32_t* pair_a, const int32_t* pair_b, int32_t n_pairs, const double* length, int32_t n_len,
                           const double* g_inertia, const double* g_mu_pair, const double* g_half, double* g_theta,
                           double* g_friction, double* g_length, void* stream);

/*
 * FP64 / FP32 FMA throughput micro-benchmark used by bench.py to measure the CUDA-core
 * roofline denominator on the box it runs on (MEASURED_PEAKS.json carries no FP64
 * figure).  Launches `blocks` x 256 threads, each running `iters` x 16 independent FMAs
 * per loop trip; writes one value per thread to out (blocks*256 elements) so the work is
 * not optimised away.  FLOPs = blocks * 256 * iters * 16 * 2.
 */
int dpll_fma_peak_f64(double* out, int32_t blocks, int64_t iters, void* stream);
int dpll_fma_peak_f32(float* out, int32_t blocks, int64_t iters, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DAIR_PLL_B200_H_ */
