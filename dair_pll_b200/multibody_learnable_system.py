"""``MultibodyLearnableSystem`` with the reference's API, backed by sm_100a kernels.

Drop-in for ``dair_pll.multibody_learnable_system.MultibodyLearnableSystem``
(multibody_learnable_system.py:41-333): same constructor, same method signatures and
output shapes, same ``nn.Parameter`` names/shapes (so ``state_dict`` checkpoints
interchange, experiment.py:530-538), same attributes (``space``, ``integrator``, ``dt``,
``multibody_terms``, ``max_batch_dim``).  The per-sample work of ``contactnets_loss``
(:104-197), ``forward_dynamics`` (:199-304) and the integrator loop runs in CUDA kernels
through ``dair_pll_b200.ops``; inputs must be CUDA tensors -- there is no CPU path.
"""
import os
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from dair_pll_b200 import ops
from dair_pll_b200.geometry import place_in_link_frame
from dair_pll_b200.integrator import VelocityIntegrator
from dair_pll_b200.multibody_terms import MultibodyTerms
from dair_pll_b200.system import System, SystemSummary

LOSS_EPS = 1e-3    # multibody_learnable_system.py:130
STEP_EPS = 1e-4    # multibody_learnable_system.py:283, 298


class KernelVelocityIntegrator(VelocityIntegrator):
    """``VelocityIntegrator`` whose time loop is one persistent rollout kernel: all
    ``steps`` of ``Integrator.simulate`` (integrator.py:95-98) run on-chip per sample."""

    def __init__(self, space, partial_step_callback, dt, rollout) -> None:
        super().__init__(space, partial_step_callback, dt)
        self._rollout = rollout

    def simulate(self, x_0: Tensor, carry_0: Tensor, steps: int) -> Tuple[Tensor, Tensor]:
        assert steps >= 0 and x_0.shape[-1] == self.space.n_x
        traj = self._rollout(x_0, steps)
        carry = carry_0.unsqueeze(-2).expand(carry_0.shape[:-1] + (steps + 1, carry_0.shape[-1]))
        return traj, carry


class MultibodyLearnableSystem(System):
    """Learnable rigid multibody system with contact (ContactNets loss + Anitescu step)."""

    def __init__(self, init_urdfs: Dict[str, str], dt: float, output_urdfs_dir: Optional[str] = None) -> None:
        multibody_terms = MultibodyTerms(init_urdfs)
        space = multibody_terms.spec.space()
        integrator = KernelVelocityIntegrator(space, self.sim_step, dt, self._rollout)
        super().__init__(space, integrator)
        self.multibody_terms = multibody_terms
        self.init_urdfs = init_urdfs
        self.output_urdfs_dir = output_urdfs_dir
        self.visualization_system = None
        self.solver = None      # the cone QP is solved inside the kernels (reference: sappy.SAPSolver(), :77)
        self.dt = dt
        self.set_carry_sampler(lambda: torch.Tensor([False]))
        self.max_batch_dim = 1
        # Extensions of the reference API (all off by default -> the reference's semantics):
        self.data_parallel = None        # parallel.PeerComm: loss.mean()/.sum() and gradients cover all ranks
        self.dynamic_schedule = False    # warps draw sample chunks in batch order (cost-ordered batches)
        self.race_expensive_head = True  # with dynamic_schedule, small launches: the first B/64 samples of the (cost-ordered)
                                         # batch are solved from eight start points at once, first to converge wins (cube)
        self.record_newton_iters = False  # BatchLoss.newton_iters: per-sample cost hint for the data set
        self.qp_warm_start = None        # (B, 6) / (B, 7) / (B, 5 + n) contiguous start points of the next contactnets_loss
                                         # call's solves (single body, elbow, trees of n links); with
                                         # record_qp_solution it is overwritten in place by the optima
        self.record_qp_solution = False  # BatchLoss.qp_solution (B, 6) / (B, 7) / (B, 5 + n): the optima, next epoch's
                                         # warm start (every system)
        self._kin_cache = {}

    # -- helpers ---------------------------------------------------------
    def _kind(self) -> str:
        return self.multibody_terms.spec.kind

    def _flat(self, t: Tensor) -> Tensor:
        return t.reshape(-1, t.shape[-1])

    def _cube_params(self, dtype: torch.dtype):
        inertia, mu, half = self.multibody_terms.kernel_parameters(dtype)
        return inertia.reshape(10), mu.reshape(1), (half[0] if half else None)

    def _body_witness_points(self, quat: Tensor):
        """(B,4) orientations -> ((B,4,3) witness points of the body geometry against the ground, n_contacts): the
        shape's support points in the direction -R^T e_z (geometry.py:560-567), rows beyond n_query zero.  A learned shape
        (DeepSupportConvex) answers through its network at the detached orientation: its support points are piecewise
        constant in the direction, so no gradient reaches the state through them (as the two-body system's)."""
        from dair_pll_b200.geometry import DeepSupportConvex
        geom = self.multibody_terms.contact_terms.geometries[0]
        learned = isinstance(geom, DeepSupportConvex)
        if learned:
            quat = quat.detach()
        if learned and geom.frame is None and quat.is_cuda and quat.dtype == torch.float64:
            # one launch for the perturbed, normalised directions; the network then evaluates them row by row
            p = geom.network(ops.body_support_directions(quat, geom.perturbations))
        else:
            w, x, y, z = quat.unbind(-1)
            s = 2.0 / (w * w + x * x + y * y + z * z)
            d = -torch.stack((s * (x * z - w * y), s * (y * z + w * x), 1 - s * (x * x + y * y)), -1)
            p = place_in_link_frame(geom, d)
        n_c = p.shape[-2]
        if n_c < 4:
            p = torch.cat((p, p.new_zeros(p.shape[:-2] + (4 - n_c, 3))), -2)
        return p, n_c

    def _elbow_kin(self, dtype: torch.dtype, device: torch.device):
        """URDF constants [joint origin | joint axis | box offsets] and the axis alone, created once per
        (dtype, device): no host->device copy (= host synchronisation) inside a step, so the elbow step can be
        captured into a CUDA graph like the cube's."""
        key = (dtype, str(device))
        if key not in self._kin_cache:
            spec = self.multibody_terms.spec
            joint = spec.joints[0]
            kin = torch.tensor([*joint.origin, *joint.axis, *spec.geometries[0].offset, *spec.geometries[1].offset],
                               dtype=dtype, device=device)
            self._kin_cache[key] = (kin, kin[3:6].clone())
        return self._kin_cache[key]

    def _elbow_params(self, dtype: torch.dtype, device: torch.device):
        inertia, mu, half = self.multibody_terms.kernel_parameters(dtype)
        kin, _ = self._elbow_kin(dtype, device)
        return inertia.reshape(20), mu.reshape(2), (torch.cat(half) if half else None), kin

    def _chain_boxes_only(self) -> bool:
        from dair_pll_b200.geometry import Box, Plane
        return all(isinstance(g, (Box, Plane)) for g in self.multibody_terms.contact_terms.geometries)

    def _chain_params(self, device: torch.device):
        """Generic kinematic tree: (inertia (n*10), mu (n), half (n*3), kin (n*31), n), float64.  The kernels have n box
        slots; the system's boxes (any distribution over the links, at most n) fill the first ones, the rest are switched off
        in the kinematic table and padded here (their gradient entries are dropped by the padding's autograd)."""
        inertia, mu, half = self.multibody_terms.kernel_parameters(torch.float64)
        spec = self.multibody_terms.spec
        n = len(spec.bodies)
        boxes = [g for g in spec.geometries if g.body >= 0]
        kin = self.multibody_terms.chain_kinematic_table(device)
        mu, half = mu.reshape(-1), torch.cat(half)
        if len(boxes) < n:
            mu = torch.cat((mu, mu.new_ones(n - len(boxes))))
            half = torch.cat((half, half.new_zeros(3 * (n - len(boxes)))))
        return inertia.reshape(-1), mu, half, kin, n

    def _elbow_witness_points(self, q: Tensor) -> Tensor:
        """(B, 8) configurations -> (B, 8, 3) witness points of the two learned geometries against the
        ground: support direction of geometry i = minus the third row of its world rotation
        (geometry.py:560-567), then ``DeepSupportConvex.get_vertices`` (:309-325)."""
        from dair_pll_b200.geometry import DeepSupportConvex
        geoms = self.multibody_terms.contact_terms.geometries
        _, axis = self._elbow_kin(q.dtype, q.device)
        if q.is_cuda and q.dtype == torch.float64 and all(isinstance(g, DeepSupportConvex) for g in geoms[:2]) \
                and geoms[0].n_query == geoms[1].n_query:
            # one launch for both links' perturbed, normalised directions; the networks then evaluate them row by row
            d0, d1 = ops.elbow_support_directions(q, axis, geoms[0].perturbations, geoms[1].perturbations)
            return torch.cat((geoms[0].network(d0), geoms[1].network(d1)), -2)
        w, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
        s = 2.0 / (w * w + x * x + y * y + z * z)
        row = torch.stack((s * (x * z - w * y), s * (y * z + w * x), 1 - s * (x * x + y * y)), -1)   # R1[2, :]
        th = q[:, 7:8]
        # third row of R2 = R1 Rot(axis, th):  r Rot = r cos + (r x a) sin + a (a.r)(1 - cos)
        row2 = row * torch.cos(th) + torch.linalg.cross(row, axis.expand_as(row)) * torch.sin(th) \
            + axis * (row @ axis)[:, None] * (1 - torch.cos(th))
        # per geometry: a learned shape answers through its network, a box (mixed box / mesh systems) with its corners --
        # ordinary torch functions of the box lengths, so the kernel's d loss / d witness point reaches them by autograd
        def points(geom, d):
            return geom.get_vertices(d) if isinstance(geom, DeepSupportConvex) else geom.support_points(d)
        return torch.cat((points(geoms[0], -row), points(geoms[1], -row2)), -2)

    # -- ContactNets loss --------------------------------------------------
    def contactnets_loss(self, x: Tensor, u: Tensor, x_plus: Tensor, loss_pool=None) -> Tensor:
        """(*, n_x), (*, 0), (*, n_x) -> (*,) ContactNets loss (:104-197)."""
        del u, loss_pool   # unactuated assets; the kernel needs no process pool
        assert x.shape[-1] == self.space.n_x and x_plus.shape == x.shape
        batch = x.shape[:-1]
        if self._kind() == 'cube' and self.multibody_terms.contact_terms.has_witness_point_geometry():
            # Sphere / Polygon / learned geometry: support points evaluated here, contact set handed to the witness-point
            # kernel, whose d loss / d points reaches the shape parameters (network weights) through autograd
            if self.data_parallel is not None:
                raise NotImplementedError('the in-kernel gradient exchange is provided for the box; use '
                                          'parallel.GradientAllReduce (NCCL) for this geometry')
            inertia, mu, _ = self._cube_params(torch.float64)
            xf, xpf = self._flat(x).to(torch.float64), self._flat(x_plus).to(torch.float64)
            pts, n_c = self._body_witness_points(xpf[:, :4])
            flags = ops.LOSS_DYNAMIC if self.dynamic_schedule else 0
            u_init = self._f64_warm_start(xf.shape[0], 6)
            res = ops.BodyWitnessPointLoss.apply(xf, xpf, inertia, mu, pts, n_c, float(self.dt), LOSS_EPS, flags,
                                                 self.record_newton_iters, u_init, self.record_qp_solution)
            loss, iters = res[0], res[1]
            out = loss.to(x.dtype).reshape(batch).as_subclass(ops.BatchLoss)
            out._dpll_fused = None           # mean() / sum() are plain reductions: the points' gradient needs the graph
            out.newton_iters = iters.reshape(batch) if self.record_newton_iters else None
            out.qp_solution = None
            if self.record_qp_solution:
                # with a warm start the optima were written back into the warm-start tensor itself
                out.qp_solution = (u_init if u_init is not None else res[2]).reshape(batch + (6,))
            return out
        if self._kind() == 'cube':
            lt, ct = self.multibody_terms.lagrangian_terms, self.multibody_terms.contact_terms
            # the learnable leaves go straight to the library (parameter preparation, multibody_terms.py:230-231,
            # 466-471, geometry.py:394-397, and its chain rule run on the device)
            leaves = (lt.inertial_parameters.to(x.dtype), ct.friction_params.to(x.dtype),
                      ct.geometries[0].length_params.to(x.dtype))
            flags = (ops.LOSS_DYNAMIC | (ops.LOSS_RACE if self.race_expensive_head else 0)) if self.dynamic_schedule else 0
            warm, self.qp_warm_start = self.qp_warm_start, None          # consumed by this call
            loss, sums, means, iters, usol = ops.CubeContactNetsLossLeaf.apply(
                self._flat(x), self._flat(x_plus), *leaves, float(self.dt), LOSS_EPS, flags, self.data_parallel,
                self.record_newton_iters, warm.reshape(-1, 6) if warm is not None else None, self.record_qp_solution)
            # loss.mean() / loss.sum() (drake_experiment.py:222-223) then come from this launch's own reduction
            out = ops.batch_loss(loss.reshape(batch), sums, means, 15, leaves,
                                 iters.reshape(batch) if self.record_newton_iters else None)
            if self.record_qp_solution:
                # with a warm start the optima were written back into the warm-start tensor itself
                out.qp_solution = (warm if warm is not None else usol).reshape(batch + (6,))
            return out
        elif self._kind() == 'elbow':
            if self.data_parallel is not None:
                raise NotImplementedError('the in-kernel gradient exchange is provided for the cube; use '
                                          'parallel.GradientAllReduce (NCCL) for this system')
            inertia, mu, half, kin = self._elbow_params(x.dtype, x.device)
            xf, xpf = self._flat(x), self._flat(x_plus)
            warm, self.qp_warm_start = self.qp_warm_start, None          # consumed by this call
            if warm is not None and (warm.shape[-1] != 7 or warm.numel() != 7 * xf.shape[0] or warm.dtype != x.dtype or
                                     (self.record_qp_solution and not warm.is_contiguous())):
                raise ValueError(f'qp_warm_start must be a contiguous ({xf.shape[0]}, 7) {x.dtype} tensor for this batch, '
                                 f'got {tuple(warm.shape)} {warm.dtype}')
            u_init = warm.reshape(-1, 7) if warm is not None else None
            if half is None:      # learned geometry: witness points from the support-function networks
                pts = self._elbow_witness_points(xpf[:, :8])
                if u_init is None and not self.record_qp_solution:
                    loss = ops.ElbowContactNetsLossPts.apply(xf, xpf, inertia, mu, pts, kin, float(self.dt), LOSS_EPS)
                    usol = None
                else:
                    loss, usol = ops.ElbowContactNetsLossPts.apply(xf, xpf, inertia, mu, pts, kin, float(self.dt), LOSS_EPS,
                                                                   u_init, self.record_qp_solution)
                out = loss.reshape(batch).as_subclass(ops.BatchLoss)
                out._dpll_fused = None           # mean() / sum() are plain reductions: the points' gradient needs the graph
                out.newton_iters = None
            else:
                flags = ops.LOSS_DYNAMIC if self.dynamic_schedule else 0
                loss, sums, means, iters, usol = ops.ElbowContactNetsLoss.apply(
                    xf, xpf, inertia, mu, half, kin, float(self.dt), LOSS_EPS, flags, self.record_newton_iters, u_init,
                    self.record_qp_solution)
                # mean() / sum() of the result reuse the launch's own reduction and fused gradient (ops.BatchLoss)
                out = ops.batch_loss(loss.reshape(batch), sums, means, 28, (inertia, mu, half),
                                     iters.reshape(batch) if self.record_newton_iters else None)
            out.qp_solution = None
            if self.record_qp_solution:
                # with a warm start the optima were written back into the warm-start tensor itself
                out.qp_solution = (warm if warm is not None else usol).reshape(batch + (7,))
            return out
        elif self._kind() == 'chain' and not self._chain_boxes_only():
            # other shapes than boxes on the links: each shape's support points (host side, ordinary torch functions of the
            # shape parameters) become the witness points of the tree kernels
            mt = self.multibody_terms
            n = len(mt.spec.bodies)
            inertia, mu, _ = mt.kernel_parameters(torch.float64)
            mu = mu.reshape(-1)
            if mu.shape[0] < n:
                mu = torch.cat((mu, mu.new_ones(n - mu.shape[0])))
            xf, xpf = self._flat(x).to(torch.float64), self._flat(x_plus).to(torch.float64)
            pts, packed = mt.chain_witness_points(xpf[:, :7 + n - 1])
            u_init = self._f64_warm_start(xf.shape[0], 5 + n)
            iters = torch.empty(xf.shape[0], dtype=torch.int32, device=x.device) if self.record_newton_iters else None
            out = ops.ChainWitnessPointLoss.apply(xf, xpf, inertia.reshape(-1), mu, pts, mt.chain_kinematic_table(x.device, True),
                                                  n, packed, float(self.dt), LOSS_EPS, u_init, self.record_qp_solution, iters)
        elif self._kind() == 'chain':
            inertia, mu, half, kin, n = self._chain_params(x.device)
            xf = self._flat(x).to(torch.float64)
            u_init = self._f64_warm_start(xf.shape[0], 5 + n)
            iters = torch.empty(xf.shape[0], dtype=torch.int32, device=x.device) if self.record_newton_iters else None
            out = ops.ChainContactNetsLoss.apply(xf, self._flat(x_plus).to(torch.float64), inertia, mu, half, kin, n,
                                                 float(self.dt), LOSS_EPS, u_init, self.record_qp_solution, iters)
        else:
            raise NotImplementedError(f'no kernel specialisation for system kind {self._kind()!r}')
        if u_init is None and not self.record_qp_solution and iters is None:
            return out.to(x.dtype).reshape(batch)
        loss, usol = out if (u_init is not None or self.record_qp_solution) else (out, None)
        result = loss.to(x.dtype).reshape(batch).as_subclass(ops.BatchLoss)
        result._dpll_fused = None                # mean() / sum() are plain reductions of the (B,) loss
        result.newton_iters = iters.reshape(batch) if iters is not None else None
        result.qp_solution = None
        if self.record_qp_solution:
            # with a warm start the optima were written back into the warm-start tensor itself
            result.qp_solution = (u_init if u_init is not None else usol).reshape(batch + (5 + n,))
        return result

    def _f64_warm_start(self, B: int, width: int):
        """Consumes ``qp_warm_start`` for the float64 kernels (trees, width 5 + n; the single body with witness points,
        width 6): None, or the (B, width) start points, contiguous when the optima are to be written into it."""
        warm, self.qp_warm_start = self.qp_warm_start, None          # consumed by this call
        if warm is None:
            return None
        if warm.shape[-1] != width or warm.numel() != width * B or warm.dtype != torch.float64 or \
                (self.record_qp_solution and not warm.is_contiguous()):
            raise ValueError(f'qp_warm_start must be a contiguous ({B}, {width}) torch.float64 tensor for this batch, '
                             f'got {tuple(warm.shape)} {warm.dtype}')
        return warm.reshape(B, width)

    # -- simulation ------------------------------------------------------
    def _rollout(self, x_0: Tensor, steps: int) -> Tensor:
        """(*, n_x) -> (*, steps+1, n_x)."""
        batch = x_0.shape[:-1]
        if self._kind() == 'cube' and self.multibody_terms.contact_terms.has_witness_point_geometry():
            # the witness points depend on the orientation: the time loop stays on the host, one step per launch
            if torch.is_grad_enabled() and (x_0.requires_grad or any(p.requires_grad for p in self.multibody_terms.parameters())):
                # differentiable (prediction loss): every step an autograd node (36-direction tangent kernel); the support
                # points are ordinary torch functions of the state and the shape parameters, so their cotangent reaches both
                inertia, mu, _ = self._cube_params(torch.float64)
                xs = [self._flat(x_0).to(torch.float64)]
                for _ in range(steps):
                    pts, n_c = self._body_witness_points(xs[-1][:, :4])
                    xs.append(ops.BodyStepPts.apply(xs[-1], inertia, mu, pts, n_c, float(self.dt), STEP_EPS))
                traj = torch.stack(xs, 1).to(x_0.dtype)
                return traj.reshape(batch + (steps + 1, self.space.n_x))
            with torch.no_grad():
                inertia, mu, _ = self._cube_params(torch.float64)
                xs = [self._flat(x_0).to(torch.float64)]
                for _ in range(steps):
                    pts, n_c = self._body_witness_points(xs[-1][:, :4])
                    xs.append(ops.body_step_pts(xs[-1], inertia, mu, pts, n_c, float(self.dt), STEP_EPS))
                traj = torch.stack(xs, 1).to(x_0.dtype)
            return traj.reshape(batch + (steps + 1, self.space.n_x))
        if self._kind() == 'cube':
            inertia, mu, half = self._cube_params(x_0.dtype)
            if torch.is_grad_enabled() and any(t.requires_grad for t in (x_0, inertia, mu, half)):
                # differentiable path (prediction loss): backward through every step's QP
                traj = ops.CubeRollout.apply(self._flat(x_0), inertia, mu, half, float(self.dt), steps, STEP_EPS)
            else:
                traj, _ = ops.cube_rollout(self._flat(x_0), inertia.detach(), mu.detach(), half.detach(),
                                           float(self.dt), steps, STEP_EPS)
        elif self._kind() == 'elbow':
            inertia, mu, half, kin = self._elbow_params(x_0.dtype, x_0.device)
            if half is None:
                # learned geometry: witness points depend on the state, so the time loop stays on the
                # host and every step is [support directions -> support networks -> one-step kernel]
                if torch.is_grad_enabled() and (x_0.requires_grad or
                                                any(p.requires_grad for p in self.multibody_terms.parameters())):
                    # differentiable (prediction loss trains the geometry): every step is an autograd node whose backward
                    # is the 61-direction tangent kernel; the points' cotangents reach the network weights through
                    # ICNNSupport (support points are piecewise constant in the direction: no chain through the state there)
                    xs = [self._flat(x_0)]
                    for _ in range(steps):
                        pts = self._elbow_witness_points(xs[-1][:, :8].detach())
                        xs.append(ops.ElbowStepPts.apply(xs[-1], inertia, mu, pts, kin, float(self.dt), STEP_EPS))
                    traj = torch.stack(xs, 1)
                else:
                    with torch.no_grad():
                        xs = [self._flat(x_0)]
                        for _ in range(steps):
                            pts = self._elbow_witness_points(xs[-1][:, :8])
                            one, _ = ops.elbow_rollout(xs[-1], inertia.detach(), mu.detach(), None, kin, float(self.dt), 1,
                                                       STEP_EPS, pts=pts)
                            xs.append(one[:, 1])
                        traj = torch.stack(xs, 1)
            elif torch.is_grad_enabled() and any(t.requires_grad for t in (x_0, inertia, mu, half)):
                traj = ops.ElbowRollout.apply(self._flat(x_0), inertia, mu, half, kin, float(self.dt), steps, STEP_EPS)
            else:
                traj, _ = ops.elbow_rollout(self._flat(x_0), inertia.detach(), mu.detach(), half.detach(), kin,
                                            float(self.dt), steps, STEP_EPS)
        elif self._kind() == 'chain' and not self._chain_boxes_only():
            # (the step with witness points exists in the device math and agrees with the reference on the host emulation;
            # its GPU entry point is not shipped: see DESIGN.md section 8)
            raise NotImplementedError('the time step of trees with non-box shapes has no GPU entry point yet (the ContactNets '
                                      'loss of such systems is provided; rollouts: boxes on trees, every shape on one or two '
                                      'bodies)')
        elif self._kind() == 'chain':
            inertia, mu, half, kin, n = self._chain_params(x_0.device)
            xf = self._flat(x_0).to(torch.float64)
            if torch.is_grad_enabled() and any(t.requires_grad for t in (x_0, inertia, mu, half)):
                traj = ops.ChainRollout.apply(xf, inertia, mu, half, kin, n, float(self.dt), steps, STEP_EPS).to(x_0.dtype)
            else:
                traj = ops.chain_rollout(xf.detach(), inertia.detach(), mu.detach(), half.detach(), kin, n, float(self.dt),
                                         steps, STEP_EPS).to(x_0.dtype)
        else:
            raise NotImplementedError(f'no kernel specialisation for system kind {self._kind()!r}')
        return traj.reshape(batch + (steps + 1, self.space.n_x))

    def forward_dynamics(self, q: Tensor, v: Tensor, u: Tensor, dynamics_pool=None) -> Tensor:
        """(*, n_q), (*, n_v) -> next velocity (*, n_v) by Anitescu's convex step (:199-304)."""
        del u, dynamics_pool
        x = self.space.x(q, v)
        return self.space.v(self._rollout(x, 1)[..., 1, :])

    def sim_step(self, x: Tensor, carry: Tensor) -> Tuple[Tensor, Tensor]:
        """``Integrator.partial_step`` callback (:306-313)."""
        q, v = self.space.q_v(x)
        return self.forward_dynamics(q, v, x.new_zeros(x.shape[:-1] + (0,))), carry

    def generate_updated_urdfs(self) -> Dict[str, str]:
        """Writes the current parameterisation back into copies of the initial URDFs (same basenames, in
        ``output_urdfs_dir``) and returns their paths, as the reference's method of the same name
        (multibody_learnable_system.py:82-102; urdf_utils.represent_multibody_terms_as_urdfs): per link the
        mass, centre of mass and inertia about it; per box collision geometry its size and friction
        coefficient.  Host side only.  Learned mesh geometries keep their original ``<mesh>`` element."""
        import xml.etree.ElementTree as ET
        assert self.output_urdfs_dir is not None
        os.makedirs(self.output_urdfs_dir, exist_ok=True)
        mt = self.multibody_terms
        pi_cm = mt.lagrangian_terms.pi_cm().detach().cpu().double()
        mu = mt.contact_terms.get_friction_coefficients().detach().cpu().double()
        fmt = lambda vals: ' '.join(repr(float(v)) for v in vals)      # noqa: E731
        new_urdfs = {}
        for name, old_path in self.init_urdfs.items():
            tree = ET.parse(old_path)
            gi = 0
            for bi, link in enumerate(tree.getroot().findall('link')):
                pi = pi_cm[bi]
                m = float(pi[0])
                inertial = link.find('inertial')
                inertial.find('mass').set('value', repr(m))
                origin = inertial.find('origin')
                if origin is None:
                    origin = ET.SubElement(inertial, 'origin')
                origin.set('xyz', fmt(pi[1:4] / m))
                origin.set('rpy', '0 0 0')
                ine = inertial.find('inertia')
                for key, val in zip(('ixx', 'iyy', 'izz', 'ixy', 'ixz', 'iyz'), pi[4:10]):
                    ine.set(key, repr(float(val)))
                for col in link.findall('collision'):
                    geometry = mt.contact_terms.geometries[gi]
                    box = col.find('geometry').find('box')
                    if box is not None:
                        box.set('size', fmt(2 * geometry.get_half_lengths().detach().cpu().double().reshape(3)))
                    for prox in col.iter():
                        if prox.tag.endswith('mu_static') or prox.tag.endswith('mu_dynamic'):
                            prox.set('value', repr(float(mu[gi])))
                    gi += 1
            new_path = os.path.join(self.output_urdfs_dir, os.path.basename(old_path))
            tree.write(new_path, xml_declaration=True, encoding='utf-8')
            new_urdfs[name] = new_path
        return new_urdfs

    def summary(self, statistics: Dict) -> SystemSummary:
        del statistics
        scalars, meshes = self.multibody_terms.scalars_and_meshes()
        return SystemSummary(scalars=scalars, videos={}, meshes=meshes)
