"""Learnable multibody parameters with the reference's module tree and parameter names.

Mirror of ``dair_pll/multibody_terms.py``: ``MultibodyTerms`` owns ``lagrangian_terms``
(``inertial_parameters`` theta, (n_bodies,10), :156) and ``contact_terms``
(``friction_params`` (n_geometries,), :317; ``geometries`` ModuleList, :312;
``collision_candidates``, :319) so ``state_dict()`` keys are identical.  The per-sample
evaluation of M, F, phi, J (``forward`` methods :214-237, :428-521, :584-609) happens in
the CUDA kernels; what stays here is the per-*batch* parameter preparation
(theta -> [m, c, I_cm/m], |friction| and Drake's pairwise combination, |length_params|),
kept in PyTorch so autograd chains the kernels' callable-level gradients to the leaves.
"""
from typing import List, Tuple

import torch
from torch import Tensor
from torch.nn import Module, ModuleList, Parameter

from dair_pll_b200.geometry import Box, DeepSupportConvex, Plane, Polygon, Sphere
from dair_pll_b200.inertia import InertialParameterConverter
from dair_pll_b200.system_spec import SystemSpec


class LagrangianTerms(Module):
    """Owns theta; ``inertia_vector()`` is what the generated callables / kernels consume."""

    def __init__(self, spec: SystemSpec) -> None:
        super().__init__()
        pi_cm = torch.stack([b.pi_cm() for b in spec.bodies])
        self.inertial_parameters = Parameter(InertialParameterConverter.pi_cm_to_theta(pi_cm),
                                             requires_grad=True)

    def pi_cm(self) -> Tensor:
        return InertialParameterConverter.theta_to_pi_cm(self.inertial_parameters)

    def inertia_vector(self) -> Tensor:
        """(n_bodies, 10) [m, c, I_cm/m] (multibody_terms.py:230-231)."""
        return InertialParameterConverter.pi_cm_to_drake_spatial_inertia(self.pi_cm())


class ContactTerms(Module):
    """Owns friction and geometry parameters."""

    def __init__(self, spec: SystemSpec) -> None:
        super().__init__()
        geoms = []
        for g in spec.geometries:
            if g.kind == 'box':
                geoms.append(Box(torch.tensor(g.half_lengths, dtype=torch.float64), 4))
            elif g.kind == 'sphere':
                geoms.append(Sphere(torch.tensor(g.radius, dtype=torch.float64)))
            elif g.kind == 'plane':
                geoms.append(Plane())
            elif g.kind == 'mesh':
                geoms.append(DeepSupportConvex(g.mesh_vertices()))
            else:
                raise NotImplementedError(f'geometry kind {g.kind!r}')
        if spec.kind == 'cube':
            # single floating body: a collision frame of its own is honoured through the witness-point kernels
            # (the multi-link kernels take the frame offsets in their kinematic table instead)
            for geom, g in zip(geoms, spec.geometries):
                if g.body >= 0 and g.has_frame():
                    geom.set_frame(torch.tensor(g.offset, dtype=torch.float64), g.rotation())
        self.geometries = ModuleList(geoms)
        self.friction_params = Parameter(torch.tensor([g.mu for g in spec.geometries], dtype=torch.float64),
                                         requires_grad=True)
        # (2, n_pairs): row 0 = geometry a (Plane sorts first, geometry.py:46), row 1 = geometry b
        self._pairs = [tuple(int(i) for i in pair) for pair in spec.collision_pairs]    # host copy: no device reads
        self.register_buffer('collision_candidates',
                             torch.tensor(spec.collision_pairs, dtype=torch.long).t().contiguous(),
                             persistent=False)

    def get_friction_coefficients(self) -> Tensor:
        return self.friction_params.abs()

    def pair_index32(self) -> Tensor:
        """(2, n_pairs) int32 copy of ``collision_candidates`` on the parameters' device (created once per device)."""
        dev = self.friction_params.device
        if getattr(self, '_pair32', None) is None or self._pair32.device != dev:
            self._pair32 = torch.tensor(list(zip(*self._pairs)), dtype=torch.int32, device=dev).reshape(2, -1).contiguous()
        return self._pair32

    def pair_friction(self) -> Tensor:
        """(n_pairs,) combined coefficient 2 mu_a mu_b / (mu_a + mu_b) (multibody_terms.py:466-471)."""
        mu = self.get_friction_coefficients()
        mu_a, mu_b = mu[self.collision_candidates[0]], mu[self.collision_candidates[1]]
        return 2 * mu_a * mu_b / (mu_a + mu_b)

    def half_lengths(self) -> List[Tensor]:
        """|length_params| (3,) of each pair's body geometry, in pair order (boxes only)."""
        return [self.geometries[b].get_half_lengths().reshape(3) for _, b in self._pairs]

    def has_learned_geometry(self) -> bool:
        return any(isinstance(g, DeepSupportConvex) for g in self.geometries)

    def has_witness_point_geometry(self) -> bool:
        """True if a body geometry is evaluated through its support points here (Sphere, Polygon, DeepSupportConvex, or
        any shape that sits in a collision frame of its own)."""
        return any(isinstance(g, (Sphere, Polygon, DeepSupportConvex)) or g.frame is not None for g in self.geometries)


class MultibodyTerms(Module):
    """Container for the learnable dynamics parameters of a URDF system."""

    def __init__(self, urdfs) -> None:
        super().__init__()
        self.urdfs = urdfs
        self.spec = SystemSpec.from_urdfs(urdfs)
        self.lagrangian_terms = LagrangianTerms(self.spec)
        self.contact_terms = ContactTerms(self.spec)
        self.geometry_body_assignment = {
            b.name: [gi for gi, g in enumerate(self.spec.geometries) if g.body == bi]
            for bi, b in enumerate(self.spec.bodies)}

    def kernel_parameters(self, dtype: torch.dtype) -> Tuple[Tensor, Tensor, List[Tensor]]:
        """Callable-level parameters in the kernels' dtype, differentiable w.r.t. the leaves.  float64 on a CUDA device:
        one launch (``ops.LeafPrepare``, and one more for the chain rule) instead of the elementwise PyTorch graph."""
        lt, ct = self.lagrangian_terms, self.contact_terms
        boxes = not (ct.has_learned_geometry() or ct.has_witness_point_geometry())
        theta = lt.inertial_parameters
        if theta.is_cuda and dtype == torch.float64 and theta.dtype == torch.float64:
            from dair_pll_b200 import ops
            if boxes:
                length = torch.cat([ct.geometries[b].length_params.reshape(3) for _, b in ct._pairs])
            else:
                length = theta.new_empty(0)
            inertia, mu, half = ops.LeafPrepare.apply(theta, ct.friction_params, ct.pair_index32(), length)
            return inertia, mu, (list(half.reshape(-1, 3).unbind(0)) if boxes else [])
        inertia = lt.inertia_vector().to(dtype)
        mu = ct.pair_friction().to(dtype)
        if not boxes:
            return inertia, mu, []
        half = [h.to(dtype) for h in ct.half_lengths()]
        return inertia, mu, half

    def forward(self, q: Tensor, v: Tensor, u: Tensor = None):
        """(delassus, M, J, phi, non_contact_acceleration) as ``MultibodyTerms.forward`` of the reference
        (multibody_terms.py:584-609), evaluated by the terms kernels (float64, no autograd; contacts
        ordered by geometry, then box-vertex index).  The loss and step kernels do not go through these matrices."""
        from dair_pll_b200 import ops
        del u
        batch = q.shape[:-1]
        inertia, mu, half = self.kernel_parameters(q.dtype)
        if self.spec.kind == 'cube':
            if self.contact_terms.has_witness_point_geometry():
                raise NotImplementedError('dense terms export is provided for a box in the link frame (other shapes and '
                                          'framed boxes go through the witness-point kernels)')
            D, M, J, phi, acc = ops.cube_terms(q.reshape(-1, 7), v.reshape(-1, 6), inertia.detach().reshape(10),
                                               mu.detach().reshape(1), half[0].detach())
        elif self.spec.kind == 'elbow':
            if not half:
                raise NotImplementedError('dense terms export is provided for box geometries (witness points of a '
                                          'learned geometry come from the support-function networks)')
            joint = self.spec.joints[0]
            kin = torch.tensor([*joint.origin, *joint.axis, *self.spec.geometries[0].offset,
                                *self.spec.geometries[1].offset], dtype=q.dtype, device=q.device)
            D, M, J, phi, acc = ops.elbow_terms(q.reshape(-1, 8), v.reshape(-1, 7), inertia.detach().reshape(20),
                                                mu.detach().reshape(2), torch.cat(half).detach(), kin)
        elif self.spec.kind == 'chain':
            if not half:
                raise NotImplementedError('dense terms export is provided for box geometries (other shapes reach the tree '
                                          'kernels as witness points)')
            n = len(self.spec.bodies)
            n_boxes = len(half)
            kin = self.chain_kinematic_table(q.device)
            mu_s, half_s = mu.detach().reshape(-1), torch.cat(half).detach()
            if n_boxes < n:                      # the kernels have n box slots; the unused ones are switched off in `kin`
                mu_s = torch.cat((mu_s, mu_s.new_ones(n - n_boxes)))
                half_s = torch.cat((half_s, half_s.new_zeros(3 * (n - n_boxes))))
            D, M, J, phi, acc = ops.chain_terms(q.reshape(-1, 7 + n - 1), v.reshape(-1, 6 + n - 1), inertia.detach().reshape(-1),
                                                mu_s, half_s, kin, n, n_boxes)
        else:
            raise NotImplementedError(f'no kernel specialisation for system kind {self.spec.kind!r}')
        n_v, k, n_c = M.shape[-1], J.shape[-2], phi.shape[-1]
        return (D.reshape(batch + (k, k)), M.reshape(batch + (n_v, n_v)), J.reshape(batch + (k, n_v)),
                phi.reshape(batch + (n_c,)), acc.reshape(batch + (n_v,)))

    def chain_kinematic_table(self, device, witness: bool = False) -> Tensor:
        """(n * 31,) float64 kinematic table of the generic tree kernels (include/dair_pll_b200.h, dpll_chain_loss_f64):
        per row the link's joint and the box slot of the same index; created once per device.  ``witness``: the table of the
        witness-point entry points -- the points arrive in link coordinates, so the slots carry no placement of their own."""
        key = (str(device), witness)
        cache = self.__dict__.setdefault('_chain_kin_cache', {})
        if key not in cache:
            spec = self.spec
            boxes = [g for g in spec.geometries if g.body >= 0]
            rows = []
            for b in range(len(spec.bodies)):
                if b == 0:
                    rows += [0.] * 3 + [1., 0., 0., 0., 1., 0., 0., 0., 1.] + [0., 0., 1.]
                    parent, sliding = 0, 0.
                else:
                    j = spec.joints[b - 1]          # joint b - 1 is the one whose child is link b (SystemSpec orders them)
                    rows += [*j.origin, *j.rotation(), *j.axis]
                    parent, sliding = j.parent, float(j.prismatic)
                if b < len(boxes) and witness:
                    rows += [0., 0., 0., float(parent), 1., 0., 0., 0., 1., 0., 0., 0., 1., sliding, float(boxes[b].body), 1.]
                elif b < len(boxes):
                    g = boxes[b]
                    rows += [*g.offset, float(parent), *g.rotation().reshape(-1).tolist(), sliding, float(g.body), 1.]
                else:
                    rows += [0., 0., 0., float(parent), 1., 0., 0., 0., 1., 0., 0., 0., 1., sliding, 0., 0.]
            cache[key] = torch.tensor(rows, dtype=torch.float64, device=device)
        return cache[key]

    def chain_link_rotations(self, q: Tensor) -> Tensor:
        """(B, n_q) configurations of a tree -> (B, n, 3, 3) world rotations of its links: R_0 from the (not necessarily unit)
        base quaternion as Drake forms it, R_b = R_parent Rfix_b Rot(axis_b, q_b) (a sliding joint keeps its joint frame's
        orientation).  Plain torch: the witness points of non-box shapes are evaluated on the host side of the kernels."""
        from dair_pll_b200.system_spec import _rpy_matrix
        w, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
        s = 2.0 / (w * w + x * x + y * y + z * z)
        R0 = torch.stack((torch.stack((1 - s * (y * y + z * z), s * (x * y - w * z), s * (x * z + w * y)), -1),
                          torch.stack((s * (x * y + w * z), 1 - s * (x * x + z * z), s * (y * z - w * x)), -1),
                          torch.stack((s * (x * z - w * y), s * (y * z + w * x), 1 - s * (x * x + y * y)), -1)), -2)
        rots = [R0]
        for b, joint in enumerate(self.spec.joints, start=1):
            Rfix = _rpy_matrix(joint.rpy).to(q)
            R = rots[joint.parent] @ Rfix
            if not joint.prismatic:
                a = torch.tensor(joint.axis, dtype=q.dtype, device=q.device)
                K = torch.zeros(3, 3, dtype=q.dtype, device=q.device)
                K[0, 1], K[0, 2], K[1, 0], K[1, 2], K[2, 0], K[2, 1] = -a[2], a[1], a[2], -a[0], -a[1], a[0]
                th = q[:, 6 + b]
                Rj = torch.eye(3, dtype=q.dtype, device=q.device) + torch.sin(th)[:, None, None] * K \
                    + (1 - torch.cos(th))[:, None, None] * (K @ K)
                R = R @ Rj
            rots.append(R)
        return torch.stack(rots, 1)

    def chain_witness_points(self, q: Tensor):
        """Witness points of every body geometry of a tree against the ground, in the frame of the geometry's LINK:
        ((B, n_slots, 4, 3) with unused rows zero, per-slot point counts packed 3 bits each) -- each shape's support points
        (geometry.py:553-582) in the direction -R_WG^T e_z, placed by the collision frame's offset and rotation."""
        R = self.chain_link_rotations(q)
        n = len(self.spec.bodies)
        pts, packed = [], 0
        bodies = [g for g in self.spec.geometries if g.body >= 0]
        for slot, (gs, geom) in enumerate(zip(bodies, self.contact_terms.geometries)):
            d_link = -R[:, gs.body, 2, :]
            Rg = gs.rotation().to(q)
            off = torch.tensor(gs.offset, dtype=q.dtype, device=q.device)
            d_geom = d_link @ Rg
            from dair_pll_b200.geometry import DeepSupportConvex
            p = geom.get_vertices(d_geom) if isinstance(geom, DeepSupportConvex) else geom.support_points(d_geom)
            k = p.shape[-2]
            p = p @ Rg.t() + off
            if k < 4:
                p = torch.cat((p, p.new_zeros(p.shape[:-2] + (4 - k, 3))), -2)
            pts.append(p)
            packed |= k << (3 * slot)
        for _ in range(n - len(bodies)):
            pts.append(q.new_zeros((q.shape[0], 4, 3)))
        return torch.stack(pts, 1), packed

    def scalars_and_meshes(self):
        """Summary scalars per body and, for learned (``DeepSupportConvex``) geometries, the extracted mesh with its
        bounding-box diameters and centre (multibody_terms.py:536-582)."""
        from dair_pll_b200.deep_support_function import extract_mesh
        from dair_pll_b200.geometry import DeepSupportConvex
        scalars, meshes = {}, {}
        mu = self.contact_terms.get_friction_coefficients()
        for body, pi in zip(self.spec.bodies, self.lagrangian_terms.pi_cm()):
            for k, val in InertialParameterConverter.pi_cm_to_scalars(pi).items():
                scalars[f'{body.name}_{k}'] = val
            for gi in self.geometry_body_assignment[body.name]:
                for k, val in self.contact_terms.geometries[gi].scalars().items():
                    scalars[f'{body.name}_{k}'] = val
                scalars[f'{body.name}_mu'] = mu[gi].item()
                geometry = self.contact_terms.geometries[gi]
                if isinstance(geometry, DeepSupportConvex):
                    mesh = extract_mesh(geometry.network)
                    meshes[body.name] = mesh
                    lo, hi = mesh.vertices.min(dim=0).values, mesh.vertices.max(dim=0).values
                    for axis, dia, cen in zip('xyz', hi - lo, lo + (hi - lo) / 2):
                        scalars[f'{body.name}_diameter_{axis}'] = dia.item()
                        scalars[f'{body.name}_center_{axis}'] = cen.item()
        return scalars, meshes
