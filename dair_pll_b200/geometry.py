"""Learnable collision geometries: parameter containers mirroring ``dair_pll/geometry.py``.

The collision maths itself (top-k support points :162-202, plane-convex collision :553-582)
runs inside the CUDA kernels; these modules own the ``nn.Parameter`` s with the reference's
names and shapes so checkpoints interchange (``Box.length_params`` (1,3) :375-397).
``DeepSupportConvex`` (:255-364) owns the learned support-function network and the fixed direction
perturbations.  ``Sphere`` (:415-456) and ``Polygon`` (:220-252) evaluate their support points here (a scale /
a top-k gather over a handful of vertices) and hand them to the witness-point kernels
(``dpll_body_loss_pts_f64``).  Mesh-mesh collision (:584-643, fcl) is not provided.
"""
from typing import Dict

import torch
from torch import Tensor
from torch.nn import Module, Parameter

from dair_pll_b200.deep_support_function import HomogeneousICNN

_TOTAL_ORDERING = ['Plane', 'Polygon', 'Box', 'Sphere', 'DeepSupportConvex']  # geometry.py:46


def place_in_link_frame(geometry: 'CollisionGeometry', directions: Tensor) -> Tensor:
    """Support points (*, n, 3) of ``geometry`` for LINK-frame directions (*, 3), in the link frame: the query direction
    goes into the collision frame (R_BG^T d), the points come back (p_BG + R_BG p).  ``geometry.frame`` is None when the
    two frames coincide (multibody_terms.py:299-303: the reference gets R_WG, p_WG from Drake per geometry frame)."""
    if geometry.frame is None:
        return geometry.support_points(directions)
    offset, rot = (t.to(directions.dtype) for t in geometry.frame)
    return geometry.support_points(directions @ rot) @ rot.t() + offset


class CollisionGeometry(Module):
    """Base class; ``>`` / ``<`` follow the reference's type ordering used to orient pairs."""

    def set_frame(self, offset: Tensor, rotation: Tensor) -> None:
        """Collision frame in the link frame (URDF ``<collision><origin xyz rpy>``): non-persistent buffers, so they follow
        ``.to(device)`` and stay out of the state_dict (the reference keeps them inside Drake's plant)."""
        self.register_buffer('frame_offset', offset.to(torch.float64).reshape(3), persistent=False)
        self.register_buffer('frame_rotation', rotation.to(torch.float64).reshape(3, 3), persistent=False)

    @property
    def frame(self):
        """(offset (3,), rotation (3, 3)) or None when the collision frame is the link frame."""
        return (self.frame_offset, self.frame_rotation) if hasattr(self, 'frame_offset') else None

    def __ge__(self, other) -> bool:
        return _TOTAL_ORDERING.index(type(self).__name__) > _TOTAL_ORDERING.index(type(other).__name__)

    def __lt__(self, other) -> bool:
        return other.__ge__(self)

    def scalars(self) -> Dict[str, float]:
        raise NotImplementedError


class Plane(CollisionGeometry):
    """Half space z <= 0 in its own frame; no parameters."""

    def scalars(self) -> Dict[str, float]:
        return {}


class Box(CollisionGeometry):
    """Cuboid; learnable ``length_params`` whose absolute values are the half lengths."""

    def __init__(self, half_lengths: Tensor, n_query: int = 4) -> None:
        super().__init__()
        assert half_lengths.numel() == 3
        self.n_query = n_query
        self.length_params = Parameter(half_lengths.detach().clone().reshape(1, 3), requires_grad=True)

    def get_half_lengths(self) -> Tensor:
        return self.length_params.abs()

    def support_points(self, directions: Tensor) -> Tensor:
        """(*, 3) directions -> (*, n_query, 3): the ``n_query`` corners with the largest support, by ascending vertex
        index i = 4 x + 2 y + z, bit set = +h (geometry.py:39-41, 162-202, 399-403).  Used when the box sits in a
        collision frame of its own (the box kernels select the corners themselves)."""
        signs = torch.tensor([[(i >> 2) & 1, (i >> 1) & 1, i & 1] for i in range(8)], dtype=directions.dtype,
                             device=directions.device) * 2 - 1
        verts = signs * self.get_half_lengths().to(directions.dtype)
        sel = torch.topk(directions @ verts.t(), self.n_query, dim=-1, sorted=False).indices
        sel, _ = torch.sort(sel, dim=-1)
        return verts[sel]

    def scalars(self) -> Dict[str, float]:
        return {f'len_{ax}': 2 * v.item() for ax, v in zip('xyz', self.get_half_lengths().reshape(-1))}


class Sphere(CollisionGeometry):
    """Sphere by its support function (geometry.py:415-456): one witness point ``direction * |length_param|``."""
    n_query = 1

    def __init__(self, radius: Tensor) -> None:
        super().__init__()
        assert radius.numel() == 1
        self.length_param = Parameter(radius.detach().clone().to(torch.float64).reshape(()), requires_grad=True)

    def get_radius(self) -> Tensor:
        return self.length_param.abs()

    def support_points(self, directions: Tensor) -> Tensor:
        """(*, 3) unit directions -> (*, 1, 3)."""
        return (directions * self.get_radius().to(directions.dtype)).unsqueeze(-2)

    def scalars(self) -> Dict[str, float]:
        return {'radius': self.get_radius().item()}


class Polygon(CollisionGeometry):
    """Convex polytope given by its vertices (geometry.py:220-252): the witness points are the ``n_query``
    vertices with the largest support in the query direction (geometry.py:162-202; returned by ascending vertex
    index, the reference's order is unspecified)."""

    def __init__(self, vertices: Tensor, n_query: int = 4) -> None:
        super().__init__()
        assert vertices.dim() == 2 and vertices.shape[1] == 3 and vertices.shape[0] >= n_query
        self.n_query = n_query
        self.vertices = Parameter(vertices.detach().clone().to(torch.float64), requires_grad=True)

    def support_points(self, directions: Tensor) -> Tensor:
        """(*, 3) directions -> (*, n_query, 3)."""
        verts = self.vertices.to(directions.dtype)
        dots = directions @ verts.t()
        sel = torch.topk(dots, self.n_query, dim=-1, sorted=False).indices
        sel, _ = torch.sort(sel, dim=-1)
        return verts[sel]

    def scalars(self) -> Dict[str, float]:
        out = {}
        for axis, values in zip('xyz', self.vertices.t()):
            for i, v in enumerate(values):
                out[f'v{i}_{axis}'] = v.item()
        return out


class DeepSupportConvex(CollisionGeometry):
    """Convex shape represented by its learned support function (geometry.py:255-325): the witness
    points against a plane are the network's support points in ``n_query`` directions -- the support
    direction itself plus ``n_query - 1`` randomly perturbed copies, fixed at construction."""

    def __init__(self, vertices: Tensor, n_query: int = 4, depth: int = 2, width: int = 256,
                 perturbation: float = 0.4) -> None:
        super().__init__()
        self.n_query = n_query
        vertices = vertices.to(torch.float64)
        length_scale = (vertices.max(dim=0).values - vertices.min(dim=0).values).norm() / 2
        self.network = HomogeneousICNN(depth, width, scale=length_scale.item())
        # plain attribute in the reference (not in state_dict); a non-persistent buffer follows .to(device)
        self.register_buffer('perturbations', torch.cat((
            torch.zeros((1, 3), dtype=torch.float64),
            perturbation * (torch.rand((n_query - 1, 3), dtype=torch.float64) - 0.5))), persistent=False)

    def get_vertices(self, directions: Tensor) -> Tensor:
        """(*, 3) support directions -> (*, n_query, 3) support points (geometry.py:309-325)."""
        perturbed = directions.unsqueeze(-2) + self.perturbations.to(directions.dtype)
        perturbed = perturbed / perturbed.norm(dim=-1, keepdim=True)
        return self.network(perturbed)

    def support_points(self, directions: Tensor) -> Tensor:
        """The witness points for (*, 3) directions, as every shape answers them (``get_vertices``)."""
        return self.get_vertices(directions)

    def scalars(self) -> Dict[str, float]:
        return {}
