"""Host-side model ingestion: URDF -> :class:`SystemSpec`.

In the reference this is done by pydrake (``drake_utils.MultibodyPlantDiagram``,
drake_utils.py:227-335) followed by symbolic derivation (multibody_terms.py:114-157,
267-319).  pydrake is not a dependency here: the two kinematic classes the kernels
specialise (a single floating body; a floating body plus one revolute child) are read
straight from the URDF XML.  Conventions reproduced from the reference:

* a ground half-space z = 0 with mu = 1 is always added (drake_utils.py:280-288) and is
  the LAST geometry; body geometries come first, in link order;
* every (ground, body-geometry) pair is a collision candidate; body-body pairs inside one
  URDF's ``collision_filter_group`` are filtered (contactnets_elbow.urdf:74-78);
* theta is initialised from the URDF inertia via pi_cm -> pi_o -> theta
  (multibody_terms.py:194-196);
* state space = ProductSpace([FixedBaseSpace(0) (world), FloatingBaseSpace(n_joints)])
  (drake_utils.py:309-335).
"""
import os
import xml.etree.ElementTree as ET
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch

from dair_pll_b200.state_space import FixedBaseSpace, FloatingBaseSpace, ProductSpace


def _floats(text: Optional[str], n: int, default: float = 0.0) -> Tuple[float, ...]:
    if text is None:
        return tuple([default] * n)
    vals = tuple(float(t) for t in text.split())
    assert len(vals) == n, f'expected {n} numbers, got {text!r}'
    return vals


@dataclass
class BodySpec:
    name: str
    mass: float
    com: Tuple[float, float, float]
    inertia_cm: Tuple[float, float, float, float, float, float]   # xx, yy, zz, xy, xz, yz

    def pi_cm(self) -> torch.Tensor:
        m = self.mass
        return torch.tensor([m, m * self.com[0], m * self.com[1], m * self.com[2], *self.inertia_cm],
                            dtype=torch.float64)


@dataclass
class GeometrySpec:
    body: int                                   # index into bodies, -1 = world
    kind: str                                   # 'box' | 'sphere' | 'mesh' | 'plane'
    offset: Tuple[float, float, float] = (0., 0., 0.)
    half_lengths: Optional[Tuple[float, float, float]] = None
    mesh_file: Optional[str] = None
    mu: float = 1.0
    radius: Optional[float] = None
    rpy: Tuple[float, float, float] = (0., 0., 0.)   # fixed rotation link frame -> collision frame (<collision><origin rpy>)

    def has_frame(self) -> bool:
        """True if the collision frame differs from the link frame."""
        return any(abs(a) > 0 for a in self.offset) or any(abs(a) > 0 for a in self.rpy)

    def rotation(self) -> torch.Tensor:
        """(3, 3) link frame <- collision frame, URDF convention R = Rz(yaw) Ry(pitch) Rx(roll)."""
        return _rpy_matrix(self.rpy)

    def mesh_vertices(self) -> torch.Tensor:
        """Vertices of the Wavefront .obj (only ``v x y z`` records are needed: the reference uses them
        for the initial length scale of the support-function network, geometry.py:303-305)."""
        verts = []
        with open(self.mesh_file) as fh:
            for line in fh:
                parts = line.split()
                if len(parts) >= 4 and parts[0] == 'v':
                    verts.append([float(v) for v in parts[1:4]])
        return torch.tensor(verts, dtype=torch.float64)


@dataclass
class JointSpec:
    parent: int
    child: int
    origin: Tuple[float, float, float]
    axis: Tuple[float, float, float]
    rpy: Tuple[float, float, float] = (0., 0., 0.)        # fixed rotation parent link -> joint frame
    prismatic: bool = False                               # slides along the axis (URDF type="prismatic") instead of turning

    def rotation(self) -> Tuple[float, ...]:
        """Row-major 3x3 of the URDF rotation R = Rz(yaw) Ry(pitch) Rx(roll)."""
        return tuple(_rpy_matrix(self.rpy).reshape(-1).tolist())


def _rpy_matrix(rpy) -> torch.Tensor:
    r, p, y = (torch.tensor(float(v), dtype=torch.float64) for v in rpy)
    cr, sr, cp, sp, cy, sy = torch.cos(r), torch.sin(r), torch.cos(p), torch.sin(p), torch.cos(y), torch.sin(y)
    Rx = torch.stack((torch.stack((torch.ones(()).double(), torch.zeros(()).double(), torch.zeros(()).double())),
                      torch.stack((torch.zeros(()).double(), cr, -sr)), torch.stack((torch.zeros(()).double(), sr, cr))))
    Ry = torch.stack((torch.stack((cp, torch.zeros(()).double(), sp)),
                      torch.stack((torch.zeros(()).double(), torch.ones(()).double(), torch.zeros(()).double())),
                      torch.stack((-sp, torch.zeros(()).double(), cp))))
    Rz = torch.stack((torch.stack((cy, -sy, torch.zeros(()).double())), torch.stack((sy, cy, torch.zeros(()).double())),
                      torch.stack((torch.zeros(()).double(), torch.zeros(()).double(), torch.ones(()).double()))))
    return Rz @ Ry @ Rx


@dataclass
class SystemSpec:
    kind: str                                   # 'cube' (1 floating body) | 'elbow' (+1 hinge) | 'chain' (generic tree, <= 6 links)
    bodies: List[BodySpec]
    joints: List[JointSpec]
    geometries: List[GeometrySpec]              # body geometries first, ground last
    collision_pairs: List[Tuple[int, int]] = field(default_factory=list)   # (ground, body geometry)

    @property
    def n_joints(self) -> int:
        return len(self.joints)

    @property
    def n_q(self) -> int:
        return 7 + self.n_joints

    @property
    def n_v(self) -> int:
        return 6 + self.n_joints

    @property
    def n_x(self) -> int:
        return self.n_q + self.n_v

    @property
    def n_contacts(self) -> int:
        return 4 * len(self.collision_pairs)    # n_query = 4 per pair (geometry.py:48-49, 491)

    def space(self) -> ProductSpace:
        return ProductSpace([FixedBaseSpace(0), FloatingBaseSpace(self.n_joints)])

    @staticmethod
    def from_urdfs(urdfs: Dict[str, str]) -> 'SystemSpec':
        if len(urdfs) != 1:
            raise NotImplementedError('one URDF (one kinematic chain) per system is supported')
        (path,) = urdfs.values()
        return SystemSpec.from_urdf(path)

    @staticmethod
    def from_urdf(path: str) -> 'SystemSpec':
        root = ET.parse(path).getroot()
        bodies, geometries, names = [], [], []
        for link in root.findall('link'):
            inertial = link.find('inertial')
            if inertial is None:
                raise NotImplementedError(f'link {link.get("name")} has no <inertial>')
            origin = inertial.find('origin')
            com = _floats(origin.get('xyz') if origin is not None else None, 3)
            ine = inertial.find('inertia')
            inertia_cm = tuple(float(ine.get(k)) for k in ('ixx', 'iyy', 'izz', 'ixy', 'ixz', 'iyz'))
            irpy = _floats(origin.get('rpy'), 3) if origin is not None else (0., 0., 0.)
            if any(abs(a) > 0 for a in irpy):
                # a rotated inertial frame only re-expresses the constant inertia tensor: I_link = R I R^T (on the host)
                xx, yy, zz, xy, xz, yz = inertia_cm
                I = torch.tensor([[xx, xy, xz], [xy, yy, yz], [xz, yz, zz]], dtype=torch.float64)
                R = _rpy_matrix(irpy)
                I = R @ I @ R.t()
                inertia_cm = (I[0, 0].item(), I[1, 1].item(), I[2, 2].item(), I[0, 1].item(), I[0, 2].item(), I[1, 2].item())
            names.append(link.get('name'))
            bodies.append(BodySpec(link.get('name'), float(inertial.find('mass').get('value')), com, inertia_cm))
            for col in link.findall('collision'):
                corigin = col.find('origin')
                offset = _floats(corigin.get('xyz') if corigin is not None else None, 3)
                crpy = _floats(corigin.get('rpy'), 3) if corigin is not None else (0., 0., 0.)
                mu = 1.0
                for prox in col.iter():
                    if prox.tag.endswith('mu_static'):
                        mu = float(prox.get('value'))
                geom = col.find('geometry')
                box, mesh, sphere = geom.find('box'), geom.find('mesh'), geom.find('sphere')
                if sphere is not None:
                    geometries.append(GeometrySpec(len(bodies) - 1, 'sphere', offset, None, None, mu,
                                                   float(sphere.get('radius')), crpy))
                elif box is not None:
                    size = _floats(box.get('size'), 3)
                    geometries.append(GeometrySpec(len(bodies) - 1, 'box', offset,
                                                   tuple(0.5 * s for s in size), None, mu, None, crpy))
                elif mesh is not None:
                    fname = mesh.get('filename')
                    if not os.path.isabs(fname):
                        fname = os.path.join(os.path.dirname(os.path.abspath(path)), fname)
                    geometries.append(GeometrySpec(len(bodies) - 1, 'mesh', offset, None, fname, mu, None, crpy))
                else:
                    raise NotImplementedError('only <box>, <sphere> and <mesh> collision geometries are supported')
        joints = []
        for joint in root.findall('joint'):
            if joint.get('type') not in ('continuous', 'revolute', 'prismatic'):
                raise NotImplementedError(f'joint type {joint.get("type")}')
            jo = joint.find('origin')
            jrpy = _floats(jo.get('rpy'), 3) if jo is not None else (0., 0., 0.)
            axis = joint.find('axis')
            ax = _floats(axis.get('xyz') if axis is not None else '1 0 0', 3)
            norm = sum(a * a for a in ax) ** 0.5
            if norm == 0:
                raise ValueError(f'joint {joint.get("name")} has a zero axis')
            joints.append(JointSpec(names.index(joint.find('parent').get('link')),
                                    names.index(joint.find('child').get('link')),
                                    _floats(jo.get('xyz') if jo is not None else None, 3),
                                    tuple(a / norm for a in ax), jrpy,   # Drake normalises the axis on parsing
                                    joint.get('type') == 'prismatic'))
        # a kinematic tree listed root first: joint k's child is link k + 1 (so joint order = link order, which is also the
        # order of the joint coordinates in the state) and its parent is any earlier link
        tree = len(joints) == len(bodies) - 1 and all(j.child == k + 1 and 0 <= j.parent <= k for k, j in enumerate(joints))
        serial = tree and all(j.parent == k for k, j in enumerate(joints))
        rotated = any(any(abs(a) > 0 for a in j.rpy) for j in joints)
        if len(bodies) == 1 and not joints:
            kind = 'cube'
        elif len(bodies) == 2 and serial and not rotated and not joints[0].prismatic \
                and [g.body for g in geometries] == [0, 1] \
                and not any(any(abs(a) > 0 for a in g.rpy) for g in geometries):
            kind = 'elbow'                      # the specialised two-body kernels (unrotated joint and collision frames)
        elif 2 <= len(bodies) <= 6 and tree:
            kind = 'chain'                      # generic tree (csrc/cn_chain.cuh): serial or branching, rotated joint frames
        else:
            raise NotImplementedError(
                'kernels cover a single floating body, a floating body with one revolute child, and kinematic trees of up '
                'to 6 links joined by revolute or prismatic joints, links listed root first with joint k leading to link k + 1; larger '
                'trees need the symbolic path (SURVEY.md section 8(f) N2)')
        if kind == 'cube':
            if len(geometries) != 1:
                raise NotImplementedError('the single-body kernels take exactly one collision geometry')
            if geometries[0].kind not in ('box', 'sphere', 'mesh'):
                raise NotImplementedError('the single-body kernels take a <box>, <sphere> or <mesh> (learned geometry) '
                                          'collision geometry (a Polygon is set through the module API)')
            # a collision frame that differs from the link frame (offset and / or rotation) is handled through the
            # witness-point kernels: the contact points are support points of the shape, moved into the link frame
        elif kind == 'chain':
            # the generic tree kernels have as many box slots as links; a slot may sit on any link, so the boxes can be spread
            # over the links in any way (several on one link, none on another) as long as there are no more boxes than links
            # (boxes go to the kernels as lengths; spheres, meshes and any mix of shapes as witness points per slot)
            if not 1 <= len(geometries) <= len(bodies):
                raise NotImplementedError('the generic tree kernels take between one collision geometry and as many as there '
                                          'are links')
        # (mixed geometry kinds: the two-body and the tree kernels take witness points per link / slot, so the links may carry
        # different kinds of shapes; a single body has one geometry)
        ground = len(geometries)
        geometries.append(GeometrySpec(-1, 'plane', (0., 0., 0.), None, None, 1.0))
        pairs = [(ground, g) for g in range(ground)]
        return SystemSpec(kind, bodies, joints, geometries, pairs)
