"""CPU: host-side mirror of the reference API (no compute calls into the CUDA library)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from dair_pll_b200 import _lib, quaternion
from dair_pll_b200.inertia import InertialParameterConverter as IPC
from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem
from dair_pll_b200.state_space import FixedBaseSpace, FloatingBaseSpace, ProductSpace
from dair_pll_b200.system_spec import SystemSpec
from oracle import contactnets_oracle as co
from tests.util import ROOT

torch.manual_seed(0)


def test_cube_spec_and_parameter_names(assets_dir):
    system = MultibodyLearnableSystem({'cube': os.path.join(assets_dir, 'cube.urdf')}, 0.0068)
    spec = system.multibody_terms.spec
    assert (spec.kind, spec.n_q, spec.n_v, spec.n_x, spec.n_contacts) == ('cube', 7, 6, 13, 4)
    # checkpoint compatibility: same state_dict keys/shapes as the reference module tree
    sd = system.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == {
        'multibody_terms.lagrangian_terms.inertial_parameters': (1, 10),
        'multibody_terms.contact_terms.friction_params': (2,),
        'multibody_terms.contact_terms.geometries.0.length_params': (1, 3)}
    assert system.space.n_x == 13 and system.max_batch_dim == 1 and system.dt == 0.0068
    assert torch.allclose(sd['multibody_terms.contact_terms.friction_params'], torch.tensor([0.15, 1.0]).double())
    mu = system.multibody_terms.contact_terms.pair_friction()
    assert abs(mu.item() - 2 * 0.15 / 1.15) < 1e-15     # SURVEY Appendix B: 0.26087
    theta = sd['multibody_terms.lagrangian_terms.inertial_parameters'][0]
    assert np.allclose(theta[:4].numpy(), [-0.4971, -3.4087, -3.4087, -3.4087], atol=5e-5)


def test_elbow_spec(assets_dir):
    spec = SystemSpec.from_urdf(os.path.join(assets_dir, 'elbow.urdf'))
    assert (spec.kind, spec.n_q, spec.n_v, spec.n_x, spec.n_contacts) == ('elbow', 8, 7, 15, 8)
    assert spec.joints[0].origin == (-0.035, 0.06, 0.0) and spec.joints[0].axis == (0.0, 1.0, 0.0)
    assert spec.geometries[1].offset == (0.035, 0.0, 0.0) and spec.geometries[-1].kind == 'plane'
    assert spec.collision_pairs == [(2, 0), (2, 1)]


def test_no_cpu_path(assets_dir):
    system = MultibodyLearnableSystem({'cube': os.path.join(assets_dir, 'cube.urdf')}, 0.0068)
    x = torch.zeros(3, 13, dtype=torch.float64)
    x[:, 0] = 1
    with pytest.raises(RuntimeError, match='no CPU path'):
        system.contactnets_loss(x, torch.zeros(3, 0), x)


def test_inertia_conversions_roundtrip_and_match_oracle():
    pi_cm = torch.tensor([[0.37, 0.37 * 0.002, -0.37 * 0.001, 0.37 * 0.003, 8.1e-4, 8.5e-4, 7.9e-4, 1e-5, -2e-5, 3e-5],
                          [1.3, 0.02, 0.01, -0.03, 2e-3, 3e-3, 2.5e-3, 1e-4, 0, -2e-4]], dtype=torch.float64)
    theta = IPC.pi_cm_to_theta(pi_cm)
    assert torch.allclose(IPC.theta_to_pi_cm(theta), pi_cm, rtol=1e-12, atol=1e-16)
    assert torch.allclose(IPC.pi_o_to_theta(IPC.theta_to_pi_o(theta)), theta, rtol=1e-12, atol=1e-14)
    assert torch.allclose(theta, co.pi_cm_to_theta(pi_cm), rtol=1e-13, atol=1e-15)
    vec = IPC.pi_cm_to_drake_spatial_inertia(IPC.theta_to_pi_cm(theta))
    assert torch.allclose(vec, co.theta_to_inertia_vector(theta), rtol=1e-12, atol=1e-16)
    assert torch.allclose(vec[:, 4:], pi_cm[:, 4:] / pi_cm[:, :1], rtol=1e-12)


def test_state_space_exponential_and_difference_are_inverse():
    space = ProductSpace([FixedBaseSpace(0), FloatingBaseSpace(1)])
    assert (space.n_q, space.n_v, space.n_x) == (8, 7, 15)
    q = torch.randn(5, 8, dtype=torch.float64)
    q[:, :4] /= q[:, :4].norm(dim=-1, keepdim=True)
    dq = 0.3 * torch.randn(5, 7, dtype=torch.float64)
    q2 = space.exponential(q, dq)
    assert torch.allclose(space.configuration_difference(q, q2), dq, atol=1e-12)
    # same quaternion update as the oracle's restatement of state_space.py:466-486
    ref = co.quat_mul(q[:, :4], co.quat_exp(dq[:, :3]))
    assert torch.allclose(q2[:, :4], ref, atol=1e-15)
    assert torch.allclose(quaternion.exp(torch.zeros(1, 3, dtype=torch.float64)),
                          torch.tensor([[1., 0, 0, 0]], dtype=torch.float64))
    x = torch.randn(5, 15, dtype=torch.float64)
    assert torch.equal(space.x(*space.q_v(x)), x)


def test_velocity_integrator_step_uses_callback():
    from dair_pll_b200.integrator import VelocityIntegrator
    space = ProductSpace([FixedBaseSpace(0), FloatingBaseSpace(0)])
    integ = VelocityIntegrator(space, lambda x, c: (space.v(x) * 0 + 1.0, c), 0.1)
    x = torch.zeros(2, 13, dtype=torch.float64)
    x[:, 0] = 1
    traj, carry = integ.simulate(x, torch.zeros(2, 1), 3)
    assert traj.shape == (2, 4, 13) and carry.shape == (2, 4, 1)
    assert torch.allclose(traj[:, -1, 4:7], torch.full((2, 3), 0.3, dtype=torch.float64))


def test_library_exports_every_declared_symbol():
    """The C-ABI shared library loads and exports each function include/*.h declares."""
    header = open(os.path.join(ROOT, 'include', 'dair_pll_b200.h')).read()
    declared = set(re.findall(r'\b(dpll_\w+)\s*\(', header))
    assert declared, 'no declarations parsed'
    assert declared == set(_lib.EXPORTS), (declared ^ set(_lib.EXPORTS))
    lib = ctypes.CDLL(_lib.lib_path())
    for name in declared:
        assert hasattr(lib, name), name
    lib.dpll_version.restype = ctypes.c_int
    lib.dpll_workspace_bytes.restype = ctypes.c_size_t
    assert lib.dpll_version() >= 100
    assert lib.dpll_workspace_bytes() >= 14 * 8


def test_device_slice_dataset_matches_reference_slicing(tmp_path):
    """Same (previous, future) pairs, in the same order, as the reference's per-index loop
    (dataset_management.py:43-59), from the reference's on-disk format (<index>.pt, file_utils.py:173-176)."""
    from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig
    gen = torch.Generator().manual_seed(0)
    trajs = [torch.randn(T, 13, generator=gen, dtype=torch.float64) for T in (9, 4, 17)]
    for i, t in enumerate(trajs):
        torch.save(t, tmp_path / f'{i}.pt')
    (tmp_path / 'notes.txt').write_text('ignored')
    for cfg in (TrajectorySliceConfig(), TrajectorySliceConfig(t_skip=2, t_history=3, t_prediction=2)):
        ds = DeviceTrajectorySliceDataset(cfg)
        assert ds.add_trajectories_from_directory(str(tmp_path)) == 3
        prev_ref, fut_ref = [], []
        for tr in trajs:                               # the reference's loop, restated
            for index in range(cfg.t_skip, tr.shape[0] - cfg.t_prediction):
                prev_ref.append(tr[index + 1 - cfg.t_history:index + 1])
                fut_ref.append(tr[index + 1:index + 1 + cfg.t_prediction])
        assert len(ds) == len(prev_ref)
        prev, fut = ds.tensors()
        assert torch.equal(prev, torch.stack(prev_ref)) and torch.equal(fut, torch.stack(fut_ref))
        p5, f5 = ds[5]
        assert torch.equal(p5, prev_ref[5]) and torch.equal(f5, fut_ref[5])
        seen = torch.cat([p[:, -1, 0] for p, _ in ds.batches(7, generator=torch.Generator().manual_seed(1))])
        assert seen.shape[0] == len(ds) and torch.equal(seen.sort().values, prev[:, -1, 0].sort().values)
        assert sum(p.shape[0] for p, _ in ds.batches(7, drop_last=True)) == (len(ds) // 7) * 7
    with pytest.raises(AssertionError):
        TrajectorySliceConfig(t_skip=0, t_history=2)


def test_icnn_weight_gradient_chain_rule_matches_autograd_of_the_oracle():
    """The host half of the support network's backward (deep_support_function.icnn_weight_gradients: the chain rule
    from the three reductions the backward kernels produce, the output weight's gradient from homogeneity) against
    autograd through the oracle restatement of deep_support_function.py:238-266, for all four weights (signed
    weights, so |.| and sign() are exercised).  The reductions themselves are formed here in torch -- on the GPU
    they come from the dpll_icnn_* kernels (tests/test_gpu_parity.py)."""
    from dair_pll_b200.deep_support_function import icnn_weight_gradients
    torch.manual_seed(3)
    W = 48
    Wd0, Wd1, Wh, wout = (torch.randn(3, W, dtype=torch.float64), torch.randn(3, W, dtype=torch.float64),
                          torch.randn(W, W, dtype=torch.float64) / W, torch.randn(W, dtype=torch.float64))
    d = torch.randn(301, 3, dtype=torch.float64)
    d = d / d.norm(dim=-1, keepdim=True)
    gp = torch.randn(301, 3, dtype=torch.float64)
    # what the kernels hand over (SURVEY.md A.6)
    lin0 = d @ Wd0
    m0 = torch.where(lin0 > 0, 1.0, 0.5).double()
    m1 = torch.where((lin0 * m0) @ Wh.abs() + d @ Wd1 > 0, 1.0, 0.5).double()
    a0 = (m1 @ (wout.abs()[:, None] * Wh.abs().t())) * m0
    g1, gWd0, G = gp.t() @ m1, gp.t() @ a0, ((gp @ Wd0) * m0).t() @ m1
    got = icnn_weight_gradients(Wd1, Wh, wout, g1, gWd0, G)
    b = [w.clone().requires_grad_() for w in (Wd0, Wd1, Wh, wout)]
    po = co.icnn_support(dict(Wd0=b[0], Wd1=b[1], Wh=b[2], wout=b[3]), d)
    (po * gp).sum().backward()
    for x, y in zip(got, b):
        assert torch.allclose(x, y.grad, rtol=1e-10, atol=1e-12)
    with pytest.raises(RuntimeError):                 # the product has no CPU path
        from dair_pll_b200.deep_support_function import ICNNSupport
        ICNNSupport.apply(d, Wd0, Wd1, Wh, wout, 0.5)


@pytest.mark.parametrize('asset', ['cube.urdf', 'elbow.urdf'])
def test_generate_updated_urdfs_round_trip(asset, tmp_path):
    """multibody_learnable_system.py:82-102: the learned parameterisation written back into the URDF is read back
    to the same inertial, geometric and friction parameters (host logic; no GPU)."""
    urdf = os.path.join(ROOT, 'dair_pll_b200', 'assets', asset)
    s = MultibodyLearnableSystem({'sys': urdf}, 0.0068, output_urdfs_dir=str(tmp_path))
    gen = torch.Generator().manual_seed(0)
    with torch.no_grad():
        mt = s.multibody_terms
        pi = mt.lagrangian_terms.pi_cm().clone()
        pi[:, 0] *= 1.2
        pi[:, 1:4] += 0.003 * pi[:, :1] * torch.randn(pi[:, 1:4].shape, generator=gen, dtype=pi.dtype)
        pi[:, 4:7] *= 1.1
        pi[:, 7:] += 1e-5
        mt.lagrangian_terms.inertial_parameters.copy_(IPC.pi_cm_to_theta(pi))
        mt.contact_terms.friction_params.mul_(0.8)
        for g in mt.contact_terms.geometries:
            if hasattr(g, 'length_params'):
                g.length_params.mul_(torch.tensor([[1.1, 0.9, 1.05]], dtype=g.length_params.dtype))
    paths = s.generate_updated_urdfs()
    assert os.path.basename(paths['sys']) == asset and os.path.dirname(paths['sys']) == str(tmp_path)
    s2 = MultibodyLearnableSystem(paths, 0.0068)
    a, b = s.multibody_terms, s2.multibody_terms
    assert torch.allclose(a.lagrangian_terms.pi_cm(), b.lagrangian_terms.pi_cm(), rtol=1e-12, atol=1e-15)
    n_body_geoms = len(a.contact_terms.geometries) - 1
    assert torch.allclose(a.contact_terms.friction_params[:n_body_geoms].abs(),
                          b.contact_terms.friction_params[:n_body_geoms].abs(), rtol=1e-12)
    for ga, gb in zip(a.contact_terms.geometries, b.contact_terms.geometries):
        if hasattr(ga, 'length_params'):
            assert torch.allclose(ga.length_params.abs(), gb.length_params.abs(), rtol=1e-12)


def test_device_slice_dataset_matches_the_reference_class_fixture():
    """tests/golden/dataset_slices.npz holds the outputs of the REFERENCE's own TrajectorySliceDataset
    (dair_pll/dataset_management.py:17-67, run through oracle/ref_shim.py by oracle/gen_golden_dataset.py) on three
    recorded tosses for four slice configurations: same pairs, same order, bit for bit."""
    from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig
    from tests.util import load_golden
    g = load_golden('dataset_slices')
    trajs = [torch.from_numpy(g[f'traj{i}']) for i in range(int(g['n_traj']))]
    for c, (skip, hist, pred) in enumerate(g['configs']):
        ds = DeviceTrajectorySliceDataset(TrajectorySliceConfig(t_skip=int(skip), t_history=int(hist), t_prediction=int(pred)))
        for t in trajs:
            ds.add_slices_from_trajectory(t)
        prev, fut = ds.tensors()
        assert torch.equal(prev, torch.from_numpy(g[f'previous{c}'])), c
        assert torch.equal(fut, torch.from_numpy(g[f'future{c}'])), c


def test_cost_ordered_batches_cover_each_slice_once_and_deal_equal_shards():
    """DeviceTrajectorySliceDataset cost hints: every batch is handed out by decreasing hint, dealt round-robin to the
    ranks, so each rank's share is itself ordered, shares differ by at most one slice and their costs by at most
    the largest single hint; together the shares are exactly the batch."""
    from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig
    gen = torch.Generator().manual_seed(5)
    ds = DeviceTrajectorySliceDataset(TrajectorySliceConfig())
    for T in (40, 23, 61):
        ds.add_slices_from_trajectory(torch.randn(T, 13, generator=gen, dtype=torch.float64))
    n = len(ds)
    cost = torch.randint(0, 40, (n,), generator=gen, dtype=torch.int32)
    ds.update_costs(None, cost)
    ds.update_costs(torch.tensor([3, 5]), torch.tensor([99, 98], dtype=torch.int32))
    cost[3], cost[5] = 99, 98
    world = 3
    for batch_size in (n, 32):
        seen = []
        for lo in range(0, n, batch_size):
            pass
        shares = [list(ds.batches(batch_size, shuffle=True, generator=torch.Generator().manual_seed(9), cost_ordered=True,
                                  return_indices=True, rank=r, world=world)) for r in range(world)]
        for b in range(len(shares[0])):
            idx = [shares[r][b][2] for r in range(world)]
            sizes = [i.numel() for i in idx]
            assert max(sizes) - min(sizes) <= 1
            for r in range(world):
                c = cost[idx[r]]
                assert torch.equal(c, c.sort(descending=True).values)               # each share is ordered
                prev, fut = ds.tensors()
                assert torch.equal(shares[r][b][0], prev[idx[r]]) and torch.equal(shares[r][b][1], fut[idx[r]])
            tot = [int(cost[i].sum()) for i in idx]
            assert max(tot) - min(tot) <= int(cost.max())
            seen.append(torch.cat(idx))
        allidx = torch.cat(seen)
        assert allidx.numel() == n and torch.equal(allidx.sort().values, torch.arange(n))
    # the first batch of the whole-set order starts with the most expensive slices
    first = next(iter(ds.batches(n, shuffle=False, cost_ordered=True, return_indices=True)))[2]
    assert first[0].item() == 3 and first[1].item() == 5


def test_peer_allreduce_protocol_model():
    """tests/host_emul/comm_model.cpp: a thread-per-rank model of the in-kernel all-reduce protocol
    (csrc/cn_comm.cuh: monotone flags, two alternating data rows, rank-ordered sums) never reads a row of the wrong
    epoch, for 2 / 4 / 8 ranks drifting at random."""
    import subprocess
    import tempfile
    out = os.path.join(tempfile.gettempdir(), f'dpll_comm_model_{os.getuid()}.so')
    subprocess.check_call(['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-pthread', '-o', out,
                           os.path.join(ROOT, 'tests', 'host_emul', 'comm_model.cpp')])
    lib = ctypes.CDLL(out)
    for world in (2, 4, 8):
        assert lib.comm_model_run(world, 5000, 17, world) == 0


def test_urdf_ingestion_rejects_what_the_kernels_do_not_model(tmp_path):
    """Models the kernels would silently mis-simulate are refused at construction (more collision geometries than links);
    a rotated collision frame sends a two-link system to the generic tree kernels (boxes as lengths, learned meshes as
    witness points); a single floating body's collision frame (offset and rotation) is carried to its geometry and
    equals the oracle tree's; a joint axis is normalised as Drake does on parsing."""
    from dair_pll_b200.geometry import place_in_link_frame
    from dair_pll_b200.system_spec import SystemSpec
    from oracle.callables import FRAMED_BODY_TREE as tree
    framed = MultibodyLearnableSystem({'body': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'framed_box.urdf')}, 0.0068)
    ct = framed.multibody_terms.contact_terms
    assert ct.has_witness_point_geometry() and ct.geometries[0].frame is not None and ct.geometries[1].frame is None
    off, rot = ct.geometries[0].frame
    assert torch.allclose(off, torch.tensor(tree.geometry_offset[0], dtype=torch.float64), atol=0, rtol=0)
    assert torch.allclose(rot, tree.geometry_rotation(0, torch.float64), atol=1e-15)
    assert 'frame_offset' not in ''.join(framed.state_dict().keys())          # checkpoint keys as the reference's
    # the lowest corners of the placed box in a direction are its support points
    d = torch.tensor([[0.3, -0.5, -0.8]], dtype=torch.float64)
    pts = place_in_link_frame(ct.geometries[0], d)[0]
    signs = torch.tensor([[(i >> 2) & 1, (i >> 1) & 1, i & 1] for i in range(8)], dtype=torch.float64) * 2 - 1
    corners = off + (signs * ct.geometries[0].get_half_lengths()) @ rot.t()
    best = torch.topk(corners @ d[0], 4).values
    assert torch.allclose(torch.sort(pts @ d[0]).values, torch.sort(best).values, atol=1e-15)
    # a rotated collision frame on a two-link system: not the specialised elbow kernels but the generic tree kernels
    elbow = open(os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow.urdf')).read()
    p = tmp_path / 'rotated.urdf'
    p.write_text(elbow.replace('<origin xyz="0.035 0 0" rpy="0 0 0"/>\n      <geometry>', '<origin xyz="0.035 0 0" rpy="0.1 0 0"/>\n      <geometry>', 1))
    assert 'rpy="0.1 0 0"' in p.read_text()
    rotated = SystemSpec.from_urdf(str(p))
    assert rotated.kind == 'chain' and rotated.geometries[1].rpy == (0.1, 0.0, 0.0)
    assert SystemSpec.from_urdf(os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow.urdf')).kind == 'elbow'
    # ... and so does a learned (mesh) geometry in a rotated collision frame: its support points become witness points
    mesh = open(os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow_mesh.urdf')).read()
    assert 'rpy="0 0 0"/>\n      <geometry><mesh' in mesh
    pm = tmp_path / 'rotated_mesh.urdf'
    pm.write_text(mesh.replace('rpy="0 0 0"/>\n      <geometry><mesh', 'rpy="0.1 0 0"/>\n      <geometry><mesh', 1)
                  .replace('elbow_half.obj', os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow_half.obj')))
    rm = SystemSpec.from_urdf(str(pm))
    assert rm.kind == 'chain' and [g.kind for g in rm.geometries] == ['mesh', 'mesh', 'plane']
    # more collision geometries than links is what the tree kernels' slots cannot hold
    two = elbow.replace('</collision>\n  </link>\n  <link name="elbow_2">',
                        '</collision>\n' + elbow[elbow.index('    <collision>'):elbow.index('</collision>') + 12] * 2
                        + '\n  </link>\n  <link name="elbow_2">', 1)
    pt = tmp_path / 'crowded.urdf'
    pt.write_text(two)
    assert len(SystemSpec.from_urdf(str(p)).geometries) == 3
    with pytest.raises(NotImplementedError):
        SystemSpec.from_urdf(str(pt))
    elbow = open(os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow.urdf')).read()
    assert 'xyz="0 1 0"' in elbow
    p2 = tmp_path / 'axis.urdf'
    p2.write_text(elbow.replace('<axis xyz="0 1 0"', '<axis xyz="0 2 0"', 1))
    spec = SystemSpec.from_urdf(str(p2))
    assert spec.joints[0].axis == (0.0, 1.0, 0.0)


def test_branching_tree_spec_and_what_is_still_refused(assets_dir, tmp_path):
    """N2: a branching four-link tree parses into the 'chain' kind with each link's parent in the kinematic table (equal to
    the oracle tree's); trees whose links are not listed root first, or with more than six links, are refused."""
    from oracle.callables import TREE4_TREE
    from tests.test_host_emulation import chain_kin_rows
    s = MultibodyLearnableSystem({'tree4': os.path.join(assets_dir, 'tree4.urdf')}, 0.0068)
    spec = s.multibody_terms.spec
    assert (spec.kind, spec.n_q, spec.n_v, spec.n_x, spec.n_contacts) == ('chain', 10, 9, 19, 16)
    assert [j.parent for j in spec.joints] == [0, 0, 2] and [j.child for j in spec.joints] == [1, 2, 3]
    _, _, _, kin, n = s._chain_params(torch.device('cpu'))
    assert n == 4 and np.allclose(kin.numpy().reshape(4, 31), chain_kin_rows(TREE4_TREE), rtol=0, atol=1e-15)
    # boxes spread unevenly over the links (two on the root, none on links 1 and 2): box slots with their own link index
    from oracle.callables import TREE4G_TREE
    sg = MultibodyLearnableSystem({'tree4g': os.path.join(assets_dir, 'tree4g.urdf')}, 0.0068)
    assert [g.body for g in sg.multibody_terms.spec.geometries] == [0, 0, 3, -1] and sg.multibody_terms.spec.n_contacts == 12
    _, mu_g, half_g, kin_g, n_g = sg._chain_params(torch.device('cpu'))
    assert n_g == 4 and mu_g.shape == (4,) and half_g.shape == (12,) and (half_g[9:] == 0).all()
    assert np.allclose(kin_g.numpy().reshape(4, 31), chain_kin_rows(TREE4G_TREE), rtol=0, atol=1e-15)
    assert sorted(k for k, _ in sg.named_parameters() if 'length_params' in k) == [
        f'multibody_terms.contact_terms.geometries.{i}.length_params' for i in range(3)]
    text = open(os.path.join(assets_dir, 'tree4.urdf')).read()
    # the joint to link 3 declared before the joint to link 2: joint order would no longer be link order
    j2 = text[text.index('<joint name="joint_2"'):text.index('<joint name="joint_3"')]
    j3 = text[text.index('<joint name="joint_3"'):text.index('</robot>')]
    p = tmp_path / 'reordered.urdf'
    p.write_text(text.replace(j2 + j3, j3 + j2))
    with pytest.raises(NotImplementedError):
        SystemSpec.from_urdf(str(p))
    # more links than the largest instantiation (six)
    link = text[text.index('  <link name="link_3">'):text.index('  <joint name="joint_1"')]
    p5 = tmp_path / 'five.urdf'
    extra = ''.join(link.replace('link_3', f'link_{k}') for k in (4, 5, 6))
    extra += ''.join(j3.replace('joint_3', f'joint_{k}').replace('child link="link_3"', f'child link="link_{k}"') for k in (4, 5, 6))
    p5.write_text(text.replace(link, link + extra.split('<joint')[0]).replace('</robot>', '<joint' + '<joint'.join(extra.split('<joint')[1:]) + '</robot>'))
    assert len(SystemSpec.from_urdf(os.path.join(assets_dir, 'tree6.urdf')).bodies) == 6
    with pytest.raises(NotImplementedError):
        SystemSpec.from_urdf(str(p5))


def test_chain_spec_carries_rotated_joint_frames(assets_dir):
    """N2 first slice: a three-link serial chain parses into the 'chain' kind; the kinematic table handed to
    dpll_chain_* (joint origin | fixed joint-frame rotation | axis | box offset per link) equals the one the
    oracle's tree code (oracle/callables.py:CHAIN3_TREE) is built from."""
    from oracle.callables import CHAIN3_TREE
    from tests.test_host_emulation import chain_kin_rows
    s = MultibodyLearnableSystem({'chain3': os.path.join(assets_dir, 'chain3.urdf')}, 0.0068)
    spec = s.multibody_terms.spec
    assert (spec.kind, spec.n_q, spec.n_v, spec.n_x, spec.n_contacts) == ('chain', 9, 8, 17, 12)
    assert spec.collision_pairs == [(3, 0), (3, 1), (3, 2)]
    inertia, mu, half, kin, n = s._chain_params(torch.device('cpu'))
    assert n == 3 and inertia.shape == (30,) and mu.shape == (3,) and half.shape == (9,)
    assert np.allclose(kin.numpy().reshape(3, 31), chain_kin_rows(CHAIN3_TREE), rtol=0, atol=1e-15)
    names = [k for k, _ in s.named_parameters()]
    assert 'multibody_terms.contact_terms.geometries.2.length_params' in names
    x = torch.zeros(2, 17, dtype=torch.float64)
    x[:, 0] = 1
    with pytest.raises(RuntimeError, match='no CPU path'):
        s.contactnets_loss(x, torch.zeros(2, 0), x)


def test_extract_mesh_of_a_box_support_function_and_cpu_refusal():
    """``extract_mesh`` (deep_support_function.py:95-122) on a closed-form support function: a box's support points are
    its corners, so the 296 sampled directions collapse to the 8 distinct vertices and the hull has 12 triangles, every
    one wound counter-clockwise seen from outside; the sampled direction set equals the reference's formula; a network of
    any depth refuses CPU tensors (there is no CPU path)."""
    from dair_pll_b200.deep_support_function import (HomogeneousICNN, extract_mesh, extract_obj, outward_normal_hyperplanes,
                                                     surface_directions)
    d = surface_directions()
    assert d.shape == (296, 3) and d.dtype == torch.float32
    assert torch.allclose(d.norm(dim=-1), torch.ones(296), atol=1e-6)
    half = torch.tensor([0.05, 0.03, 0.02], dtype=torch.float64)
    box = lambda dirs: torch.where(dirs >= 0, half, -half)   # noqa: E731
    mesh = extract_mesh(box)
    assert mesh.vertices.shape == (8, 3) and mesh.faces.shape == (12, 3)
    normals, backwards, offsets = outward_normal_hyperplanes(mesh.vertices, mesh.faces)
    assert not backwards.any()
    a, b, c = (mesh.vertices[mesh.faces[:, i]] for i in range(3))
    assert ((torch.linalg.cross(b - a, c - a) * normals).sum(-1) > 0).all()
    # every face plane is one of the six box planes
    assert torch.allclose(offsets, (normals.abs() * half).sum(-1), atol=1e-15)
    text = extract_obj(box)
    assert text.count('\nf ') + text.startswith('f ') == 12 and text.count('v ') == 8 and text.count('vn ') == 12
    for depth in (1, 2, 3):
        net = HomogeneousICNN(depth, 16)
        assert len(net.hidden_weights) == depth - 1 and len(net.input_weights) == depth
        with pytest.raises(RuntimeError, match='no CPU path'):
            net(torch.zeros(4, 3, dtype=torch.float64))


def test_mixed_box_and_mesh_elbow_parses(assets_dir):
    """A box on one link and a learned mesh on the other is the two-body kind with witness points per link (no box lengths
    in the kernel-level parameters: the box's corners reach the kernels as points); mixed kinds on other systems are refused."""
    from dair_pll_b200.geometry import Box, DeepSupportConvex
    s = MultibodyLearnableSystem({'elbow': os.path.join(assets_dir, 'elbow_mixed.urdf')}, 0.0068)
    spec = s.multibody_terms.spec
    assert spec.kind == 'elbow' and [g.kind for g in spec.geometries] == ['box', 'mesh', 'plane']
    geoms = s.multibody_terms.contact_terms.geometries
    assert isinstance(geoms[0], Box) and isinstance(geoms[1], DeepSupportConvex)
    _, _, half = s.multibody_terms.kernel_parameters(torch.float64)
    assert half == []
    names = [k for k, _ in s.named_parameters()]
    assert 'multibody_terms.contact_terms.geometries.0.length_params' in names
    assert 'multibody_terms.contact_terms.geometries.1.network.output_weight' in names


def test_bench_dump_outputs_files_and_row_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: one float .npy per output; above DUMP_MAX_ROWS per-sample losses the same seeded,
    ordered subset of rows is written on every run."""
    import bench
    monkeypatch.setattr(bench, 'DUMP_MAX_ROWS', 5)
    loss = torch.arange(12, dtype=torch.float64)
    grads = [torch.ones(1, 10, dtype=torch.float64), torch.zeros(2, dtype=torch.float64)]
    for out in (tmp_path / 'a', tmp_path / 'b'):
        bench.dump_outputs(str(out), loss, loss.mean(), grads, ['p.first', 'p.second'])
    assert sorted(os.listdir(tmp_path / 'a')) == ['grad.p.first.npy', 'grad.p.second.npy', 'loss.npy', 'loss_mean.npy']
    rows = np.load(tmp_path / 'a' / 'loss.npy')
    assert rows.dtype == np.float64 and rows.shape == (5,) and np.all(np.diff(rows) > 0) and set(rows) <= set(range(12))
    assert np.array_equal(rows, np.load(tmp_path / 'b' / 'loss.npy'))
    assert np.load(tmp_path / 'a' / 'loss_mean.npy') == 5.5
    assert np.array_equal(np.load(tmp_path / 'a' / 'grad.p.first.npy'), np.ones((1, 10)))


@pytest.mark.parametrize('argv', [['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'out']])
def test_bench_refuses_arguments_it_cannot_honour(argv, monkeypatch):
    """No timed step to report, or a dump the CPU reference path would not write: refused before any work."""
    import bench
    monkeypatch.setattr('sys.argv', ['bench.py'] + argv)
    with pytest.raises(SystemExit) as e:
        bench.parse_args()
    assert e.value.code == 2
