"""GPU, round 2: the regions round 1 left untested -- the bench batch itself against the oracle, the elbow at
scale and in the fp32 variant, long rollouts, the training-loop entry point (row strides, cost-ordered dynamic
scheduling, in-kernel exchange at world size 1), the device data set against the reference class's outputs."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
from dair_pll_b200 import ops, synthetic  # noqa: E402
from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem  # noqa: E402
from tests.util import kernel_level_params, load_golden, max_rel_to_scale, rel_err  # noqa: E402

DEV = 'cuda:0'
DT = 0.0068


def _leaf_grads(system):
    mt = system.multibody_terms
    out = [mt.lagrangian_terms.inertial_parameters.grad, mt.contact_terms.friction_params.grad]
    out += [g.length_params.grad for g in mt.contact_terms.geometries if hasattr(g, 'length_params')]
    return [t.detach().cpu().numpy().copy() for t in out]


def test_bench_batch_subset_matches_oracle():
    """The headline workload itself: bench.py's 1,048,576-pair batch (same generator, seed and parameters) goes
    through the public API once; a random 16,384-sample subset of its per-sample losses, and the parameter
    gradient of that subset, are compared with the CPU oracle at 1e-9 (north_star)."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle import contactnets_oracle as co
    from oracle.callables import CUBE_TREE, TreeCallables
    system = bench.make_system(torch.device(DEV), torch.float64)
    x, xp = bench.make_batch(system, 1 << 20, seed=0, device=torch.device(DEV), dtype=torch.float64)
    loss = system.contactnets_loss(x, None, xp).detach()
    idx = torch.randperm(1 << 20, generator=torch.Generator().manual_seed(123))[:16384].to(DEV)
    xs, xps = x[idx].contiguous(), xp[idx].contiguous()
    sub = system.contactnets_loss(xs, None, xps)
    assert torch.equal(sub.detach(), loss[idx])                  # per-sample results do not depend on the batch
    sub.sum().backward()
    mt = system.multibody_terms
    P = co.OracleParams(mt.lagrangian_terms.inertial_parameters.detach().cpu().clone(),
                        mt.contact_terms.friction_params.detach().cpu().clone(),
                        [mt.contact_terms.geometries[0].length_params.detach().cpu().clone()]).requires_grad_()
    lo = co.contactnets_loss(TreeCallables(CUBE_TREE), P, xs.cpu(), xps.cpu(), DT)
    lo.sum().backward()
    assert rel_err(sub.detach().cpu().numpy(), lo.detach().numpy(), 1e-9).max() < 1e-9
    gt, gf, gl = _leaf_grads(system)
    assert max_rel_to_scale(gt, P.inertial_parameters.grad.numpy()) < 1e-9
    assert max_rel_to_scale(gf, P.friction_params.grad.numpy()) < 1e-9
    assert max_rel_to_scale(gl, P.length_params[0].grad.numpy()) < 1e-9


@pytest.mark.parametrize('mode', [['--order', 'cost'], ['--order', 'natural', '--no-graph']])
def test_bench_dump_outputs_are_the_last_timed_step(mode, tmp_path):
    """bench.py --dump-outputs writes the per-sample losses (in generator order), the mean loss and the gradients of a
    timed step (every step computes the same values, so which one is not checked): the same as the public API's on the
    same seeded batch.  20,000 pairs fit the L2, so the graphed run cycles through many captured copies of the batch."""
    import json
    import subprocess
    sys.path.insert(0, ROOT)
    import bench
    run = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '3', '--warmup', '1', '--batch', '20000',
                          '--no-secondary', '--no-cpu-baseline', '--dump-outputs', str(tmp_path)] + mode,
                         check=True, stdout=subprocess.PIPE, text=True)
    assert json.loads(run.stdout)['config']['timed_steps'] == 3
    system = bench.make_system(torch.device(DEV), torch.float64)
    x, xp = bench.make_batch(system, 20000, seed=0, device=torch.device(DEV), dtype=torch.float64)
    loss = system.contactnets_loss(x, None, xp)
    mean = loss.mean()
    mean.backward()
    assert rel_err(np.load(tmp_path / 'loss.npy'), loss.detach().cpu().numpy(), 1e-9).max() < 1e-12
    assert rel_err(np.load(tmp_path / 'loss_mean.npy'), mean.item()) < 1e-12
    for name, p in system.named_parameters():
        got = np.load(tmp_path / f'grad.{name}.npy')
        assert got.dtype == np.float64 and max_rel_to_scale(got, p.grad.cpu().numpy()) < 1e-12, name


def _elbow_random(n, assets_dir, seed):
    from dair_pll_b200.inertia import InertialParameterConverter as IPC
    pi, fr, half = synthetic.elbow_learnables_perturbed(seed)
    s = MultibodyLearnableSystem({'elbow': os.path.join(assets_dir, 'elbow.urdf')}, DT)
    s.load_state_dict({
        'multibody_terms.lagrangian_terms.inertial_parameters': IPC.pi_cm_to_theta(pi),
        'multibody_terms.contact_terms.friction_params': fr,
        'multibody_terms.contact_terms.geometries.0.length_params': half[0].reshape(1, 3),
        'multibody_terms.contact_terms.geometries.1.length_params': half[1].reshape(1, 3)})
    s = s.to(DEV)
    x = synthetic.elbow_states(n, seed=seed + 10, device=DEV)
    with torch.no_grad():
        traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(n, 1, device=DEV), 1)
    xp = synthetic.perturb_next_state(traj[:, 1], seed=seed + 11, n_q=8)
    return s, (pi, fr, half), x, xp, traj


def test_elbow_matches_cpu_oracle_on_random_inputs(assets_dir):
    """Two-body system at scale: 65,536 random state pairs (all contact regimes of both boxes) -- per-sample
    losses, every parameter gradient and the one-step next states against the CPU oracle at 1e-9."""
    from oracle import contactnets_oracle as co
    from oracle.callables import ELBOW_TREE, TreeCallables
    n = 65536
    s, (pi, fr, half), x, xp, traj = _elbow_random(n, assets_dir, 1)
    loss = s.contactnets_loss(x, None, xp)
    loss.sum().backward()
    calls = TreeCallables(ELBOW_TREE)
    P = co.OracleParams(co.pi_cm_to_theta(pi), fr.clone(), [h.reshape(1, 3).clone() for h in half]).requires_grad_()
    lo = co.contactnets_loss(calls, P, x.cpu(), xp.cpu(), DT)
    lo.sum().backward()
    assert rel_err(loss.detach().cpu().numpy(), lo.detach().numpy(), 1e-9).max() < 1e-9
    g = _leaf_grads(s)
    assert max_rel_to_scale(g[0], P.inertial_parameters.grad.numpy()) < 1e-9
    assert max_rel_to_scale(g[1], P.friction_params.grad.numpy()) < 1e-9
    assert max_rel_to_scale(np.stack([a.reshape(3) for a in g[2:]]),
                            np.stack([p.grad.numpy().reshape(3) for p in P.length_params])) < 1e-9
    with torch.no_grad():
        step_o = co.sim_step(calls, P, x[:8192].cpu(), DT)
    assert np.abs(traj[:8192, 1].cpu().numpy() - step_o.numpy()).max() < 1e-9


def test_elbow_fp32_variant(assets_dir):
    """fp32 variant of the two-body entry points (dpll_elbow_loss_f32 / dpll_elbow_rollout_f32: fp32 storage, fp64
    arithmetic): losses, gradients and next states within 1e-4 (north_star) of the fp64 results."""
    n = 8192
    s, _, x, xp, traj = _elbow_random(n, assets_dir, 2)
    loss64 = s.contactnets_loss(x, None, xp)
    loss64.mean().backward()
    g64 = _leaf_grads(s)
    for p in s.parameters():
        p.grad = None
    loss32 = s.contactnets_loss(x.float(), None, xp.float())
    assert loss32.dtype == torch.float32
    loss32.mean().backward()
    g32 = _leaf_grads(s)
    l64, l32 = loss64.detach().cpu().numpy(), loss32.detach().cpu().numpy().astype(np.float64)
    assert np.abs(l32 - l64).max() < 1e-4 * max(np.abs(l64).max(), 1e-3)
    assert abs(l32.mean() - l64.mean()) < 1e-4 * abs(l64.mean())
    for a, b in zip(g32, g64):
        assert max_rel_to_scale(a, b) < 1e-4
    with torch.no_grad():
        t32, _ = s.simulate(x.float().unsqueeze(-2), torch.zeros(n, 1, device=DEV), 1)
    assert t32.dtype == torch.float32
    ref = traj[:, 1].cpu().numpy()
    assert np.abs(t32[:, 1].cpu().numpy() - ref).max() < 1e-4 * max(1.0, np.abs(ref).max())


def test_elbow_learned_geometry_width_256_matches_oracle(assets_dir):
    """Config 3's system as configured (support networks of width 256, reference initialisation): loss and the
    gradients of inertia, friction and all network weights against autograd through the CPU oracle."""
    from oracle import contactnets_oracle as co
    from oracle.callables import ELBOW_TREE, TreeCallables
    torch.manual_seed(0)
    s = MultibodyLearnableSystem({'elbow': os.path.join(assets_dir, 'elbow_mesh.urdf')}, DT).to(DEV)
    n = 2048
    x = synthetic.elbow_states(n, seed=31, device=DEV)
    with torch.no_grad():
        traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(n, 1, device=DEV), 1)
    xp = synthetic.perturb_next_state(traj[:, 1], seed=32, n_q=8)
    loss = s.contactnets_loss(x, None, xp)
    loss.sum().backward()
    mt = s.multibody_terms
    nets = []
    for gi in range(2):
        geom = mt.contact_terms.geometries[gi]
        net = geom.network
        nets.append(dict(Wd0=net.input_weights[0].detach().cpu().clone().requires_grad_(),
                         Wd1=net.input_weights[1].detach().cpu().clone().requires_grad_(),
                         Wh=net.hidden_weights[0].detach().cpu().clone().requires_grad_(),
                         wout=net.output_weight.detach().cpu().clone().requires_grad_(),
                         perturbations=geom.perturbations.detach().cpu().clone()))
    P = co.OracleParams(mt.lagrangian_terms.inertial_parameters.detach().cpu().clone(),
                        mt.contact_terms.friction_params.detach().cpu().clone(), [], icnn=nets).requires_grad_()
    lo = co.contactnets_loss(TreeCallables(ELBOW_TREE), P, x.cpu(), xp.cpu(), DT)
    lo.sum().backward()
    assert rel_err(loss.detach().cpu().numpy(), lo.detach().numpy(), 1e-9).max() < 1e-9
    assert max_rel_to_scale(mt.lagrangian_terms.inertial_parameters.grad.cpu().numpy(), P.inertial_parameters.grad.numpy()) < 1e-9
    assert max_rel_to_scale(mt.contact_terms.friction_params.grad.cpu().numpy(), P.friction_params.grad.numpy()) < 1e-9
    for gi in range(2):
        net = mt.contact_terms.geometries[gi].network
        for k, p in (('Wd0', net.input_weights[0]), ('Wd1', net.input_weights[1]), ('Wh', net.hidden_weights[0]),
                     ('wout', net.output_weight)):
            assert max_rel_to_scale(p.grad.cpu().numpy(), nets[gi][k].grad.numpy()) < 1e-9, (gi, k)


def test_long_rollout_matches_oracle_with_growth_bound(assets_dir):
    """Config 4's horizon: 256 tosses x 80 steps (the example's initial-condition sampler, contactnets_simple.py:56-63)
    against the CPU oracle's own 80-step simulation.  Each step is held to 1e-9; over a trajectory the difference
    may grow through contact events (a toss has a handful of impacts; measured sensitivity of an impact step to
    its input is <= ~30x), so the whole trajectory is held to 1e-9 * 30^k with k the impacts seen -- stated here
    as: median over tosses <= 1e-9, maximum <= 1e-5 -- and one-step agreement is re-checked ALONG the
    trajectory by stepping the oracle from the kernel's own states."""
    from oracle import contactnets_oracle as co
    from oracle.callables import CUBE_TREE, TreeCallables
    g = load_golden('cube_real_nominal')
    s = MultibodyLearnableSystem({'cube': os.path.join(assets_dir, 'cube.urdf')}, DT).to(DEV)
    n, steps = 256, 80
    gen = torch.Generator().manual_seed(7)
    x0 = torch.tensor([1., 0., 0., 0., 0., 0., 0.21, 0., 0., 0., 0., 0., -.075], dtype=torch.float64).repeat(n, 1)
    x0[:, 7:] += 0.1 * (2 * torch.rand(n, 6, generator=gen, dtype=torch.float64) - 1) * torch.tensor([30., 30, 30, 10, 10, 10])
    quat = x0[:, :4] + 0.3 * torch.randn(n, 4, generator=gen, dtype=torch.float64)
    x0[:, :4] = quat / quat.norm(dim=-1, keepdim=True)
    with torch.no_grad():
        traj, _ = s.simulate(x0.to(DEV).unsqueeze(-2), torch.zeros(n, 1, device=DEV), steps)
    mt = s.multibody_terms
    P = co.OracleParams(mt.lagrangian_terms.inertial_parameters.detach().cpu(), mt.contact_terms.friction_params.detach().cpu(),
                        [mt.contact_terms.geometries[0].length_params.detach().cpu()])
    calls = TreeCallables(CUBE_TREE)
    with torch.no_grad():
        tro = co.simulate(calls, P, x0, DT, steps)
    t = traj.cpu()
    assert (t[:, -1, 6] < 0.2).all()                         # the tosses did come down and hit the ground
    err = (t - tro).abs().amax(dim=(1, 2))
    assert err.median().item() < 1e-9 and err.max().item() < 1e-5
    # one-step parity along the kernel's own trajectory (no accumulation): every 8th state of every toss
    xs = t[:, 0:steps:8].reshape(-1, 13)
    with torch.no_grad():
        nxt = co.sim_step(calls, P, xs, DT)
    assert (nxt - t[:, 1:steps + 1:8].reshape(-1, 13)).abs().max().item() < 1e-9
    del g


def test_tiled_real_data_matches_reference_golden(assets_dir):
    """The reference's recorded tosses (478 consecutive real pairs, 83% in contact) tiled 512 times: every tile's
    per-sample losses are the golden ones and the gradient of the mean is the golden gradient."""
    g = load_golden('cube_real_nominal')
    s = MultibodyLearnableSystem({'cube': os.path.join(assets_dir, 'cube.urdf')}, float(g['dt']))
    s.load_state_dict({
        'multibody_terms.lagrangian_terms.inertial_parameters': torch.from_numpy(g['theta']),
        'multibody_terms.contact_terms.friction_params': torch.from_numpy(g['friction_params']),
        'multibody_terms.contact_terms.geometries.0.length_params': torch.from_numpy(g['half_lengths']).reshape(1, 3)})
    s = s.to(DEV)
    k = 512
    x = torch.from_numpy(np.tile(g['x'], (k, 1))).to(DEV)
    xp = torch.from_numpy(np.tile(g['x_plus'], (k, 1))).to(DEV)
    loss = s.contactnets_loss(x, None, xp)
    loss.mean().backward()
    l = loss.detach().cpu().numpy().reshape(k, -1)
    assert np.abs(l - g['loss'][None]).max() < 1e-13
    gt, gf, gl = _leaf_grads(s)
    assert max_rel_to_scale(gt, g['grad_theta']) < 1e-9
    assert max_rel_to_scale(gf, g['grad_friction']) < 1e-9
    assert max_rel_to_scale(gl, g['grad_length']) < 1e-9


def test_training_entry_point_strides_order_and_exchange(assets_dir):
    """dpll_cube_loss_leaf_dp_*: (1) row-strided views (the reference's x_past[..., -1, :]) give the bits of the
    contiguous call; (2) a cost-ordered batch with dynamic chunk scheduling gives the same per-sample losses and
    the same sums to rounding; (3) a world-size-1 communicator is the identity; (4) means = sums / count."""
    from dair_pll_b200 import parallel
    g = load_golden('cube_synthetic')
    theta = torch.from_numpy(g['theta']).to(DEV)
    fr = torch.from_numpy(g['friction_params']).to(DEV)
    ln = torch.from_numpy(g['half_lengths']).reshape(1, 3).to(DEV)
    inertia, mu, half = (torch.from_numpy(a).to(DEV) for a in kernel_level_params(g))
    n = 300001
    x = synthetic.cube_states(n, seed=61, device=DEV)
    traj, _ = ops.cube_rollout(x, inertia, mu, half, DT, 1)
    xp = synthetic.perturb_next_state(traj[:, 1], seed=62)
    base = ops.cube_loss_leaf_dp_raw(x, xp, theta, fr, ln, DT, 1e-3, want_iters=True)
    loss, sums, means, local, iters = base
    assert sums[16].item() == n and torch.equal(local, sums[:16])
    assert torch.allclose(means, sums[:16] / n, rtol=1e-15, atol=0)
    old = ops.cube_loss_leaf_raw(x, xp, theta, fr, ln, DT, 1e-3)
    assert torch.equal(old[0], loss) and torch.equal(old[1], sums[:15]) and torch.equal(old[2], sums[15:16])
    # (1) strided rows
    past, fut = torch.stack((x, x + 1.0), 1), torch.stack((xp, xp - 1.0), 1)
    xv, xpv = past[:, 0, :], fut[:, 0, :]
    assert not xv.is_contiguous()
    st = ops.cube_loss_leaf_dp_raw(xv, xpv, theta, fr, ln, DT, 1e-3)
    assert torch.equal(st[0], loss) and torch.equal(st[1], sums)
    # (2) cost order + dynamic scheduling
    order = torch.argsort(iters, descending=True, stable=True)
    xo, xpo = x[order].contiguous(), xp[order].contiguous()
    dyn = ops.cube_loss_leaf_dp_raw(xo, xpo, theta, fr, ln, DT, 1e-3, flags=ops.LOSS_DYNAMIC, want_iters=True)
    assert torch.equal(dyn[0], loss[order]) and torch.equal(dyn[4], iters[order])
    assert max_rel_to_scale(dyn[1].cpu().numpy(), sums.cpu().numpy()) < 1e-12
    for m in (1, 31, 32, 33, 4097):
        a = ops.cube_loss_leaf_dp_raw(xo[:m], xpo[:m], theta, fr, ln, DT, 1e-3, flags=ops.LOSS_DYNAMIC)
        b = ops.cube_loss_leaf_dp_raw(xo[:m], xpo[:m], theta, fr, ln, DT, 1e-3)
        assert torch.equal(a[0], b[0]) and max_rel_to_scale(a[1].cpu().numpy(), b[1].cpu().numpy()) < 1e-12, m
    # (3) communicator of one rank
    comm = parallel.PeerComm(torch.device(DEV))
    try:
        for _ in range(3):                                   # epochs advance, buffers alternate
            c = ops.cube_loss_leaf_dp_raw(x, xp, theta, fr, ln, DT, 1e-3, comm=comm)
            assert torch.equal(c[1], sums) and torch.equal(c[2], means) and torch.equal(c[3], local)
        v = torch.arange(15, dtype=torch.float64, device=DEV)
        assert torch.equal(comm.all_reduce_sum(v, 0.5), v * 0.5)
        comm.check()
    finally:
        comm.close()
    # module API: the options change nothing but the schedule
    s = MultibodyLearnableSystem({'cube': os.path.join(assets_dir, 'cube.urdf')}, DT)
    s.load_state_dict({
        'multibody_terms.lagrangian_terms.inertial_parameters': torch.from_numpy(g['theta']),
        'multibody_terms.contact_terms.friction_params': torch.from_numpy(g['friction_params']),
        'multibody_terms.contact_terms.geometries.0.length_params': torch.from_numpy(g['half_lengths']).reshape(1, 3)})
    s = s.to(DEV)
    s.record_newton_iters = True
    l0 = s.contactnets_loss(xv, None, xpv)
    assert torch.equal(l0.newton_iters, iters)
    l0.mean().backward()
    g0 = _leaf_grads(s)
    for p in s.parameters():
        p.grad = None
    s.dynamic_schedule = True
    l1 = s.contactnets_loss(xo, None, xpo)
    l1.mean().backward()
    assert abs(l1.mean().item() - l0.mean().item()) <= 1e-13 * abs(l0.mean().item())
    for a, b in zip(_leaf_grads(s), g0):
        assert max_rel_to_scale(a, b) < 1e-12


def test_device_dataset_matches_reference_fixture_on_the_gpu():
    """SURVEY 8(f) N3: the device-resident slice data set holds exactly the (previous, future) pairs the reference's
    TrajectorySliceDataset produced (fixture generated by the reference's own class, oracle/gen_golden_dataset.py),
    and cost-ordered batches feed the loss without leaving the device."""
    from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig
    g = load_golden('dataset_slices')
    trajs = [torch.from_numpy(g[f'traj{i}']) for i in range(int(g['n_traj']))]
    for c, (skip, hist, pred) in enumerate(g['configs']):
        ds = DeviceTrajectorySliceDataset(TrajectorySliceConfig(t_skip=int(skip), t_history=int(hist), t_prediction=int(pred)),
                                          device=torch.device(DEV))
        for t in trajs:
            ds.add_slices_from_trajectory(t)
        prev, fut = ds.tensors()
        assert prev.is_cuda and torch.equal(prev.cpu(), torch.from_numpy(g[f'previous{c}']))
        assert torch.equal(fut.cpu(), torch.from_numpy(g[f'future{c}']))
    # an epoch through the loss: hints recorded from the first pass order the second
    ds = DeviceTrajectorySliceDataset(TrajectorySliceConfig(t_skip=1, t_history=2, t_prediction=1), device=torch.device(DEV))
    for t in trajs:
        ds.add_slices_from_trajectory(t)
    s = MultibodyLearnableSystem({'cube': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'cube.urdf')}, DT).to(DEV)
    s.record_newton_iters = True
    total = 0.0
    for prev, fut, idx in ds.batches(16, shuffle=True, generator=torch.Generator(device=DEV).manual_seed(0), return_indices=True):
        loss = s.contactnets_loss(prev[..., -1, :], None, fut[..., 0, :])
        ds.update_costs(idx, loss.newton_iters)
        total += loss.sum().item()
    s.dynamic_schedule = True
    total2, costs = 0.0, []
    for prev, fut, idx in ds.batches(16, shuffle=True, generator=torch.Generator(device=DEV).manual_seed(1), cost_ordered=True,
                                     return_indices=True):
        loss = s.contactnets_loss(prev[..., -1, :], None, fut[..., 0, :])
        costs.append(loss.newton_iters.cpu())
        total2 += loss.sum().item()
    assert abs(total - total2) <= 1e-12 * abs(total)
    assert all(torch.equal(c, c.sort(descending=True).values) for c in costs)


@pytest.mark.parametrize('name', ['elbow_nominal', 'elbow_perturbed'])
def test_elbow_dense_terms_match_oracle(name, assets_dir):
    """MultibodyTerms.forward for the two-body system (multibody_terms.py:584-609; dpll_elbow_terms_f64): the
    (delassus, M, J, phi, acceleration) tuple against the oracle's tree code at the golden states."""
    from oracle import contactnets_oracle as co
    from oracle.callables import ELBOW_TREE, TreeCallables
    from tests.util import oracle_params_from_golden
    g = load_golden(name)
    s = MultibodyLearnableSystem({'elbow': os.path.join(assets_dir, 'elbow.urdf')}, float(g['dt']))
    s.load_state_dict({
        'multibody_terms.lagrangian_terms.inertial_parameters': torch.from_numpy(g['theta']),
        'multibody_terms.contact_terms.friction_params': torch.from_numpy(g['friction_params']),
        'multibody_terms.contact_terms.geometries.0.length_params': torch.from_numpy(g['half_lengths'][0]).reshape(1, 3),
        'multibody_terms.contact_terms.geometries.1.length_params': torch.from_numpy(g['half_lengths'][1]).reshape(1, 3)})
    s = s.to(DEV)
    xp = torch.from_numpy(g['x_plus']).to(DEV)
    D, M, J, phi, acc = s.multibody_terms(xp[:, :8], xp[:, 8:], None)
    assert D.shape[1:] == (24, 24) and M.shape[1:] == (7, 7) and J.shape[1:] == (24, 7) and phi.shape[1:] == (8,)
    P = oracle_params_from_golden(g, requires_grad=False)
    with torch.no_grad():
        Mo, Jo, phio, acco = co.multibody_terms(TreeCallables(ELBOW_TREE), P, xp.cpu()[:, :8], xp.cpu()[:, 8:])
        Do = Jo @ torch.linalg.solve(Mo, Jo.transpose(-1, -2))
    assert np.abs(M.cpu().numpy() - Mo.numpy()).max() < 1e-14 * max(1.0, np.abs(Mo.numpy()).max())
    assert np.abs(J.cpu().numpy() - Jo.numpy()).max() < 1e-13
    assert np.abs(phi.cpu().numpy() - phio.numpy()).max() < 1e-14
    assert np.abs(acc.cpu().numpy() - acco.numpy()).max() < 1e-9 * max(1.0, np.abs(acco.numpy()).max())
    assert np.abs(D.cpu().numpy() - Do.numpy()).max() < 1e-9 * np.abs(Do.numpy()).max()


def test_reverse_mode_rollout_backward_matches_forward_mode(assets_dir):
    """K7: dpll_cube_rollout_backward_f64 (reverse-mode adjoint, one 6x6 solve per step) against
    dpll_cube_rollout_grad_f64 (27 dual-number rollouts per toss) through the autograd Function, 256 tosses x 24
    steps from the example's initial-condition sampler: every gradient to 1e-10; and the module API
    (``simulate`` under autograd) uses the reverse-mode path."""
    g = load_golden('cube_real_perturbed')
    inertia, mu, half = (torch.from_numpy(a).to(DEV) for a in kernel_level_params(g))
    n, steps = 256, 24
    gen = torch.Generator().manual_seed(3)
    x0 = torch.tensor([1., 0., 0., 0., 0., 0., 0.12, 0., 0., 0., 0., 0., -.4], dtype=torch.float64).repeat(n, 1)
    x0[:, 7:] += (2 * torch.rand(n, 6, generator=gen, dtype=torch.float64) - 1) * torch.tensor([3., 3, 3, 1, 1, 1])
    quat = x0[:, :4] + 0.3 * torch.randn(n, 4, generator=gen, dtype=torch.float64)
    x0[:, :4] = quat / quat.norm(dim=-1, keepdim=True)
    w = torch.randn(n, steps + 1, 13, generator=gen, dtype=torch.float64).to(DEV)
    grads = []
    for forward_mode in (True, False):
        leaves = [t.clone().requires_grad_() for t in (x0.to(DEV), inertia, mu, half)]
        traj = ops.CubeRollout.apply(leaves[0], leaves[1], leaves[2], leaves[3], DT, steps, 1e-4, forward_mode)
        (traj * w).sum().backward()
        grads.append([t.grad.cpu().numpy() for t in leaves])
        assert (traj[:, -1, 6] < 0.11).any()                      # tosses reach the ground within the horizon
    for a, b in zip(grads[1], grads[0]):
        assert max_rel_to_scale(a, b) < 1e-10
    s = MultibodyLearnableSystem({'cube': os.path.join(assets_dir, 'cube.urdf')}, DT).to(DEV)
    xs = x0[:32].to(DEV).requires_grad_()
    traj, _ = s.simulate(xs.unsqueeze(-2), torch.zeros(32, 1, device=DEV), 6)
    assert traj.requires_grad
    traj.sum().backward()
    assert xs.grad is not None and torch.isfinite(xs.grad).all()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in s.parameters())


@pytest.mark.parametrize('name', ['shape_sphere', 'shape_polygon', 'shape_framed_box'])
def test_sphere_and_polygon_geometries_match_reference_golden(name, assets_dir):
    """SURVEY 8(f) N4, plane-convex half: a floating body with the reference's Sphere (geometry.py:415-456) or Polygon
    (:220-252) collision geometry through the module API -- the geometry module evaluates the support points, the
    witness-point kernels (dpll_body_loss_pts_f64 / dpll_body_step_pts_f64) do the rest -- against goldens produced by
    the reference's own classes: losses, gradients of theta / friction / radius or vertices, next states, at 1e-9."""
    from dair_pll_b200.geometry import Polygon
    g = load_golden(name)
    urdf = 'framed_box.urdf' if name == 'shape_framed_box' else 'sphere.urdf'
    s = MultibodyLearnableSystem({'body': os.path.join(assets_dir, urdf)}, float(g['dt']))
    ct = s.multibody_terms.contact_terms
    if name == 'shape_framed_box':
        # a Box in a collision frame offset and rotated in the link (URDF <collision><origin xyz rpy>): the frame comes
        # from the URDF, the contact points are the placed box's support points
        with torch.no_grad():
            ct.geometries[0].length_params.copy_(torch.from_numpy(g['shape_param']))
        leaf = lambda: ct.geometries[0].length_params       # noqa: E731
    elif name == 'shape_polygon':
        ct.geometries[0] = Polygon(torch.from_numpy(g['shape_param']), 4)
        leaf = lambda: ct.geometries[0].vertices            # noqa: E731
    else:
        with torch.no_grad():
            ct.geometries[0].length_param.copy_(torch.from_numpy(g['shape_param']))
        leaf = lambda: ct.geometries[0].length_param        # noqa: E731
    with torch.no_grad():
        s.multibody_terms.lagrangian_terms.inertial_parameters.copy_(torch.from_numpy(g['theta']))
        ct.friction_params.copy_(torch.from_numpy(g['friction_params']))
    s = s.to(DEV)
    x, xp = torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)
    loss = s.contactnets_loss(x, None, xp)
    loss.mean().backward()
    l = loss.detach().cpu().numpy()
    assert np.abs(l - g['loss']).max() < 1e-12
    assert rel_err(l, g['loss'], 1e-9).max() < 1e-9
    mt = s.multibody_terms
    assert max_rel_to_scale(mt.lagrangian_terms.inertial_parameters.grad.cpu().numpy(), g['grad_theta']) < 1e-9
    assert max_rel_to_scale(mt.contact_terms.friction_params.grad.cpu().numpy(), g['grad_friction']) < 1e-9
    assert max_rel_to_scale(leaf().grad.cpu().numpy(), g['grad_shape_param']) < 1e-9
    with torch.no_grad():
        traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(x.shape[0], 1, device=DEV), 2)
    assert np.abs(traj[:, 1].cpu().numpy() - g['x_next']).max() < 1e-9
    assert torch.isfinite(traj).all()
    # prediction-loss path: 3-step rollout, gradients of theta / friction / shape parameter / initial state against the
    # reference's own integrator differentiated by autograd (the support points depend on the state: a sphere's d r)
    for p in s.parameters():
        p.grad = None
    x0 = torch.from_numpy(g['roll_x0']).to(DEV).requires_grad_()
    w = torch.from_numpy(g['roll_w']).to(DEV)
    steps = w.shape[1]
    tr, _ = s.simulate(x0.unsqueeze(-2), torch.zeros(x0.shape[0], 1, device=DEV), steps)
    (tr[:, 1:] * w).sum().backward()
    assert np.abs(tr[:, 1:].detach().cpu().numpy() - g['roll_traj']).max() < 1e-8
    tol = 1e-7      # the reference form of the velocity update loses ~cond(Q) eps of the derivatives (DESIGN.md section 2)
    assert max_rel_to_scale(x0.grad.cpu().numpy(), g['roll_grad_x0']) < tol
    assert max_rel_to_scale(mt.lagrangian_terms.inertial_parameters.grad.cpu().numpy(), g['roll_grad_theta']) < tol
    assert max_rel_to_scale(mt.contact_terms.friction_params.grad.cpu().numpy(), g['roll_grad_friction']) < tol
    assert max_rel_to_scale(leaf().grad.cpu().numpy(), g['roll_grad_shape_param']) < tol


def test_warm_started_solves_give_the_same_results_in_fewer_iterations(assets_dir):
    """dpll_cube_loss_leaf_dp_* with u_init / u_out: started from the optima found with slightly different parameters
    (a training loop's previous epoch) the solves reach the same losses and gradients (the QP's optimum is unique) in
    fewer Newton iterations; through the module API the data set carries the solutions."""
    from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig
    g = load_golden('cube_synthetic')
    theta = torch.from_numpy(g['theta']).to(DEV)
    fr = torch.from_numpy(g['friction_params']).to(DEV)
    ln = torch.from_numpy(g['half_lengths']).reshape(1, 3).to(DEV)
    inertia, mu, half = (torch.from_numpy(a).to(DEV) for a in kernel_level_params(g))
    n = 100003
    x = synthetic.cube_states(n, seed=81, device=DEV)
    traj, _ = ops.cube_rollout(x, inertia, mu, half, DT, 1)
    xp = synthetic.perturb_next_state(traj[:, 1], seed=82)
    cold = ops.cube_loss_leaf_dp_raw(x, xp, theta, fr, ln, DT, 1e-3, want_iters=True, want_u=True)
    assert cold[5].shape == (n, 6) and (cold[5][cold[4] == 0] == 0).all()
    # same parameters: already optimal -> no Newton direction is taken, bits of the loss unchanged to rounding
    same = ops.cube_loss_leaf_dp_raw(x, xp, theta, fr, ln, DT, 1e-3, want_iters=True, u_init=cold[5], want_u=True)
    assert int(same[4].max()) <= 1 and torch.allclose(same[0], cold[0], rtol=1e-12, atol=1e-18)
    # moved parameters: same answers as a cold solve, far fewer iterations
    theta2, fr2, ln2 = theta * 1.001, fr * 0.999, ln * 1.0005
    ref = ops.cube_loss_leaf_dp_raw(x, xp, theta2, fr2, ln2, DT, 1e-3, want_iters=True)
    warm = ops.cube_loss_leaf_dp_raw(x, xp, theta2, fr2, ln2, DT, 1e-3, want_iters=True, u_init=cold[5])
    assert rel_err(warm[0].cpu().numpy(), ref[0].cpu().numpy(), 1e-9).max() < 1e-10
    assert max_rel_to_scale(warm[1].cpu().numpy(), ref[1].cpu().numpy()) < 1e-11
    assert warm[4].double().mean().item() < 0.6 * ref[4].double().mean().item()
    # a bad start is only slower, never wrong
    junk = ops.cube_loss_leaf_dp_raw(x, xp, theta2, fr2, ln2, DT, 1e-3, u_init=torch.randn(n, 6, dtype=torch.float64, device=DEV))
    assert rel_err(junk[0].cpu().numpy(), ref[0].cpu().numpy(), 1e-9).max() < 1e-9
    # module API + data set
    ds = DeviceTrajectorySliceDataset(TrajectorySliceConfig(), device=torch.device(DEV))
    ds.add_slices_from_trajectory(torch.stack((x[:5000], xp[:5000]), 1).reshape(-1, 13)[:2])   # placeholder trajectory
    s = MultibodyLearnableSystem({'cube': os.path.join(assets_dir, 'cube.urdf')}, DT).to(DEV)
    s.record_qp_solution = True
    l0 = s.contactnets_loss(x[:5000], None, xp[:5000])
    assert l0.qp_solution.shape == (5000, 6)
    s.qp_warm_start = l0.qp_solution
    s.record_newton_iters = True
    l1 = s.contactnets_loss(x[:5000], None, xp[:5000])
    assert s.qp_warm_start is None and int(l1.newton_iters.max()) <= 1
    assert torch.allclose(l1.detach(), l0.detach(), rtol=1e-12, atol=1e-18)
    ds.update_solutions(torch.tensor([0]), l0.qp_solution[:1])
    assert ds.warm_start(torch.tensor([0])).shape == (1, 6)


def _chain_system(g, urdf, n):
    s = MultibodyLearnableSystem({'chain': urdf}, float(g['dt']))
    sd = {'multibody_terms.lagrangian_terms.inertial_parameters': torch.from_numpy(g['theta']),
          'multibody_terms.contact_terms.friction_params': torch.from_numpy(g['friction_params'])}
    for i in range(g['half_lengths'].shape[0]):      # one entry per box (tree4g: fewer boxes than links)
        sd[f'multibody_terms.contact_terms.geometries.{i}.length_params'] = torch.from_numpy(g['half_lengths'][i]).reshape(1, 3)
    s.load_state_dict(sd)
    return s.to(DEV)


@pytest.mark.parametrize('name, n_links', [('chain3', 3), ('chain3r', 3), ('slider3', 3), ('tree4', 4), ('tree4g', 4),
                                           ('tree6', 6)])
def test_generic_chain_and_tree_match_reference_golden(name, n_links, assets_dir):
    """N2: a three-link URDF with a rotated, off-axis second joint, and a BRANCHING four-link URDF (two links off the
    root, a third off one of them), go URDF -> SystemSpec -> the generic tree kernels; losses, every parameter gradient
    and a time step against the reference's own contactnets_loss / sim_step (tests/golden/{chain3,tree4}.npz,
    oracle/gen_golden_chain.py)."""
    g = load_golden(name)
    s = _chain_system(g, os.path.join(assets_dir, f'{name}.urdf'), n_links)
    assert s._kind() == 'chain' and s.space.n_x == 13 + 2 * (n_links - 1)
    x, xp = torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)
    loss = s.contactnets_loss(x, None, xp)
    loss.mean().backward()
    l = loss.detach().cpu().numpy()
    assert np.abs(l - g['loss']).max() < 1e-12
    assert rel_err(l, g['loss'], 1e-9).max() < 1e-9
    gt, gf, *gl = _leaf_grads(s)
    assert max_rel_to_scale(gt, g['grad_theta']) < 1e-9
    assert max_rel_to_scale(gf, g['grad_friction']) < 1e-9
    assert max_rel_to_scale(np.stack([a.reshape(3) for a in gl]), g['grad_length']) < 1e-9
    with torch.no_grad():
        traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(x.shape[0], 1, device=DEV), 3)
    t = traj.cpu().numpy()
    assert np.abs(t[:, 1] - g['x_next']).max() < 1e-9
    assert np.isfinite(t).all() and np.abs(np.linalg.norm(t[:, :, :4], axis=-1) - 1).max() < 1e-12
    # the rollout is the step applied repeatedly
    with torch.no_grad():
        one, _ = s.simulate(traj[:, 1:2], torch.zeros(x.shape[0], 1, device=DEV), 1)
    assert (one[:, 1] - traj[:, 2]).abs().max().item() < 1e-12
    # prediction-loss path: 3-step rollout gradients (forward-mode tangents, dpll_chain_rollout_grad_f64) against the
    # reference's own integrator differentiated by autograd
    for p in s.parameters():
        p.grad = None
    x0 = torch.from_numpy(g['roll_x0']).to(DEV).requires_grad_()
    w = torch.from_numpy(g['roll_w']).to(DEV)
    tr, _ = s.simulate(x0.unsqueeze(-2), torch.zeros(x0.shape[0], 1, device=DEV), w.shape[1])
    (tr[:, 1:] * w).sum().backward()
    assert np.abs(tr[:, 1:].detach().cpu().numpy() - g['roll_traj']).max() < 1e-8
    tol = 1e-7      # the reference form of the velocity update loses ~cond(Q) eps of the derivatives (DESIGN.md section 2)
    gt, gf, *gl = _leaf_grads(s)
    assert max_rel_to_scale(x0.grad.cpu().numpy(), g['roll_grad_x0']) < tol
    assert max_rel_to_scale(gt, g['roll_grad_theta']) < tol
    assert max_rel_to_scale(gf, g['roll_grad_friction']) < tol
    assert max_rel_to_scale(np.stack([a.reshape(3) for a in gl]), g['roll_grad_length']) < tol


@pytest.mark.parametrize('name', ['chain3r', 'slider3', 'tree4g', 'tree6'])
def test_tree_dense_terms_match_oracle(name, assets_dir):
    """MultibodyTerms.forward for the generic trees (multibody_terms.py:584-609; dpll_chain_terms_f64) through the module
    API: the (delassus, M, J, phi, acceleration) tuple against the oracle's tree callables at the golden states -- rotated
    collision frames, the sliding joint, fewer boxes than links, six links."""
    from oracle import contactnets_oracle as co
    from oracle.callables import CHAIN3R_TREE, SLIDER3_TREE, TREE4G_TREE, TREE6_TREE, TreeCallables
    from tests.util import oracle_params_from_golden
    tree = {'chain3r': CHAIN3R_TREE, 'slider3': SLIDER3_TREE, 'tree4g': TREE4G_TREE, 'tree6': TREE6_TREE}[name]
    n, n_boxes = tree.n_bodies, len(tree.geometry_body) - 1
    g = load_golden(name)
    s = _chain_system(g, os.path.join(assets_dir, f'{name}.urdf'), n)
    xp = torch.from_numpy(g['x_plus']).to(DEV)
    nq, nv, k = 7 + n - 1, 6 + n - 1, 12 * n_boxes
    D, M, J, phi, acc = s.multibody_terms(xp[:, :nq], xp[:, nq:], None)
    assert D.shape[1:] == (k, k) and M.shape[1:] == (nv, nv) and J.shape[1:] == (k, nv) and phi.shape[1:] == (4 * n_boxes,)
    P = oracle_params_from_golden(g, requires_grad=False)
    with torch.no_grad():
        Mo, Jo, phio, acco = co.multibody_terms(TreeCallables(tree), P, xp.cpu()[:, :nq], xp.cpu()[:, nq:])
        Do = Jo @ torch.linalg.solve(Mo, Jo.transpose(-1, -2))
    assert np.abs(M.cpu().numpy() - Mo.numpy()).max() < 1e-14 * max(1.0, np.abs(Mo.numpy()).max())
    assert np.abs(J.cpu().numpy() - Jo.numpy()).max() < 1e-13
    assert np.abs(phi.cpu().numpy() - phio.numpy()).max() < 1e-14
    assert np.abs(acc.cpu().numpy() - acco.numpy()).max() < 1e-9 * max(1.0, np.abs(acco.numpy()).max())
    assert np.abs(D.cpu().numpy() - Do.numpy()).max() < 1e-9 * np.abs(Do.numpy()).max()


@pytest.mark.parametrize('name', ['elbow_nominal', 'elbow_perturbed'])
def test_generic_chain_two_links_reproduces_the_elbow_kernels(name, assets_dir):
    """The generic recursion at N = 2 against the reference goldens of the elbow AND against the specialised kernels."""
    g = load_golden(name)
    x, xp = torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)
    s = _chain_system(g, os.path.join(assets_dir, 'elbow.urdf'), 2)
    inertia, mu, half, kin = (t.detach() for t in s._elbow_params(torch.float64, torch.device(DEV)))
    eye = [1, 0, 0, 0, 1, 0, 0, 0, 1]
    kin18 = torch.tensor([0, 0, 0, *eye, 0, 0, 1, *kin[6:9].tolist(), 0, *eye, 0, 0, 1,
                          *kin[0:3].tolist(), *eye, *kin[3:6].tolist(), *kin[9:12].tolist(), 0, *eye, 0, 1, 1],
                         dtype=torch.float64, device=DEV)      # ... | parent | collision-frame rotation | type | box link | used
    inertia.requires_grad_(); mu.requires_grad_(); half.requires_grad_()
    loss = ops.ChainContactNetsLoss.apply(x, xp, inertia, mu, half, kin18, 2, float(g['dt']), 1e-3)
    loss.sum().backward()
    l = loss.detach().cpu().numpy()
    assert rel_err(l, g['loss'], 1e-9).max() < 1e-9
    ref_loss, ref_grad, _, _, _ = ops.elbow_loss_raw(x, xp, inertia.detach(), mu.detach(), half.detach(), kin,
                                                     float(g['dt']), 1e-3)
    assert rel_err(l, ref_loss.cpu().numpy(), 1e-9).max() < 1e-10
    mine = torch.cat((inertia.grad.reshape(-1), mu.grad, half.grad.reshape(-1))).cpu().numpy()
    assert max_rel_to_scale(mine, ref_grad.cpu().numpy()) < 1e-10


def _icnn_weights(width, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(3, width, generator=g, dtype=torch.float64), torch.randn(3, width, generator=g, dtype=torch.float64),
            torch.randn(width, width, generator=g, dtype=torch.float64) / width, torch.randn(width, generator=g, dtype=torch.float64)]


@pytest.mark.parametrize('slope', [0.5, 0.25, 0.0])
def test_tensor_core_support_points_match_the_fp64_layer_path(slope):
    """csrc/cn_icnn_tc.cu (int8 digit-plane products on tcgen05, fp64 reconstruction) against the FP64 layer path
    (dpll_icnn_* + library GEMMs) and the oracle: empty, single-row, ragged and multi-tile batches, three slopes.
    Tolerance 1e-11 of the point scale (the 42-bit Jacobian quantisation is below 1e-12)."""
    from oracle import contactnets_oracle as co
    ws = _icnn_weights(256, 5)
    wd = [w.to(DEV) for w in ws]
    for rows in (0, 1, 127, 128, 129, 20000):
        d = torch.randn(rows, 3, generator=torch.Generator().manual_seed(rows), dtype=torch.float64)
        d = d / d.norm(dim=-1, keepdim=True).clamp(min=1e-300)
        got = ops.icnn_support_points_tc(d.to(DEV), *wd, slope)
        assert got.shape == (rows, 3)
        if rows == 0:
            continue
        ref = ops.icnn_support_forward(d.to(DEV), *wd, slope)[0]
        scale = ref.abs().max().item()
        assert (got - ref).abs().max().item() < 1e-11 * scale
        if rows <= 129 and slope == 0.5:
            po = co.icnn_support(dict(Wd0=ws[0], Wd1=ws[1], Wh=ws[2], wout=ws[3]), d)
            assert (got.cpu() - po).abs().max().item() < 1e-11 * scale
    # a zero direction row (what a padded tile sees) gives a finite point -- the one of the all-negative mask -- not NaN
    zero = torch.zeros(3, 3, dtype=torch.float64, device=DEV)
    z = ops.icnn_support_points_tc(zero, *wd, slope)
    assert torch.isfinite(z).all()
    assert (z - ops.icnn_support_forward(zero, *wd, slope)[0]).abs().max().item() < 1e-11 * scale
    # the rare-path fallback on EVERY entry: directions scaled by 1e-12 put every |z1| below its tolerance, so every
    # (row, column group) is redone in plain fp64 after the tile loop; support points are homogeneous of degree 0 in the
    # direction, so the answer is the one of the unscaled directions
    d = torch.randn(300, 3, generator=torch.Generator().manual_seed(77), dtype=torch.float64).to(DEV)
    tiny = ops.icnn_support_points_tc(d * 1e-12, *wd, slope)
    ref = ops.icnn_support_forward(d, *wd, slope)[0]
    assert (tiny - ref).abs().max().item() < 1e-11 * ref.abs().max().item()


def test_support_network_backward_visits_only_rows_with_a_cotangent():
    """ICNNSupport.backward gathers the rows whose cotangent is non-zero (3.7% of the rows of the config-3 batch) and
    re-evaluates only those: the weight gradients equal autograd through the oracle with the same sparse cotangent;
    an all-zero cotangent gives zero gradients."""
    from dair_pll_b200.deep_support_function import ICNNSupport
    from oracle import contactnets_oracle as co
    ws = _icnn_weights(256, 9)
    rows = 6000
    g = torch.Generator().manual_seed(1)
    d = torch.randn(rows, 3, generator=g, dtype=torch.float64)
    d = d / d.norm(dim=-1, keepdim=True)
    gp = torch.randn(rows, 3, generator=g, dtype=torch.float64)
    gp[torch.rand(rows, generator=g) < 0.9] = 0
    a = [w.clone().to(DEV).requires_grad_() for w in ws]
    p = ICNNSupport.apply(d.to(DEV), a[0], a[1], a[2], a[3], 0.5)
    (p * gp.to(DEV)).sum().backward()
    b = [w.clone().requires_grad_() for w in ws]
    po = co.icnn_support(dict(Wd0=b[0], Wd1=b[1], Wh=b[2], wout=b[3]), d)
    (po * gp).sum().backward()
    for x, y in zip(a, b):
        assert (x.grad.cpu() - y.grad).abs().max() <= 1e-10 * y.grad.abs().max()
    a2 = [w.clone().to(DEV).requires_grad_() for w in ws]
    p2 = ICNNSupport.apply(d.to(DEV), a2[0], a2[1], a2[2], a2[3], 0.5)
    (p2 * 0).sum().backward()
    assert all((x.grad == 0).all() for x in a2)


def test_elbow_support_directions_kernel_matches_the_tensor_formula(assets_dir):
    """dpll_elbow_support_directions_f64 against the host formula it replaces (minus the third row of each link's
    rotation, perturbed and normalised, geometry.py:309-325, 560-567), through a strided view of the state batch."""
    torch.manual_seed(0)
    s = MultibodyLearnableSystem({'elbow': os.path.join(assets_dir, 'elbow_mesh.urdf')}, DT).to(DEV)
    x = synthetic.elbow_states(3001, seed=5, device=DEV)
    q = x[:, :8]
    geoms = s.multibody_terms.contact_terms.geometries
    _, axis = s._elbow_kin(torch.float64, torch.device(DEV))
    d0, d1 = ops.elbow_support_directions(q, axis, geoms[0].perturbations, geoms[1].perturbations)
    w, xx, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    sc = 2.0 / (w * w + xx * xx + y * y + z * z)
    row = torch.stack((sc * (xx * z - w * y), sc * (y * z + w * xx), 1 - sc * (xx * xx + y * y)), -1)
    th = q[:, 7:8]
    row2 = row * torch.cos(th) + torch.linalg.cross(row, axis.expand_as(row)) * torch.sin(th) \
        + axis * (row @ axis)[:, None] * (1 - torch.cos(th))
    for got, base, geom in ((d0, row, geoms[0]), (d1, row2, geoms[1])):
        ref = -base.unsqueeze(-2) + geom.perturbations
        ref = ref / ref.norm(dim=-1, keepdim=True)
        assert (got - ref).abs().max().item() < 1e-14


@pytest.mark.parametrize('name', ['cube', 'elbow', 'chain3', 'tree4', 'tree4g', 'tree6'])
def test_leaf_preparation_kernels_match_the_host_parameter_graph(name, assets_dir):
    """dpll_leaf_prepare_f64 / dpll_leaf_backward_f64 (one launch each) against the PyTorch graph they replace --
    theta -> [m, c, I_cm/m] (inertia.py:205-234, 304-331, 376-382), pairwise friction (multibody_terms.py:466-471),
    |length_params| (geometry.py:394-397) -- values and the chain rule to the leaves, with perturbed (sign-mixed) leaves."""
    s = MultibodyLearnableSystem({name: os.path.join(assets_dir, f'{name}.urdf')}, DT).to(DEV)
    mt = s.multibody_terms
    gen = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for p in mt.parameters():
            p.mul_(1 + 0.2 * (torch.rand(p.shape, generator=gen, dtype=p.dtype) - 0.5).to(DEV))
        mt.contact_terms.friction_params[0].neg_()               # |.| and its sign in the chain rule
        mt.contact_terms.geometries[mt.contact_terms._pairs[0][1]].length_params[0, 1].neg_()
    inertia, mu, half = mt.kernel_parameters(torch.float64)                         # the kernels
    ref_in = mt.lagrangian_terms.inertia_vector()
    ref_mu = mt.contact_terms.pair_friction()
    ref_half = mt.contact_terms.half_lengths()
    assert max_rel_to_scale(inertia.detach().cpu().numpy(), ref_in.detach().cpu().numpy()) < 1e-14
    assert max_rel_to_scale(mu.detach().cpu().numpy(), ref_mu.detach().cpu().numpy()) < 1e-15
    assert len(half) == len(ref_half)
    wi, wm = torch.randn_like(ref_in), torch.randn_like(ref_mu)
    wh = [torch.randn_like(h) for h in ref_half]
    for h, r in zip(half, ref_half):
        assert torch.equal(h.detach(), r.detach())
    grads = []
    for (a, b, c) in ((inertia, mu, half), (ref_in, ref_mu, ref_half)):
        for p in mt.parameters():
            p.grad = None
        ((a * wi).sum() + (b * wm).sum() + sum((h * w).sum() for h, w in zip(c, wh))).backward()
        grads.append(_leaf_grads(s))
    for got, ref in zip(*grads):
        assert max_rel_to_scale(got, ref) < 1e-13


def test_learned_geometry_rollout_is_differentiable_and_matches_oracle_autograd(assets_dir):
    """Prediction-loss path with learned (support-function) geometry (multibody_learnable_system.py:293-304 through
    geometry.py:309-325): a 3-step rollout of the two-body system with two width-256 networks through the module API --
    trajectory, and the gradients of theta, friction, every network weight and the initial state -- against autograd
    through the CPU oracle's simulate()."""
    from oracle import contactnets_oracle as co
    from oracle.callables import ELBOW_TREE, TreeCallables
    torch.manual_seed(0)
    s = MultibodyLearnableSystem({'elbow': os.path.join(assets_dir, 'elbow_mesh.urdf')}, DT).to(DEV)
    n, steps = 24, 3
    x0 = synthetic.elbow_states(n, seed=41, device=DEV).requires_grad_()
    gen = torch.Generator().manual_seed(5)
    target = torch.randn(n, steps, 15, generator=gen, dtype=torch.float64).to(DEV)
    traj, _ = s.simulate(x0.unsqueeze(-2), torch.zeros(n, 1, device=DEV), steps)
    ((traj[:, 1:] - target) ** 2).sum().backward()
    mt = s.multibody_terms
    nets = []
    for gi in range(2):
        geom = mt.contact_terms.geometries[gi]
        net = geom.network
        nets.append(dict(Wd0=net.input_weights[0].detach().cpu().clone().requires_grad_(),
                         Wd1=net.input_weights[1].detach().cpu().clone().requires_grad_(),
                         Wh=net.hidden_weights[0].detach().cpu().clone().requires_grad_(),
                         wout=net.output_weight.detach().cpu().clone().requires_grad_(),
                         perturbations=geom.perturbations.detach().cpu().clone()))
    P = co.OracleParams(mt.lagrangian_terms.inertial_parameters.detach().cpu().clone(),
                        mt.contact_terms.friction_params.detach().cpu().clone(), [], icnn=nets).requires_grad_()
    x0o = x0.detach().cpu().clone().requires_grad_()
    tro = co.simulate(TreeCallables(ELBOW_TREE), P, x0o, DT, steps)
    ((tro[:, 1:] - target.cpu()) ** 2).sum().backward()
    assert np.abs(traj.detach().cpu().numpy() - tro.detach().numpy()).max() < 1e-8
    # tolerance: the reference form of the velocity update loses ~cond(Q) eps of the derivatives (DESIGN.md section 2)
    tol = 1e-7
    assert max_rel_to_scale(mt.lagrangian_terms.inertial_parameters.grad.cpu().numpy(), P.inertial_parameters.grad.numpy()) < tol
    assert max_rel_to_scale(mt.contact_terms.friction_params.grad.cpu().numpy(), P.friction_params.grad.numpy()) < tol
    assert max_rel_to_scale(x0.grad.cpu().numpy(), x0o.grad.numpy()) < tol
    seen = 0
    for gi in range(2):
        net = mt.contact_terms.geometries[gi].network
        for k, p in (('Wd0', net.input_weights[0]), ('Wd1', net.input_weights[1]), ('Wh', net.hidden_weights[0]),
                     ('wout', net.output_weight)):
            ref = nets[gi][k].grad.numpy()
            assert max_rel_to_scale(p.grad.cpu().numpy(), ref) < tol, (gi, k)
            seen += int(np.abs(ref).max() > 0)
    assert seen >= 4          # the batch does train the geometry (contacts carry force during the rollout)


def test_racing_kernel_for_the_expensive_head_gives_the_same_results(assets_dir):
    """DPLL_LOSS_RACE: the first B/64 samples of a cost-ordered batch are solved from eight start points at once (first to
    converge wins) on a second stream.  The optimum is unique, so per-sample losses, the summed loss and the leaf
    gradients must equal the plain dynamic launch's to solver tolerance -- eagerly and replayed from a CUDA graph."""
    import bench
    from dair_pll_b200 import parallel
    system = bench.make_system(torch.device(DEV), torch.float64)
    x, xp = bench.make_batch(system, 65536, 123, torch.device(DEV), torch.float64)
    lt, ct = system.multibody_terms.lagrangian_terms, system.multibody_terms.contact_terms
    leaves = [t.detach() for t in (lt.inertial_parameters, ct.friction_params, ct.geometries[0].length_params)]
    it = ops.cube_loss_leaf_dp_raw(x, xp, *leaves, DT, 1e-3, want_iters=True)[4]
    order = torch.argsort(it, descending=True, stable=True)
    xo, xpo = x.index_select(0, order).contiguous(), xp.index_select(0, order).contiguous()
    ref = ops.cube_loss_leaf_dp_raw(xo, xpo, *leaves, DT, 1e-3, flags=ops.LOSS_DYNAMIC, want_iters=True)
    got = ops.cube_loss_leaf_dp_raw(xo, xpo, *leaves, DT, 1e-3, flags=ops.LOSS_DYNAMIC | ops.LOSS_RACE, want_iters=True)
    torch.cuda.synchronize()
    head = 65536 // 64
    scale = ref[0].abs().max().item()
    assert (got[0] - ref[0]).abs().max().item() < 1e-11 * scale                  # per-sample losses
    assert torch.equal(got[0][head:], ref[0][head:])                             # the wavefront part is the same computation
    assert max_rel_to_scale(got[1].cpu().numpy(), ref[1].cpu().numpy()) < 1e-10  # [leaf gradients | loss sum | count]
    assert int(got[4][:head].max()) < int(ref[4][:head].max())                   # the worst chain did get shorter
    # public API + graph capture (fork / join of the second stream inside the capture)
    system.dynamic_schedule = True
    params = list(system.parameters())

    def step():
        for p in params:
            p.grad = None
        m = system.contactnets_loss(xo, None, xpo).mean()
        m.backward()
        return m.detach()
    eager = step().clone()
    g_eager = [p.grad.clone() for p in params]
    graphed = parallel.GraphedStep(step, torch.device(DEV))
    for _ in range(3):
        out = graphed()
    torch.cuda.synchronize()
    assert abs(out.item() - eager.item()) < 1e-12 * abs(eager.item())
    for p, g in zip(params, g_eager):
        assert max_rel_to_scale(p.grad.cpu().numpy(), g.cpu().numpy()) < 1e-10
    system.race_expensive_head = False
    plain = step()
    assert abs(plain.item() - eager.item()) < 1e-11 * abs(eager.item())


@pytest.mark.parametrize('depth', [1, 3, 4])
def test_support_network_of_other_depths_matches_the_reference_class(depth):
    """``HomogeneousICNN`` at depths other than the default 2 (deep_support_function.py:125-266): support points and the
    gradients of a linear functional of them with respect to EVERY weight against the reference's own class
    (tests/golden/icnn_depth.npz, oracle/gen_golden_icnn_depth.py), 1e-12."""
    from dair_pll_b200.deep_support_function import HomogeneousICNN
    g = load_golden('icnn_depth')
    width = int(g['width'])
    net = HomogeneousICNN(depth, width, negative_slope=0.5)
    with torch.no_grad():
        for i, w in enumerate(net.input_weights):
            w.copy_(torch.from_numpy(g[f'd{depth}_in{i}']))
        for i, w in enumerate(net.hidden_weights):
            w.copy_(torch.from_numpy(g[f'd{depth}_hid{i}']))
        net.output_weight.copy_(torch.from_numpy(g[f'd{depth}_out']))
    net = net.to(DEV)
    d = torch.from_numpy(g['directions']).to(DEV)
    c = torch.from_numpy(g['cotangent']).to(DEV)
    p = net(d)
    assert max_rel_to_scale(p.detach().cpu().numpy(), g[f'd{depth}_p']) < 1e-12
    (p * c).sum().backward()
    for i, w in enumerate(net.input_weights):
        assert max_rel_to_scale(w.grad.cpu().numpy(), g[f'd{depth}_gin{i}']) < 1e-12, ('input', i)
    for i, w in enumerate(net.hidden_weights):
        assert max_rel_to_scale(w.grad.cpu().numpy(), g[f'd{depth}_ghid{i}']) < 1e-12, ('hidden', i)
    assert max_rel_to_scale(net.output_weight.grad.cpu().numpy(), g[f'd{depth}_gout']) < 1e-12


def test_summary_mesh_matches_the_reference_extraction():
    """``extract_mesh`` (deep_support_function.py:95-122) of a depth-3 network evaluated on the device against the mesh
    the reference's own function extracted from the same weights: same vertices (1e-10 absolute), same set of
    outward-wound triangles."""
    from dair_pll_b200.deep_support_function import HomogeneousICNN, extract_mesh
    g = load_golden('icnn_depth')
    net = HomogeneousICNN(3, int(g['width']), negative_slope=0.5)
    with torch.no_grad():
        for i, w in enumerate(net.input_weights):
            w.copy_(torch.from_numpy(g[f'd3_in{i}']))
        for i, w in enumerate(net.hidden_weights):
            w.copy_(torch.from_numpy(g[f'd3_hid{i}']))
        net.output_weight.copy_(torch.from_numpy(g['d3_out']))
    mesh = extract_mesh(net.to(DEV))
    gv, gf = g['d3_mesh_vertices'], g['d3_mesh_faces']
    key = lambda v: tuple(np.round(np.asarray(v) * 1e10).astype(np.int64).tolist())   # noqa: E731  (shape is ~0.1 across)
    assert {key(v) for v in mesh.vertices.numpy()} == {key(v) for v in gv}

    def canon(vertices, faces):   # oriented triangles by vertex coordinates, rotation-invariant
        out = set()
        for f in faces.tolist():
            tri = [key(vertices[i]) for i in f]
            k = tri.index(min(tri))
            out.add((tri[k], tri[(k + 1) % 3], tri[(k + 2) % 3]))
        return out
    assert canon(mesh.vertices.numpy(), mesh.faces.numpy()) == canon(gv, gf)


def test_elbow_mesh_summary_carries_the_learned_meshes(assets_dir):
    """``MultibodyLearnableSystem.summary`` for the learned-geometry elbow (multibody_learnable_system.py:313-333,
    multibody_terms.py:566-580): one mesh per link from the default depth-2 tensor-core networks, with the bounding-box
    scalars; every mesh is a closed convex surface (Euler characteristic 2) whose vertices are support points."""
    system = MultibodyLearnableSystem({'elbow': os.path.join(assets_dir, 'elbow_mesh.urdf')}, DT).to(DEV)
    summary = system.summary({})
    assert len(summary.meshes) == 2
    for name, mesh in summary.meshes.items():
        v, f = mesh.vertices.shape[0], mesh.faces.shape[0]
        edges = {tuple(sorted((tri[i], tri[(i + 1) % 3]))) for tri in mesh.faces.tolist() for i in range(3)}
        assert v - len(edges) + f == 2
        for axis in 'xyz':
            assert summary.scalars[f'{name}_diameter_{axis}'] > 0
            assert f'{name}_center_{axis}' in summary.scalars


def test_mixed_box_and_learned_geometry_elbow_matches_reference_golden(assets_dir):
    """The two-body system with a Box on the first link and a DeepSupportConvex on the second (mixed collision geometry):
    the box's corners and the network's support points meet as witness points of the same kernels; loss, the gradients of
    theta, friction, the BOX LENGTHS and every network weight, and a 3-step rollout against a golden produced by the
    reference's own classes (oracle/gen_golden_mixed.py), 1e-9."""
    from dair_pll_b200.deep_support_function import HomogeneousICNN
    from dair_pll_b200.geometry import Box, DeepSupportConvex
    g = load_golden('elbow_mixed_w64')
    s = MultibodyLearnableSystem({'elbow': os.path.join(assets_dir, 'elbow_mixed.urdf')}, float(g['dt']))
    geoms = s.multibody_terms.contact_terms.geometries
    assert isinstance(geoms[0], Box) and isinstance(geoms[1], DeepSupportConvex) and s._kind() == 'elbow'
    geoms[1].network = HomogeneousICNN(2, 64)
    geoms[1].perturbations = torch.from_numpy(g['net_perturbations'])
    pre = 'multibody_terms.contact_terms.geometries.'
    s.load_state_dict({'multibody_terms.lagrangian_terms.inertial_parameters': torch.from_numpy(g['theta']),
                       'multibody_terms.contact_terms.friction_params': torch.from_numpy(g['friction_params']),
                       pre + '0.length_params': torch.from_numpy(g['box_length_params']),
                       pre + '1.network.input_weights.0': torch.from_numpy(g['net_Wd0']),
                       pre + '1.network.input_weights.1': torch.from_numpy(g['net_Wd1']),
                       pre + '1.network.hidden_weights.0': torch.from_numpy(g['net_Wh']),
                       pre + '1.network.output_weight': torch.from_numpy(g['net_wout'])})
    s = s.to(DEV)
    x, xp = torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)
    loss = s.contactnets_loss(x, None, xp)
    loss.mean().backward()
    l = loss.detach().cpu().numpy()
    assert np.abs(l - g['loss']).max() < 1e-12
    assert rel_err(l, g['loss'], 1e-9).max() < 1e-9
    mt = s.multibody_terms
    assert max_rel_to_scale(mt.lagrangian_terms.inertial_parameters.grad.cpu().numpy(), g['grad_theta']) < 1e-9
    assert max_rel_to_scale(mt.contact_terms.friction_params.grad.cpu().numpy(), g['grad_friction']) < 1e-9
    assert max_rel_to_scale(geoms[0].length_params.grad.cpu().numpy(), g['grad_box_length_params']) < 1e-9
    net = geoms[1].network
    for k, p_ in (('Wd0', net.input_weights[0]), ('Wd1', net.input_weights[1]), ('Wh', net.hidden_weights[0]),
                  ('wout', net.output_weight)):
        assert max_rel_to_scale(p_.grad.cpu().numpy(), g[f'net_grad_{k}']) < 1e-9, k
    x0 = torch.from_numpy(g['sim_x0']).to(DEV)
    with torch.no_grad():
        traj, _ = s.simulate(x0.unsqueeze(-2), torch.zeros(x0.shape[0], 1, device=DEV), g['sim_traj'].shape[1] - 1)
    t = traj.cpu().numpy()
    assert np.abs(t[:, 1] - g['sim_traj'][:, 1]).max() < 1e-9
    assert np.abs(t - g['sim_traj']).max() < 1e-6


def test_tree_with_sphere_and_polygon_links_matches_reference_golden(assets_dir):
    """Any plane-convex shape on any link of a tree (witness-point form of the tree kernels, dpll_chain_loss_pts_f64): the three-link chain with the reference's Box on link 0, Sphere on link 1 and Polygon on link 2
    through the module API -- the shapes' support points from the host side (torch forward kinematics + the geometry
    classes), everything else in the kernels -- against a golden produced by the reference's own classes
    (oracle/gen_golden_chain.py:make_shapes): losses and the gradients of theta, friction, box lengths, radius and vertices at 1e-9."""
    from dair_pll_b200.geometry import Polygon, Sphere
    g = load_golden('chain3s')
    s = MultibodyLearnableSystem({'chain3': os.path.join(assets_dir, 'chain3.urdf')}, float(g['dt']))
    ct = s.multibody_terms.contact_terms
    ct.geometries[1] = Sphere(torch.from_numpy(g['sphere_radius']))
    ct.geometries[2] = Polygon(torch.from_numpy(g['polygon_vertices']), 4)
    with torch.no_grad():
        s.multibody_terms.lagrangian_terms.inertial_parameters.copy_(torch.from_numpy(g['theta']))
        ct.friction_params.copy_(torch.from_numpy(g['friction_params']))
        ct.geometries[0].length_params.copy_(torch.from_numpy(g['box_length_params']))
    s = s.to(DEV)
    x, xp = torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)
    loss = s.contactnets_loss(x, None, xp)
    loss.mean().backward()
    l = loss.detach().cpu().numpy()
    assert np.abs(l - g['loss']).max() < 1e-12
    assert rel_err(l, g['loss'], 1e-9).max() < 1e-9
    mt = s.multibody_terms
    assert max_rel_to_scale(mt.lagrangian_terms.inertial_parameters.grad.cpu().numpy(), g['grad_theta']) < 1e-9
    assert max_rel_to_scale(mt.contact_terms.friction_params.grad.cpu().numpy(), g['grad_friction']) < 1e-9
    assert max_rel_to_scale(ct.geometries[0].length_params.grad.cpu().numpy(), g['grad_box_length_params']) < 1e-9
    assert max_rel_to_scale(ct.geometries[1].length_param.grad.cpu().numpy(), g['grad_sphere_radius']) < 1e-9
    assert max_rel_to_scale(ct.geometries[2].vertices.grad.cpu().numpy(), g['grad_polygon_vertices']) < 1e-9
    # (the time step of such systems has no GPU entry point yet: refused, not approximated)
    with pytest.raises(NotImplementedError), torch.no_grad():
        s.simulate(x.unsqueeze(-2), torch.zeros(x.shape[0], 1, device=DEV), 2)
