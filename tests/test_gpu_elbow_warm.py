"""GPU: warm-started solves of the two-body (elbow) ContactNets loss (dpll_elbow_loss_warm_*): the optimum of every cone QP
is unique, so a start point changes the number of Newton directions and nothing else -- against cold solves of the same
kernel, the reference goldens and a cold training loop."""
import numpy as np
import pytest
import torch

from dair_pll_b200 import ops, synthetic
from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig
from tests.test_gpu_parity import _elbow_system, _mesh_system
from tests.test_gpu_parity_r2 import _elbow_random, _leaf_grads
from tests.util import load_golden, max_rel_to_scale, rel_err

pytestmark = pytest.mark.gpu

DEV = 'cuda:0'
DT = 0.0068


def _np(t):
    return t.detach().cpu().numpy()


def _warm_raw(x, xp, inertia, mu, half, kin, u_init, u_out, flags=0, dtype=torch.float64):
    """Direct call of dpll_elbow_loss_warm_* with both pointers as given (NULL included): loss, grad, force, iters."""
    B, dev = x.shape[0], x.device
    loss, grad, loss_sum = (torch.empty(n, dtype=dtype, device=dev) for n in (B, 28, 1))
    force = torch.empty((B, 24), dtype=dtype, device=dev)
    iters = torch.empty(B, dtype=torch.int32, device=dev)
    ops._call('dpll_elbow_loss_warm', dev, x, xp, None, inertia, mu, half, kin, None, DT, 1e-3, B, flags, loss, force, None,
              iters, grad, loss_sum, None, u_init, u_out, dtype=dtype, workspace=True)
    return loss, grad, force, iters


def _cases(assets_dir):
    """(name, kernel-level parameters, x, x_plus): 65,536 random pairs and the two reference goldens."""
    out = []
    s, _, x, xp, _ = _elbow_random(65536, assets_dir, 1)
    out.append(('random', [t.detach() for t in s._elbow_params(torch.float64, torch.device(DEV))], x, xp))
    for name in ('elbow_nominal', 'elbow_perturbed'):
        g = load_golden(name)
        s = _elbow_system(g, assets_dir)
        out.append((name, [t.detach() for t in s._elbow_params(torch.float64, torch.device(DEV))],
                    torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)))
    return out


def _moved(params):
    inertia, mu, half, kin = params
    return [inertia * 1.001, mu * 0.999, half * 1.0005, kin]


def _full(params, x, xp, **kw):
    """loss, grad, force, iters of elbow_loss_raw"""
    loss, grad, _, force, iters = ops.elbow_loss_raw(x, xp, *params, DT, 1e-3, want_force=True, want_iters=True, **kw)
    return loss, grad, force, iters


def _force_err(a, b):
    a, b = _np(a), _np(b)
    return (np.abs(a - b) / np.maximum(np.abs(b).max(axis=1, keepdims=True), 1e-6)).max()


def test_null_warm_pointers_launch_the_cold_kernel_bit_for_bit(assets_dir):
    for name, params, x, xp in _cases(assets_dir):
        cold = _full(params, x, xp)
        warm = _warm_raw(x, xp, *params, None, None)
        for a, b in zip(cold, warm):
            assert torch.equal(a, b), name


def test_warm_started_solves_give_the_cold_results(assets_dir):
    """Started from the cold optima (same parameters) or from the optima of parameters moved by 1e-3 (one Adam step of the
    reference's learning rate), the solves reach the cold losses, forces and gradients in fewer Newton directions.
    Free-flight samples record exactly zero."""
    for name, params, x, xp in _cases(assets_dir):
        B = x.shape[0]
        cold = _full(params, x, xp)
        u = torch.full((B, 7), float('nan'), dtype=torch.float64, device=DEV)
        rec = _full(params, x, xp, u_out=u)                    # the warm instance from the feasible-segment start
        for a, b in zip(cold, rec):
            assert torch.equal(a, b), name
        assert not torch.isnan(u).any() and bool((u[cold[3] == 0] == 0).all()), name
        same = _full(params, x, xp, u_init=u)
        assert rel_err(_np(same[0]), _np(cold[0]), 1e-9).max() < 1e-12, name
        assert max_rel_to_scale(_np(same[1]), _np(cold[1])) < 1e-12, name
        assert _force_err(same[2], cold[2]) < 1e-8, name
        assert int(same[3].max()) <= 1 and same[3].double().mean() < cold[3].double().mean(), name
        # moved parameters: the optima of the old ones as start points
        moved = _moved(params)
        ref = _full(moved, x, xp)
        warm = _full(moved, x, xp, u_init=u)
        assert rel_err(_np(warm[0]), _np(ref[0]), 1e-9).max() < 1e-10, name
        assert np.abs(_np(warm[0]) - _np(ref[0])).max() <= 1e-12 * np.abs(_np(ref[0])).max(), name
        assert max_rel_to_scale(_np(warm[1]), _np(ref[1])) < 1e-10, name
        assert _force_err(warm[2], ref[2]) < 1e-7, name
        assert warm[3].double().mean() < ref[3].double().mean(), name


def test_in_place_dynamic_schedule_and_fp32_storage(assets_dir):
    _, params, x, xp = _cases(assets_dir)[0]
    B = x.shape[0]
    u0 = torch.empty((B, 7), dtype=torch.float64, device=DEV)
    _full(params, x, xp, u_out=u0)
    moved = _moved(params)
    ref = _full(moved, x, xp)
    u_sep = torch.empty_like(u0)
    sep = _full(moved, x, xp, u_init=u0.clone(), u_out=u_sep)
    for flags in (0, ops.LOSS_DYNAMIC):
        buf = u0.clone()
        got = _full(moved, x, xp, u_init=buf, u_out=buf, flags=flags)          # in place
        assert rel_err(_np(got[0]), _np(ref[0]), 1e-9).max() < 1e-10, flags
        assert max_rel_to_scale(_np(got[1]), _np(ref[1])) < 1e-10, flags
        assert max_rel_to_scale(_np(buf), _np(u_sep)) < 1e-12, flags
        if flags == 0:            # static ranges: in place and out of place are the same launch
            for a, b in zip(got, sep):
                assert torch.equal(a, b)
    # fp32 storage (fp64 arithmetic): within 1e-4 of the fp64 results
    p32 = [t.float() for t in moved]
    u32 = u0.float()
    l32, g32, f32, _ = _warm_raw(x.float(), xp.float(), *p32, u32, u32, dtype=torch.float32)
    l64 = _np(ref[0])
    assert np.abs(_np(l32).astype(np.float64) - l64).max() < 1e-4 * max(np.abs(l64).max(), 1e-3)
    assert max_rel_to_scale(_np(g32).astype(np.float64), _np(ref[1])) < 1e-4
    assert max_rel_to_scale(_np(u32).astype(np.float64), _np(u_sep)) < 1e-4


def _module_grads(s):
    return [_np(p.grad).copy() for p in s.parameters() if p.grad is not None]


@pytest.mark.parametrize('golden', ['elbow_mesh_w64', 'elbow_mixed_w64'])
def test_learned_geometry_goldens_with_warm_starts(golden, assets_dir):
    """Learned and mixed geometry through the module: a second call warm-started from the first call's recorded optima
    matches the reference golden at 1e-9; free-flight rows record exactly zero."""
    g = load_golden(golden)
    if golden == 'elbow_mesh_w64':
        s = _mesh_system(g, assets_dir, 64)
    else:
        from dair_pll_b200.deep_support_function import HomogeneousICNN
        import os
        from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem
        s = MultibodyLearnableSystem({'elbow': os.path.join(assets_dir, 'elbow_mixed.urdf')}, float(g['dt']))
        geoms = s.multibody_terms.contact_terms.geometries
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
    s.record_qp_solution = True
    first = s.contactnets_loss(x, None, xp)
    first.mean().backward()
    g_cold = _module_grads(s)
    u = first.qp_solution
    assert isinstance(first, ops.BatchLoss) and u.shape == (x.shape[0], 7)
    for p in s.parameters():
        p.grad = None
    s.qp_warm_start = u
    loss = s.contactnets_loss(x, None, xp)
    assert s.qp_warm_start is None and loss.qp_solution.data_ptr() == u.data_ptr()      # in place
    loss.mean().backward()
    l = _np(loss)
    assert np.abs(l - g['loss']).max() < 1e-12 and rel_err(l, g['loss'], 1e-9).max() < 1e-9
    assert max_rel_to_scale(_np(s.multibody_terms.lagrangian_terms.inertial_parameters.grad), g['grad_theta']) < 1e-9
    assert max_rel_to_scale(_np(s.multibody_terms.contact_terms.friction_params.grad), g['grad_friction']) < 1e-9
    for a, b in zip(_module_grads(s), g_cold):
        assert max_rel_to_scale(a, b) < 1e-10
    with pytest.raises(ValueError):
        s.qp_warm_start = torch.zeros((x.shape[0], 6), dtype=torch.float64, device=DEV)
        s.contactnets_loss(x, None, xp)


def test_free_flight_rows_record_zero_through_the_module(assets_dir):
    s, _, x, xp, _ = _elbow_random(16384, assets_dir, 3)
    s.record_qp_solution = s.record_newton_iters = True
    loss = s.contactnets_loss(x, None, xp)
    u, it = loss.qp_solution, loss.newton_iters
    assert u.shape == (16384, 7) and 0 < int((it == 0).sum()) < 16384
    assert bool((u[it == 0] == 0).all()) and bool((u[it > 0].abs().sum(1) > 0).all())


def test_adam_epochs_with_data_set_warm_starts_match_cold_solves(assets_dir):
    """Three Adam epochs (lr 1e-3) through DeviceTrajectorySliceDataset, every batch warm-started from the optima the data
    set recorded for its slices in the previous epoch; at every batch a twin system loaded with the same parameters solves
    cold: losses and gradients agree to 1e-10."""
    s_data, _, x, _, _ = _elbow_random(64, assets_dir, 5)
    with torch.no_grad():
        traj, _ = s_data.simulate(x.unsqueeze(-2), torch.zeros(64, 1, device=DEV), 40)
    ds = DeviceTrajectorySliceDataset(TrajectorySliceConfig(), device=torch.device(DEV))
    for k in range(64):
        ds.add_slices_from_trajectory(synthetic.perturb_next_state(traj[k], seed=k, n_q=8))
    s, _, _, _, _ = _elbow_random(8, assets_dir, 6)
    twin, _, _, _, _ = _elbow_random(8, assets_dir, 6)
    s.record_qp_solution = s.record_newton_iters = True
    opt = torch.optim.Adam(s.parameters(), lr=1e-3)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(0)
    its = []
    for epoch in range(3):
        n_warm = 0
        for prev, fut, idx in ds.batches(640, generator=gen, return_indices=True):
            twin.load_state_dict(s.state_dict())
            warm = ds.warm_start(idx)
            n_warm += warm is not None
            s.qp_warm_start = warm
            opt.zero_grad()
            loss = s.contactnets_loss(prev[:, -1], None, fut[:, 0])
            loss.mean().backward()
            ds.update_solutions(idx, loss.qp_solution)
            ref = twin.contactnets_loss(prev[:, -1], None, fut[:, 0])
            ref.mean().backward()
            assert rel_err(_np(loss), _np(ref), 1e-9).max() < 1e-10, epoch
            for a, b in zip(_leaf_grads(s), _leaf_grads(twin)):
                assert max_rel_to_scale(a, b) < 1e-10, epoch
            for p in twin.parameters():
                p.grad = None
            its.append((epoch, loss.newton_iters.double().mean().item()))
            opt.step()
        # epoch 0: the first batch solves cold, later ones start from the zeros of slices not recorded yet
        assert n_warm == len(range(0, len(ds), 640)) - (epoch == 0)
    first = np.mean([m for e, m in its if e == 0])
    later = np.mean([m for e, m in its if e > 0])
    assert later < first
    assert ds.warm_start().shape == (len(ds), 7)
    with pytest.raises(ValueError):
        ds.update_solutions(None, torch.zeros((len(ds), 6), dtype=torch.float64, device=DEV))


def test_warm_elbow_step_replays_as_cuda_graph(assets_dir):
    from dair_pll_b200 import parallel
    s, _, x, xp, _ = _elbow_random(65536, assets_dir, 7)
    s.record_qp_solution = True
    u = s.contactnets_loss(x, None, xp).qp_solution.clone()
    params = list(s.parameters())

    def step():
        for p in params:
            p.grad = None
        s.qp_warm_start = u
        m = s.contactnets_loss(x, None, xp).mean()
        m.backward()
        return m.detach()
    eager = step().clone()
    g_eager = [p.grad.clone() for p in params]
    u_eager = u.clone()
    graphed = parallel.GraphedStep(step, torch.device(DEV))
    for _ in range(3):
        out = graphed()
    torch.cuda.synchronize()
    assert abs(out.item() - eager.item()) <= 1e-12 * abs(eager.item())
    for p, g in zip(params, g_eager):
        assert max_rel_to_scale(_np(p.grad), _np(g)) < 1e-10
    assert max_rel_to_scale(_np(u), _np(u_eager)) < 1e-12


def test_non_uniform_upstream_gradient_gives_the_cold_weighted_gradient(assets_dir):
    _, params, x, xp = _cases(assets_dir)[0]
    inertia, mu, half, kin = params
    B = x.shape[0]
    u = torch.empty((B, 7), dtype=torch.float64, device=DEV)
    _full(params, x, xp, u_out=u)
    moved = [t.clone().requires_grad_() for t in _moved(params)[:3]]
    w = torch.rand(B, dtype=torch.float64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(4))
    loss, _, _, _, usol = ops.ElbowContactNetsLoss.apply(x, xp, *moved, kin, DT, 1e-3, 0, False, u, True)
    assert usol.numel() == 0                                   # recorded into u in place
    (loss * w).sum().backward()
    got = torch.cat([t.grad.reshape(-1) for t in moved])
    ref = ops.elbow_loss_raw(x, xp, *(t.detach() for t in moved), kin, DT, 1e-3, weight=w)[1]
    assert max_rel_to_scale(_np(got), _np(ref)) < 1e-10
    # learned-geometry Function: same protocol, points' gradient scaled by the weights
    pts = torch.randn(B, 8, 3, dtype=torch.float64, device=DEV) * 0.02
    loss_p, usol_p = ops.ElbowContactNetsLossPts.apply(x, xp, moved[0].detach().requires_grad_(),
                                                       moved[1].detach().requires_grad_(), pts, kin, DT, 1e-3, None, True)
    assert usol_p.shape == (B, 7)
    ref_p = ops.elbow_loss_raw(x, xp, moved[0].detach(), moved[1].detach(), None, kin, DT, 1e-3, pts=pts)[0]
    assert rel_err(_np(loss_p), _np(ref_p), 1e-9).max() < 1e-12
