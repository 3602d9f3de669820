"""GPU: warm-started QP solves and recorded optima of the tree losses (boxes: dpll_chain_loss_warm_f64; witness points:
dpll_chain_loss_pts_warm_f64), through the module's warm-start API and the data set.  The optimum of every pair's cone QP is
unique, so a start point changes the Newton count, not the losses, gradients or optima (to the solver's tolerance)."""
import os

import numpy as np
import pytest
import torch

from dair_pll_b200 import ops
from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem
from tests.test_gpu_parity_r2 import _chain_system
from tests.util import load_golden, max_rel_to_scale

DEV = 'cuda:0'
pytestmark = pytest.mark.gpu


def _system(name, assets_dir):
    g = load_golden(name)
    if name != 'chain3s':
        n = {'chain3': 3, 'tree4': 4}[name]
        return g, _chain_system(g, os.path.join(assets_dir, f'{name}.urdf'), n), n
    from dair_pll_b200.geometry import Polygon, Sphere
    s = MultibodyLearnableSystem({'chain3': os.path.join(assets_dir, 'chain3.urdf')}, float(g['dt']))
    ct = s.multibody_terms.contact_terms
    ct.geometries[1] = Sphere(torch.from_numpy(g['sphere_radius']))
    ct.geometries[2] = Polygon(torch.from_numpy(g['polygon_vertices']), 4)
    with torch.no_grad():
        s.multibody_terms.lagrangian_terms.inertial_parameters.copy_(torch.from_numpy(g['theta']))
        ct.friction_params.copy_(torch.from_numpy(g['friction_params']))
        ct.geometries[0].length_params.copy_(torch.from_numpy(g['box_length_params']))
    return g, s.to(DEV), 3


def _grads(s):
    return torch.cat([p.grad.reshape(-1) for p in s.parameters() if p.grad is not None]).cpu().numpy()


def _run(s, x, xp, warm=None, record=False):
    for p in s.parameters():
        p.grad = None
    s.qp_warm_start, s.record_qp_solution = warm, record
    loss = s.contactnets_loss(x, None, xp)
    assert s.qp_warm_start is None                       # consumed by the call
    loss.mean().backward()
    return loss.detach().cpu().numpy(), _grads(s), getattr(loss, 'qp_solution', None)


def _moved_optima(s, x, xp):
    """the optima of the parameters moved by 1e-3: last epoch's, in a training loop"""
    with torch.no_grad():
        saved = [p.detach().clone() for p in s.parameters()]
        for p in s.parameters():
            p.mul_(1.001)
        s.record_qp_solution = True
        u = s.contactnets_loss(x, None, xp).qp_solution.clone()
        for p, v in zip(s.parameters(), saved):
            p.copy_(v)
    return u


@pytest.mark.parametrize('name', ['chain3', 'tree4', 'chain3s'])
def test_warm_started_tree_loss_matches_cold(name, assets_dir):
    g, s, n = _system(name, assets_dir)
    x, xp = torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)
    B = x.shape[0]
    l_c, g_c, none = _run(s, x, xp)
    assert none is None and np.abs(l_c - g['loss']).max() < 1e-12
    l_r, g_r, u_c = _run(s, x, xp, record=True)                     # cold solve, optima recorded
    assert tuple(u_c.shape) == (B, 5 + n) and np.array_equal(l_r, l_c)
    u_c = u_c.cpu().numpy()
    u_moved = _moved_optima(s, x, xp)
    for what, start in (('zero', torch.zeros_like(u_moved)), ('cold optimum', torch.from_numpy(u_c).to(DEV)),
                        ('moved optimum', u_moved.clone())):
        buf = start.clone()
        l_w, g_w, u_w = _run(s, x, xp, warm=buf, record=True)
        assert u_w.data_ptr() == buf.data_ptr()                       # written into the warm-start tensor itself
        assert np.abs(l_w - l_c).max() <= 1e-13 * np.abs(l_c).max(), what
        assert max_rel_to_scale(g_w, g_c) < 1e-10, what
        assert max_rel_to_scale(buf.cpu().numpy(), u_c) < 1e-9, what
        l_n, g_n, u_n = _run(s, x, xp, warm=start.clone())            # a start, nothing recorded
        assert u_n is None and np.abs(l_n - l_c).max() <= 1e-13 * np.abs(l_c).max()
        assert max_rel_to_scale(g_n, g_c) < 1e-10, what
    for bad in (torch.zeros(B, 4 + n, dtype=torch.float64, device=DEV), torch.zeros(B, 5 + n, device=DEV),
                torch.zeros(5 + n, B, dtype=torch.float64, device=DEV).t()):
        s.qp_warm_start, s.record_qp_solution = bad, True
        with pytest.raises(ValueError):
            s.contactnets_loss(x, None, xp)
        assert s.qp_warm_start is None


@pytest.mark.parametrize('name', ['chain3', 'tree4', 'chain3s'])
def test_warm_start_cuts_the_newton_count(name, assets_dir):
    """Newton directions per sample (the iters output of the warm entry points): started from the optima of parameters
    moved by 1e-3 the mean is below the cold solve's; free flight takes none from any start."""
    g, s, n = _system(name, assets_dir)
    x, xp = torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)
    B = x.shape[0]
    u_moved = _moved_optima(s, x, xp)
    mt = s.multibody_terms

    def iters(start):
        it = torch.zeros(B, dtype=torch.int32, device=DEV)
        loss = torch.empty(B, dtype=torch.float64, device=DEV)
        with torch.no_grad():
            if name == 'chain3s':
                inertia, mu, _ = mt.kernel_parameters(torch.float64)
                pts, packed = mt.chain_witness_points(xp[:, :9])
                ops._call('dpll_chain_loss_pts_warm_f64', x.device, n, x, xp, None, inertia.reshape(-1).contiguous(),
                          mu.reshape(-1).contiguous(), mt.chain_kinematic_table(x.device, True), pts.contiguous(), packed,
                          float(s.dt), 1e-3, B, loss, None, None, None, start, None, it, workspace=True)
            else:
                inertia, mu, half, kin, _ = s._chain_params(x.device)
                ops._call('dpll_chain_loss_warm_f64', x.device, n, x, xp, None, inertia.contiguous(), mu.contiguous(),
                          half.contiguous(), kin, float(s.dt), 1e-3, B, loss, None, it, None, None, start, None,
                          workspace=True)
        return it.cpu().numpy(), loss.cpu().numpy()

    it_c, l_c = iters(None)
    it_w, l_w = iters(u_moved)
    free = it_c == 0
    assert 0 < free.sum() < B and np.all(it_w[free] == 0)
    assert it_w.mean() < it_c.mean(), (it_w.mean(), it_c.mean())
    assert np.abs(l_w - l_c).max() <= 1e-13 * np.abs(l_c).max()


def test_data_set_training_loop_with_warm_starts_reproduces_cold(assets_dir):
    """A few Adam epochs through DeviceTrajectorySliceDataset on the four-link tree: warm-started from the optima the data
    set records, the losses are the cold loop's."""
    from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig
    g = load_golden('tree4')
    x, xp = torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)
    B = x.shape[0]
    data = DeviceTrajectorySliceDataset(TrajectorySliceConfig(), device=DEV)
    for a, b in zip(x, xp):                              # one two-state trajectory per pair
        data.add_slices_from_trajectory(torch.stack((a, b)))

    def loop(warm):
        s = _chain_system(g, os.path.join(assets_dir, 'tree4.urdf'), 4)
        opt = torch.optim.Adam(s.parameters(), lr=1e-3)
        out = []
        for _ in range(4):
            prev, fut, idx = next(data.batches(B, shuffle=False, return_indices=True))
            opt.zero_grad(set_to_none=True)
            if warm:
                s.record_qp_solution = True
                s.qp_warm_start = data.warm_start(idx)
            loss = s.contactnets_loss(prev[:, -1], None, fut[:, 0])
            if warm:
                assert loss.qp_solution.shape == (B, 9)
                data.update_solutions(idx, loss.qp_solution)
            loss.mean().backward()
            opt.step()
            out.append(loss.detach().cpu().numpy())
        return np.stack(out)

    cold, warm = loop(False), loop(True)
    assert np.abs(warm - cold).max() <= 1e-10 * np.abs(cold).max()


@pytest.mark.parametrize('name', ['tree4', 'chain3s'])
def test_tree_batch_loss_records_newton_counts(name, assets_dir):
    """record_newton_iters gives the tree losses their (B,) Newton counts (the data set's cost hint), with and without a
    warm start; the loss does not change."""
    g, s, n = _system(name, assets_dir)
    x, xp = torch.from_numpy(g['x']).to(DEV), torch.from_numpy(g['x_plus']).to(DEV)
    ref = s.contactnets_loss(x, None, xp).detach()
    s.record_newton_iters = True
    loss = s.contactnets_loss(x, None, xp)
    it = loss.newton_iters
    assert it.shape == (x.shape[0],) and it.dtype == torch.int32 and (it == 0).any() and (it > 0).any()
    assert torch.equal(loss.detach(), ref)
    s.record_qp_solution = True
    u = loss.qp_solution if loss.qp_solution is not None else s.contactnets_loss(x, None, xp).qp_solution.clone()
    s.qp_warm_start = u
    warm = s.contactnets_loss(x, None, xp)
    assert warm.newton_iters.max() <= 1
