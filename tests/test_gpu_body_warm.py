"""GPU: warm-started QP solves and recorded optima of the single floating body with witness points
(dpll_body_loss_pts_warm_f64): cube-mesh (learned geometry, width 256), Sphere, Polygon and a box in a placed collision
frame; both schedules and both unroll instances, in place, CUDA-graph capture of the warm training step, the module's
warm-start API and the data set.  The optimum of every pair's cone QP is unique, so a start point changes the Newton
count, not the losses, gradients or optima (to the solver's tolerance)."""
import os

import numpy as np
import pytest
import torch

from dair_pll_b200 import ops
from dair_pll_b200.multibody_learnable_system import LOSS_EPS
from tests.test_cube_mesh_host import _shape_inputs
from tests.test_gpu_cube_mesh import DT, _batch, _system
from tests.util import max_rel_to_scale

DEV = 'cuda:0'
pytestmark = pytest.mark.gpu


def _check_same(cold, warm, what):
    """loss within 1e-12 of its largest value (as the elbow's GPU tests); gradient, grad_pts within 1e-10 of their largest entries"""
    assert (warm[0] - cold[0]).abs().max().item() <= 1e-12 * cold[0].abs().max().item(), what
    assert max_rel_to_scale(warm[1].cpu().numpy(), cold[1].cpu().numpy()) < 1e-10, what
    assert max_rel_to_scale(warm[3].cpu().numpy(), cold[3].cpu().numpy()) < 1e-10, what


def _scenario(args, flags):
    """cold (optima recorded), the optima of the parameters moved by 1e-3, warm from them (distinct output and in place)"""
    x, xp, inertia, mu, pts, n_c, dt = args
    B = x.shape[0]
    raw = lambda **kw: ops.body_loss_pts_raw(x, xp, kw.pop('inertia', inertia), kw.pop('mu', mu), pts, n_c, dt, LOSS_EPS,
                                             flags=flags, want_iters=True, **kw)
    u_c = torch.empty(B, 6, dtype=torch.float64, device=DEV)
    cold = raw(u_out=u_c)
    plain = raw()
    assert torch.equal(plain[0], cold[0]) and torch.equal(plain[4], cold[4])      # recording changes nothing
    u_moved = torch.empty_like(u_c)
    raw(inertia=inertia * 1.001, mu=mu * 0.999, u_out=u_moved)
    free = cold[4] == 0
    assert free.any() and (~free).any() and torch.all(u_c[free] == 0)
    u_w = torch.full_like(u_c, float('nan'))
    warm = raw(u_init=u_moved, u_out=u_w)
    _check_same(cold, warm, 'moved optimum')
    assert max_rel_to_scale(u_w.cpu().numpy(), u_c.cpu().numpy()) < 1e-9 and torch.all(u_w[free] == 0)
    assert torch.all(warm[4][free] == 0)
    assert warm[4].double().mean() < cold[4].double().mean(), (warm[4].double().mean(), cold[4].double().mean())
    buf = u_moved.clone()
    inplace = raw(u_init=buf, u_out=buf)
    _check_same(cold, inplace, 'in place')
    assert torch.equal(inplace[4], warm[4]) and max_rel_to_scale(buf.cpu().numpy(), u_c.cpu().numpy()) < 1e-9
    start_only = raw(u_init=u_moved)
    _check_same(cold, start_only, 'start, nothing recorded')
    return cold, warm


@pytest.mark.parametrize('name', ['shape_sphere', 'shape_polygon', 'shape_framed_box'])
def test_shapes_warm_equals_cold(name):
    g, x, xp, inertia, mu, pts, n_c = _shape_inputs(name)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    cold, _ = _scenario((t(x), t(xp), t(inertia), t(mu), t(pts), n_c, float(g['dt'])), 0)
    assert np.abs(cold[0].cpu().numpy() - g['loss']).max() < 1e-12


@pytest.mark.parametrize('n', [65536, 524288])
@pytest.mark.parametrize('flags', [0, ops.LOSS_DYNAMIC])
def test_cube_mesh_warm_equals_cold_both_instances_and_schedules(n, flags):
    """65,536 pairs run the unrolled instance, 524,288 the rolled one (the switch is near 380,000 pairs); the static and
    the dynamic schedule"""
    s = _system()
    x, xp = _batch(s, n, 31)
    inertia, mu, _ = s._cube_params(torch.float64)
    with torch.no_grad():
        pts, n_c = s._body_witness_points(xp[:, :4])
    _scenario((x, xp, inertia.detach(), mu.detach(), pts, n_c, DT), flags)


def _grads(s):
    return torch.cat([p.grad.reshape(-1) for p in s.parameters() if p.grad is not None]).cpu().numpy()


def test_cube_mesh_module_warm_start_api():
    s = _system()
    x, xp = _batch(s, 4096, 41)
    B = x.shape[0]

    def run(warm=None, record=False):
        for p in s.parameters():
            p.grad = None
        s.qp_warm_start, s.record_qp_solution = warm, record
        loss = s.contactnets_loss(x, None, xp)
        assert s.qp_warm_start is None                      # consumed by the call
        loss.mean().backward()
        return loss.detach(), _grads(s), loss.qp_solution

    l_c, g_c, none = run()
    assert none is None
    l_r, _, u_c = run(record=True)
    assert tuple(u_c.shape) == (B, 6) and torch.equal(l_r, l_c)
    for what, start in (('zero', torch.zeros_like(u_c)), ('cold optimum', u_c.clone())):
        buf = start.clone()
        l_w, g_w, u_w = run(buf, True)
        assert u_w.data_ptr() == buf.data_ptr()              # written into the warm-start tensor itself
        assert (l_w - l_c).abs().max().item() <= 1e-12 * l_c.abs().max().item(), what
        assert max_rel_to_scale(g_w, g_c) < 1e-10, what
        assert max_rel_to_scale(buf.cpu().numpy(), u_c.cpu().numpy()) < 1e-9, what
        l_n, g_n, u_n = run(start.clone())
        assert u_n is None and (l_n - l_c).abs().max().item() <= 1e-12 * l_c.abs().max().item()
        assert max_rel_to_scale(g_n, g_c) < 1e-10, what
    for bad in (torch.zeros(B, 7, dtype=torch.float64, device=DEV), torch.zeros(B, 6, device=DEV),
                torch.zeros(6, B, dtype=torch.float64, device=DEV).t()):
        s.qp_warm_start, s.record_qp_solution = bad, True
        with pytest.raises(ValueError):
            s.contactnets_loss(x, None, xp)
        assert s.qp_warm_start is None


def test_cube_mesh_warm_training_step_replays_as_cuda_graph():
    """The training step with a warm start recorded in place (one buffer per batch) captured with parallel.GraphedStep and
    replayed equals the eager step."""
    from dair_pll_b200 import parallel
    s = _system()
    x, xp = _batch(s, 65536, 51)
    s.record_qp_solution = True
    u = s.contactnets_loss(x, None, xp).qp_solution.clone()
    params = list(s.parameters())

    def step():
        for p in params:
            p.grad = None
        s.qp_warm_start, s.record_qp_solution = u, True
        m = s.contactnets_loss(x, None, xp).mean()
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


def test_cube_mesh_data_set_loop_with_warm_starts_reproduces_cold():
    """A few Adam epochs through DeviceTrajectorySliceDataset (one two-state trajectory per pair): warm-started from the
    optima the data set recorded, the losses are the cold loop's."""
    from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig
    x, xp = _batch(_system(), 1024, 61)
    data = DeviceTrajectorySliceDataset(TrajectorySliceConfig(), device=DEV)
    for a, b in zip(x, xp):
        data.add_slices_from_trajectory(torch.stack((a, b)))

    def loop(warm):
        s = _system()
        opt = torch.optim.Adam(s.parameters(), lr=1e-3)
        s.record_qp_solution = warm
        out = []
        for _ in range(3):
            for prev, fut, idx in data.batches(256, shuffle=False, return_indices=True):
                if warm:
                    s.qp_warm_start = data.warm_start(idx)
                opt.zero_grad(set_to_none=True)
                loss = s.contactnets_loss(prev[:, -1], None, fut[:, 0])
                if warm:
                    assert loss.qp_solution.shape == (idx.shape[0], 6)
                    data.update_solutions(idx, loss.qp_solution)
                loss.mean().backward()
                opt.step()
                out.append(loss.detach().cpu().numpy())
        return np.concatenate(out)

    cold, warm = loop(False), loop(True)
    assert np.abs(warm - cold).max() <= 1e-10 * np.abs(cold).max()
