"""GPU: the single floating body with learned (DeepSupportConvex, width 256) geometry -- cube_mesh.urdf through the module
API against the CPU oracle (loss, parameter and network gradients, one step, a differentiable rollout), the support-
direction kernel, and the witness-point instance of the wavefront loss kernel at scale (static vs dynamic schedule, both
unroll instances, CUDA-graph capture of the whole training step)."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
from dair_pll_b200 import ops, synthetic  # noqa: E402
from dair_pll_b200.multibody_learnable_system import LOSS_EPS, MultibodyLearnableSystem  # noqa: E402
from tests.util import max_rel_to_scale, rel_err  # noqa: E402

DEV = 'cuda:0'
DT = 0.0068
CUBE_MESH = os.path.join(ROOT, 'dair_pll_b200', 'assets', 'cube_mesh.urdf')


def _system(seed=0):
    torch.manual_seed(seed)
    return MultibodyLearnableSystem({'cube': CUBE_MESH}, DT).to(DEV)


def _batch(s, n, seed):
    x = synthetic.cube_states(n, seed=seed, device=DEV)
    with torch.no_grad():
        traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(n, 1, device=DEV), 1)
    return x, synthetic.perturb_next_state(traj[:, 1], seed=seed + 1)


def _oracle_params(s):
    from oracle import contactnets_oracle as co
    mt = s.multibody_terms
    geom = mt.contact_terms.geometries[0]
    net = geom.network
    nets = [dict(Wd0=net.input_weights[0].detach().cpu().clone().requires_grad_(),
                 Wd1=net.input_weights[1].detach().cpu().clone().requires_grad_(),
                 Wh=net.hidden_weights[0].detach().cpu().clone().requires_grad_(),
                 wout=net.output_weight.detach().cpu().clone().requires_grad_(),
                 perturbations=geom.perturbations.detach().cpu().clone())]
    return co.OracleParams(mt.lagrangian_terms.inertial_parameters.detach().cpu().clone(),
                           mt.contact_terms.friction_params.detach().cpu().clone(), [], icnn=nets).requires_grad_(), nets


def _net_params(s):
    net = s.multibody_terms.contact_terms.geometries[0].network
    return (('Wd0', net.input_weights[0]), ('Wd1', net.input_weights[1]), ('Wh', net.hidden_weights[0]),
            ('wout', net.output_weight))


def test_cube_mesh_width_256_matches_oracle():
    """The ContactNets loss of cube_mesh.urdf through the module API: per-sample losses and the gradients of theta,
    friction and every network weight against autograd through the CPU oracle (CUBE_TREE with the network's support
    points), 1e-9."""
    from oracle import contactnets_oracle as co
    from oracle.callables import CUBE_TREE, TreeCallables
    s = _system()
    x, xp = _batch(s, 2048, 31)
    loss = s.contactnets_loss(x, None, xp)
    loss.sum().backward()
    P, nets = _oracle_params(s)
    lo = co.contactnets_loss(TreeCallables(CUBE_TREE), P, x.cpu(), xp.cpu(), DT)
    lo.sum().backward()
    mt = s.multibody_terms
    assert rel_err(loss.detach().cpu().numpy(), lo.detach().numpy(), 1e-9).max() < 1e-9
    assert max_rel_to_scale(mt.lagrangian_terms.inertial_parameters.grad.cpu().numpy(), P.inertial_parameters.grad.numpy()) < 1e-9
    assert max_rel_to_scale(mt.contact_terms.friction_params.grad.cpu().numpy(), P.friction_params.grad.numpy()) < 1e-9
    seen = 0
    for k, p in _net_params(s):
        ref = nets[0][k].grad.numpy()
        assert max_rel_to_scale(p.grad.cpu().numpy(), ref) < 1e-9, k
        seen += int(np.abs(ref).max() > 0)
    assert seen == 4


def test_cube_mesh_simulate_and_differentiable_rollout_match_oracle():
    """One simulate() step within 1e-9 of the oracle; a 3-step differentiable rollout and the gradients of theta, friction,
    every network weight and the initial state against oracle autograd within 1e-7 (DESIGN.md section 2)."""
    from oracle import contactnets_oracle as co
    from oracle.callables import CUBE_TREE, TreeCallables
    s = _system()
    calls = TreeCallables(CUBE_TREE)
    x = synthetic.cube_states(512, seed=7, device=DEV)
    with torch.no_grad():
        traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(512, 1, device=DEV), 1)
    P, nets = _oracle_params(s)
    with torch.no_grad():
        step_o = co.sim_step(calls, P, x.cpu(), DT)
    assert np.abs(traj[:, 1].cpu().numpy() - step_o.numpy()).max() < 1e-9

    n, steps = 24, 3
    x0 = synthetic.cube_states(n, seed=41, device=DEV).requires_grad_()
    target = torch.randn(n, steps, 13, generator=torch.Generator().manual_seed(5), dtype=torch.float64).to(DEV)
    traj, _ = s.simulate(x0.unsqueeze(-2), torch.zeros(n, 1, device=DEV), steps)
    ((traj[:, 1:] - target) ** 2).sum().backward()
    P, nets = _oracle_params(s)
    x0o = x0.detach().cpu().clone().requires_grad_()
    tro = co.simulate(calls, P, x0o, DT, steps)
    ((tro[:, 1:] - target.cpu()) ** 2).sum().backward()
    assert np.abs(traj.detach().cpu().numpy() - tro.detach().numpy()).max() < 1e-8
    mt = s.multibody_terms
    tol = 1e-7
    assert max_rel_to_scale(mt.lagrangian_terms.inertial_parameters.grad.cpu().numpy(), P.inertial_parameters.grad.numpy()) < tol
    assert max_rel_to_scale(mt.contact_terms.friction_params.grad.cpu().numpy(), P.friction_params.grad.numpy()) < tol
    assert max_rel_to_scale(x0.grad.cpu().numpy(), x0o.grad.numpy()) < tol
    seen = 0
    for k, p in _net_params(s):
        ref = nets[0][k].grad.numpy()
        assert max_rel_to_scale(p.grad.cpu().numpy(), ref) < tol, k
        seen += int(np.abs(ref).max() > 0)
    assert seen >= 1          # the rollout does train the geometry


def test_body_support_directions_kernel_matches_torch_formula():
    s = _system()
    geom = s.multibody_terms.contact_terms.geometries[0]
    q = synthetic.cube_states(4096, seed=3, device=DEV)
    q[:, :4] *= 1.0 + 0.1 * torch.rand(4096, 1, device=DEV, dtype=torch.float64)      # unnormalised quaternions
    d = ops.body_support_directions(q, geom.perturbations)                              # row stride 13
    w, a, b, c = q[:, :4].unbind(-1)
    sc = 2.0 / (w * w + a * a + b * b + c * c)
    base = -torch.stack((sc * (a * c - w * b), sc * (b * c + w * a), 1 - sc * (a * a + b * b)), -1)
    ref = base.unsqueeze(-2) + geom.perturbations
    ref = ref / ref.norm(dim=-1, keepdim=True)
    assert (d - ref).abs().max().item() < 1e-15


def _raw(s, x, xp, flags=0, want_iters=False):
    inertia, mu, _ = s._cube_params(torch.float64)
    with torch.no_grad():
        pts, n_c = s._body_witness_points(xp[:, :4])
    return ops.body_loss_pts_raw(x, xp, inertia.detach(), mu.detach(), pts, n_c, DT, LOSS_EPS, flags=flags,
                                 want_iters=want_iters)


def _oracle_rows(s, x, xp, rows):
    from oracle import contactnets_oracle as co
    from oracle.callables import CUBE_TREE, TreeCallables
    P, _ = _oracle_params(s)
    with torch.no_grad():
        return co.contactnets_loss(TreeCallables(CUBE_TREE), P, x[rows].cpu(), xp[rows].cpu(), DT).numpy()


def test_static_and_dynamic_schedule_at_262144_pairs():
    """DPLL_LOSS_DYNAMIC moves samples between warps, not the per-sample arithmetic: losses, iteration counts and grad_pts are
    bit-identical to the static schedule's, the summed gradients agree to rounding, and 4,096 rows match the oracle."""
    s = _system()
    x, xp = _batch(s, 262144, 11)
    ref = _raw(s, x, xp, want_iters=True)
    dyn = _raw(s, x, xp, flags=ops.LOSS_DYNAMIC, want_iters=True)
    torch.cuda.synchronize()
    assert torch.equal(ref[0], dyn[0]) and torch.equal(ref[3], dyn[3]) and torch.equal(ref[4], dyn[4])
    assert max_rel_to_scale(dyn[1].cpu().numpy(), ref[1].cpu().numpy()) < 1e-12
    assert abs(dyn[2].item() - ref[2].item()) < 1e-12 * abs(ref[2].item())
    assert (ref[4] == 0).any() and (ref[4] > 0).any()            # free-flight triage and solver both taken
    rows = torch.randperm(262144, generator=torch.Generator().manual_seed(0))[:4096].to(DEV)
    lo = _oracle_rows(s, x, xp, rows)
    assert rel_err(ref[0][rows].cpu().numpy(), lo, 1e-9).max() < 1e-9


@pytest.mark.parametrize('n', [65536, 1048576])
def test_both_unroll_instances_match_oracle(n):
    """Launches of up to ~320 samples per warp run the instance with the per-contact loops unrolled, larger ones the rolled
    instance: 65,536 and 1,048,576 pairs take one each.  A 2,048-row subset of each against the oracle; the sums of the
    launch equal the sums of its own per-sample outputs."""
    s = _system()
    x, xp = _batch(s, n, 21)
    loss, grad, loss_sum, gpts, _, _ = _raw(s, x, xp)
    torch.cuda.synchronize()
    assert torch.isfinite(loss).all() and torch.isfinite(grad).all() and torch.isfinite(gpts).all()
    assert abs(loss_sum.item() - loss.sum().item()) < 1e-11 * abs(loss_sum.item())
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(1))[:2048].to(DEV)
    lo = _oracle_rows(s, x, xp, rows)
    assert rel_err(loss[rows].cpu().numpy(), lo, 1e-9).max() < 1e-9


def test_cube_mesh_training_step_replays_as_cuda_graph():
    """The whole step -- directions kernel, support network, loss kernel, backward through the kernel and the network --
    captured with parallel.GraphedStep and replayed equals the eager step (cost-ordered batch, dynamic schedule)."""
    from dair_pll_b200 import parallel
    s = _system()
    x, xp = _batch(s, 65536, 51)
    s.record_newton_iters = True
    it = s.contactnets_loss(x, None, xp).newton_iters
    assert it is not None and it.shape == (65536,)
    s.record_newton_iters = False
    order = torch.argsort(it, descending=True, stable=True)
    xo, xpo = x.index_select(0, order).contiguous(), xp.index_select(0, order).contiguous()
    s.dynamic_schedule = True
    params = list(s.parameters())

    def step():
        for p in params:
            p.grad = None
        m = s.contactnets_loss(xo, None, xpo).mean()
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


def test_example_trains_learned_cube_geometry():
    sys.path.insert(0, os.path.join(ROOT, 'examples'))
    import contactnets_simple
    out = contactnets_simple.run(epochs=2, n_pop=16, verbose=False, system='cube', geometry='mesh')
    assert len(out['history']) == 2 and all(np.isfinite(out['history']))
