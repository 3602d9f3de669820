"""ContactNets parameter learning from simulated tosses -- the B200 counterpart of the reference's
``examples/contactnets_simple.py`` (BASELINE config 1), with the reference's settings (256 tosses of 80 / 120 steps
sampled uniformly around CUBE_X_0 / ELBOW_X_0, dt = 0.0068, Adam, lr 1e-3, batch 256; contactnets_simple.py:52-86),
for the cube and the two-body elbow, with box geometries or learned (mesh, ``DeepSupportConvex``) ones, with the
ContactNets loss or the prediction loss.

The reference generates its ground truth with Drake; here the ground-truth tosses come from the learnable system
itself at the URDF's parameters (the same Anitescu step, multibody_learnable_system.py:199-304), and the learned
system starts from perturbed inertia / friction / geometry.  Everything after data generation stays on the GPU:
trajectories -> ``DeviceTrajectorySliceDataset`` -> ``contactnets_loss(...).mean().backward()`` -> Adam.

    python examples/contactnets_simple.py --epochs 200 [--system elbow] [--geometry mesh] [--prediction --t-prediction 2]

With ``--geometry mesh`` the ground truth is still the box system; the learned system's geometry is a support-function
network initialised from the box's mesh (cube_mesh.urdf / elbow_mesh.urdf), as in the reference's *_mesh experiments.
"""
import argparse
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig  # noqa: E402
from dair_pll_b200.inertia import InertialParameterConverter as IPC  # noqa: E402
from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem  # noqa: E402

DT = 0.0068
N_POP = 256
CUBE_X_0 = torch.tensor([-0.525, 0.394, -0.296, -0.678, 0.186, 0.026, 0.222, 1.463, -4.854, 9.870, 0.014, 1.291, -0.212],
                        dtype=torch.float64)
CUBE_SAMPLER_RANGE = 0.1 * torch.ones(12, dtype=torch.float64)
ELBOW_X_0 = torch.tensor([1., 0., 0., 0., 0., 0., 0.21 + .015, math.pi, 0., 0., 0., 0., 0., -.075, 0.], dtype=torch.float64)
ELBOW_SAMPLER_RANGE = torch.tensor([2 * math.pi, 2 * math.pi, 2 * math.pi, .03, .03, .015, math.pi, 6., 6., 6., .5, .5,
                                    .075, 6.], dtype=torch.float64)
X_0S = {'cube': CUBE_X_0, 'elbow': ELBOW_X_0}
SAMPLER_RANGES = {'cube': CUBE_SAMPLER_RANGE, 'elbow': ELBOW_SAMPLER_RANGE}
TRAJECTORY_LENGTHS = {'cube': 80, 'elbow': 120}
URDFS = {'cube': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'cube.urdf'),
         'elbow': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow.urdf')}
MESH_URDFS = {'cube': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'cube_mesh.urdf'),
              'elbow': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow_mesh.urdf')}


def sample_initial_states(system, kind: str, n: int, seed: int, device) -> torch.Tensor:
    """``UniformSampler(space, x_0, ranges)`` of the reference (state_space.py:900-948): a uniform perturbation in
    the tangent space of x_0, applied with the space's exponential map."""
    gen = torch.Generator().manual_seed(seed)
    space = system.space
    dx = (2 * (torch.rand((n, 2 * space.n_v), generator=gen, dtype=torch.float64) - 0.5) * SAMPLER_RANGES[kind]).to(device)
    x0 = X_0S[kind].to(device).expand(n, -1)
    q = space.exponential(space.q(x0), dx[:, :space.n_v])
    return space.x(q, space.v(x0) + dx[:, space.n_v:])


def parameter_report(system) -> dict:
    mt = system.multibody_terms
    pi = IPC.theta_to_pi_cm(mt.lagrangian_terms.inertial_parameters.detach())
    half = [g.length_params.detach().abs().reshape(-1).tolist() for g in mt.contact_terms.geometries
            if hasattr(g, 'length_params')]
    return {'mass': pi[..., 0].reshape(-1).tolist(), 'friction': mt.contact_terms.friction_params.detach().abs().tolist(),
            'half_lengths': [v for h in half for v in h]}


def run(epochs: int = 100, n_pop: int = N_POP, batch_size: int = 256, lr: float = 1e-3, seed: int = 0,
        perturbation: float = 0.3, device: str = 'cuda:0', verbose: bool = True, contactnets: bool = True,
        t_prediction: int = 1, system: str = 'cube', geometry: str = 'box') -> dict:
    """``contactnets=False`` trains on the prediction loss instead (experiment.py:292-320: mean squared velocity
    error of the ``t_prediction``-step rollout from the last past state), differentiating through every step's
    QP (``simulate`` -> ``dpll_cube_rollout_grad_f64``)."""
    dev = torch.device(device)
    truth = MultibodyLearnableSystem({system: URDFS[system]}, DT).to(dev)
    x0 = sample_initial_states(truth, system, n_pop, seed, dev)
    with torch.no_grad():
        trajectories, _ = truth.simulate(x0.unsqueeze(-2), torch.zeros(n_pop, 1, device=dev), TRAJECTORY_LENGTHS[system])
    data = DeviceTrajectorySliceDataset(TrajectorySliceConfig(t_prediction=1 if contactnets else t_prediction), dev)
    for traj in trajectories:
        data.add_slices_from_trajectory(traj)

    # the learned system starts from multiplicatively perturbed parameters of the same URDF
    learned = MultibodyLearnableSystem({system: (MESH_URDFS if geometry == 'mesh' else URDFS)[system]}, DT)
    gen_p = torch.Generator().manual_seed(seed + 1)

    def jitter(n):
        return 1 + perturbation * (2 * torch.rand(n, generator=gen_p, dtype=torch.float64) - 1)
    state = learned.state_dict()
    pi = IPC.theta_to_pi_cm(state['multibody_terms.lagrangian_terms.inertial_parameters']).clone()
    n_b = pi.shape[0]
    pi[..., 0] *= jitter(n_b)                                  # masses
    pi[..., 4:7] *= jitter(3 * n_b).reshape(n_b, 3)            # principal moments
    state['multibody_terms.lagrangian_terms.inertial_parameters'] = IPC.pi_cm_to_theta(pi)
    key = 'multibody_terms.contact_terms.friction_params'
    state[key] = state[key] * jitter(state[key].numel())
    for key in [k for k in state if k.endswith('length_params')]:
        state[key] = state[key] * jitter(3).reshape(1, 3)
    learned.load_state_dict(state)
    learned = learned.to(dev)
    initial = parameter_report(learned)
    optimizer = torch.optim.Adam(learned.parameters(), lr=lr)
    gen = torch.Generator(device=dev).manual_seed(seed)
    history = []
    start = time.time()
    for epoch in range(epochs):
        total, count = 0.0, 0
        for x_past, x_future in data.batches(batch_size, generator=gen):
            optimizer.zero_grad(set_to_none=True)
            if contactnets:     # the experiment's loss callback (drake_experiment.py:202-224)
                loss = learned.contactnets_loss(x_past[:, -1, :], None, x_future[:, 0, :]).mean()
            else:               # experiment.prediction_loss (experiment.py:292-320)
                steps = x_future.shape[1]
                predicted, _ = learned.simulate(x_past[:, -1:, :], torch.zeros(x_past.shape[0], 1, device=dev), steps)
                space = learned.space
                loss = ((space.v(predicted[:, 1:, :]) - space.v(x_future)) ** 2).sum() / space.v(x_future).numel()
            loss.backward()
            optimizer.step()
            total += loss.detach() * x_past.shape[0]
            count += x_past.shape[0]
        history.append((total / count).item())
        if verbose and (epoch % max(1, epochs // 10) == 0 or epoch == epochs - 1):
            print(f'epoch {epoch:4d}  training loss {history[-1]:.6e}  {parameter_report(learned)}')
    return {'history': history, 'truth': parameter_report(truth), 'initial': initial, 'learned': parameter_report(learned),
            'pairs': len(data), 'seconds': time.time() - start}


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--epochs', type=int, default=100)
    ap.add_argument('--n-pop', type=int, default=N_POP)
    ap.add_argument('--batch-size', type=int, default=256)
    ap.add_argument('--lr', type=float, default=1e-3)
    ap.add_argument('--perturbation', type=float, default=0.3)
    ap.add_argument('--system', choices=['cube', 'elbow'], default='cube')
    ap.add_argument('--geometry', choices=['box', 'mesh'], default='box',
                    help='geometry of the learned system: boxes, or support-function networks initialised from them')
    ap.add_argument('--prediction', action='store_true', help='prediction loss instead of the ContactNets loss')
    ap.add_argument('--t-prediction', type=int, default=1)
    a = ap.parse_args()
    out = run(a.epochs, a.n_pop, a.batch_size, a.lr, perturbation=a.perturbation, contactnets=not a.prediction,
              t_prediction=a.t_prediction, system=a.system, geometry=a.geometry)
    print(f"{out['pairs']} pairs, {a.epochs} epochs in {out['seconds']:.1f} s")
    print('truth  ', out['truth'])
    print('learned', out['learned'])
