"""Cold versus warm-started solves of the four-link tree's ContactNets loss (tree4.urdf, the golden's parameters and
states tiled to 65,536 pairs, as bench.py's tree4 measurement) and of the single body with learned geometry (cube_mesh.urdf,
--body-batch synthetic pairs, dpll_body_loss_pts_{,warm_}f64).

1. Kernel time (CUDA events over --reps launches of dpll_chain_loss_{,warm_}f64, after warm-up) and mean / max Newton
   counts, in natural and in cost order (the cold Newton counts, descending), for a cold solve and for a solve started
   from the optima of the parameters before one Adam step (lr 1e-3) of the loss.
2. A short Adam loop through DeviceTrajectorySliceDataset, with and without warm starts from the optima the data set
   recorded in the previous epoch: step time (CUDA events) and the largest loss difference to the cold loop.

Prints one line per measurement and a JSON summary, with the device's name, power limit and maximum SM clock.  Writes
nothing into the repository (--out: optional JSON file)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from dair_pll_b200 import ops  # noqa: E402
from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig  # noqa: E402
from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem  # noqa: E402
from tools.time_elbow_warm import gpu_info, time_ms  # noqa: E402


def tree_system(g, dev):
    s = MultibodyLearnableSystem({'chain': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'tree4.urdf')}, float(g['dt']))
    sd = {'multibody_terms.lagrangian_terms.inertial_parameters': torch.from_numpy(g['theta']),
          'multibody_terms.contact_terms.friction_params': torch.from_numpy(g['friction_params'])}
    for i in range(g['half_lengths'].shape[0]):
        sd[f'multibody_terms.contact_terms.geometries.{i}.length_params'] = torch.from_numpy(g['half_lengths'][i]).reshape(1, 3)
    s.load_state_dict(sd)
    return s.to(dev)


def body_kernels(dev, batch, reps, res):
    """cube-mesh: kernel time and Newton counts, cold and from the optima before one Adam step, natural and cost order"""
    from dair_pll_b200 import synthetic
    from dair_pll_b200.multibody_learnable_system import LOSS_EPS
    torch.manual_seed(0)
    s = MultibodyLearnableSystem({'cube': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'cube_mesh.urdf')}, 0.0068).to(dev)
    x = synthetic.cube_states(batch, seed=3, device=dev)
    with torch.no_grad():
        traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(batch, 1, device=dev), 1)
    xp = synthetic.perturb_next_state(traj[:, 1], seed=4)
    s.record_qp_solution = True
    opt = torch.optim.Adam(s.parameters(), lr=1e-3)
    loss = s.contactnets_loss(x, None, xp)
    u_before = loss.qp_solution.clone()
    loss.mean().backward()
    opt.step()
    inertia, mu, _ = [t.detach() if torch.is_tensor(t) else t for t in s._cube_params(torch.float64)]
    with torch.no_grad():
        pts, n_c = s._body_witness_points(xp[:, :4])
    raw = lambda xx, xxp, pp, **kw: ops.body_loss_pts_raw(xx, xxp, inertia, mu, pp, n_c, 0.0068, LOSS_EPS, **kw)
    it_cold = raw(x, xp, pts, want_iters=True)[4]
    order = torch.argsort(it_cold, descending=True, stable=True)
    for label, perm, flags in (('natural', None, 0), ('cost', order, ops.LOSS_DYNAMIC)):
        sel = (lambda t: t) if perm is None else (lambda t: t.index_select(0, perm).contiguous())
        xx, xxp, pp, u0 = sel(x), sel(xp), sel(pts), sel(u_before)
        ref = raw(xx, xxp, pp, want_iters=True, flags=flags)
        warm = raw(xx, xxp, pp, want_iters=True, flags=flags, u_init=u0)
        dl = ((warm[0] - ref[0]).abs().max() / ref[0].abs().max()).item()
        dg = ((warm[1] - ref[1]).abs().max() / ref[1].abs().max()).item()
        u_out = torch.empty_like(u0)
        ms_c = time_ms(lambda: raw(xx, xxp, pp, flags=flags), reps)
        ms_w = time_ms(lambda: raw(xx, xxp, pp, flags=flags, u_init=u0, u_out=u_out), reps)
        ms_c2 = time_ms(lambda: raw(xx, xxp, pp, flags=flags), reps)
        r = {'cold_ms': min(ms_c, ms_c2), 'cold_ms_runs': [ms_c, ms_c2], 'warm_ms': ms_w,
             'cold_newton_mean': ref[4].double().mean().item(), 'cold_newton_max': int(ref[4].max()),
             'warm_newton_mean': warm[4].double().mean().item(), 'warm_newton_max': int(warm[4].max()),
             'warm_vs_cold_loss_rel': dl, 'warm_vs_cold_grad_rel': dg}
        res[f'cube_mesh_{label}_order'] = r
        print(f'cube-mesh {label:7s} order: cold {ms_c:.3f} / {ms_c2:.3f} ms (Newton mean {r["cold_newton_mean"]:.2f} max '
              f'{r["cold_newton_max"]}), warm {ms_w:.3f} ms (Newton mean {r["warm_newton_mean"]:.2f} max '
              f'{r["warm_newton_max"]}); warm vs cold: loss {dl:.1e}, gradient {dg:.1e}')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=65536)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--epochs', type=int, default=5)
    ap.add_argument('--loop-batch', type=int, default=16384)
    ap.add_argument('--body-batch', type=int, default=262144)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    dev = torch.device('cuda', 0)
    res = {'device': gpu_info(), 'batch': a.batch, 'body_batch': a.body_batch}
    print('device:', res['device'])
    body_kernels(dev, a.body_batch, a.reps, res)
    g = dict(np.load(os.path.join(ROOT, 'tests', 'golden', 'tree4.npz')))
    reps = (a.batch + g['x'].shape[0] - 1) // g['x'].shape[0]
    x = torch.from_numpy(g['x']).to(dev).repeat(reps, 1)[:a.batch].contiguous()
    xp = torch.from_numpy(g['x_plus']).to(dev).repeat(reps, 1)[:a.batch].contiguous()
    B, n, dt = a.batch, 4, float(g['dt'])

    s = tree_system(g, dev)
    s.record_qp_solution = True
    opt = torch.optim.Adam(s.parameters(), lr=1e-3)
    loss = s.contactnets_loss(x, None, xp)
    u_before = loss.qp_solution.clone()
    loss.mean().backward()
    opt.step()
    s.record_qp_solution = False
    inertia, mu, half, kin, _ = [t.detach() if torch.is_tensor(t) else t for t in s._chain_params(dev)]

    def launch(xx, xxp, u0=None, u_out=None, iters=None, grad=None):
        out = torch.empty(B, dtype=torch.float64, device=dev)
        if u0 is None and u_out is None:
            ops._call('dpll_chain_loss_f64', dev, n, xx, xxp, None, inertia, mu, half, kin, dt, 1e-3, B, out, None, iters,
                      grad, None, workspace=True)
        else:
            ops._call('dpll_chain_loss_warm_f64', dev, n, xx, xxp, None, inertia, mu, half, kin, dt, 1e-3, B, out, None,
                      iters, grad, None, u0, u_out, workspace=True)
        return out

    def solve(xx, xxp, u0=None):
        it = torch.empty(B, dtype=torch.int32, device=dev)
        grad = torch.empty(14 * n, dtype=torch.float64, device=dev)
        l = launch(xx, xxp, u0, None, it, grad)
        return l, grad, it

    it_cold = solve(x, xp)[2]
    order = torch.argsort(it_cold, descending=True, stable=True)
    for label, perm in (('natural', None), ('cost', order)):
        xx, xxp = (x, xp) if perm is None else (x.index_select(0, perm).contiguous(), xp.index_select(0, perm).contiguous())
        u0 = u_before if perm is None else u_before.index_select(0, perm).contiguous()
        ref, warm = solve(xx, xxp), solve(xx, xxp, u0)
        dl = ((warm[0] - ref[0]).abs().max() / ref[0].abs().max()).item()
        dg = ((warm[1] - ref[1]).abs().max() / ref[1].abs().max()).item()
        u_out = torch.empty_like(u0)      # every timed warm launch starts from the same point
        grad = torch.empty(14 * n, dtype=torch.float64, device=dev)
        ms_c = time_ms(lambda: launch(xx, xxp, grad=grad), a.reps)
        ms_w = time_ms(lambda: launch(xx, xxp, u0, u_out, grad=grad), a.reps)
        ms_c2 = time_ms(lambda: launch(xx, xxp, grad=grad), a.reps)
        r = {'cold_ms': min(ms_c, ms_c2), 'cold_ms_runs': [ms_c, ms_c2], 'warm_ms': ms_w,
             'cold_newton_mean': ref[2].double().mean().item(), 'cold_newton_max': int(ref[2].max()),
             'warm_newton_mean': warm[2].double().mean().item(), 'warm_newton_max': int(warm[2].max()),
             'warm_vs_cold_loss_rel': dl, 'warm_vs_cold_grad_rel': dg}
        res[f'kernel_{label}_order'] = r
        print(f'{label:7s} order: cold {ms_c:.3f} / {ms_c2:.3f} ms (Newton mean {r["cold_newton_mean"]:.2f} max '
              f'{r["cold_newton_max"]}), warm {ms_w:.3f} ms (Newton mean {r["warm_newton_mean"]:.2f} max '
              f'{r["warm_newton_max"]}); warm vs cold: loss {dl:.1e}, gradient {dg:.1e}')

    losses = {}
    for mode in ('cold', 'warm'):
        ds = DeviceTrajectorySliceDataset(TrajectorySliceConfig(), device=dev)
        for p0, p1 in zip(x, xp):                 # one two-state trajectory per pair
            ds.add_slices_from_trajectory(torch.stack((p0, p1)))
        m = tree_system(g, dev)
        m.record_qp_solution = mode == 'warm'
        opt = torch.optim.Adam(m.parameters(), lr=1e-3)
        per_epoch, ls = [], []
        for epoch in range(a.epochs):
            st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k = 0
            st.record()
            for prev, fut, idx in ds.batches(a.loop_batch, shuffle=False, return_indices=True):
                if mode == 'warm':
                    m.qp_warm_start = ds.warm_start(idx)
                opt.zero_grad()
                loss = m.contactnets_loss(prev[:, -1], None, fut[:, 0])
                loss.mean().backward()
                opt.step()
                if mode == 'warm':
                    ds.update_solutions(idx, loss.qp_solution)
                ls.append(loss.detach())
                k += 1
            en.record()
            torch.cuda.synchronize()
            per_epoch.append({'step_ms': st.elapsed_time(en) / k})
            print(f'adam loop {mode}: epoch {epoch} {per_epoch[-1]["step_ms"]:.3f} ms per step')
        res[f'adam_loop_{mode}'] = per_epoch
        losses[mode] = torch.cat(ls)
    res['adam_loop_warm_vs_cold_loss_rel'] = ((losses['warm'] - losses['cold']).abs().max() /
                                              losses['cold'].abs().max()).item()
    print('adam loop warm vs cold loss:', res['adam_loop_warm_vs_cold_loss_rel'])
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
