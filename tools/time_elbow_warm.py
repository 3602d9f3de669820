"""Cold versus warm-started solves of the two-body (elbow) ContactNets loss, on the bench's elbow batch (262,144 box
pairs, synthetic.elbow_states seed 3, default elbow.urdf parameters).

1. Kernel time (CUDA events over --reps launches, after warm-up) and mean / max Newton counts, in natural and in cost
   order (cost order = the cold Newton counts, descending, with the dynamic schedule), for a cold solve and for a solve
   started from the optima of the parameters before one Adam step (lr 1e-3) of the loss.
2. A short Adam loop through DeviceTrajectorySliceDataset, with and without warm starts from the optima the data set
   recorded in the previous epoch: step time (CUDA events) and mean Newton count per epoch.

Prints one line per measurement and a JSON summary, with the device's name, power limit and maximum SM clock.  Writes
nothing into the repository (--out: optional JSON file)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from dair_pll_b200 import ops, synthetic  # noqa: E402
from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig  # noqa: E402
from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem  # noqa: E402

DT = 0.0068


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = torch.cuda.get_device_name(0)
    return q


def time_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st.record()
    for _ in range(reps):
        fn()
    en.record()
    torch.cuda.synchronize()
    return st.elapsed_time(en) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=262144)
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--epochs', type=int, default=6)
    ap.add_argument('--loop-batch', type=int, default=65536)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    dev = torch.device('cuda', 0)
    res = {'device': gpu_info(), 'batch': a.batch}
    print('device:', res['device'])

    s = MultibodyLearnableSystem({'elbow': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow.urdf')}, DT).to(dev)
    x = synthetic.elbow_states(a.batch, seed=3, device=dev)
    with torch.no_grad():
        traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(a.batch, 1, device=dev), 1)
    xp = synthetic.perturb_next_state(traj[:, 1], seed=4, n_q=8)

    # the optima before one Adam step, the parameters after it
    s.record_qp_solution = True
    opt = torch.optim.Adam(s.parameters(), lr=1e-3)
    loss = s.contactnets_loss(x, None, xp)
    u_before = loss.qp_solution.clone()
    loss.mean().backward()
    opt.step()
    s.record_qp_solution = False
    params = [t.detach() for t in s._elbow_params(torch.float64, dev)]
    it_cold = ops.elbow_loss_raw(x, xp, *params, DT, 1e-3, want_iters=True)[4]
    order = torch.argsort(it_cold, descending=True, stable=True)
    for label, perm, flags in (('natural', None, 0), ('cost', order, ops.LOSS_DYNAMIC)):
        xx, xxp = (x, xp) if perm is None else (x.index_select(0, perm).contiguous(), xp.index_select(0, perm).contiguous())
        u0 = u_before if perm is None else u_before.index_select(0, perm).contiguous()
        ref = ops.elbow_loss_raw(xx, xxp, *params, DT, 1e-3, want_iters=True, flags=flags)
        warm = ops.elbow_loss_raw(xx, xxp, *params, DT, 1e-3, want_iters=True, flags=flags, u_init=u0)
        dl = ((warm[0] - ref[0]).abs().max() / ref[0].abs().max()).item()
        dg = ((warm[1] - ref[1]).abs().max() / ref[1].abs().max()).item()
        # warm launches read u0 and write the optima elsewhere, so every timed launch starts from the same point
        u_out = torch.empty_like(u0)
        ms_c = time_ms(lambda: ops.elbow_loss_raw(xx, xxp, *params, DT, 1e-3, flags=flags), a.reps)
        ms_w = time_ms(lambda: ops.elbow_loss_raw(xx, xxp, *params, DT, 1e-3, flags=flags, u_init=u0, u_out=u_out), a.reps)
        ms_c2 = time_ms(lambda: ops.elbow_loss_raw(xx, xxp, *params, DT, 1e-3, flags=flags), a.reps)
        r = {'cold_ms': min(ms_c, ms_c2), 'cold_ms_runs': [ms_c, ms_c2], 'warm_ms': ms_w,
             'cold_newton_mean': ref[4].double().mean().item(), 'cold_newton_max': int(ref[4].max()),
             'warm_newton_mean': warm[4].double().mean().item(), 'warm_newton_max': int(warm[4].max()),
             'warm_vs_cold_loss_rel': dl, 'warm_vs_cold_grad_rel': dg}
        res[f'kernel_{label}_order'] = r
        print(f'{label:7s} order: cold {ms_c:.3f} / {ms_c2:.3f} ms (Newton mean {r["cold_newton_mean"]:.2f} max '
              f'{r["cold_newton_max"]}), warm {ms_w:.3f} ms (Newton mean {r["warm_newton_mean"]:.2f} max '
              f'{r["warm_newton_max"]}); warm vs cold: loss {dl:.1e}, gradient {dg:.1e}')

    # training loop through the data set: slices (x, x_plus) of two-state trajectories
    ds = DeviceTrajectorySliceDataset(TrajectorySliceConfig(), device=dev)
    ds._previous.append(x.unsqueeze(1))           # one slice per pair, without a Python loop over 262,144 trajectories
    ds._future.append(xp.unsqueeze(1))
    for mode in ('cold', 'warm'):
        m = MultibodyLearnableSystem({'elbow': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow.urdf')}, DT).to(dev)
        m.record_newton_iters = True
        m.record_qp_solution = mode == 'warm'
        ds._usol = None
        opt = torch.optim.Adam(m.parameters(), lr=1e-3)
        per_epoch = []
        for epoch in range(a.epochs):
            st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            its, n = [], 0
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
                its.append(loss.newton_iters.double().mean())
                n += 1
            en.record()
            torch.cuda.synchronize()
            per_epoch.append({'step_ms': st.elapsed_time(en) / n, 'newton_mean': torch.stack(its).mean().item()})
            print(f'adam loop {mode}: epoch {epoch} {per_epoch[-1]["step_ms"]:.3f} ms per step, Newton mean '
                  f'{per_epoch[-1]["newton_mean"]:.2f}')
        res[f'adam_loop_{mode}'] = per_epoch
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
