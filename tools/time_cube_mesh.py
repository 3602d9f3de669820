"""Single floating body with learned geometry (cube_mesh.urdf, width-256 support network): the ContactNets training step
(loss + backward) at B = 262,144 pairs, in cost order (dynamic schedule) and in natural order, eager and replayed as one CUDA
graph (CUDA events); then, in a torch.profiler run of its own, the kernel time of each part of the step -- support directions,
support-network forward, loss, support-network backward.  With --parent-lib, the witness-point loss of an earlier build of
the library (the one-sample-per-thread kernel, ABI 213) and of this one, in alternating runs, for a Sphere and a Polygon at
1,048,576 pairs.  Prints the card's name and power limit first."""
import argparse
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from dair_pll_b200 import _lib, parallel, synthetic  # noqa: E402
from dair_pll_b200.multibody_learnable_system import LOSS_EPS, MultibodyLearnableSystem  # noqa: E402

DT = 0.0068
ap = argparse.ArgumentParser()
ap.add_argument('--batch', type=int, default=262144)
ap.add_argument('--reps', type=int, default=20)
ap.add_argument('--parent-lib', default=None, help='libdair_pll_b200.so of an earlier build (ABI 213) for the A/B')
ap.add_argument('--ab-batch', type=int, default=1048576)
ap.add_argument('--ab-rounds', type=int, default=5)
a = ap.parse_args()
dev = torch.device('cuda', 0)
smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                     capture_output=True, text=True).stdout.strip()
print(f'GPU: {smi}')


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st.record()
    for _ in range(reps):
        fn()
    en.record()
    torch.cuda.synchronize()
    return st.elapsed_time(en) / reps


torch.manual_seed(0)
s = MultibodyLearnableSystem({'cube': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'cube_mesh.urdf')}, DT).to(dev)
x = synthetic.cube_states(a.batch, seed=0, device=dev)
with torch.no_grad():
    traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(a.batch, 1, device=dev), 1)
xp = synthetic.perturb_next_state(traj[:, 1], seed=1)
s.record_newton_iters = True
iters = s.contactnets_loss(x, None, xp).newton_iters
s.record_newton_iters = False
print(f'B = {a.batch}: {(iters == 0).float().mean().item():.1%} free flight, mean {iters.float().mean().item():.2f} '
      f'Newton directions per sample, max {int(iters.max())}')
order = torch.argsort(iters, descending=True, stable=True)
batches = {'natural': (x, xp, False),
           'cost': (x.index_select(0, order).contiguous(), xp.index_select(0, order).contiguous(), True)}
params = list(s.parameters())


def make_step(xb, xpb):
    def step():
        for p in params:
            p.grad = None
        m = s.contactnets_loss(xb, None, xpb).mean()
        m.backward()
        return m.detach()
    return step


for name, (xb, xpb, dyn) in batches.items():
    s.dynamic_schedule = dyn
    step = make_step(xb, xpb)
    ms_eager = timed(step, a.reps)
    g = parallel.GraphedStep(step, dev)
    ms_graph = timed(g, a.reps)
    del g
    print(f'step, {name} order: eager {ms_eager:.3f} ms   graph {ms_graph:.3f} ms   ({a.batch / ms_graph / 1e3:.1f} M pairs/s)')

# kernel time of each part (a profiled run of its own: the numbers above are taken without the profiler).  icnn_tc_kernel
# runs twice per step: over every direction row (forward) and over the rows with a cotangent (the backward's mask record).
from torch.profiler import ProfilerActivity, profile  # noqa: E402


def part_of(name, icnn_seen):
    if 'icnn_tc_kernel' in name:
        return 'ICNN forward' if icnn_seen % 2 == 0 else 'ICNN backward'
    for part, keys in (('directions', ('body_support_directions',)), ('loss', ('cube_loss_wf_kernel', 'reduce_partials')),
                       ('ICNN backward', ('bwd_',))):
        if any(k in name for k in keys):
            return part
    return 'other'


PARTS = ('directions', 'ICNN forward', 'loss', 'ICNN backward', 'other')
for name, (xb, xpb, dyn) in batches.items():
    s.dynamic_schedule = dyn
    step = make_step(xb, xpb)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    n_prof = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            step()
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                     key=lambda e: e.time_range.start)
    per, seen, by_name = {}, 0, {}
    for e in kernels:
        part = part_of(e.name, seen)
        seen += int('icnn_tc_kernel' in e.name)
        us = e.time_range.elapsed_us() / n_prof
        per[part] = per.get(part, 0.0) + us
        by_name[e.name[:60]] = by_name.get(e.name[:60], 0.0) + us
    print(f'kernel time per step, {name} order (torch.profiler): ' +
          '  '.join(f'{p} {per.get(p, 0.0) / 1e3:.3f} ms' for p in PARTS) + f'   sum {sum(per.values()) / 1e3:.3f} ms')
    top = sorted(((us, k) for k, us in by_name.items()), reverse=True)[:6]
    print('   largest kernels: ' + '; '.join(f'{k} {us / 1e3:.3f} ms' for us, k in top))

if a.parent_lib:
    # the witness-point loss of the parent build vs this build, Sphere (1 point) and Polygon (4 points), alternating runs
    from dair_pll_b200.geometry import Polygon, Sphere
    old = ctypes.CDLL(os.path.abspath(a.parent_lib))
    f64, i32, i64, vp, sz = ctypes.c_double, ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p, ctypes.c_size_t
    old.dpll_body_loss_pts_f64.argtypes = [vp] * 6 + [i32, f64, f64, i64] + [vp] * 6 + [vp, sz, vp]
    old.dpll_body_loss_pts_f64.restype = ctypes.c_int
    assert old.dpll_version() == 213
    B = a.ab_batch
    box = MultibodyLearnableSystem({'cube': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'cube.urdf')}, DT).to(dev)
    xs = synthetic.cube_states(B, seed=2, device=dev)
    with torch.no_grad():
        tr, _ = box.simulate(xs.unsqueeze(-2), torch.zeros(B, 1, device=dev), 1)
    xps = synthetic.perturb_next_state(tr[:, 1], seed=3)
    inertia, mu, _ = box._cube_params(torch.float64)
    inertia, mu = inertia.detach().contiguous(), mu.detach().contiguous()
    gen = torch.Generator().manual_seed(4)
    shapes = {'Sphere': Sphere(torch.tensor(0.0524, dtype=torch.float64)),
              'Polygon': Polygon(0.06 * (2 * torch.rand(10, 3, generator=gen, dtype=torch.float64) - 1), 4)}
    ws = torch.empty(_lib.load().dpll_workspace_bytes(), dtype=torch.uint8, device=dev)
    for sname, geom in shapes.items():
        geom = geom.to(dev)
        w, q1, q2, q3 = xps[:, :4].unbind(-1)
        sc = 2.0 / (w * w + q1 * q1 + q2 * q2 + q3 * q3)
        d = -torch.stack((sc * (q1 * q3 - w * q2), sc * (q2 * q3 + w * q1), 1 - sc * (q1 * q1 + q2 * q2)), -1)
        with torch.no_grad():
            p = geom.support_points(d)
        n_c = p.shape[-2]
        pts = torch.cat((p, p.new_zeros(B, 4 - n_c, 3)), -2).contiguous() if n_c < 4 else p.contiguous()
        outs = {k: (torch.empty(B, dtype=torch.float64, device=dev), torch.empty(11, dtype=torch.float64, device=dev),
                    torch.empty(1, dtype=torch.float64, device=dev), torch.empty((B, 4, 3), dtype=torch.float64, device=dev))
                for k in ('parent', 'new')}

        def run_old():
            lo, g, ls, gp = outs['parent']
            rc = old.dpll_body_loss_pts_f64(xs.data_ptr(), xps.data_ptr(), None, inertia.data_ptr(), mu.data_ptr(),
                                            pts.data_ptr(), n_c, DT, LOSS_EPS, B, lo.data_ptr(), None, gp.data_ptr(), None,
                                            g.data_ptr(), ls.data_ptr(), ws.data_ptr(), ws.numel(),
                                            torch.cuda.current_stream().cuda_stream)
            assert rc == 0

        def run_new():
            lo, g, ls, gp = outs['new']
            rc = _lib.load().dpll_body_loss_pts_f64(xs.data_ptr(), xps.data_ptr(), None, inertia.data_ptr(), mu.data_ptr(),
                                                    pts.data_ptr(), n_c, DT, LOSS_EPS, B, 0, lo.data_ptr(), None,
                                                    gp.data_ptr(), None, g.data_ptr(), ls.data_ptr(), None, ws.data_ptr(),
                                                    ws.numel(), torch.cuda.current_stream().cuda_stream)
            assert rc == 0
        times = {'parent': [], 'new': []}
        for _ in range(a.ab_rounds):
            times['parent'].append(timed(run_old, 10))
            times['new'].append(timed(run_new, 10))
        lo_o, g_o, _, gp_o = outs['parent']
        lo_n, g_n, _, gp_n = outs['new']
        dl = ((lo_n - lo_o).abs().max() / lo_o.abs().max()).item()
        dg = ((g_n - g_o).abs().max() / g_o.abs().max()).item()
        dp = ((gp_n - gp_o).abs().max() / gp_o.abs().max()).item()
        print(f'{sname} ({n_c} points), B = {B}: parent {min(times["parent"]):.3f} ms (runs ' +
              ', '.join(f'{t:.3f}' for t in times['parent']) + f')   new {min(times["new"]):.3f} ms (runs ' +
              ', '.join(f'{t:.3f}' for t in times['new']) + f')   max rel diff loss {dl:.1e} grad {dg:.1e} grad_pts {dp:.1e}')
