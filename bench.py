#!/usr/bin/env python
"""Benchmark of the hot path: ContactNets loss + backward, cube, fp64 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--dtype f64|f32] [--impl reference]
                    [--dump-outputs DIR]

One step = one pass of ``system.contactnets_loss(x, u, x_plus).mean().backward()`` over one
synthetic batch (SURVEY.md section 8(d)) of B state pairs per GPU.  Prints ONE JSON line (rank 0).
The headline figure is the mean over exactly K timed steps after W (at least 3) untimed ones; the default K = 3000
makes that window about 1 s at the default batch (0.35 ms per step on a B200 at its 1,000 W power limit), long enough
for the clock sampler (nvidia-smi every 100 ms) to sample inside it.  The eager, kernel-only and end-to-end timings take
their step counts from K as well.
For N > 1 launch with ``python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N``:
one process per GPU, the batch sharded by sample (each rank its own B samples: weak scaling),
NCCL all-reduce of the 15-double gradient/loss buffer inside every step.

``--dump-outputs DIR`` writes what the last timed step computed: ``loss.npy`` (the per-sample losses in
generator order; a fixed, seeded sample of 4,194,304 of them when the batch is larger), ``loss_mean.npy`` and
``grad.<parameter name>.npy``.  The inputs depend only on the arguments, so two builds run with the same
arguments can be compared output for output: the per-sample losses repeat bit for bit, the gradients only to
rounding (they are sums in the order the dynamic schedule hands out the work).

``--impl reference`` times the reference's CPU path instead: the oracle port
(oracle/contactnets_oracle.py: the reference's algorithm restated in batched fp64 PyTorch +
the C cone-QP solver standing in for sappy) on all host cores, on a bounded sample of the
same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

DT = 0.0068
# Algorithmic FLOPs per sample (SURVEY.md section 8(d); FMA = 2): F = F0 + F_IT * newton_iters
F0_CUBE, FIT_CUBE = 4600.0, 2100.0
BYTES_PER_SAMPLE = {torch.float64: 2 * 13 * 8 + 8, torch.float32: 2 * 13 * 4 + 4}
METRIC = 'ContactNets loss+backward samples/s, cube'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3000, help='timed steps of the headline measurement')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--batch', type=int, default=1 << 20, help='samples per step: global (strong scaling) or per GPU (weak)')
    ap.add_argument('--dtype', choices=['f64', 'f32'], default='f64')
    ap.add_argument('--impl', choices=['b200', 'reference'], default='b200')
    ap.add_argument('--cpu-sample', type=int, default=65536, help='samples in the CPU baseline step')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-secondary', action='store_true', help='skip the other BASELINE.json configs')
    ap.add_argument('--no-graph', action='store_true', help='time eager launches instead of the CUDA-graph replay')
    ap.add_argument('--variant', type=int, default=0, help='0 = wavefront loss kernel, 1 = one sample per thread')
    ap.add_argument('--scaling', choices=['strong', 'weak'], default=None,
                    help='strong: --batch is the GLOBAL batch, sharded over the ranks (default for N > 1); '
                         'weak: --batch pairs per GPU (default for N = 1)')
    ap.add_argument('--allreduce', choices=['peer', 'nccl'], default='peer',
                    help='gradient exchange: in-kernel peer-memory all-reduce (default) or NCCL after the step')
    ap.add_argument('--order', choices=['cost', 'natural'], default='cost',
                    help='batch order: by decreasing Newton count of the previous pass (default) or generator order')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the loss and the gradients of the last timed step as DIR/<name>.npy (one process only)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs is not None and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the CUDA path: not with --impl reference')
    return args


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        clocks, reasons, smax, power = [], set(), None, []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                clocks.append(float(r[1]))
                smax = float(r[2])
                power.append(float(r[3]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        clocks.sort()
        med = clocks[len(clocks) // 2] if clocks else None
        return {'sm_mhz': med, 'sm_max_mhz': smax, 'reasons': sorted(reasons), 'samples': len(clocks),
                'power_w_max': max(power) if power else None}


def make_system(device, dtype):
    from dair_pll_b200 import synthetic
    from dair_pll_b200.inertia import InertialParameterConverter as IPC
    from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem
    system = MultibodyLearnableSystem({'cube': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'cube.urdf')}, DT)
    pi, fr, half = synthetic.cube_learnables_perturbed(0)
    system.load_state_dict({
        'multibody_terms.lagrangian_terms.inertial_parameters': IPC.pi_cm_to_theta(pi),
        'multibody_terms.contact_terms.friction_params': fr,
        'multibody_terms.contact_terms.geometries.0.length_params': half.reshape(1, 3)})
    return system.to(device)


def make_batch(system, batch, seed, device, dtype):
    """x: seeded synthetic states; x_plus: one learnable-system step + measurement noise."""
    from dair_pll_b200 import synthetic
    x = synthetic.cube_states(batch, seed=seed, device=device, dtype=torch.float64)
    with torch.no_grad():
        traj, _ = system.simulate(x.unsqueeze(-2), torch.zeros(batch, 1, device=device), 1)
    xp = synthetic.perturb_next_state(traj[:, 1], seed=seed + 7919)
    return x.to(dtype).contiguous(), xp.to(dtype).contiguous()


def _time_gpu(fn, device, reps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(device)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize(device)
    return s.elapsed_time(e) / reps


def measured_bf16_tflops():
    """Dense bf16 tensor throughput measured by the driver on this pool (MEASURED_PEAKS.json), else the profiling recipe's
    nominal fallback."""
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['bf16_tflops'])
    except (OSError, KeyError, ValueError):
        return 2250.0


def _roofline(flops, ms, peak_flops, extra=None):
    out = {'bound': 'fp64_cuda_core', 'achieved': flops / (ms * 1e-3) / 1e12, 'peak': peak_flops / 1e12, 'unit': 'TFLOP/s',
           'frac': flops / (ms * 1e-3) / peak_flops, 'kernel_ms': ms}
    if extra:
        out.update(extra)
    return out


def secondary_configs(device, peak_flops):
    """The other BASELINE.json configs, measured through the public API on device-resident inputs
    (CUDA events; context for the headline number, not part of it).  Every entry carries the roofline of
    its dominant kernel by the survey's algorithmic FLOP model (SURVEY.md section 8(d)) and the mean
    Newton count the model is evaluated at."""
    import numpy as np
    from dair_pll_b200 import ops, synthetic
    from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem
    out = {}
    system = make_system(device, torch.float64)
    params = list(system.parameters())
    lt, ct = system.multibody_terms.lagrangian_terms, system.multibody_terms.contact_terms

    def leaves(dtype):
        return [t.detach().to(dtype) for t in (lt.inertial_parameters, ct.friction_params, ct.geometries[0].length_params)]

    def cube_entry(xx, xxp, ordered):
        """graph-replayed public-API step + kernel-only roofline on one batch"""
        from dair_pll_b200 import parallel
        system.dynamic_schedule = ordered
        if ordered:
            it = ops.cube_loss_leaf_dp_raw(xx, xxp, *leaves(xx.dtype), DT, 1e-3, want_iters=True)[4]
            idx = torch.argsort(it, descending=True, stable=True)
            xx, xxp = xx.index_select(0, idx).contiguous(), xxp.index_select(0, idx).contiguous()

        def step():
            for p in params:
                p.grad = None
            mean = system.contactnets_loss(xx, None, xxp).mean()
            mean.backward()
            return mean
        ms_eager = _time_gpu(step, device, 10)
        graphed = parallel.GraphedStep(step, device)
        n = xx.shape[0]
        ms = _time_gpu(graphed, device, max(20, int(100.0 / max(ms_eager, 0.05))))
        flags = (ops.LOSS_DYNAMIC | ops.LOSS_RACE) if ordered else 0
        it = ops.cube_loss_leaf_dp_raw(xx, xxp, *leaves(xx.dtype), DT, 1e-3, flags=flags, want_iters=True)[4]
        mean_it = it.double().mean().item()
        ms_k = _time_gpu(lambda: ops.cube_loss_leaf_dp_raw(xx, xxp, *leaves(xx.dtype), DT, 1e-3, flags=flags), device,
                         max(20, int(100.0 / max(ms_eager, 0.05))))
        system.dynamic_schedule = False
        return {'ms': ms, 'samples_per_s': n / ms * 1e3, 'eager_ms': ms_eager, 'mean_newton_iters': mean_it,
                'order': 'cost' if ordered else 'natural',
                'roofline': _roofline(n * (F0_CUBE + FIT_CUBE * mean_it), ms_k, peak_flops,
                                      {'kernel': 'cube_loss_wf_kernel', 'flops_per_sample': F0_CUBE + FIT_CUBE * mean_it})}

    # config 2: cube loss + backward at B = 65,536, fp64 and the fp32 variant (fp32 storage, fp64 arithmetic)
    x, xp = make_batch(system, 65536, 11, device, torch.float64)
    for name, (xx, xxp) in {'f64': (x, xp), 'f32_storage': (x.float(), xp.float())}.items():
        for ordered in (False, True):
            out[f'cube_loss_backward_B65536_{name}_{"cost" if ordered else "natural"}_order'] = cube_entry(xx, xxp, ordered)
    # the real contact distribution: the reference's recorded tosses (assets/contactnets_cube, 478 consecutive pairs
    # kept as a test fixture), tiled to the headline batch size, nominal URDF parameters
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'cube_real_nominal.npz'))
    reps = (1 << 20) // g['x'].shape[0] + 1
    perm = torch.randperm(reps * g['x'].shape[0], generator=torch.Generator().manual_seed(0))[:1 << 20]
    xr = torch.from_numpy(np.tile(g['x'], (reps, 1)))[perm].to(device).contiguous()
    xpr = torch.from_numpy(np.tile(g['x_plus'], (reps, 1)))[perm].to(device).contiguous()
    saved = {k: v.detach().clone() for k, v in system.state_dict().items()}
    system.load_state_dict({
        'multibody_terms.lagrangian_terms.inertial_parameters': torch.from_numpy(g['theta']).to(device),
        'multibody_terms.contact_terms.friction_params': torch.from_numpy(g['friction_params']).to(device),
        'multibody_terms.contact_terms.geometries.0.length_params': torch.from_numpy(g['half_lengths']).reshape(1, 3).to(device)})
    for ordered in (False, True):
        out[f'cube_real_tiled_B1048576_f64_{"cost" if ordered else "natural"}_order'] = cube_entry(xr, xpr, ordered)
    system.load_state_dict(saved)

    # a training loop on the headline batch: Adam steps (lr 1e-3, the reference example's optimiser,
    # contactnets_simple.py:79-86) move the parameters every step; the batch is in cost order and every pair's solve
    # starts from the optimum of the previous step (system.qp_warm_start, updated in place).  Same losses and
    # gradients as cold solves (unique optimum) -- only the Newton counts change.
    xt, xpt = make_batch(system, 1 << 20, 0, device, torch.float64)
    it0 = ops.cube_loss_leaf_dp_raw(xt, xpt, *leaves(torch.float64), DT, 1e-3, want_iters=True)[4]
    order = torch.argsort(it0, descending=True, stable=True)
    xt, xpt = xt.index_select(0, order).contiguous(), xpt.index_select(0, order).contiguous()
    saved_t = {k: v.detach().clone() for k, v in system.state_dict().items()}
    system.dynamic_schedule = True
    train = {}
    from dair_pll_b200 import parallel
    for mode in ('cold', 'warm'):
        system.load_state_dict(saved_t)
        opt = torch.optim.Adam(params, lr=1e-3, capturable=True)
        usol = torch.zeros(1 << 20, 6, dtype=torch.float64, device=device)
        system.record_qp_solution = system.record_newton_iters = mode == 'warm'
        holder = {}

        def train_step():
            opt.zero_grad(set_to_none=True)
            if mode == 'warm':
                system.qp_warm_start = usol
            loss = system.contactnets_loss(xt, None, xpt)
            mean = loss.mean()
            mean.backward()
            opt.step()
            holder['iters'] = loss.newton_iters
            return mean
        graphed = parallel.GraphedStep(train_step, device)      # the whole iteration, optimiser included, as one graph
        for _ in range(5):
            graphed()
        torch.cuda.synchronize(device)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(200):
            graphed()
        s1.record()
        torch.cuda.synchronize(device)
        ms_t = s0.elapsed_time(s1) / 200
        train[mode] = {'ms_per_step': ms_t, 'samples_per_s': (1 << 20) / ms_t * 1e3,
                       'mean_newton_iters_last_step': (holder['iters'].double().mean().item() if mode == 'warm' else
                                                       it0.double().mean().item())}
    system.record_qp_solution = system.record_newton_iters = False
    system.dynamic_schedule = False
    system.load_state_dict(saved_t)
    out['cube_training_loop_adam_B1048576_f64'] = {
        **train, 'note': 'loss.mean().backward() + Adam step per iteration (CUDA graph replay), cost-ordered batch; warm = every '
                         'solve starts from the previous step\'s optimum (in-place (B,6) buffer)'}

    # config 4: rollout, 4,096 cube tosses x 80 steps
    x0 = synthetic.cube_states(4096, seed=5, device=device)
    carry = torch.zeros(4096, 1, device=device)

    def roll():
        with torch.no_grad():
            system.simulate(x0.unsqueeze(-2), carry, 80)
    ms = _time_gpu(roll, device, 10)
    inertia, mu, half = (t.detach() for t in system._cube_params(torch.float64))
    it_total = torch.empty(4096, dtype=torch.int32, device=device)
    ops.cube_rollout(x0, inertia, mu, half, DT, 80, 1e-4, iters_out=it_total)
    mean_it = it_total.double().mean().item() / 80
    out['cube_rollout_4096x80_f64'] = {
        'ms': ms, 'steps_per_s': 4096 * 80 / ms * 1e3, 'mean_newton_iters_per_step': mean_it,
        'roofline': _roofline(4096 * 80 * (1600.0 + FIT_CUBE * mean_it + 150.0), ms, peak_flops,
                              {'kernel': 'cube_rollout_kernel', 'flops_per_step': 1600.0 + FIT_CUBE * mean_it + 150.0,
                               'note': '4,096 sequential chains of 80 dependent steps: latency-bound (a lone toss advances at '
                                       '~20 us per step); 65,536 tosses reach 4.5x this rate'})}
    # prediction loss: rollout + backward through every step's QP (K7)
    x0g = x0[:4096].clone().requires_grad_()
    target = torch.zeros(4096, 81, 13, device=device, dtype=torch.float64)

    def pred_step():
        for p in params:
            p.grad = None
        x0g.grad = None
        traj, _ = system.simulate(x0g.unsqueeze(-2), carry, 80)
        ((traj - target) ** 2).mean().backward()
    ms = _time_gpu(pred_step, device, 3, warmup=1)
    out['cube_prediction_loss_4096x80_f64'] = {'ms': ms, 'steps_per_s': 4096 * 80 / ms * 1e3,
                                               'note': 'forward rollout keeping every QP optimum + reverse-mode backward through every step '
                                                       '(dpll_cube_rollout_saved_f64 / dpll_cube_rollout_backward_f64) + the torch MSE on the '
                                                       'trajectory'}
    # elbow (two bodies, 8 contacts) with box geometries, loss + backward at B = 262,144
    FO_EL, FIT_EL = 12000.0, 4700.0
    ebox = MultibodyLearnableSystem({'elbow': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow.urdf')}, DT).to(device)
    Be = 262144
    xe = synthetic.elbow_states(Be, seed=3, device=device)
    with torch.no_grad():
        te, _ = ebox.simulate(xe.unsqueeze(-2), torch.zeros(Be, 1, device=device), 1)
    xpe = synthetic.perturb_next_state(te[:, 1], seed=4, n_q=8)

    params_e = list(ebox.parameters())
    ine, mue, halfe, kin = ebox._elbow_params(torch.float64, device)
    ine, mue, halfe = ine.detach(), mue.detach(), halfe.detach()
    it_e = ops.elbow_loss_raw(xe, xpe, ine, mue, halfe, kin, DT, 1e-3, want_iters=True)[4]
    mean_it = it_e.double().mean().item()
    order_e = torch.argsort(it_e, descending=True, stable=True)
    for ordered in (False, True):
        xx, xxp = (xe.index_select(0, order_e).contiguous(), xpe.index_select(0, order_e).contiguous()) if ordered else (xe, xpe)
        ebox.dynamic_schedule = ordered
        flags = ops.LOSS_DYNAMIC if ordered else 0

        def ebox_step():
            for p in params_e:
                p.grad = None
            mean = ebox.contactnets_loss(xx, None, xxp).mean()
            mean.backward()
            return mean
        ms_eager_e = _time_gpu(ebox_step, device, 10)
        from dair_pll_b200 import parallel
        ms = _time_gpu(parallel.GraphedStep(ebox_step, device), device, 50)   # parameter preparation (theta -> inertia
        # vectors, ~100 tiny torch kernels with their autograd) is host-bound when launched eagerly
        ms_k = _time_gpu(lambda: ops.elbow_loss_raw(xx, xxp, ine, mue, halfe, kin, DT, 1e-3, flags=flags), device, 20)
        out[f'elbow_box_loss_backward_B262144_f64_{"cost" if ordered else "natural"}_order'] = {
            'ms': ms, 'samples_per_s': Be / ms * 1e3, 'eager_ms': ms_eager_e, 'mean_newton_iters': mean_it,
            'order': 'cost' if ordered else 'natural', 'step': 'CUDA graph replay of the public-API step',
            'roofline': _roofline(Be * (FO_EL + FIT_EL * mean_it), ms_k, peak_flops,
                                  {'kernel': 'elbow_loss_wf_kernel', 'flops_per_sample': FO_EL + FIT_EL * mean_it})}
    ebox.dynamic_schedule = False
    # config 3: elbow with learned (ICNN, width 256) geometry, loss + backward at B = 262,144
    torch.manual_seed(0)
    elbow = MultibodyLearnableSystem({'elbow': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'elbow_mesh.urdf')}, DT).to(device)
    with torch.no_grad():
        te, _ = elbow.simulate(xe.unsqueeze(-2), torch.zeros(Be, 1, device=device), 1)
    xpm = synthetic.perturb_next_state(te[:, 1], seed=4, n_q=8)

    params_m = list(elbow.parameters())

    def elbow_step():
        for p in params_m:
            p.grad = None
        loss = elbow.contactnets_loss(xe, None, xpm)
        loss.mean().backward()
        return loss.detach()       # (a live autograd graph of an eager step would break the later capture)
    ms_eager_m = _time_gpu(elbow_step, device, 3, warmup=1)
    ms = _time_gpu(parallel.GraphedStep(elbow_step, device), device, 10)
    # dominant kernel: the support-point kernel of ONE network over its D = 4 B direction rows (two such launches per step)
    net = elbow.multibody_terms.contact_terms.geometries[0].network
    ws = [net.input_weights[0].detach(), net.input_weights[1].detach(), net.hidden_weights[0].detach(), net.output_weight.detach()]
    Dm = 4 * Be
    dirs = torch.randn(Dm, 3, dtype=torch.float64, device=device)
    dirs = dirs / dirs.norm(dim=-1, keepdim=True)
    prepared = ops.icnn_tc_prepare(*ws, net.negative_slope)
    ms_k = _time_gpu(lambda: ops.icnn_support_points_tc(dirs, *ws, net.negative_slope, prepared), device, 10)
    TC_OPS_PER_ROW = 2.0 * 3 * 6 * 256 * 256        # 3 input coordinates x 6 int8 digit planes x (256 x 256) MACs
    int8_peak = 2.0 * measured_bf16_tflops() * 1e12
    out['elbow_mesh_loss_backward_B262144_f64'] = {
        'ms': ms, 'samples_per_s': Be / ms * 1e3, 'eager_ms': ms_eager_m, 'step': 'CUDA graph replay of the public-API step',
        'roofline': {'bound': 'tensor', 'kernel': 'icnn_tc_kernel (support points of one network, D = 1,048,576 rows; 2 launches '
                                                  'per step)',
                     'achieved': Dm * TC_OPS_PER_ROW / (ms_k * 1e-3) / 1e12, 'peak': int8_peak / 1e12, 'unit': 'TOP/s (int8)',
                     'frac': Dm * TC_OPS_PER_ROW / (ms_k * 1e-3) / int8_peak, 'kernel_ms': ms_k,
                     'ops_per_row': TC_OPS_PER_ROW,
                     'peak_source': '2 x MEASURED_PEAKS.json bf16_tflops (tcgen05 kind::i8 issues at twice the bf16 rate; no '
                                    'measured int8 figure exists)',
                     'note': 'exact fp64 result from int8 digit-plane products; FP64-equivalent work of the replaced GEMMs: '
                             '4.28e6 FLOP per sample'}}
    # generic kinematic tree (SURVEY 8(f) N2; one sample per thread, the general path, not a tuned one): the branching
    # four-link tree of the tests, its fixture states tiled to 65,536 pairs
    import numpy as np
    fx = np.load(os.path.join(ROOT, 'tests', 'golden', 'tree4.npz'))
    tree = MultibodyLearnableSystem({'tree4': os.path.join(ROOT, 'dair_pll_b200', 'assets', 'tree4.urdf')}, DT)
    sd = {'multibody_terms.lagrangian_terms.inertial_parameters': torch.from_numpy(fx['theta']),
          'multibody_terms.contact_terms.friction_params': torch.from_numpy(fx['friction_params'])}
    for i in range(4):
        sd[f'multibody_terms.contact_terms.geometries.{i}.length_params'] = torch.from_numpy(fx['half_lengths'][i]).reshape(1, 3)
    tree.load_state_dict(sd)
    tree = tree.to(device)
    Bt = 65536
    reps = (Bt + fx['x'].shape[0] - 1) // fx['x'].shape[0]
    xt = torch.from_numpy(fx['x']).to(device).repeat(reps, 1)[:Bt].contiguous()
    xpt = torch.from_numpy(fx['x_plus']).to(device).repeat(reps, 1)[:Bt].contiguous()
    params_t = list(tree.parameters())

    def tree_step():
        for p in params_t:
            p.grad = None
        loss = tree.contactnets_loss(xt, None, xpt)
        loss.mean().backward()
        return loss.detach()
    ms = _time_gpu(tree_step, device, 5, warmup=2)
    out['tree4_loss_backward_B65536_f64'] = {
        'ms': ms, 'samples_per_s': Bt / ms * 1e3, 'step': 'eager public-API step',
        'note': 'generic tree kernels (csrc/cn_chain.cuh): four links, 16 contacts, 9 velocities; fixture states tiled'}
    return out


DUMP_MAX_ROWS = 1 << 22      # per-sample losses written by --dump-outputs: 32 MB in float64, the dump stays under 64 MB


def dump_outputs(out_dir, loss, mean, grads, names):
    """Writes out_dir/<name>.npy: the per-sample losses (a fixed, seeded sample of DUMP_MAX_ROWS of them when there
    are more), the mean loss and the gradient of every parameter."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    if loss.shape[0] > DUMP_MAX_ROWS:
        pick = torch.randperm(loss.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ROWS].sort().values
        loss = loss.index_select(0, pick.to(loss.device))
    arrays = {'loss': loss, 'loss_mean': mean, **{f'grad.{n}': g for n, g in zip(names, grads)}}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().cpu().numpy())


def cpu_reference_step(batch, threads):
    """Builds the oracle-port step (loss + backward) on the host; returns a callable."""
    from dair_pll_b200 import synthetic
    from oracle import contactnets_oracle as co
    from oracle.callables import CUBE_TREE, TreeCallables
    from oracle.cone_qp import OracleSAPSolver
    torch.set_num_threads(threads)
    calls = TreeCallables(CUBE_TREE)
    pi, fr, half = synthetic.cube_learnables_perturbed(0)
    P = co.OracleParams(co.pi_cm_to_theta(pi), fr.clone(), [half.reshape(1, 3).clone()]).requires_grad_()
    solver = OracleSAPSolver(nthreads=threads)
    x = synthetic.cube_states(batch, seed=0)
    with torch.no_grad():
        xp = synthetic.perturb_next_state(co.sim_step(calls, P, x, DT, solver), seed=7919)

    def step():
        for t in P.leaves():
            t.grad = None
        loss = co.contactnets_loss(calls, P, x, xp, DT, solver)
        loss.mean().backward()
        return loss
    return step


def time_cpu(step, steps, warmup):
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) / steps


def run_reference(args, out):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    B = args.cpu_sample
    step = cpu_reference_step(B, threads)
    # bounded: keep the whole run within a few minutes
    steps = max(1, min(args.steps, 10))
    warmup = max(1, min(args.warmup, 2))
    sec = time_cpu(step, steps, warmup)
    value = B / sec
    scaling = args.scaling or ('strong' if args.gpus > 1 else 'weak')
    workload = (f'cube_contactnets_loss_backward_B{args.batch}_global' if scaling == 'strong'
                else f'cube_contactnets_loss_backward_B{args.batch}_per_gpu')
    sample = f'{B} cube state pairs per step (same generator/parameters as the GPU arm), {steps} steps'
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC + ' fp64', 'value': value, 'unit': 'samples/s', 'n_gpus': args.gpus,
        'steps': steps, 'warmup': warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': scaling,
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': workload, 'batch': args.batch,
                   'dt': DT, 'eps': 1e-3, 'cpu_sample_per_step': B,
                   'note': 'same workload as the GPU arm; each CPU step is a bounded sample of it'},
        'cpu_baseline': {'value': value, 'unit': 'samples/s', 'cores': threads, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}), file=out, flush=True)


def _claim_stdout():
    """stdout carries exactly ONE JSON line: everything else written to file descriptor 1 by this process or the
    libraries it loads (NCCL prints its version banner there) is sent to stderr.  Returns a writer for the line."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, 'w')


def main():
    args = parse_args()
    out = _claim_stdout()
    if args.impl == 'reference':
        run_reference(args, out)
        return
    import torch.distributed as dist
    if hasattr(torch.autograd.graph, 'set_warn_on_accumulate_grad_stream_mismatch'):
        torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)    # graph capture runs on a side stream by design
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('launch N>1 with torch.distributed.run --nproc-per-node N')
    if args.dump_outputs is not None and world > 1:
        raise SystemExit('--dump-outputs needs a single process (--gpus 1)')
    # N < visible GPUs: spread the ranks over the box (rank r -> GPU r * stride).  On the HGX boards of this pool four GPUs
    # share one PCIe root (measured: ~105 GB/s of pinned host->device copies per group of four, 51 GB/s per GPU), so four
    # ranks on GPUs 0-3 get half the end-to-end copy bandwidth of four ranks on GPUs 0, 2, 4, 6; NVLink is all-to-all.
    visible = torch.cuda.device_count()
    dev_index = local_rank * (visible // world) if (world > 1 and visible >= 2 * world) else local_rank
    torch.cuda.set_device(dev_index)
    device = torch.device('cuda', dev_index)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')   # keep stdout to the single JSON line
        dist.init_process_group('nccl', device_id=device)
    dtype = torch.float64 if args.dtype == 'f64' else torch.float32
    from dair_pll_b200 import ops, parallel
    # one process per GPU: keep each rank (and the pinned staging buffers it allocates) on its GPU's NUMA node
    host_binding = parallel.bind_host_to_gpu(dev_index) if world > 1 else None
    ops.set_loss_variant(args.variant)
    scaling = args.scaling or ('strong' if world > 1 else 'weak')
    system = make_system(device, dtype)

    # ---- the batch ------------------------------------------------------------------------------------------
    # strong scaling (BASELINE.json config 5): ONE global batch of args.batch pairs, the same for every N, each
    # rank evaluating its share; weak scaling: args.batch pairs per rank (rank r draws seed r).
    if scaling == 'strong':
        Bg = args.batch
        xg, xpg = make_batch(system, Bg, seed=0, device=device, dtype=dtype)
    else:
        Bg = args.batch * world
        xg, xpg = make_batch(system, args.batch, seed=rank, device=device, dtype=dtype)
    # cost hints = the Newton counts of a previous pass over the same pairs (what a training loop has from its
    # last epoch; dataset_management.DeviceTrajectorySliceDataset.update_costs), computed OUTSIDE the timed region
    system.record_newton_iters = True
    with torch.no_grad():
        hint = system.contactnets_loss(xg, None, xpg).newton_iters.reshape(-1)
    system.record_newton_iters = False

    def shard(order):
        """This rank's (x, x_plus) in the given order and their rows of the generated batch (None: all, in order)."""
        if scaling == 'strong':
            if order == 'cost':      # dealt round-robin from the cost-ordered global batch: equally expensive shards
                idx = torch.argsort(hint, descending=True, stable=True)[rank::world]
            else:
                lo, hi = parallel.shard_bounds(Bg, world, rank)
                idx = torch.arange(lo, hi, device=device)
        else:
            idx = torch.argsort(hint, descending=True, stable=True) if order == 'cost' else None
        if idx is None:
            return xg, xpg, None
        return xg.index_select(0, idx).contiguous(), xpg.index_select(0, idx).contiguous(), idx

    comm = None
    if world > 1 and args.allreduce == 'peer':
        comm = parallel.PeerComm(device)
    params = [p for p in system.parameters()]
    reducer = parallel.GradientAllReduce(params, device, world) if (world > 1 and comm is None) else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed(fn, steps, warmup):
        """Mean ms per call of fn over `steps` calls after `warmup` untimed ones (device time, CUDA events, max
        over ranks)."""
        for _ in range(warmup):
            fn()
        barrier()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(steps):
            fn()
        stop.record()
        barrier()
        ms = torch.tensor([start.elapsed_time(stop)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / steps

    L2_BYTES = 126e6

    def make_step(order):
        """The public-API step on this rank's shard: loss.mean().backward() -> (global) mean loss + param.grad.
        A shard that would fit the L2 (strong scaling, N > 1) is replicated into enough distinct buffers that consecutive
        steps never read rows still resident from the previous ones: the steps cycle through > 2 L2 sizes of inputs."""
        x, xp, rows = shard(order)
        step_bytes = 2 * x.shape[0] * 13 * x.element_size()
        copies = 1 if step_bytes > L2_BYTES else int(2.5 * L2_BYTES / step_bytes) + 1
        bufs = [(x, xp)] + [(x.clone(), xp.clone()) for _ in range(copies - 1)]
        u = torch.zeros(x.shape[0], 0, device=device, dtype=dtype)
        system.dynamic_schedule = order == 'cost'
        system.data_parallel = comm
        turn = {'eager': 0, 'graph': 0}

        def make_local(xx, xxp):
            def step_local():
                if reducer is not None:
                    reducer.zero()
                else:
                    for p in params:
                        p.grad = None
                loss = system.contactnets_loss(xx, u, xxp)
                mean = loss.mean()
                mean.backward()
                # once captured, these are the graph's own output buffers: every replay rewrites them
                step_local.outputs = (loss.detach(), mean.detach(), [p.grad for p in params])
                return reducer.stage(mean) if reducer is not None else mean
            return step_local
        locals_ = [make_local(xx, xxp) for xx, xxp in bufs]

        def in_generator_order(outputs):
            loss, mean, grads = outputs
            if rows is not None:
                loss = torch.empty_like(loss).index_copy_(0, rows, loss)
            return loss, mean, grads

        def step_eager():
            turn['eager'] = (turn['eager'] + 1) % copies
            out = locals_[turn['eager']]()
            return reducer.reduce() if reducer is not None else out
        if args.no_graph:
            return step_eager, step_eager, x, xp, copies, lambda: in_generator_order(locals_[turn['eager']].outputs)
        # with the in-kernel exchange the WHOLE step is one CUDA graph; with NCCL the all-reduce follows the replay
        graphs = [parallel.GraphedStep(fn, device) for fn in locals_]
        # a capture's outputs are its graph's own buffers, rewritten by every replay (eager steps rebind fn.outputs)
        captured = [fn.outputs for fn in locals_]

        def step_graphed():
            turn['graph'] = (turn['graph'] + 1) % copies
            out = graphs[turn['graph']]()
            return reducer.reduce() if reducer is not None else out
        return step_graphed, step_eager, x, xp, copies, lambda: in_generator_order(captured[turn['graph']])

    # ---- device-resident throughput (value): both batch orders, the configured one is the headline ----------
    orders = {}
    sampler = ClockSampler(dev_index)
    for order in (['natural', 'cost'] if args.order == 'cost' else ['cost', 'natural']):   # headline order last
        step, step_eager, x, xp, input_copies, last_outputs = make_step(order)
        ms_eager = timed(step_eager, args.steps, max(args.warmup, 3))
        headline = order == args.order
        if headline and rank == 0:
            sampler.start()
        ms_step = timed(step, args.steps, max(args.warmup, 3))
        if headline:
            clocks = sampler.stop() if rank == 0 else None
            if args.dump_outputs is not None:
                dump_outputs(args.dump_outputs, *last_outputs(), [n for n, _ in system.named_parameters()])
        orders[order] = {'ms_per_step': ms_step, 'value': Bg / (ms_step * 1e-3), 'eager_ms_per_step': ms_eager,
                         'timed_steps': args.steps}
    if comm is not None:
        comm.check()
    ms_step, value = orders[args.order]['ms_per_step'], orders[args.order]['value']
    B = x.shape[0]                       # this rank's samples per step (headline order: built last)

    # ---- end to end through the public API with HOST buffers ------------------------------------------------
    xh, xph = x.cpu().pin_memory(), xp.cpu().pin_memory()
    system.data_parallel = None          # chunks are summed locally; ONE exchange per step follows
    loader = parallel.HostBatchPipeline(system, device, dtype, B)
    n_flat = sum(p.numel() for p in params) + 1
    out_host = torch.empty(n_flat, dtype=torch.float64).pin_memory()

    e2e_note = 'one CUDA graph: chunked H2D copies (side stream) + loss launches + backward + exchange + D2H'
    if comm is not None or world == 1:
        graphed_e2e = loader.capture_step(xh, xph, params, float(Bg), out_host, comm)

        def step_e2e():
            graphed_e2e()
            torch.cuda.current_stream().synchronize()      # the user reads the loss / gradients on the host
    else:
        e2e_note = 'eager chunk launches + NCCL all-reduce'

        def step_e2e():
            for p in params:
                p.grad = None
            total = loader.loss_sum_from_host(xh, xph)
            mean = total / Bg
            mean.backward()
            flat = torch.cat([p.grad.reshape(-1) for p in params] + [mean.detach().reshape(1)])
            dist.all_reduce(flat)
            out_host.copy_(flat, non_blocking=True)
            torch.cuda.current_stream().synchronize()      # the user reads the loss / gradients on the host
    # an end-to-end step lasts ~12 device-resident steps (the PCIe copy of the batch): a tenth of the steps keeps the window
    ms_e2e = timed(step_e2e, max(3, args.steps // 10), 3)
    e2e_value = Bg / (ms_e2e * 1e-3)
    h2d = 2 * B * 13 * x.element_size()
    d2h = out_host.numel() * 8

    # ---- the reference's own call pattern: x = x_past[..., -1, :], x_plus = x_future[..., 0, :] views --------
    strided = None
    if rank == 0 and world == 1 and not args.no_secondary:
        past = torch.stack((x, x), 1)                # (B, 2, 13): t_history = 2, the loss reads the last
        fut = torch.stack((xp, xp), 1)
        xv, xpv = past[..., -1, :], fut[..., 0, :]

        def step_views():
            for p in params:
                p.grad = None
            system.contactnets_loss(xv, None, xpv).mean().backward()
        ms_views = timed(step_views, args.steps, 3)
        strided = {'ms_per_step_eager': ms_views, 'contiguous_eager_ms_per_step': orders[args.order]['eager_ms_per_step'],
                   'note': 'row strides go through the ABI (dpll_cube_loss_leaf_dp_*): no .contiguous() copy'}

    # ---- kernel-only timing for the roofline (CUDA events around the raw launch) ----------------------------
    lt, ct = system.multibody_terms.lagrangian_terms, system.multibody_terms.contact_terms
    leaves = [t.detach().to(dtype) for t in (lt.inertial_parameters, ct.friction_params, ct.geometries[0].length_params)]
    flags = (ops.LOSS_DYNAMIC | ops.LOSS_RACE) if args.order == 'cost' else 0
    iters = ops.cube_loss_leaf_dp_raw(x, xp, *leaves, DT, 1e-3, flags=flags, want_iters=True)[4]
    mean_iters = iters.double().mean().item()

    def kernel_only():
        ops.cube_loss_leaf_dp_raw(x, xp, *leaves, DT, 1e-3, flags=flags)
    ms_kernel = timed(kernel_only, args.steps, 3)
    flops_per_sample = F0_CUBE + FIT_CUBE * mean_iters
    achieved_tflops = B * flops_per_sample / (ms_kernel * 1e-3) / 1e12
    sms = torch.cuda.get_device_properties(device).multi_processor_count
    # the arithmetic is fp64 for both storage types (the fp32 variant is fp32 STORAGE), so is the roofline
    peak_flops = ops.fma_peak(torch.float64, device, sms * 8, 200000)
    hbm_gbs = B * BYTES_PER_SAMPLE[dtype] / (ms_kernel * 1e-3) / 1e9
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except (OSError, ValueError):
        pass
    hbm_peak = peaks.get('hbm_gbs', 6650.0)
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, 'profiles', 'r2_traffic.json')))
        key = f"cube_loss_wf_kernel_{args.dtype}_B{B}_{args.order}"
        if args.variant == 0 and key in tr:
            traffic = tr[key]['dram_bytes_read'] + tr[key]['dram_bytes_write']     # one ncu --set full capture, per launch
    except (OSError, ValueError, KeyError):
        pass

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        Bc = args.cpu_sample
        sec = time_cpu(cpu_reference_step(Bc, threads), 3, 1)
        cpu_baseline = {'value': Bc / sec, 'unit': 'samples/s', 'cores': threads, 'kind': 'port',
                        'sample': f'{Bc} cube state pairs per step x 3 steps, oracle port (batched fp64 torch + C cone-QP '
                                  f'solver, {threads} threads), same generator/parameters'}

    secondary = None
    if world == 1 and not args.no_secondary:
        system.dynamic_schedule, system.data_parallel = False, None
        secondary = secondary_configs(device, peak_flops)
        secondary['reference_call_pattern_strided_views'] = strided

    exchange = ('in-kernel peer-memory all-reduce (dpll_comm, NVLink P2P stores + flags) inside the reduction kernel'
                if comm is not None else ('NCCL all-reduce after the graph replay' if world > 1 else 'none (1 GPU)'))
    workload = (f'cube_contactnets_loss_backward_B{Bg}_global' if scaling == 'strong'
                else f'cube_contactnets_loss_backward_B{args.batch}_per_gpu')
    line = {
        'metric': METRIC + (' fp64' if dtype == torch.float64 else ' fp32'),
        'value': value, 'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': workload, 'batch_per_gpu': B, 'global_batch': Bg, 'dt': DT, 'eps': 1e-3,
                   'parallelism': f'dp{world}',
                   'l2_policy': (f'inputs larger than L2 ({2 * B * 13 * x.element_size() / 1e6:.0f} MB per step vs 126 MB)'
                                 if input_copies == 1 else
                                 f'inputs of {2 * B * 13 * x.element_size() / 1e6:.0f} MB per step would fit the 126 MB L2: the steps '
                                 f'cycle through {input_copies} distinct copies of the shard '
                                 f'({input_copies * 2 * B * 13 * x.element_size() / 1e6:.0f} MB), one captured graph per copy'),
                   'mean_newton_iters': mean_iters, 'storage': args.dtype,
                   'order': (args.order + ': batch handed to the kernel by decreasing Newton count of the previous pass '
                             '(cost hints as a training loop has them from its last epoch, computed outside the timed '
                             'region), warps draw chunks in batch order' if args.order == 'cost' else
                             'natural: generator order, static sample ranges per warp'),
                   'by_order': orders,
                   'timed_steps': orders[args.order]['timed_steps'],
                   'exchange': exchange,
                   'step': 'eager launches' if args.no_graph else 'CUDA graph replay of the public-API step',
                   'eager_ms_per_step': orders[args.order]['eager_ms_per_step']},
        'e2e': {'value': e2e_value, 'unit': 'samples/s', 'ms_per_step': ms_e2e, 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': d2h, 'step': e2e_note, 'chunks': loader.chunks,
                'host_binding': host_binding,
                # what bounds it: the pinned-memory copy of every step's inputs over this rank's PCIe link
                'h2d_gb_per_s': h2d / ms_e2e / 1e6},
        'gpu_launches': 3 * orders[args.order]['timed_steps'],   # per step: parameter preparation + loss/backward +
                                                                  # reduce/chain rule(/exchange)
        'roofline': {'bound': 'fp64_cuda_core',
                     'achieved': achieved_tflops, 'peak': peak_flops / 1e12, 'unit': 'TFLOP/s',
                     'frac': achieved_tflops / (peak_flops / 1e12), 'traffic': traffic,
                     'algorithmic_bytes': B * BYTES_PER_SAMPLE[dtype],
                     'kernel': 'cube_loss_wf_kernel' if args.variant == 0 else 'cube_loss_kernel', 'kernel_ms': ms_kernel,
                     'flops_per_sample': flops_per_sample,
                     'peak_source': 'measured in this run: dpll_fma_peak (dependent-free FMA chains, all SMs)',
                     'hbm': {'achieved_gbs': hbm_gbs, 'peak_gbs': hbm_peak, 'frac': hbm_gbs / hbm_peak,
                             'bytes_per_sample': BYTES_PER_SAMPLE[dtype]}},
        'cpu_baseline': cpu_baseline,
        'clocks': clocks,
        'secondary': secondary,
    }
    print(json.dumps(line), file=out, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
