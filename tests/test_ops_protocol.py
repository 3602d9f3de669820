"""The shared pieces of the Python binding: the fused-backward protocol of the loss Functions (on CPU with a fake
re-launch, and on the GPU for every Function that uses it) and the ctypes signatures read from the C header."""
import contextlib
import ctypes
import os
import re
import types
import weakref

import pytest
import torch

from dair_pll_b200 import _lib, ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = 'cuda:0'


# -- fused backward, host logic ----------------------------------------------------------------------------------------

class _Rerun:
    """Stands in for the weighted re-launch: records its arguments and writes a marker gradient unless skipped."""

    def __init__(self):
        self.calls = []

    def __call__(self, weight, skip_flag, grad_out):
        self.calls.append((weight.clone(), skip_flag.clone()))
        if int(skip_flag) == 0:
            grad_out.copy_(torch.arange(grad_out.numel(), dtype=grad_out.dtype) + 100.0)


GRAD = torch.tensor([1.0, -2.0, 0.5, 4.0], dtype=torch.float64)


def test_fused_grad_stride0_scales_without_relaunch():
    rerun = _Rerun()
    g = ops._fused_grad(GRAD, torch.tensor(0.25, dtype=torch.float64).expand(7), rerun)
    assert torch.equal(g, GRAD * 0.25) and rerun.calls == []


def test_fused_grad_materialised_uniform_sets_skip_flag_and_scales():
    rerun = _Rerun()
    w = torch.full((7,), 0.25, dtype=torch.float64)
    g = ops._fused_grad(GRAD, w, rerun)
    assert torch.equal(g, GRAD * 0.25)
    (weight, skip), = rerun.calls
    assert torch.equal(weight, w) and skip.dtype == torch.int32 and int(skip) == 1


def test_fused_grad_non_uniform_takes_the_weighted_relaunch():
    rerun = _Rerun()
    w = torch.tensor([0.5, 9.0, 1.5, 9.0, -2.0], dtype=torch.float64)[::2]        # a strided upstream gradient
    g = ops._fused_grad(GRAD, w, rerun)
    assert torch.equal(g, torch.arange(4, dtype=torch.float64) + 100.0)
    (weight, skip), = rerun.calls
    assert weight.is_contiguous() and torch.equal(weight, w) and int(skip) == 0


def test_fused_grad_empty_batch_is_zero():
    rerun = _Rerun()
    for empty in (torch.empty(0, dtype=torch.float64), torch.tensor(1.0, dtype=torch.float64).expand(0)):
        g = ops._fused_grad(GRAD, empty, rerun)
        assert torch.equal(g, torch.zeros_like(GRAD))
    assert rerun.calls == []


# -- ctypes signatures from the header ---------------------------------------------------------------------------------

def _header_text():
    with open(os.path.join(ROOT, 'include', 'dair_pll_b200.h')) as f:
        return f.read()


def test_header_signatures_parse_with_the_header_argument_counts():
    text = re.sub(r'/\*.*?\*/', ' ', _header_text(), flags=re.S)
    protos = dict(re.findall(r'\b(dpll_\w+)\s*\(([^)]*)\)\s*;', text))
    assert len(protos) >= 50 and set(protos) == set(_lib.EXPORTS)
    for name, params in protos.items():
        n = 0 if params.strip() in ('', 'void') else params.count(',') + 1
        argtypes, _ = _lib.EXPORTS[name]
        assert len(argtypes) == n, name


def test_header_signatures_spot_checks():
    args, ret = _lib.EXPORTS['dpll_cube_loss_f32']
    assert args[6] is ctypes.c_float and args[7] is ctypes.c_float and args[8] is ctypes.c_int64
    assert all(a is ctypes.c_void_p for a in args[:6]) and args[-2] is ctypes.c_size_t and ret is ctypes.c_int32
    args, _ = _lib.EXPORTS['dpll_cube_loss_f64']
    assert args[6] is ctypes.c_double and args[7] is ctypes.c_double
    args, _ = _lib.EXPORTS['dpll_comm_create']
    assert args == [ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p]
    assert _lib.EXPORTS['dpll_workspace_bytes'] == ([], ctypes.c_size_t)
    assert _lib.EXPORTS['dpll_comm_device_state'] == ([ctypes.c_void_p], ctypes.c_void_p)
    assert _lib.EXPORTS['dpll_chain_loss_pts_f64'][0][8] is ctypes.c_uint32


def test_header_version_is_the_binding_version():
    version = int(re.search(r'#define\s+DPLL_VERSION\s+(\d+)', _header_text()).group(1))
    assert version == _lib.ABI_VERSION


@pytest.mark.parametrize('decl', ['long double x', 'const double x[3]', 'double*** x'])
def test_unknown_c_type_raises(tmp_path, decl):
    header = tmp_path / 'h.h'
    header.write_text(f'int dpll_ok(double a, const float* b);\nint dpll_bad({decl});\n')
    with pytest.raises(TypeError, match=f'dpll_bad in {re.escape(str(header))}'):
        _lib._signatures(str(header))


# -- call path and gradient split, host logic ---------------------------------------------------------------------------

@pytest.fixture
def stub_entry(monkeypatch):
    """Routes ops._call to a Python stand-in of the library on the CPU; records, per call, its arguments and whether
    every tensor registered in ``live`` was still alive when the entry point ran."""
    live, calls = [], []

    def entry(*args):
        calls.append((args, [r() is not None for r in live]))
        return 0
    monkeypatch.setattr(_lib, 'load', lambda: types.SimpleNamespace(dpll_stub_f64=entry, dpll_stub_grad_f64=entry))
    monkeypatch.setattr(torch.cuda, 'device', lambda device: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, 'current_stream', lambda: types.SimpleNamespace(cuda_stream=7))
    return live, calls


def test_call_keeps_inline_temporaries_alive_until_the_entry_point_runs(stub_entry):
    live, calls = stub_entry

    def temporary(t):
        live.append(weakref.ref(t))
        return t
    ops._call('dpll_stub', 'cpu', temporary(torch.ones(4) * 2), None, 3, dtype=torch.float64)
    (args, alive), = calls
    assert alive == [True] and args[1:] == (None, 3, 7) and isinstance(args[0], int)


def test_summed_backward_keeps_its_float64_copies_alive(stub_entry, monkeypatch):
    live, calls = stub_entry
    cast = ops._f64

    def recorded_cast(t):
        out = cast(t)
        live.append(weakref.ref(out))
        return out
    monkeypatch.setattr(ops, '_f64', recorded_cast)
    x, p, q = torch.zeros(5, 3, dtype=torch.float32), torch.ones(2, 2, dtype=torch.float32), torch.ones(1)
    gp, gq, gx = ops._summed_backward('dpll_stub_grad_f64', x, (p, q), (5, 3), x, p, q, 0.1, 5, x[:, :2].t())
    (args, alive), = calls
    assert len(alive) == 4 and all(alive) and args[-6:-4] == (0.1, 5) and args[-1] == 7
    assert gp.shape == p.shape and gp.dtype == torch.float32 and gq.dtype == q.dtype and gx.shape == (5, 3)


def test_fused_reduction_splits_by_the_leaves_shapes_and_does_not_hold_them():
    vec = torch.arange(8, dtype=torch.float64)
    a = torch.zeros(2, 3, dtype=torch.float64, requires_grad=True)
    b = torch.zeros(1, dtype=torch.float64, requires_grad=True)
    out = ops._FusedReduction.apply(vec, 7, a, b)
    with torch.no_grad():
        a.add_(1.0)                      # an update between the reduction and its backward is not an error
    (out * 2).backward()
    assert out.item() == 7.0 and torch.equal(a.grad, 2 * vec[:6].reshape(2, 3)) and torch.equal(b.grad, 2 * vec[6:7])


# -- fused backward of every loss Function, on the GPU -----------------------------------------------------------------

ASSETS = os.path.join(ROOT, 'dair_pll_b200', 'assets')
DT = 0.0068
N = 5003


def _system_and_pair(urdf, states, n_q, seed):
    from dair_pll_b200 import synthetic
    from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem
    kind = 'cube' if n_q == 7 else 'elbow'
    s = MultibodyLearnableSystem({kind: os.path.join(ASSETS, urdf)}, DT).to(DEV)
    x = getattr(synthetic, states)(N, seed=seed, device=DEV)
    with torch.no_grad():
        traj, _ = s.simulate(x.unsqueeze(-2), torch.zeros(N, 1, device=DEV), 1)
    return s, x, synthetic.perturb_next_state(traj[:, 1], seed=seed + 1, n_q=n_q)


def _cube_box():
    s, x, xp = _system_and_pair('cube.urdf', 'cube_states', 7, 10)
    params = tuple(t.detach() for t in s._cube_params(torch.float64))
    return (lambda p: ops.CubeContactNetsLoss.apply(x, xp, *p, DT, 1e-3), params,
            lambda w: ops.cube_loss_raw(x, xp, *params, DT, 1e-3, weight=w)[1])


def _cube_box_leaves():
    s, x, xp = _system_and_pair('cube.urdf', 'cube_states', 7, 20)
    ct = s.multibody_terms.contact_terms
    params = (s.multibody_terms.lagrangian_terms.inertial_parameters.detach(), ct.friction_params.detach(),
              ct.geometries[0].length_params.detach())
    return (lambda p: ops.CubeContactNetsLossLeaf.apply(x, xp, *p, DT, 1e-3, 0, None, False)[0], params,
            lambda w: ops.cube_loss_leaf_raw(x, xp, *params, DT, 1e-3, weight=w)[1])


def _elbow_box():
    s, x, xp = _system_and_pair('elbow.urdf', 'elbow_states', 8, 30)
    inertia, mu, half, kin = (t.detach() for t in s._elbow_params(torch.float64, torch.device(DEV)))
    return (lambda p: ops.ElbowContactNetsLoss.apply(x, xp, *p, kin, DT, 1e-3)[0], (inertia, mu, half),
            lambda w: ops.elbow_loss_raw(x, xp, inertia, mu, half, kin, DT, 1e-3, weight=w)[1])


def _elbow_mesh():
    torch.manual_seed(0)
    s, x, xp = _system_and_pair('elbow_mesh.urdf', 'elbow_states', 8, 40)
    inertia, mu, _, kin = (t.detach() if t is not None else None for t in s._elbow_params(torch.float64, torch.device(DEV)))
    with torch.no_grad():
        pts = s._elbow_witness_points(xp[:, :8])
    return (lambda p: ops.ElbowContactNetsLossPts.apply(x, xp, *p, pts, kin, DT, 1e-3), (inertia, mu),
            lambda w: ops.elbow_loss_raw(x, xp, inertia, mu, None, kin, DT, 1e-3, weight=w, pts=pts)[1][:22])


def _body_mesh():
    torch.manual_seed(0)
    s, x, xp = _system_and_pair('cube_mesh.urdf', 'cube_states', 7, 50)
    inertia, mu, _ = s._cube_params(torch.float64)
    inertia, mu = inertia.detach(), mu.detach()
    with torch.no_grad():
        pts, n_c = s._body_witness_points(xp[:, :4])
    return (lambda p: ops.BodyWitnessPointLoss.apply(x, xp, *p, pts, n_c, DT, 1e-3)[0], (inertia, mu),
            lambda w: ops.body_loss_pts_raw(x, xp, inertia, mu, pts, n_c, DT, 1e-3, weight=w, want_grad_pts=False)[1])


FUSED = {'cube': _cube_box, 'cube_leaves': _cube_box_leaves, 'elbow': _elbow_box, 'elbow_mesh': _elbow_mesh,
         'body_mesh': _body_mesh}


@pytest.mark.gpu
@pytest.mark.parametrize('case', list(FUSED))
def test_fused_backward_weighted_and_materialised_uniform(case):
    """Non-uniform weights: the backward is the raw function's weighted launch, bit for bit.  A materialised uniform
    upstream gradient c: the backward is c times the forward launch's own gradient (the weighted pass is skipped on the
    device), bit for bit."""
    apply, params, raw = FUSED[case]()

    def grad_of(upstream):
        leaves = [p.clone().requires_grad_() for p in params]
        (apply(leaves) * upstream).sum().backward()
        return torch.cat([p.grad.reshape(-1) for p in leaves])

    w = torch.rand(N, dtype=torch.float64, device=DEV, generator=torch.Generator(DEV).manual_seed(1)) + 0.5
    assert torch.equal(grad_of(w), raw(w))
    c = torch.full((N,), 0.37, dtype=torch.float64, device=DEV)
    assert torch.equal(grad_of(c), raw(None) * c[0])
