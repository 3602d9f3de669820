"""CPU: the warm-started tree losses.  Their C entry points live in their own header (include/dair_pll_b200_warm_body_tree.h),
outside the prototype sets of the main and elbow warm-start headers; their argument codes are checked without a device; and
the per-sample arithmetic of the kernel's warm instance (chain_loss_sample with a start point), compiled for the host, gives
the cold results from any start point."""
import ctypes
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

from dair_pll_b200 import _lib
from tests.test_abi_args import EINVAL, EWORKSPACE, OK, WS, _RUNNER, _library
from tests.test_elbow_warm_host import _prototypes
from tests.test_host_emulation import chain_kernel_level_params, chain_kin_rows
from tests.util import ROOT, dptr, load_golden, max_rel_to_scale

WARM = ('dpll_chain_loss_warm_f64', 'dpll_chain_loss_pts_warm_f64')


def test_warm_body_tree_header_parses_into_its_own_table():
    assert set(_lib.WARM_BODY_TREE_EXPORTS) == set(WARM) | {"dpll_body_loss_pts_warm_f64"}
    assert not set(_lib.WARM_BODY_TREE_EXPORTS) & (set(_lib.EXPORTS) | set(_lib.WARM_EXPORTS))
    cold = _lib.EXPORTS['dpll_chain_loss_f64'][0]
    warm, ret = _lib.WARM_BODY_TREE_EXPORTS['dpll_chain_loss_warm_f64']
    # the cold arguments, then u_init / u_out before the workspace, its size and the stream
    assert ret is ctypes.c_int32 and warm == cold[:16] + [ctypes.c_void_p, ctypes.c_void_p] + cold[16:]
    cold_pts = _lib.EXPORTS['dpll_chain_loss_pts_f64'][0]
    warm_pts, _ = _lib.WARM_BODY_TREE_EXPORTS['dpll_chain_loss_pts_warm_f64']
    assert warm_pts == cold_pts[:16] + [ctypes.c_void_p] * 3 + cold_pts[16:]
    names = _prototypes(_lib.WARM_BODY_TREE_HEADER)
    assert names['dpll_chain_loss_warm_f64'] == _prototypes(_lib.HEADER)['dpll_chain_loss_f64'][:16] + \
        ['u_init', 'u_out', 'workspace', 'workspace_bytes', 'stream']
    assert names['dpll_chain_loss_pts_warm_f64'] == _prototypes(_lib.HEADER)['dpll_chain_loss_pts_f64'][:16] + \
        ['u_init', 'u_out', 'iters', 'workspace', 'workspace_bytes', 'stream']


N = None
BASE = dict(n_links=3, B=16, dt=0.01, eps=1e-3, n_pts_packed=0, workspace_bytes=WS, stream=None)
CASES = {
    'dpll_chain_loss_warm_f64': [
        (dict(x=N), EINVAL), (dict(B=-1), EINVAL), (dict(kin=N), EINVAL), (dict(half=N), EINVAL),
        (dict(n_links=1), EINVAL), (dict(n_links=7), EINVAL),
        (dict(workspace_bytes=WS - 1), EWORKSPACE), (dict(workspace_bytes=WS - 1, u_init=N, u_out=N), EWORKSPACE),
        (dict(B=0, grad=N, loss_sum=N), OK), (dict(B=0, grad=N, loss_sum=N, u_init=N), OK),
        (dict(B=0, grad=N, loss_sum=N, u_out=N), OK),
    ],
    'dpll_chain_loss_pts_warm_f64': [
        (dict(x=N), EINVAL), (dict(pts=N), EINVAL), (dict(B=-1), EINVAL), (dict(mu_pair=N), EINVAL),
        (dict(n_links=1), EINVAL), (dict(workspace_bytes=WS - 1), EWORKSPACE),
        (dict(B=0), OK), (dict(B=0, u_init=N, u_out=N, iters=N), OK),
    ],
}


def test_warm_tree_entry_points_return_their_argument_codes():
    """Every call is rejected (or returns) before a pointer is used; no CUDA device is visible to the subprocess."""
    _library()
    protos = _prototypes(_lib.WARM_BODY_TREE_HEADER)
    calls, expected = [], []
    for name in WARM:
        for over, code in CASES[name]:
            assert set(over) <= set(protos[name]), over
            calls.append((name, [over.get(p, BASE.get(p, 'P')) for p in protos[name]], None))
            expected.append(code)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    proc = subprocess.run([sys.executable, '-c', _RUNNER],
                          input=json.dumps(calls), capture_output=True, text=True, cwd=ROOT, env=env, timeout=300)
    assert proc.returncode == 0, proc.stderr
    out = json.loads(proc.stdout.strip().splitlines()[-1])
    bad = [(c[0], c[1], w, g) for c, w, g in zip(calls, expected, out['codes']) if w != g]
    assert not bad, bad
    assert out['workspace_bytes'] == WS and out['version'] == _lib.ABI_VERSION == 214


_EMUL = None


def _emulation():
    """g++ build of tests/host_emul/emul_chain_warm.cpp, with the flags of the main host emulation library."""
    global _EMUL
    if _EMUL is None:
        out = os.path.join(tempfile.gettempdir(), f'dpll_emul_chain_warm_{os.getuid()}.so')
        src = os.path.join(ROOT, 'tests', 'host_emul', 'emul_chain_warm.cpp')
        gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
        subprocess.check_call([gxx, '-O2', '-std=c++17', '-fPIC', '-shared', '-ffp-contract=off', '-o', out, src])
        _EMUL = ctypes.CDLL(out)
    return _EMUL


def _case(name, assets_dir):
    """(n, x, x+, kernel-level params (inertia, mu, half), kin, pts | None, packed, dt) of a golden: the box trees, or
    chain3s (Box + Sphere + Polygon as witness points, from the product's own host code)."""
    g = load_golden(name)
    x, xp = np.ascontiguousarray(g['x']), np.ascontiguousarray(g['x_plus'])
    if name != 'chain3s':
        from oracle.callables import CHAIN3_TREE, TREE4_TREE
        tree = {'chain3': CHAIN3_TREE, 'tree4': TREE4_TREE}[name]
        n = tree.n_bodies
        return n, x, xp, chain_kernel_level_params(g, n), chain_kin_rows(tree), None, 0, float(g['dt'])
    from dair_pll_b200.geometry import Polygon, Sphere
    from dair_pll_b200.multibody_learnable_system import MultibodyLearnableSystem
    s = MultibodyLearnableSystem({'chain3': os.path.join(assets_dir, 'chain3.urdf')}, float(g['dt']))
    mt = s.multibody_terms
    ct = mt.contact_terms
    ct.geometries[1] = Sphere(torch.from_numpy(g['sphere_radius']))
    ct.geometries[2] = Polygon(torch.from_numpy(g['polygon_vertices']), 4)
    with torch.no_grad():
        mt.lagrangian_terms.inertial_parameters.copy_(torch.from_numpy(g['theta']))
        ct.friction_params.copy_(torch.from_numpy(g['friction_params']))
        ct.geometries[0].length_params.copy_(torch.from_numpy(g['box_length_params']))
        pts, packed = mt.chain_witness_points(torch.from_numpy(xp[:, :9]))
        kin = np.ascontiguousarray(mt.chain_kinematic_table(torch.device('cpu'), witness=True).numpy())
        inertia = mt.lagrangian_terms.inertia_vector().reshape(30).numpy().copy()
        mu = ct.pair_friction().reshape(3).numpy().copy()
    return 3, x, xp, (inertia, mu, np.zeros(9)), kin, np.ascontiguousarray(pts.numpy()), packed, float(g['dt'])


def _loss(case, params, u_init=None, record=True, in_place=False):
    n, x, xp, _, kin, pts, packed, dt = case
    inertia, mu, half = params
    B = x.shape[0]
    loss, grad, iters = np.zeros(B), np.zeros(14 * n), np.zeros(B, np.int32)
    gp = np.zeros((B, n, 4, 3))
    u_out = (u_init if in_place else np.full((B, 5 + n), np.nan)) if record else None
    rc = _emulation().emul_chain_loss_warm_f64(
        ctypes.c_int(n), dptr(x), dptr(xp), dptr(inertia), dptr(mu), dptr(half), dptr(kin),
        dptr(pts) if pts is not None else None, ctypes.c_uint(packed), ctypes.c_double(dt), ctypes.c_double(1e-3),
        ctypes.c_int64(B), dptr(u_init) if u_init is not None else None, dptr(u_out) if u_out is not None else None,
        dptr(loss), dptr(grad), dptr(gp), dptr(iters))
    assert rc == 0
    return loss, grad, gp, iters, u_out


@pytest.mark.parametrize('name', ['chain3', 'tree4', 'chain3s'])
def test_any_start_point_gives_the_cold_tree_loss_and_gradient(name, assets_dir):
    """From zero, from the cold optimum (also in place) and from the optimum of parameters moved by 1e-3 the solves reach
    the cold loss and gradients; free-flight samples record exactly zero whatever their start; the cold optimum is a start
    that needs at most one Newton direction.  Two start points end within the solver's 1e-12 gradient tolerance of the
    optimum, not on the same bits: losses agree to 1e-13 of their largest value and the gradients, whose contact terms
    carry the forces' 1/eps, to about 1e-11 of their largest entry."""
    case = _case(name, assets_dir)
    n, x, params, g = case[0], case[1], case[3], load_golden(name)
    B = x.shape[0]
    loss_c, grad_c, gp_c, it_c, u_c = _loss(case, params)
    assert np.abs(loss_c - g['loss']).max() < 1e-12                      # the cold path is the golden's
    free = it_c == 0
    assert 0 < free.sum() < B and np.all(u_c[free] == 0) and not np.isnan(u_c).any()
    inertia, mu, half = params
    _, _, _, _, u_moved = _loss(case, (inertia * 1.001, mu * 0.999, half * 1.0005))
    rng = np.random.default_rng(0)
    starts = {'zero': np.zeros((B, 5 + n)), 'cold optimum': u_c.copy(), 'moved optimum': u_moved,
              'noise in free flight': np.where(free[:, None], rng.standard_normal((B, 5 + n)), u_c)}
    for what, u0 in starts.items():
        loss, grad, gp, iters, u = _loss(case, params, u_init=u0)
        assert np.abs(loss - loss_c).max() <= 1e-13 * np.abs(loss_c).max(), what
        assert max_rel_to_scale(grad, grad_c) < 1e-10, what
        assert max_rel_to_scale(gp, gp_c) < 1e-10, what
        assert max_rel_to_scale(u, u_c) < 1e-9, what
        assert np.all(u[free] == 0) and np.all(iters[free] == 0), what
    _, _, _, it_same, _ = _loss(case, params, u_init=u_c.copy())
    assert it_same.max() <= 1
    _, _, _, it_moved, _ = _loss(case, params, u_init=u_moved.copy())
    assert it_moved.mean() < it_c.mean()
    u_buf = u_moved.copy()
    loss, grad, _, _, u = _loss(case, params, u_init=u_buf, in_place=True)
    assert u is u_buf and max_rel_to_scale(u_buf, u_c) < 1e-9
    assert np.abs(loss - loss_c).max() <= 1e-13 * np.abs(loss_c).max() and max_rel_to_scale(grad, grad_c) < 1e-10


def test_data_set_keeps_tree_solutions_of_their_own_width():
    """update_solutions takes its width from the first solution: 5 + n (here 9) for a tree of n links."""
    from dair_pll_b200.dataset_management import DeviceTrajectorySliceDataset, TrajectorySliceConfig
    data = DeviceTrajectorySliceDataset(TrajectorySliceConfig())
    data.add_slices_from_trajectory(torch.randn(12, 19, dtype=torch.float64))
    n = len(data)
    assert data.warm_start() is None
    idx = torch.arange(0, n, 2)
    u = torch.randn(len(idx), 9, dtype=torch.float64)
    data.update_solutions(idx, u)
    w = data.warm_start(torch.arange(n))
    assert w.shape == (n, 9) and torch.equal(w[idx], u) and torch.all(w[1::2] == 0)
    with pytest.raises(ValueError):
        data.update_solutions(idx, torch.zeros(len(idx), 6, dtype=torch.float64))
