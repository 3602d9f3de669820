"""CPU: the warm-started witness-point loss of the single floating body (cube-mesh, Sphere, Polygon, a box in a placed
collision frame).  Its C entry point's argument layout and codes are checked without a device, and the per-sample arithmetic
of body_loss_pts_warm_kernel, compiled for the host, gives the cold results from any start point."""
import ctypes
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from dair_pll_b200 import _lib
from tests.test_abi_args import EINVAL, EWORKSPACE, OK, WS, _RUNNER, _library
from tests.test_cube_mesh_host import _shape_inputs
from tests.test_elbow_warm_host import _prototypes
from tests.util import ROOT, dptr, max_rel_to_scale

NAME = 'dpll_body_loss_pts_warm_f64'


def test_body_warm_entry_point_layout():
    cold = _lib.EXPORTS['dpll_body_loss_pts_f64'][0]
    warm, ret = _lib.WARM_BODY_TREE_EXPORTS[NAME]
    # the cold arguments, then u_init / u_out before the workspace, its size and the stream
    assert ret is ctypes.c_int32 and warm == cold[:18] + [ctypes.c_void_p, ctypes.c_void_p] + cold[18:]
    assert _prototypes(_lib.WARM_BODY_TREE_HEADER)[NAME] == _prototypes(_lib.HEADER)['dpll_body_loss_pts_f64'][:18] + \
        ['u_init', 'u_out', 'workspace', 'workspace_bytes', 'stream']


N = None
BASE = dict(n_contacts=4, B=16, flags=0, dt=0.01, eps=1e-3, workspace_bytes=WS, stream=None, skip_flag=None)
CASES = [
    (dict(x=N), EINVAL), (dict(pts=N), EINVAL), (dict(B=-1), EINVAL), (dict(inertia=N), EINVAL),
    (dict(n_contacts=0), EINVAL), (dict(n_contacts=5), EINVAL),
    (dict(workspace_bytes=WS - 1), EWORKSPACE), (dict(grad=N, loss_sum=N, flags=1, workspace=N), EWORKSPACE),
    (dict(workspace_bytes=WS - 1, u_init=N, u_out=N), EWORKSPACE),
    (dict(B=0, grad=N, loss_sum=N), OK), (dict(B=0, grad=N, loss_sum=N, u_init=N), OK),
]


def test_body_warm_entry_point_returns_its_argument_codes():
    """Every call is rejected (or returns) before a pointer is used; no CUDA device is visible to the subprocess."""
    _library()
    protos = _prototypes(_lib.WARM_BODY_TREE_HEADER)[NAME]
    calls, expected = [], []
    for over, code in CASES:
        assert set(over) <= set(protos), over
        calls.append((NAME, [over.get(p, BASE.get(p, 'P')) for p in protos], None))
        expected.append(code)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    proc = subprocess.run([sys.executable, '-c', _RUNNER],
                          input=json.dumps(calls), capture_output=True, text=True, cwd=ROOT, env=env, timeout=300)
    assert proc.returncode == 0, proc.stderr
    out = json.loads(proc.stdout.strip().splitlines()[-1])
    bad = [(c[1], w, g) for c, w, g in zip(calls, expected, out['codes']) if w != g]
    assert not bad, bad


_EMUL = None


def _emulation():
    global _EMUL
    if _EMUL is None:
        out = os.path.join(tempfile.gettempdir(), f'dpll_emul_body_pts_warm_{os.getuid()}.so')
        src = os.path.join(ROOT, 'tests', 'host_emul', 'emul_body_pts_warm.cpp')
        gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
        subprocess.check_call([gxx, '-O2', '-std=c++17', '-fPIC', '-shared', '-ffp-contract=off', '-o', out, src])
        _EMUL = ctypes.CDLL(out)
    return _EMUL


def _loss(inp, inertia, mu, u_init=None, record=True, in_place=False):
    x, xp, pts, n_c, dt = inp
    B = x.shape[0]
    loss, grad, gp, iters = np.zeros(B), np.zeros(11), np.zeros((B, 4, 3)), np.zeros(B, np.int32)
    u_out = (u_init if in_place else np.full((B, 6), np.nan)) if record else None
    _emulation().emul_body_loss_pts_warm_f64(
        dptr(x), dptr(xp), dptr(inertia), dptr(mu), dptr(pts), ctypes.c_int(n_c), ctypes.c_double(dt),
        ctypes.c_double(1e-3), ctypes.c_int64(B), dptr(u_init) if u_init is not None else None,
        dptr(u_out) if u_out is not None else None, dptr(loss), dptr(grad), dptr(gp), dptr(iters))
    return loss, grad, gp, iters, u_out


@pytest.mark.parametrize('name', ['shape_sphere', 'shape_polygon', 'shape_framed_box'])
def test_any_start_point_gives_the_cold_body_loss_and_gradient(name):
    """From zero, from the cold optimum (also in place), from the optimum of parameters moved by 1e-3 and from random
    starts in free flight the solves reach the cold loss and gradients; free flight records exactly zero.  Two start points
    end within the solver's 1e-12 gradient tolerance of the optimum: losses agree to 1e-13 of their largest value and the
    gradients, whose contact terms carry the forces' 1/eps, to about 1e-11 of their largest entry."""
    g, x, xp, inertia, mu, pts, n_c = _shape_inputs(name)
    inp = (x, xp, pts, n_c, float(g['dt']))
    B = x.shape[0]
    loss_c, grad_c, gp_c, it_c, u_c = _loss(inp, inertia, mu)
    assert np.abs(loss_c - g['loss']).max() < 1e-12
    free = it_c == 0
    assert 0 < free.sum() < B and np.all(u_c[free] == 0) and not np.isnan(u_c).any()
    _, _, _, _, u_moved = _loss(inp, inertia * 1.001, mu * 0.999)
    rng = np.random.default_rng(0)
    starts = {'zero': np.zeros((B, 6)), 'cold optimum': u_c.copy(), 'moved optimum': u_moved,
              'noise in free flight': np.where(free[:, None], rng.standard_normal((B, 6)), u_c)}
    for what, u0 in starts.items():
        loss, grad, gp, iters, u = _loss(inp, inertia, mu, u_init=u0)
        assert np.abs(loss - loss_c).max() <= 1e-13 * np.abs(loss_c).max(), what
        assert max_rel_to_scale(grad, grad_c) < 1e-10, what
        assert max_rel_to_scale(gp, gp_c) < 1e-10, what
        assert max_rel_to_scale(u, u_c) < 1e-9, what
        assert np.all(u[free] == 0) and np.all(iters[free] == 0), what
    _, _, _, it_same, _ = _loss(inp, inertia, mu, u_init=u_c.copy())
    assert it_same.max() <= 1
    _, _, _, it_moved, _ = _loss(inp, inertia, mu, u_init=u_moved.copy())
    assert it_moved.mean() < it_c.mean()
    u_buf = u_moved.copy()
    loss, grad, _, _, u = _loss(inp, inertia, mu, u_init=u_buf, in_place=True)
    assert u is u_buf and max_rel_to_scale(u_buf, u_c) < 1e-9
    assert np.abs(loss - loss_c).max() <= 1e-13 * np.abs(loss_c).max() and max_rel_to_scale(grad, grad_c) < 1e-10
