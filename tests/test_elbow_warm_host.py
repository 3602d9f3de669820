"""CPU: the warm-started two-body (elbow) loss.  Its C entry points live in their own header
(include/dair_pll_b200_warm.h), outside the main header's prototype set; their argument codes are checked without a
device; and the per-sample arithmetic of the kernel's warm instance, compiled for the host, gives the cold results from
any start point."""
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from dair_pll_b200 import _lib
from tests.test_abi_args import EINVAL, EWORKSPACE, OK, WS, _RUNNER, _library
from tests.test_host_emulation import ELBOW_KIN, elbow_kernel_level_params
from tests.util import ROOT, dptr, load_golden, max_rel_to_scale

WARM = ('dpll_elbow_loss_warm_f64', 'dpll_elbow_loss_warm_f32')


def _prototypes(path):
    with open(path) as f:
        text = re.sub(r'/\*.*?\*/|//[^\n]*', ' ', f.read(), flags=re.S)
    return {name: [re.split(r'[\s*]+', p.strip())[-1] for p in params.split(',') if p.strip() not in ('', 'void')]
            for name, params in re.findall(r'\b(dpll_\w+)\s*\(([^)]*)\)\s*;', text)}


def test_warm_header_parses_into_its_own_table():
    assert set(_lib.WARM_EXPORTS) == set(WARM)
    assert not set(_lib.WARM_EXPORTS) & set(_lib.EXPORTS)
    assert set(_lib.EXPORTS) == set(_prototypes(_lib.HEADER))            # the main table is the main header's, alone
    cold = _lib.EXPORTS['dpll_elbow_loss_f64'][0]
    warm, ret = _lib.WARM_EXPORTS['dpll_elbow_loss_warm_f64']
    # the cold arguments, then u_init / u_out before the workspace, its size and the stream
    assert ret is ctypes.c_int32 and warm == cold[:19] + [ctypes.c_void_p, ctypes.c_void_p] + cold[19:]
    names = _prototypes(_lib.WARM_HEADER)['dpll_elbow_loss_warm_f32']
    assert names == _prototypes(_lib.HEADER)['dpll_elbow_loss_f32'][:19] + ['u_init', 'u_out'] + \
        ['workspace', 'workspace_bytes', 'stream']


N = None
BASE = dict(B=16, flags=0, dt=0.01, eps=1e-3, workspace_bytes=WS, stream=None, skip_flag=None)
CASES = [
    (dict(x=N), EINVAL), (dict(B=-1), EINVAL), (dict(kin=N), EINVAL), (dict(half=N, pts=N), EINVAL),
    (dict(grad=N), EINVAL),                                                 # grad_pts needs grad
    (dict(workspace_bytes=WS - 1), EWORKSPACE), (dict(workspace_bytes=WS - 1, u_init=N, u_out=N), EWORKSPACE),
    (dict(grad_pts=N, grad=N, loss_sum=N, flags=1, workspace=N), EWORKSPACE),
    (dict(B=0, grad=N, grad_pts=N, loss_sum=N), OK), (dict(B=0, grad=N, grad_pts=N, loss_sum=N, u_init=N), OK),
    (dict(B=0, grad=N, grad_pts=N, loss_sum=N, u_out=N), OK),
]


def test_warm_entry_points_return_their_argument_codes():
    """Every call is rejected (or returns) before a pointer is used; no CUDA device is visible to the subprocess."""
    _library()
    protos = _prototypes(_lib.WARM_HEADER)
    calls, expected = [], []
    for name in WARM:
        for over, code in CASES:
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
    """g++ build of tests/host_emul/emul_elbow_warm.cpp, with the flags of the main host emulation library."""
    global _EMUL
    if _EMUL is None:
        out = os.path.join(tempfile.gettempdir(), f'dpll_emul_elbow_warm_{os.getuid()}.so')
        src = os.path.join(ROOT, 'tests', 'host_emul', 'emul_elbow_warm.cpp')
        gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
        subprocess.check_call([gxx, '-O2', '-std=c++17', '-fPIC', '-shared', '-ffp-contract=off', '-o', out, src])
        _EMUL = ctypes.CDLL(out)
    return _EMUL


def _loss(g, params, u_init=None, record=True, in_place=False):
    inertia, mu, half = params
    x, xp = np.ascontiguousarray(g['x']), np.ascontiguousarray(g['x_plus'])
    B = x.shape[0]
    loss, grad, iters = np.zeros(B), np.zeros(28), np.zeros(B, np.int32)
    u_out = (u_init if in_place else np.full((B, 7), np.nan)) if record else None
    _emulation().emul_elbow_loss_warm_f64(
        dptr(x), dptr(xp), dptr(inertia), dptr(mu), dptr(half), dptr(ELBOW_KIN), None, ctypes.c_double(float(g['dt'])),
        ctypes.c_double(1e-3), ctypes.c_int64(B), dptr(u_init) if u_init is not None else None,
        dptr(u_out) if u_out is not None else None, dptr(loss), dptr(grad), dptr(iters))
    return loss, grad, iters, u_out


def _perturbed(params):
    inertia, mu, half = params
    return inertia * 1.001, mu * 0.999, half * 1.0005


@pytest.mark.parametrize('name', ['elbow_nominal', 'elbow_perturbed'])
def test_any_start_point_gives_the_cold_loss_and_gradient(name):
    """From zero, from the cold optimum (also in place) and from the optimum of parameters moved by 1e-3 the solves reach
    the cold loss and gradient; the optimum of a free-flight sample is exactly zero, and the cold optimum is a start that
    needs at most one Newton direction.  The solver stops at a scaled gradient of 1e-12, so two start points end within
    that tolerance of the optimum, not on the same bits: losses then agree to 1e-13 of their largest value and the
    gradient, whose contact terms carry the forces' 1/eps, to about 2e-11 of its largest entry."""
    g = load_golden(name)
    params = elbow_kernel_level_params(g)
    B = g['x'].shape[0]
    loss_c, grad_c, it_c, u_c = _loss(g, params, record=True)
    assert np.abs(loss_c - g['loss']).max() < 1e-12
    solved = it_c > 0
    assert 0 < solved.sum() < B                                          # triage and solver both exercised
    assert np.all(u_c[~solved] == 0) and not np.isnan(u_c).any()
    moved = _perturbed(params)
    _, _, _, u_moved = _loss(g, moved, record=True)
    starts = {'zero': np.zeros((B, 7)), 'cold optimum': u_c.copy(), 'moved optimum': u_moved}
    for what, u0 in starts.items():
        loss, grad, iters, u = _loss(g, params, u_init=u0)
        assert np.abs(loss - loss_c).max() <= 1e-12 * np.abs(loss_c).max(), what
        assert max_rel_to_scale(grad, grad_c) < (1e-14 if what == 'cold optimum' else 1e-10), what
        assert max_rel_to_scale(u, u_c) < 1e-11, what
        assert np.all(u[~solved] == 0), what
    _, _, it_same, _ = _loss(g, params, u_init=u_c.copy())
    assert it_same.max() <= 1
    u_buf = u_moved.copy()
    loss, grad, _, u = _loss(g, params, u_init=u_buf, in_place=True)
    assert u is u_buf and max_rel_to_scale(u_buf, u_c) < 1e-9
    assert np.abs(loss - loss_c).max() <= 1e-12 * np.abs(loss_c).max() and max_rel_to_scale(grad, grad_c) < 1e-10
