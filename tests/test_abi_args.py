"""Argument checks of the C ABI: every ``dpll_*`` entry point is called through ctypes with invalid argument sets and
must return its exact code (``DPLL_EINVAL``, ``DPLL_EWORKSPACE``) or, for an empty batch it returns early from,
``DPLL_OK``.  Every call is rejected (or returns) before its pointers are used, so only NULL or a host scratch buffer is
passed, and ``comm`` is always NULL (a non-NULL ``comm`` is dereferenced on the host).  The calls run in a subprocess
in which no CUDA device is visible, so no call can reach a GPU whatever the library does."""
import json
import os
import re
import shutil
import subprocess
import sys

import pytest

from dair_pll_b200 import _lib
from dair_pll_b200 import build as _build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, EINVAL, EWORKSPACE = 0, -1, -2
DYNAMIC = 1
WS = 606352              # dpll_workspace_bytes(): per-block partials, prepared parameters, chunk counter

# Arguments of the base call of every entry point, by parameter name (header names).  Pointers not listed here get
# the host scratch buffer; the cases below override single arguments.
BASE = dict(B=16, D=16, n=16, capacity=16, steps=1, n_links=3, n_boxes=1, n_contacts=4, n_pts_packed=0, flags=0,
            x_row_stride=13, xp_row_stride=13, q_stride=8, n_query=4, W=256, ldk=128, slope=0.01, dt=0.01, eps=1e-6,
            workspace_bytes=WS, n_bodies=1, n_pairs=1, n_len=1, n_geoms=1, blocks=1, iters=1, rank=0, world=1, scale=1.0,
            comm=None, stream=None, skip_flag=None, u_init=None, u_out=None)

N = None
# (entry point, overrides, expected code); an entry point name ending in '*' stands for its _f64 and _f32 pair
CASES = [
    ('dpll_set_loss_variant', dict(variant=3), EINVAL),
    ('dpll_set_loss_variant', dict(variant=-1), EINVAL),
    # the single box
    *[(f'dpll_cube_loss*', o, e) for o, e in [
        (dict(x=N), EINVAL), (dict(x_plus=N), EINVAL), (dict(inertia=N), EINVAL), (dict(mu_pair=N), EINVAL),
        (dict(half=N), EINVAL), (dict(B=-1), EINVAL), (dict(workspace_bytes=WS - 1), EWORKSPACE),
        (dict(workspace=N), EWORKSPACE), (dict(grad=N, workspace_bytes=WS - 1), EWORKSPACE)]],
    *[(f'dpll_cube_loss_leaf*', o, e) for o, e in [
        (dict(theta=N), EINVAL), (dict(friction=N), EINVAL), (dict(length=N), EINVAL), (dict(x=N), EINVAL),
        (dict(B=-1), EINVAL), (dict(grad_leaf=N, loss_sum=N, workspace_bytes=WS - 1), EWORKSPACE),
        (dict(workspace=N), EWORKSPACE)]],
    *[(f'dpll_cube_loss_leaf_dp*', o, e) for o, e in [
        (dict(x_row_stride=12), EINVAL), (dict(xp_row_stride=12), EINVAL), (dict(sums=N, means=N), EINVAL),
        (dict(theta=N), EINVAL), (dict(B=-1), EINVAL), (dict(x_plus=N), EINVAL),
        (dict(workspace_bytes=WS - 1), EWORKSPACE), (dict(sums=N, workspace=N), EWORKSPACE),
        (dict(loss_variant=1, u_init='P'), EINVAL), (dict(loss_variant=1, u_out='P'), EINVAL)]],
    *[(f'dpll_cube_rollout*', o, e) for o, e in [
        (dict(B=-1), EINVAL), (dict(steps=-1), EINVAL), (dict(x0=N), EINVAL), (dict(traj=N), EINVAL),
        (dict(inertia=N), EINVAL), (dict(B=0), OK)]],
    ('dpll_cube_rollout_saved_f64', dict(usol=N), EINVAL),
    ('dpll_cube_rollout_saved_f64', dict(steps=-1), EINVAL),
    ('dpll_cube_rollout_saved_f64', dict(B=0), OK),
    ('dpll_cube_rollout_grad_f64', dict(B=-1), EINVAL),
    ('dpll_cube_rollout_grad_f64', dict(steps=-1), EINVAL),
    ('dpll_cube_rollout_grad_f64', dict(xbar=N), EINVAL),
    ('dpll_cube_rollout_grad_f64', dict(half=N), EINVAL),
    ('dpll_cube_rollout_grad_f64', dict(B=0), OK),
    ('dpll_cube_rollout_backward_f64', dict(B=-1), EINVAL),
    ('dpll_cube_rollout_backward_f64', dict(steps=-1), EINVAL),
    ('dpll_cube_rollout_backward_f64', dict(usol=N), EINVAL),
    ('dpll_cube_rollout_backward_f64', dict(traj=N), EINVAL),
    ('dpll_cube_rollout_backward_f64', dict(B=0), OK),
    ('dpll_cube_terms_f64', dict(B=-1), EINVAL),
    ('dpll_cube_terms_f64', dict(M=N), EINVAL),
    ('dpll_cube_terms_f64', dict(half=N), EINVAL),
    ('dpll_cube_terms_f64', dict(B=0), OK),
    # the single body with witness points
    *[('dpll_body_loss_pts_f64', o, e) for o, e in [
        (dict(n_contacts=0), EINVAL), (dict(n_contacts=5), EINVAL), (dict(B=-1), EINVAL), (dict(x=N), EINVAL),
        (dict(pts=N), EINVAL), (dict(inertia=N), EINVAL), (dict(workspace_bytes=WS - 1), EWORKSPACE),
        (dict(grad=N, loss_sum=N, flags=DYNAMIC, workspace_bytes=WS - 1), EWORKSPACE)]],
    ('dpll_body_step_pts_f64', dict(n_contacts=0), EINVAL),
    ('dpll_body_step_pts_f64', dict(n_contacts=5), EINVAL),
    ('dpll_body_step_pts_f64', dict(B=-1), EINVAL),
    ('dpll_body_step_pts_f64', dict(x_next=N), EINVAL),
    ('dpll_body_step_pts_f64', dict(B=0), OK),
    ('dpll_body_step_pts_grad_f64', dict(n_contacts=-1), EINVAL),
    ('dpll_body_step_pts_grad_f64', dict(n_contacts=5), EINVAL),
    ('dpll_body_step_pts_grad_f64', dict(gpts=N), EINVAL),
    ('dpll_body_step_pts_grad_f64', dict(B=0), OK),
    ('dpll_body_support_directions_f64', dict(q_stride=3), EINVAL),
    ('dpll_body_support_directions_f64', dict(n_query=0), EINVAL),
    ('dpll_body_support_directions_f64', dict(dirs=N), EINVAL),
    ('dpll_body_support_directions_f64', dict(B=0), OK),
    # the two-body tree
    *[(f'dpll_elbow_loss*', o, e) for o, e in [
        (dict(B=-1), EINVAL), (dict(x=N), EINVAL), (dict(kin=N), EINVAL), (dict(half=N, pts=N), EINVAL),
        (dict(pts=N), EINVAL), (dict(grad=N), EINVAL), (dict(workspace_bytes=WS - 1), EWORKSPACE),
        (dict(grad_pts=N, grad=N, loss_sum=N, flags=DYNAMIC, workspace=N), EWORKSPACE)]],
    *[(f'dpll_elbow_rollout*', o, e) for o, e in [
        (dict(B=-1), EINVAL), (dict(steps=-1), EINVAL), (dict(steps=2), EINVAL), (dict(x0=N), EINVAL),
        (dict(half=N, pts=N), EINVAL), (dict(pts=N, B=0), OK)]],
    ('dpll_elbow_rollout_saved_f64', dict(pts=N, usol=N), EINVAL),
    ('dpll_elbow_rollout_saved_f64', dict(pts=N, kin=N), EINVAL),
    ('dpll_elbow_rollout_saved_f64', dict(B=0), OK),
    ('dpll_elbow_rollout_grad_saved_f64', dict(steps=-1), EINVAL),
    ('dpll_elbow_rollout_grad_saved_f64', dict(gx0=N), EINVAL),
    ('dpll_elbow_rollout_grad_saved_f64', dict(B=0), OK),
    ('dpll_elbow_step_pts_grad_f64', dict(B=-1), EINVAL),
    ('dpll_elbow_step_pts_grad_f64', dict(pts=N), EINVAL),
    ('dpll_elbow_step_pts_grad_f64', dict(B=0), OK),
    ('dpll_elbow_terms_f64', dict(kin=N), EINVAL),
    ('dpll_elbow_terms_f64', dict(q=N), EINVAL),
    ('dpll_elbow_terms_f64', dict(B=0), OK),
    ('dpll_elbow_support_directions_f64', dict(q_stride=7), EINVAL),
    ('dpll_elbow_support_directions_f64', dict(pert1=N), EINVAL),
    ('dpll_elbow_support_directions_f64', dict(B=0), OK),
    # generic chains
    *[('dpll_chain_loss_f64', o, e) for o, e in [
        (dict(n_links=1), EINVAL), (dict(n_links=7), EINVAL), (dict(B=-1), EINVAL), (dict(x=N), EINVAL),
        (dict(half=N), EINVAL), (dict(workspace_bytes=WS - 1), EWORKSPACE),
        (dict(n_links=7, workspace_bytes=WS - 1), EINVAL)]],
    *[('dpll_chain_loss_pts_f64', o, e) for o, e in [
        (dict(n_links=1), EINVAL), (dict(n_links=7), EINVAL), (dict(B=-1), EINVAL), (dict(pts=N), EINVAL),
        (dict(workspace_bytes=WS - 1), EWORKSPACE), (dict(n_links=7, B=0), OK)]],
    *[(f'dpll_chain_{fn}_f64', o, e) for fn in ('rollout', 'rollout_grad') for o, e in [
        (dict(n_links=1), EINVAL), (dict(n_links=7), EINVAL), (dict(B=-1), EINVAL), (dict(steps=-1), EINVAL),
        (dict(x0=N), EINVAL), (dict(n_links=7, B=0), OK)]],
    *[('dpll_chain_terms_f64', o, e) for o, e in [
        (dict(n_boxes=4), EINVAL), (dict(n_boxes=0), EINVAL), (dict(n_links=7, n_boxes=1), EINVAL),
        (dict(n_links=1, n_boxes=1), EINVAL), (dict(B=-1), EINVAL), (dict(acc=N), EINVAL), (dict(B=0), OK)]],
    # parameter preparation
    ('dpll_leaf_prepare_f64', dict(n_bodies=-1), EINVAL),
    ('dpll_leaf_prepare_f64', dict(theta=N), EINVAL),
    ('dpll_leaf_prepare_f64', dict(pair_b=N), EINVAL),
    ('dpll_leaf_backward_f64', dict(n_geoms=-1), EINVAL),
    ('dpll_leaf_backward_f64', dict(g_friction=N), EINVAL),
    # support network
    ('dpll_icnn_input_f64', dict(D=-1), EINVAL),
    ('dpll_icnn_input_f64', dict(W=0), EINVAL),
    ('dpll_icnn_input_f64', dict(d=N), EINVAL),
    ('dpll_icnn_input_f64', dict(D=0), OK),
    ('dpll_icnn_mask_f64', dict(n=-1), EINVAL),
    ('dpll_icnn_mask_f64', dict(z=N), EINVAL),
    ('dpll_icnn_mask_f64', dict(n=0), OK),
    ('dpll_icnn_output_f64', dict(W=0), EINVAL),
    ('dpll_icnn_output_f64', dict(m1=N), EINVAL),
    ('dpll_icnn_output_f64', dict(D=0), OK),
    ('dpll_icnn_backward_f64', dict(D=-1), EINVAL),
    ('dpll_icnn_backward_f64', dict(part=N), EINVAL),
    ('dpll_icnn_backward_f64', dict(D=0), OK),
    ('dpll_icnn_tc_prepare_f64', dict(W=128), EINVAL),
    ('dpll_icnn_tc_prepare_f64', dict(image=N), EINVAL),
    ('dpll_icnn_tc_support_f64', dict(W=128), EINVAL),
    ('dpll_icnn_tc_support_f64', dict(D=-1), EINVAL),
    ('dpll_icnn_tc_support_f64', dict(p=N), EINVAL),
    ('dpll_icnn_tc_support_f64', dict(D=0), OK),
    ('dpll_icnn_tc_record_f64', dict(ldk=100), EINVAL),
    ('dpll_icnn_tc_record_f64', dict(capacity=256), EINVAL),
    ('dpll_icnn_tc_record_f64', dict(n_rows=N), EINVAL),
    ('dpll_icnn_tc_record_f64', dict(m0t=N), EINVAL),
    ('dpll_icnn_tc_record_f64', dict(capacity=0), OK),
    ('dpll_icnn_tc_bwd_f64', dict(ldk=0), EINVAL),
    ('dpll_icnn_tc_bwd_f64', dict(ldk=100), EINVAL),
    ('dpll_icnn_tc_bwd_f64', dict(ldk=128 * 10 ** 7), EINVAL),
    ('dpll_icnn_tc_bwd_f64', dict(C=N), EINVAL),
    # data-parallel exchange
    ('dpll_comm_create', dict(world=0), EINVAL),
    ('dpll_comm_create', dict(rank=1), EINVAL),
    ('dpll_comm_create', dict(comm_out=N), EINVAL),
    ('dpll_comm_connect', dict(), EINVAL),
    ('dpll_comm_destroy', dict(), EINVAL),
    ('dpll_comm_error', dict(), EINVAL),
    ('dpll_comm_allreduce_f64', dict(), EINVAL),
    # peak-rate probe
    *[(f'dpll_fma_peak*', o, e) for o, e in [
        (dict(out=N), EINVAL), (dict(blocks=0), EINVAL), (dict(iters=-1), EINVAL)]],
]


def _expand(cases):
    out = []
    for name, over, code in cases:
        names = [name[:-1] + s for s in ('_f64', '_f32')] if name.endswith('*') else [name]
        out += [(n, over, code) for n in names]
    return out


def _param_names():
    """name -> parameter names of every dpll_* prototype of the C header."""
    with open(_lib.HEADER) as f:
        text = re.sub(r'/\*.*?\*/|//[^\n]*', ' ', f.read(), flags=re.S)
    out = {}
    for name, params in re.findall(r'\b(dpll_\w+)\s*\(([^)]*)\)\s*;', text):
        out[name] = [re.split(r'[\s*]+', p.strip())[-1] for p in params.split(',') if p.strip() not in ('', 'void')]
    return out


# Runs in the subprocess: loads the library, makes each call, prints the return codes as JSON.
_RUNNER = r'''
import ctypes, json, sys
from dair_pll_b200 import _lib
lib = _lib.load()
calls = json.load(sys.stdin)
scratch = ctypes.create_string_buffer(1 << 16)
P = ctypes.addressof(scratch)
out = {"workspace_bytes": lib.dpll_workspace_bytes(), "version": lib.dpll_version(), "codes": []}
for name, args, variant in calls:
    if variant is not None:
        assert lib.dpll_set_loss_variant(variant) == 0
    fn = getattr(lib, name)
    args = [(P if t is ctypes.c_void_p else ctypes.cast(P, t)) if a == "P" else a for a, t in zip(args, fn.argtypes)]
    out["codes"].append(fn(*args))
    if variant is not None:
        assert lib.dpll_set_loss_variant(0) == 0
print(json.dumps(out))
'''


def _library():
    path = _lib.lib_path()
    if path == _build.LIB_PATH and _build.is_stale():
        if not _build.sources_present() or shutil.which(_build._nvcc()) is None:
            pytest.skip('the CUDA library is not built and nvcc is absent')
        _build.build()
    if not os.path.exists(path):
        pytest.skip(f'{path} not found')
    return path


@pytest.fixture(scope='module')
def results():
    _library()
    names = _param_names()
    calls, expected = [], []
    for name, over, code in _expand(CASES):
        params = names[name]
        assert set(over) - {'loss_variant'} <= set(params), (name, over)
        args = []
        for p in params:
            v = over.get(p, BASE.get(p, 'P'))
            args.append(v)
        calls.append((name, args, over.get('loss_variant')))
        expected.append(code)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    proc = subprocess.run([sys.executable, '-c', _RUNNER], input=json.dumps(calls), capture_output=True, text=True,
                          cwd=ROOT, env=env, timeout=300)
    assert proc.returncode == 0, proc.stderr
    return json.loads(proc.stdout.strip().splitlines()[-1]), calls, expected


def test_invalid_arguments_return_their_codes(results):
    out, calls, expected = results
    bad = [(name, args, want, got) for (name, args, _), want, got in zip(calls, expected, out['codes']) if want != got]
    assert not bad, '\n'.join(f'{n}{tuple(a)}: expected {w}, got {g}' for n, a, w, g in bad)


def test_every_entry_point_with_arguments_is_covered():
    covered = {n for n, _, _ in _expand(CASES)}
    no_args = {n for n, p in _param_names().items() if not p}
    rest = set(_param_names()) - covered - no_args - {'dpll_comm_device_state', 'dpll_icnn_backward_blocks'}
    assert not rest, sorted(rest)


def test_workspace_bytes(results):
    out, _, _ = results
    assert out['workspace_bytes'] == WS
    assert out['version'] == _lib.ABI_VERSION
