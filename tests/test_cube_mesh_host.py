"""Single floating body with learned (mesh) geometry, on the host: the cube-mesh asset and the witness-point pieces of the
wavefront loss kernel (cn_cube.cuh: body_loss_{free_flight,prologue,epilogue}_pts) composed per sample by the host
emulation (tests/host_emul/emul_body_pts_wf.cpp), against body_loss_sample_pts and the reference goldens of the Sphere / Polygon / framed-box shapes."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from oracle import contactnets_oracle as co
from tests.util import ROOT, dptr, host_emulation_lib, load_golden, max_rel_to_scale

ASSETS = os.path.join(ROOT, 'dair_pll_b200', 'assets')
_WF_LIB = None


def wf_emulation_lib():
    """g++ build of tests/host_emul/emul_body_pts_wf.cpp (the kernel's witness-point pieces composed per sample), with the
    flags of the main host emulation library."""
    global _WF_LIB
    if _WF_LIB is None:
        out = os.path.join(tempfile.gettempdir(), f'dpll_emul_body_pts_wf_{os.getuid()}.so')
        src = os.path.join(ROOT, 'tests', 'host_emul', 'emul_body_pts_wf.cpp')
        gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
        subprocess.check_call([gxx, '-O2', '-std=c++17', '-fPIC', '-shared', '-ffp-contract=off', '-o', out, src])
        _WF_LIB = ctypes.CDLL(out)
    return _WF_LIB


def test_cube_mesh_urdf_parses_to_single_body_with_learned_geometry():
    from dair_pll_b200.geometry import DeepSupportConvex
    from dair_pll_b200.multibody_terms import MultibodyTerms
    from dair_pll_b200.system_spec import SystemSpec
    spec = SystemSpec.from_urdfs({'cube': os.path.join(ASSETS, 'cube_mesh.urdf')})
    assert spec.kind == 'cube'
    body_geoms = [g for g in spec.geometries if g.body >= 0]
    assert [g.kind for g in body_geoms] == ['mesh']
    assert spec.n_contacts == 4
    verts = body_geoms[0].mesh_vertices()
    assert verts.shape == (8, 3) and torch.allclose(verts.abs(), torch.full((8, 3), 0.0524, dtype=torch.float64))
    mt = MultibodyTerms({'cube': os.path.join(ASSETS, 'cube_mesh.urdf')})
    ct = mt.contact_terms
    assert isinstance(ct.geometries[0], DeepSupportConvex) and ct.has_witness_point_geometry()
    assert ct.geometries[0].n_query == 4
    # the reference's parameter names for a DeepSupportConvex body (geometry.py:255-325, deep_support_function.py:125-186)
    assert sorted(mt.state_dict().keys()) == sorted([
        'lagrangian_terms.inertial_parameters', 'contact_terms.friction_params',
        'contact_terms.geometries.0.network.hidden_weights.0', 'contact_terms.geometries.0.network.input_weights.0',
        'contact_terms.geometries.0.network.input_weights.1', 'contact_terms.geometries.0.network.output_weight'])


def _shape_inputs(name):
    """golden states, kernel-level parameters and the shape's witness points at x+ and x (host torch)"""
    from dair_pll_b200.geometry import Box, Polygon, Sphere, place_in_link_frame
    g = load_golden(name)
    p = torch.from_numpy(g['shape_param'])
    if name == 'shape_framed_box':
        from oracle.callables import FRAMED_BODY_TREE as tree
        geom = Box(p.reshape(3), 4)
        geom.set_frame(torch.tensor(tree.geometry_offset[0], dtype=torch.float64), tree.geometry_rotation(0, torch.float64))
    else:
        geom = Sphere(p) if name == 'shape_sphere' else Polygon(p, 4)
    theta = torch.from_numpy(g['theta'])
    inertia = co.theta_to_inertia_vector(theta).reshape(10).numpy().copy()
    m = np.abs(g['friction_params'])
    mu = np.array([2 * m[0] * m[1] / (m[0] + m[1])])
    x, xp = np.ascontiguousarray(g['x']), np.ascontiguousarray(g['x_plus'])

    def witness(states):
        w, a, b, c = torch.from_numpy(states[:, :4]).unbind(-1)
        s = 2.0 / (w * w + a * a + b * b + c * c)
        d = -torch.stack((s * (a * c - w * b), s * (b * c + w * a), 1 - s * (a * a + b * b)), -1)
        pts = place_in_link_frame(geom, d).detach()
        n_c = pts.shape[-2]
        if n_c < 4:
            pts = torch.cat((pts, pts.new_zeros(pts.shape[0], 4 - n_c, 3)), -2)
        return np.ascontiguousarray(pts.numpy()), n_c
    pts, n_c = witness(xp)
    return g, x, xp, inertia, mu, pts, n_c


def _run(fn_name, x, xp, inertia, mu, pts, n_c, dt, flags=None):
    lib = wf_emulation_lib() if fn_name == 'emul_body_loss_pts_wf_f64' else host_emulation_lib()
    B = x.shape[0]
    loss, g11, gp = np.zeros(B), np.zeros(11), np.zeros((B, 4, 3))
    args = [dptr(x), dptr(xp), dptr(inertia), dptr(mu), dptr(pts), ctypes.c_int(n_c), ctypes.c_double(dt),
            ctypes.c_double(1e-3), ctypes.c_int64(B), dptr(loss), dptr(g11), dptr(gp)]
    if fn_name == 'emul_body_loss_pts_wf_f64':
        args.append(dptr(flags) if flags is not None else None)
    getattr(lib, fn_name)(*args)
    return loss, g11, gp


@pytest.mark.parametrize('name', ['shape_sphere', 'shape_polygon', 'shape_framed_box'])
def test_wavefront_pts_pieces_match_generic_path_and_golden(name):
    """The per-sample composition the PTS instance of the wavefront kernel runs (triage, prologue, feasible-segment start,
    Newton visits, epilogue) against body_loss_sample_pts (Newton from u = 0, one pass) and the reference golden."""
    g, x, xp, inertia, mu, pts, n_c = _shape_inputs(name)
    dt = float(g['dt'])
    B = x.shape[0]
    flags = np.zeros(B, np.int32)
    loss_w, g_w, gp_w = _run('emul_body_loss_pts_wf_f64', x, xp, inertia, mu, pts, n_c, dt, flags)
    loss_r, g_r, gp_r = _run('emul_body_loss_pts_f64', x, xp, inertia, mu, pts, n_c, dt)
    assert np.abs(loss_w - loss_r).max() < 1e-12
    assert np.abs(loss_w - g['loss']).max() < 1e-12
    assert max_rel_to_scale(g_w, g_r) < 1e-9
    assert max_rel_to_scale(gp_w, gp_r) < 1e-9
    assert np.all(gp_w[:, n_c:] == 0)
    assert 0 < flags.sum() < B                    # both the free-flight triage and the solver are exercised


@pytest.mark.parametrize('n_c', [1, 2, 3, 4])
def test_wavefront_pts_pieces_every_contact_count(n_c):
    """n_contacts 1..4: the first n_c of the Polygon's four witness points; the rows beyond are switched off."""
    g, x, xp, inertia, mu, pts, _ = _shape_inputs('shape_polygon')
    pts = np.ascontiguousarray(pts.copy())
    pts[:, n_c:] = 0.0
    dt = float(g['dt'])
    loss_w, g_w, gp_w = _run('emul_body_loss_pts_wf_f64', x, xp, inertia, mu, pts, n_c, dt)
    loss_r, g_r, gp_r = _run('emul_body_loss_pts_f64', x, xp, inertia, mu, pts, n_c, dt)
    assert np.abs(loss_w - loss_r).max() < 1e-12
    assert max_rel_to_scale(g_w, g_r) < 1e-9
    assert max_rel_to_scale(gp_w, gp_r) < 1e-9
    assert np.all(gp_w[:, n_c:] == 0) and np.abs(gp_w[:, :n_c]).max() > 0


def test_free_flight_triage_equals_generic_path_on_flight_samples():
    """On samples the triage finalises, its loss, parameter gradient and grad_pts equal the generic path's."""
    g, x, xp, inertia, mu, pts, n_c = _shape_inputs('shape_polygon')
    xp = xp.copy()
    xp[:40, 6] -= 0.05                              # some penetrations: the flight test must still hold exactly
    xp = np.ascontiguousarray(xp)
    dt = float(g['dt'])
    B = x.shape[0]
    flags = np.zeros(B, np.int32)
    _run('emul_body_loss_pts_wf_f64', x, xp, inertia, mu, pts, n_c, dt, flags)
    free = flags == 1
    assert 0 < free.sum() < B
    xs, xps, ps = (np.ascontiguousarray(a[free]) for a in (x, xp, pts))
    loss_w, g_w, gp_w = _run('emul_body_loss_pts_wf_f64', xs, xps, inertia, mu, ps, n_c, dt)
    loss_r, g_r, gp_r = _run('emul_body_loss_pts_f64', xs, xps, inertia, mu, ps, n_c, dt)
    assert np.abs(loss_w - loss_r).max() <= 1e-14 * np.abs(loss_r).max()
    assert np.abs(g_w - g_r).max() <= 1e-12 * np.abs(g_r).max()
    assert np.abs(gp_w - gp_r).max() <= 1e-12 * np.abs(gp_r).max()
    assert np.abs(gp_r).max() > 0                  # the penetration term is exercised
