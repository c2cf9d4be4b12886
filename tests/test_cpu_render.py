"""CPU tests of camera rendering: the camera matrices, a single box against its analytic image, and prb_render's kernel
source (under the SIMT emulator) against the independent numpy ray caster tests/np_render.py."""
import os

import numpy as np
import pytest

import emu_render
import np_render
from emu_lib import EmuSim
from oracle.oracle import Oracle
from roboticsplayroompybullet_b200.camera import (Camera, default_camera, default_palette, gripper_camera,
                                                  projection_matrix_fov, view_matrix, view_matrix_from_yaw_pitch_roll,
                                                  yaw_pitch_eye)
from roboticsplayroompybullet_b200.model import load_model

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
MAX_AMBIGUOUS = 0.02
DEPTH_REL = 1e-5


def _mat(v):
    return np.asarray(v, np.float64).reshape(4, 4).T


def _ndc(P, V, x):
    c = _mat(P) @ _mat(V) @ np.r_[x, 1.0]
    return c[:3] / c[3]


def test_matrix_helpers():
    eye, target, up = np.array([0.4, -1.1, 0.9]), np.array([0.05, 0.2, 0.1]), np.array([0.0, 0.0, 1.0])
    V = view_matrix(eye, target, up)
    P = projection_matrix_fov(55.0, 4 / 3, 0.1, 4.0)
    assert np.allclose(_ndc(P, V, target)[:2], 0.0, atol=1e-6)
    f = (target - eye) / np.linalg.norm(target - eye)
    assert abs(_ndc(P, V, eye + 0.1 * f)[2] + 1.0) < 1e-5           # near plane -> NDC z = -1
    assert abs(_ndc(P, V, eye + 4.0 * f)[2] - 1.0) < 1e-5           # far plane -> +1
    # the view is rigid: eye at the origin, looking down -z
    assert np.allclose(_mat(V) @ np.r_[eye, 1.0], [0, 0, 0, 1], atol=1e-6)
    for yaw, pitch, dist in ((0.0, -30.0, 1.2), (47.0, -65.0, 0.8), (-120.0, 20.0, 2.0)):
        e, u = yaw_pitch_eye(target, dist, yaw, pitch)
        assert abs(np.linalg.norm(e - target) - dist) < 1e-9
        assert np.allclose(view_matrix_from_yaw_pitch_roll(target, dist, yaw, pitch, 0.0), view_matrix(e, target, u), atol=1e-6)
    # yaw 0, pitch -30: the eye is behind the target along -y and above it
    e, _ = yaw_pitch_eye(target, 1.0, 0.0, -30.0)
    assert np.allclose(e - target, [0.0, -np.cos(np.radians(30)), 0.5], atol=1e-9)


def test_single_box_depth_and_silhouette():
    """UR5Reach's ground plane (a thin 4 m box) seen from below fills the view at the analytic depth; the
    same collider turned into a cube of half extent h at distance D straight ahead: centre depth D - h, and the
    silhouette within one perimeter of the analytic square."""
    m = load_model('UR5Reach-v0')
    n = int(m['n_col'])
    ground = [c for c in range(n) if m['col_body'][c] < 0][0]
    gz = float(m['col_pos'].reshape(n, 3)[ground][2])
    dist, W = 0.8, 64
    eye = np.array([0.0, 0.0, gz - dist])
    cam = Camera(W, W, view_matrix(eye, eye + [0, 0, 1.0], [0, 1.0, 0]), projection_matrix_fov(60.0, 1.0, 0.05, 5.0))
    sim = EmuSim(m, 1)
    out = emu_render.render(m, sim.state, cam, default_palette(m), depth=True, segmentation=True)
    assert (out['segmentation'][0] == ground).all()
    below = dist - float(m['col_half'].reshape(n, 3)[ground][2])         # underside of the plate
    assert np.abs(out['depth'][0] - below).max() < 1e-5 * below

    D, h = 0.6, 0.05
    m.d['col_pos'] = m['col_pos'].copy()
    m.d['col_half'] = m['col_half'].copy()
    m.d['col_pos'].reshape(n, 3)[ground] = eye + [0.0, 0.0, D]
    m.d['col_half'].reshape(n, 3)[ground] = [h, h, h]
    sim = EmuSim(m, 1)
    out = emu_render.render(m, sim.state, cam, default_palette(m), depth=True, segmentation=True)
    seg, depth = out['segmentation'][0], out['depth'][0]
    assert abs(depth[W // 2, W // 2] - (D - h)) < 1e-5 * (D - h)
    assert np.allclose(depth[seg < 0], 5.0, rtol=1e-5)              # background: the far plane
    # front face: a square of side 2h at depth D - h, W / (2 (D - h) tan 30deg) pixels per metre there
    side_px = 2 * h * W / (2 * (D - h) * np.tan(np.radians(30)))
    assert abs((seg == ground).sum() - side_px ** 2) <= 4 * side_px


def _states(env_id, n, seed):
    m = load_model(env_id)
    out = []
    for i in range(n):
        o = Oracle(m, seed=seed + i)
        o.reset()
        out.append(np.asarray(o.state, np.float32))
    return m, np.stack(out)


def _check(m, states, cams):
    sim = EmuSim(m, len(states))
    sim.state[:, :sim.state_dim] = states
    pal = default_palette(m)
    before = sim.state.copy()
    for cam in cams:
        out = emu_render.render(m, sim.state, cam, pal, depth=True, segmentation=True)
        for i in range(len(states)):
            ref = np_render.render(m, states[i], cam, pal)
            r = np_render.compare((out['rgb'][i], out['depth'][i], out['segmentation'][i]), ref)
            assert r['seg_mismatch'] == 0, r
            assert r['ambiguous'] <= MAX_AMBIGUOUS, r
            assert r['depth_rel'] <= DEPTH_REL, r
            assert r['rgb'] <= 1, r
    assert before.tobytes() == sim.state.tobytes()          # read only


@pytest.mark.parametrize('env_id', ['UR5PlayAbsRPY1Obj-v0', 'pandaPick-v0', 'UR5Reach-v0'])
def test_emu_render_matches_numpy_reset_states(env_id):
    m, states = _states(env_id, 3, seed=11)
    _check(m, states, [default_camera(m, 48, 48), gripper_camera(m, 48, 48)])


@pytest.mark.parametrize('golden', ['heavy_step_r1.npz', 'many_contacts.npz'])
def test_emu_render_matches_numpy_golden_states(golden):
    """Stored play states with the fingers closed on the block and many contacts (tests/golden)."""
    m = load_model('UR5PlayAbsRPY1Obj-v0')
    st = np.load(os.path.join(GOLDEN, golden))['state'][:6]
    _check(m, st, [default_camera(m, 48, 48), gripper_camera(m, 48, 48)])


def _visible_bodies(env_id, seed=5, size=96):
    m, st = _states(env_id, 1, seed)
    sim = EmuSim(m, 1)
    sim.state[:, :sim.state_dim] = st
    seg = emu_render.render(m, sim.state, default_camera(m, size, size), default_palette(m), segmentation=True)['segmentation'][0]
    return m, set(np.unique(seg).tolist()) - {-1}


def test_default_camera_shows_the_play_scene():
    m, seen = _visible_bodies('UR5PlayAbsRPY1Obj-v0')
    n = int(m['n_col'])
    body, half = np.asarray(m['col_body']), m['col_half'].reshape(n, 3)
    static = [c for c in range(n) if body[c] < 0 and half[c].max() < 1.0]
    table_top = max(static, key=lambda c: half[c][0] * half[c][1] if half[c][2] < 0.01 else 0)
    assert table_top in seen
    for b in range(1, 1 + int(m['n_free']) + int(m['n_slide'])):    # block, drawer, door, button, dial
        assert any(body[c] == b for c in seen), b
    assert any(body[c] == 0 for c in seen)                           # the arm


def test_default_camera_shows_the_pick_scene():
    m, seen = _visible_bodies('pandaPick-v0')
    n = int(m['n_col'])
    body, half, pos = np.asarray(m['col_body']), m['col_half'].reshape(n, 3), m['col_pos'].reshape(n, 3)
    ground = [c for c in range(n) if body[c] < 0 and half[c].max() >= 1.0][0]
    # the tray's four walls; its floor lies below the ground plane's top
    tray = [c for c in range(n) if body[c] < 0 and c != ground and pos[c][2] + half[c][2] > pos[ground][2] + half[ground][2]]
    assert len(tray) == 4 and all(c in seen for c in tray), (tray, seen)
    assert any(body[c] == 1 for c in seen)                           # the cube
    gripper = [c for c in range(n) if body[c] == 0 and m['col_link'][c] >= m['site_link'][0]]   # hand and fingers
    assert any(c in seen for c in gripper)


def test_emu_render_rejects_bad_cameras():
    m = load_model('UR5Reach-v0')
    sim = EmuSim(m, 1)
    pal = default_palette(m)
    good = default_camera(m, 16, 16)
    bad = [Camera(0, 16, good.view, good.proj), Camera(16, 1025, good.view, good.proj),
           Camera(16, 16, np.zeros(16), good.proj), Camera(16, 16, good.view, np.zeros(16)),
           Camera(16, 16, good.view, good.proj, light_dir=(0, 0, 0))]
    for cam in bad:
        with pytest.raises(ValueError):
            emu_render.render(m, sim.state, cam, pal)
    emu_render.render(m, sim.state, good, pal)
