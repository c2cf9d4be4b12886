"""CPU tests of ray casting (prb_ray_test): its kernel source (csrc/prb_rays.cuh, under the SIMT emulator) against the
independent numpy reference tests/np_rays.py, known answers on a single box, the gripper_proprioception ray of the
step, the camera's segmentation, launch shapes, invalid input, and the Python surface's checks."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import emu_rays
import emu_render
import np_rays
import np_render
from emu_lib import EmuSim
from helpers import random_actions
from oracle.oracle import Oracle
from roboticsplayroompybullet_b200 import lib
from roboticsplayroompybullet_b200.camera import default_camera, default_palette
from roboticsplayroompybullet_b200.envs import check_rays
from roboticsplayroompybullet_b200.model import load_model

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
PLAY = 'UR5PlayAbsRPY1Obj-v0'


def _states(env_id, n, seed):
    m = load_model(env_id)
    out = []
    for i in range(n):
        o = Oracle(m, seed=seed + i)
        o.reset()
        out.append(np.asarray(o.state, np.float32))
    return m, np.stack(out)


def _got(out, i):
    return out['collider'][i], out['fraction'][i], out['position'][i], out['normal'][i]


def _check_sets(m, states, seed=0):
    """The three ray sets on every state: the emulated kernel against np_rays (CPU criterion 4).  The 2 % cap on
    ambiguous rays holds per ray set over all states: two boxes with coplanar faces (a block resting flush on another)
    tie exactly, which can make a few rays of one small set in one env ambiguous."""
    rng = np.random.default_rng(seed)
    N = len(states)
    rnd = [np_rays.random_segments(m, states[i], 256, rng) for i in range(N)]
    ff, ft = np_rays.site_fan()
    hf, ht = np_rays.height_scan(m)
    sets = [(np.stack([r[0] for r in rnd]), np.stack([r[1] for r in rnd]), None), (ff, ft, 0), (hf, ht, None)]
    for frm, to, site in sets:
        out = emu_rays.ray_test(m, states, frm, to, site=site)
        amb = []
        for i in range(N):
            f, t = (frm[i], to[i]) if frm.ndim == 3 else (frm, to)
            amb.append(np_rays.assert_agrees(_got(out, i), np_rays.ray_test(m, states[i], f, t, site=site), None)['ambiguous'])
        assert np.mean(amb) <= 0.02, amb
    assert (out['collider'] >= 0).mean() > 0.9                 # the height scan lies over the table


@pytest.mark.parametrize('env_id', [PLAY, 'pandaPick-v0', 'UR5Reach-v0'])
def test_emu_rays_match_numpy_reset_states(env_id):
    m, states = _states(env_id, 3, seed=41)
    _check_sets(m, states)


@pytest.mark.parametrize('golden', ['heavy_step_r1.npz', 'many_contacts.npz'])
def test_emu_rays_match_numpy_golden_states(golden):
    m = load_model(PLAY)
    _check_sets(m, np.load(os.path.join(GOLDEN, golden))['state'][:6], seed=1)


# ------------------------------------------------------------------ known answers on one box
C, H = np.array([0.25, -0.5, 1.0]), 0.0625       # exact in fp32: box coordinates are exact for axis-aligned rays


def _one_box():
    """UR5Reach with its ground plane turned into an axis-aligned cube of half extent H at C; (model, state, its index)."""
    m = load_model('UR5Reach-v0')
    n = int(m['n_col'])
    box = [c for c in range(n) if m['col_body'][c] < 0][0]
    for k in ('col_pos', 'col_half', 'col_rot'):
        m.d[k] = m[k].copy()
    m.d['col_pos'].reshape(n, 3)[box] = C
    m.d['col_half'].reshape(n, 3)[box] = H
    m.d['col_rot'].reshape(n, 3, 3)[box] = np.eye(3)
    sim = EmuSim(m, 1)
    return m, sim.state[:, :sim.state_dim].copy(), box


def test_known_answers_single_box():
    m, st, box = _one_box()
    mask = 1 << box
    nan = np.nan
    # from, to (relative to C), expected collider hit, fraction, normal
    cases = [
        ((0, 0, -0.5), (0, 0, 0.5), True, (0.5 - H) / 1.0, (0, 0, -1)),               # axis-aligned, from below
        ((0.5, 0, 0), (-0.5, 0, 0), True, (0.5 - H) / 1.0, (1, 0, 0)),                # axis-aligned, from +x
        ((-0.5, -0.1, 0.05), (0.5, 0.1, -0.05), True, (0.5 - H) / 1.0, (-1, 0, 0)),    # oblique through the -x face
        ((0, 0, 0), (0.3, 0.1, 0.0), True, 0.0, None),                                  # start inside: 0, -direction
        ((-0.5, 0, H), (0.5, 0, H), True, (0.5 - H) / 1.0, (-1, 0, 0)),                 # parallel, in the +z face plane
        ((-0.5, 0, H + 1e-3), (0.5, 0, H + 1e-3), False, None, None),                   # parallel, just above it
        ((0.01, 0.02, 0.03), (0.01, 0.02, 0.03), True, 0.0, (0, 0, 0)),                # zero length, inside
        ((0, 0, 0.5), (0, 0, 0.5), False, None, None),                                  # zero length, outside
        ((0, 0, -0.5), (0, 0, -H), False, None, None),                                  # the hit exactly at `to`
        ((0, 0, -0.5), (0, 0, -H + 1e-3), True, (0.5 - H) / (0.5 - H + 1e-3), (0, 0, -1)),
        ((nan, 0, -0.5), (0, 0, 0.5), False, None, None),                               # non-finite endpoint
        ((0, 0, -0.5), (0, np.inf, 0.5), False, None, None),
    ]
    frm = np.array([C + np.array(c[0], float) for c in cases])
    to = np.array([C + np.array(c[1], float) for c in cases])
    out = emu_rays.ray_test(m, st, frm, to, mask=mask)
    col, frac, pos, nrm = _got(out, 0)
    for k, (f, t, hit, s, n) in enumerate(cases):
        if not hit:
            assert col[k] == -1 and frac[k] == 1.0 and not pos[k].any() and not nrm[k].any(), k
            continue
        assert col[k] == box and abs(frac[k] - s) <= 1e-6, (k, col[k], frac[k], s)
        d = np.array(t, float) - np.array(f, float)
        if n is None:
            n = -d / np.linalg.norm(d)
        assert np.abs(nrm[k] - n).max() <= 1e-6, (k, nrm[k], n)
        assert np.abs(pos[k] - (frm[k] + s * d)).max() <= 1e-6, k
    # the numpy reference gives the same answers (its non-finite rays are misses too)
    ref = np_rays.ray_test(m, st[0], frm, to, mask=np.arange(int(m['n_col'])) == box)
    assert (ref['collider'] == col).all()
    # a masked-out box is never hit, even from inside
    out = emu_rays.ray_test(m, st, frm, to, mask=~mask)
    assert (out['collider'][0] != box).all()


# ------------------------------------------------------------------ gripper_proprioception and the camera
def _proprio_check(m, states):
    """phase_observe's flag (the emulated step's observation) == the rule applied to the fp64 ray cast by the ray kernel,
    on every env whose ray is unambiguous."""
    N = len(states)
    sim = EmuSim(m, N)
    sim.state[:, :sim.state_dim] = states
    flag = sim.observe()['gripper_proprioception'][:, 0]
    rays = [np_rays.proprio_ray(m, states[i]) for i in range(N)]
    frm = np.stack([r[0] for r in rays])[:, None, :]
    to = np.stack([r[1] for r in rays])[:, None, :]
    out = emu_rays.ray_test(m, states, frm, to)
    checked = 0
    for i in range(N):
        if np_rays.ray_test(m, states[i], frm[i], to[i])['ambiguous'][0]:
            continue
        assert np_rays.proprio_flag(m, out['collider'][i, 0], out['fraction'][i, 0]) == flag[i], i
        checked += 1
    assert checked >= N - 1, (checked, N)
    return flag


def test_proprioception_matches_step_observation():
    m, states = _states(PLAY, 4, seed=3)
    gold = [np.load(os.path.join(GOLDEN, g))['state'][:8] for g in ('heavy_step_r1.npz', 'many_contacts.npz')]
    # a short rollout that closes the gripper on whatever lies below it
    sim = EmuSim(m, 8, seed=5)
    sim.reset()
    rng = np.random.default_rng(7)
    for _ in range(3):
        sim.step(random_actions(rng, 8, PLAY))
    roll = sim.state[:, :sim.state_dim].copy()
    flags = np.concatenate([_proprio_check(m, s) for s in [states] + gold + [roll]])
    assert flags.min() == 0.0 and flags.max() == 1.0          # both outcomes occur


def test_camera_rays_match_segmentation():
    m, states = _states(PLAY, 2, seed=9)
    cam = default_camera(m, 32, 32)
    pal = default_palette(m)
    seg = emu_render.render(m, states, cam, pal, segmentation=True)['segmentation']
    V = np_render._mat(cam.view)
    Pm = np_render._mat(cam.proj)
    Minv = np.linalg.inv(Pm @ V)
    eye = np.linalg.inv(V)[:3, 3]
    jj, ii = np.meshgrid(np.arange(32), np.arange(32))
    xn, yn = 2 * (jj.ravel() + 0.5) / 32 - 1, 1 - 2 * (ii.ravel() + 0.5) / 32
    far = np.stack([xn, yn, np.ones_like(xn), np.ones_like(xn)], 1) @ Minv.T
    to = far[:, :3] / far[:, 3:]
    frm = np.tile(eye, (len(to), 1))
    out = emu_rays.ray_test(m, states, frm, to)
    for i in range(len(states)):
        ref_r = np_rays.ray_test(m, states[i], frm, to)
        ref_c = np_render.render(m, states[i], cam, pal)
        ok = ~ref_r['ambiguous'] & ~ref_c[3].ravel()
        assert ok.mean() > 0.95
        assert (out['collider'][i][ok] == seg[i].ravel()[ok]).all()


# ------------------------------------------------------------------ same bits, launch shapes, invalid input, layout
def test_shared_and_per_env_and_launch_shapes_give_the_same_bits():
    m, states = _states(PLAY, 3, seed=13)
    rng = np.random.default_rng(3)
    frm, to = np_rays.random_segments(m, states[0], 1500, rng)
    big = emu_rays.ray_test(m, states, frm, to)                             # block per env, 2 chunks of blockIdx.y
    per = emu_rays.ray_test(m, states, np.broadcast_to(frm, (3,) + frm.shape), np.broadcast_to(to, (3,) + to.shape))
    for k in big:
        assert big[k].tobytes() == per[k].tobytes(), k
    for lo in (0, 30, 1470):                                                # warp per env (R <= 32) on slices
        small = emu_rays.ray_test(m, states, frm[lo:lo + 30], to[lo:lo + 30])
        forced = emu_rays.ray_test(m, states, frm[lo:lo + 30], to[lo:lo + 30], force_large=True)
        for k in big:
            assert small[k].tobytes() == big[k][:, lo:lo + 30].tobytes() == forced[k].tobytes(), (lo, k)
    # in a site frame too
    ff, ft = np_rays.site_fan(4)
    a, b = emu_rays.ray_test(m, states, ff, ft, site=2), emu_rays.ray_test(m, states, ff, ft, site=2, force_large=True)
    assert all(a[k].tobytes() == b[k].tobytes() for k in a)


def test_invalid_calls_are_rejected():
    m, states = _states('UR5Reach-v0', 1, seed=1)
    f = np.zeros((4, 3), np.float32)
    t = np.ones((4, 3), np.float32)
    bad = [(lib.PrbRays(0, 0, -1, 0, ~0 & 0xFFFFFFFFFFFFFFFF), 'num_rays'), (lib.PrbRays(16385, 0, -1, 0, 1), 'num_rays'),
           (lib.PrbRays(4, 2, -1, 0, 1), 'per_env'), (lib.PrbRays(4, 0, -2, 0, 1), 'frame'), (lib.PrbRays(4, 0, 4, 0, 1), 'frame'),
           (lib.PrbRays(4, 0, -1, 1, 1), 'reserved')]
    for r, word in bad:
        with pytest.raises(ValueError, match=word):
            emu_rays.ray_test(m, states, f, t, rays=r)
    for name in ('from', 'to', 'collider', 'fraction'):
        with pytest.raises(ValueError, match='required'):
            emu_rays.ray_test(m, states, f, t, null=(name,))
    out = emu_rays.ray_test(m, states, f, t, null=('position', 'normal'))     # the optional outputs
    assert out['collider'].shape == (1, 4)


def test_struct_layout_matches_c(tmp_path):
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "prb.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n",'
           ' sizeof(prb_rays), offsetof(prb_rays, per_env), offsetof(prb_rays, frame), offsetof(prb_rays, reserved),'
           ' offsetof(prb_rays, collider_mask));return 0;}\n')
    exe = str(tmp_path / 'prb_rays_probe')
    open(exe + '.c', 'w').write(src)
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', exe, exe + '.c'])
    got = list(map(int, subprocess.check_output([exe]).split()))
    R = lib.PrbRays
    assert got == [ctypes.sizeof(R), R.per_env.offset, R.frame.offset, R.reserved.offset, R.collider_mask.offset]
    assert 'prb_ray_test' in lib.SYMBOLS


def test_check_rays():
    m = load_model(PLAY)
    nc = int(m['n_col'])
    body = np.asarray(m['col_body'])[:nc]
    f = np.zeros((5, 3))
    assert check_rays(m, 2, f, f) == (0, 5, (1 << nc) - 1)
    assert check_rays(m, 2, np.zeros((2, 5, 3)), np.zeros((2, 5, 3)), site=3)[:2] == (1, 5)
    per_env, R, mask = check_rays(m, 2, f, f, exclude_bodies=(0, 1))
    assert all(((mask >> c) & 1) == (body[c] not in (0, 1)) for c in range(nc))
    for kw in ({'ray_from': f, 'ray_to': np.zeros((4, 3))}, {'ray_from': np.zeros((3, 5, 3)), 'ray_to': np.zeros((3, 5, 3))},
               {'ray_from': np.zeros((5, 2)), 'ray_to': np.zeros((5, 2))}, {'ray_from': np.zeros((0, 3)), 'ray_to': np.zeros((0, 3))},
               {'ray_from': np.zeros((16385, 3)), 'ray_to': np.zeros((16385, 3))}, {'site': 4}, {'site': -1}, {'site': True},
               {'ray_to': np.full((5, 3), np.nan)}, {'exclude_bodies': (99,)}):
        args = {'ray_from': f, 'ray_to': f, **kw}
        with pytest.raises(ValueError):
            check_rays(m, 2, **args)
