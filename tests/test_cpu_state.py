"""CPU tests of the link and joint state calls (prb_body_states, prb_write_state, prb_restore_state): the kernel source
(csrc/prb_state.cuh, under the SIMT emulator) against an fp64 numpy reference built on tests/np_arm_dynamics.py's
forward kinematics, exact equalities with the state and with prb_arm_dynamics, the write semantics against the host
path (edit the rows, set the state, observe), restores, invalid calls, the struct layouts and the Python checks."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import emu_arm
import emu_lib
import emu_state as S
import np_arm_dynamics as R
from emu_lib import EmuSim
from np_state import host_edit as _host_edit, normalised as _normalised, quat_mat as _quat_mat, reference_rows
from helpers import random_actions
from oracle.oracle import Oracle
from roboticsplayroompybullet_b200 import lib
from roboticsplayroompybullet_b200.envs import check_frame, check_joints, check_state_value, state_ids
from roboticsplayroompybullet_b200.model import load_model

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
PLAY = 'UR5PlayAbsRPY1Obj-v0'
WORLDS = [PLAY, 'pandaPick-v0', 'UR5Reach-v0']
U32 = 2.0 ** -24          # fp32 unit roundoff
# Kernel against the fp64 reference: |got - ref| <= TOL * max(1, max |ref|) per env and quantity.  Frames are composed
# over <= 8 links in fp32 (a few ulps per link), the COM velocity adds one cross product and the quaternion comes from
# the rotation matrix; prb_arm_dynamics' kernel, on the same forward kinematics, is held to the same 64u.
TOL = 64 * U32
OUT_KEYS = ('obs_quat', 'achieved_goal', 'desired_goal', 'controllable_achieved_goal', 'full_positional_state', 'joints',
            'velocity', 'observation', 'gripper_proprioception', 'reward', 'is_success')
WORST = {}


def _check_reads(m, sim, tag):
    """Both frames of every row against the reference; free-body rows and joint arrays equal the state bit for bit."""
    nd, nf, ns = int(m['nd']), int(m['n_free']), int(m['n_slide'])
    st = sim.state
    so = 5 * nd + 13 * nf
    for frame in (0, 1):
        out = S.body_states(sim, frame)
        body = out['body']
        for i in range(sim.N):
            rots, vec = reference_rows(m, st[i], frame)
            got = np.concatenate([body[i, :, 0:3], body[i, :, 7:13]], 1)
            scale = max(1.0, np.abs(vec).max())
            err = np.abs(got - vec).max() / scale
            qn = np.linalg.norm(body[i, :, 3:7].astype(np.float64), axis=1)
            rerr = max(np.abs(_quat_mat(body[i, k, 3:7]) - rots[k]).max() for k in range(len(rots)))
            rerr = max(rerr, np.abs(qn - 1.0).max())
            for key, e in (('vectors', err), ('rotations', rerr)):
                WORST[(tag, frame, key)] = max(WORST.get((tag, frame, key), 0.0), e / U32)
                assert e <= TOL, (tag, frame, key, i, e / U32)
            assert body[i, nd:nd + nf].tobytes() == st[i, 5 * nd:5 * nd + 13 * nf].tobytes()
        jq = np.concatenate([st[:, :nd], st[:, so:so + 2 * ns:2]], 1)
        jqd = np.concatenate([st[:, nd:2 * nd], st[:, so + 1:so + 2 * ns:2]], 1)
        assert out['q'].tobytes() == jq.tobytes() and out['qd'].tobytes() == jqd.tobytes()
    print(tag, {k[1:]: round(v, 2) for k, v in WORST.items() if k[0] == tag})


def _oracle_reset_sim(env_id, n, seed):
    m = load_model(env_id)
    s = EmuSim(m, n)
    for i in range(n):
        o = Oracle(m, seed=seed + i)
        o.reset()
        s.state[i, :s.state_dim] = np.asarray(o.state, np.float32)
    return m, s


def _stepped(env_id, n, seed, steps=6):
    m = load_model(env_id)
    s = EmuSim(m, n, seed=seed)
    s.reset()
    rng = np.random.default_rng(seed)
    for _ in range(steps):
        s.step(random_actions(rng, n, env_id))
    return m, s


# ------------------------------------------------------------------ reads against the reference
@pytest.mark.parametrize('env_id', WORLDS)
def test_reads_match_reference_reset_and_stepped_states(env_id):
    m, s = _oracle_reset_sim(env_id, 4, seed=21)
    _check_reads(m, s, env_id + ' reset')
    m, s = _stepped(env_id, 8, seed=4)
    _check_reads(m, s, env_id + ' stepped')


@pytest.mark.parametrize('golden', ['heavy_step_r1.npz', 'many_contacts.npz'])
def test_reads_match_reference_golden_states(golden):
    st = np.load(os.path.join(GOLDEN, golden))['state'][:6]
    m = load_model(PLAY)
    s = EmuSim(m, len(st))
    s.state[:, :s.state_dim] = st
    _check_reads(m, s, golden)


@pytest.mark.parametrize('env_id', [PLAY, 'pandaPlayAbsRPY1Obj-v0'])
def test_link_points_and_com_velocity_agree_with_arm_dynamics(env_id):
    """Link-frame positions are calculate_jacobian's zero-offset link points bit for bit (both take lp from phase_fk);
    the COM frame's position and velocity agree with the COM point's position and J qd within the bound."""
    m, s = _stepped(env_id, 8, seed=17)
    nd = int(m['nd'])
    st = s.state[:, :s.state_dim].copy()
    link = S.body_states(s, 0, outputs=('body',))['body']
    com = S.body_states(s, 1, outputs=('body',))['body']
    zero = emu_arm.arm_dynamics(m, st, [(l, -1, (0.0, 0.0, 0.0)) for l in range(nd)], outputs=('position',))['position']
    assert zero.tobytes() == np.ascontiguousarray(link[:, :nd, :3]).tobytes()
    coms = np.asarray(m['arm_com'], np.float64).reshape(-1, 3)[:nd]
    at = emu_arm.arm_dynamics(m, st, [(l, -1, tuple(coms[l])) for l in range(nd)], outputs=('position', 'velocity'))
    scale = max(1.0, np.abs(at['velocity']).max())
    assert np.abs(at['position'] - com[:, :nd, :3]).max() <= TOL
    assert np.abs(at['velocity'][:, :, :3] - com[:, :nd, 7:10]).max() <= TOL * scale
    assert np.abs(at['velocity'][:, :, 3:] - com[:, :nd, 10:13]).max() <= TOL * scale
    assert link[:, :nd, 10:13].tobytes() == com[:, :nd, 10:13].tobytes()


# ------------------------------------------------------------------ writes
def _twin(s):
    t = EmuSim(s.m, s.N, seed=s.seed)
    t.state[:] = s.state
    for k in s.out:
        t.out[k][:] = s.out[k]
    return t


def _random_inputs(m, s, rng):
    K, nj = S.sizes(m)
    nd = int(m['nd'])
    jq = rng.uniform(-1.5, 1.5, (s.N, nj)).astype(np.float32)
    jqd = rng.uniform(-2.0, 2.0, (s.N, nj)).astype(np.float32)
    body = S.body_states(s, 0, outputs=('body',))['body']
    body[:, nd:, :3] += rng.uniform(-0.05, 0.05, (s.N, K - nd, 3)).astype(np.float32)
    body[:, nd:, 3:7] = rng.normal(size=(s.N, K - nd, 4)).astype(np.float32) * 2.5       # not unit: normalised
    body[:, nd:, 7:] = rng.uniform(-0.5, 0.5, (s.N, K - nd, 6)).astype(np.float32)
    return jq, jqd, body


def _groups(m):
    nd, nf, ns = int(m['nd']), int(m['n_free']), int(m['n_slide'])
    allj, allf = (1 << (nd + ns)) - 1, (1 << nf) - 1
    W = lib.PrbStateWrite
    return {'joint_positions': W(allj, 0, 0, 0, 0), 'joint_velocities': W(0, allj, 0, 0, 0),
            'free_poses': W(0, 0, allf, 0, 0), 'free_velocities': W(0, 0, 0, allf, 0),
            'mixed': W(0b1010011, 0b11, 1, allf, 0), 'everything': W(allj, allj, allf, allf, 0)}


@pytest.mark.parametrize('env_id', [PLAY, 'pandaPick-v0'])
def test_masked_write_equals_host_path(env_id):
    m, s = _stepped(env_id, 8, seed=8)
    rng = np.random.default_rng(1)
    for name, w in _groups(m).items():
        if (w.free_poses | w.free_velocities) and int(m['n_free']) == 0:
            continue
        jq, jqd, body = _random_inputs(m, s, rng)
        mask = (rng.random(s.N) < 0.5).astype(np.uint8)
        mask[0], mask[1] = 1, 0
        a, h = _twin(s), _twin(s)
        before = {k: v.copy() for k, v in a.out.items()}
        st0 = a.state.copy()
        status = S.write_state(a, w, jq, jqd, body, mask)
        assert (status == mask).all(), name
        h.state[:, :h.state_dim] = _host_edit(m, h.state[:, :h.state_dim], w, jq, jqd, body, mask)
        h.observe()
        on, off = mask == 1, mask == 0
        assert a.state[on].tobytes() == h.state[on].tobytes(), name
        assert a.state[off].tobytes() == st0[off].tobytes(), name
        for k in OUT_KEYS:
            assert a.out[k][on].tobytes() == h.out[k][on].tobytes(), (name, k)
            assert a.out[k][off].tobytes() == before[k][off].tobytes(), (name, k)
        # the quaternions written are unit to fp32 rounding
        if w.free_poses:
            nd, nf = int(m['nd']), int(m['n_free'])
            qs = a.state[on][:, 5 * nd:5 * nd + 13 * nf].reshape(-1, nf, 13)[:, :, 3:7].astype(np.float64)
            assert np.abs(np.linalg.norm(qs, axis=2) - 1.0).max() <= 4 * U32
        s = a           # the next group starts from the written state


def test_rejected_envs_are_unchanged_and_null_mask_writes_all():
    m, s = _stepped(PLAY, 8, seed=2)
    nd, K = int(m['nd']), S.sizes(m)[0]
    rng = np.random.default_rng(5)
    jq, jqd, body = _random_inputs(m, s, rng)
    jq[1, 3] = np.nan                     # a selected joint position
    jqd[2, 13] = np.inf                   # a selected slide velocity
    body[3, nd, 3:7] = 0.0                # a zero quaternion
    body[4, nd + 1, 3:7] = 1e-7           # norm 2e-7 < 1e-6
    body[5, nd + 1, 8] = np.nan           # a selected velocity word
    jqd[6, 0] = np.nan                    # not selected below (joint_velocities bit 0 clear): no effect
    body[7, 0, :] = np.nan                # an arm row of body_dev is never read
    w = lib.PrbStateWrite((1 << 15) - 1, (1 << 15) - 2, 3, 3, 0)
    a = _twin(s)
    before = {k: v.copy() for k, v in a.out.items()}
    st0 = a.state.copy()
    status = S.write_state(a, w, jq, jqd, body)
    assert list(status) == [1, 2, 2, 2, 2, 2, 1, 1]
    rej = status == 2
    assert a.state[rej].tobytes() == st0[rej].tobytes()
    for k in OUT_KEYS:
        assert a.out[k][rej].tobytes() == before[k][rej].tobytes(), k
    ok = status == 1
    h = _twin(s)
    h.state[:, :h.state_dim] = _host_edit(m, h.state[:, :h.state_dim], w, jq, jqd, body, ok.astype(np.uint8))
    h.observe()
    assert a.state[ok].tobytes() == h.state[ok].tobytes()


def test_read_then_write_of_the_same_values_round_trips():
    """Everything read and written back: the state keeps its bits except the free-body quaternion words, which are
    renormalised in fp32 (within a few ulps of the stored ones); the outputs are those of an observe."""
    m, s = _stepped(PLAY, 8, seed=12)
    nd, nf, ns = int(m['nd']), int(m['n_free']), int(m['n_slide'])
    r = S.body_states(s, 0)
    a = _twin(s)
    st0 = a.state.copy()
    allj = (1 << (nd + ns)) - 1
    status = S.write_state(a, lib.PrbStateWrite(allj, allj, 3, 3, 0), r['q'], r['qd'], r['body'])
    assert (status == 1).all()
    qw = np.zeros(a.stride, bool)
    for b in range(nf):
        qw[5 * nd + 13 * b + 3:5 * nd + 13 * b + 7] = True
    assert a.state[:, ~qw].tobytes() == st0[:, ~qw].tobytes()
    assert a.state[:, qw].tobytes() == _normalised(st0[:, qw].reshape(-1, 4)).tobytes()
    assert np.abs(a.state[:, qw] - st0[:, qw]).max() <= 4 * U32
    h = _twin(a)
    h.observe()
    for k in OUT_KEYS:
        assert a.out[k].tobytes() == h.out[k].tobytes(), k


def test_restore_equals_snapshot_and_masks():
    m, s = _stepped(PLAY, 8, seed=6, steps=3)
    snap = s.state.copy()
    snap_out = {k: v.copy() for k, v in s.out.items()}
    rng = np.random.default_rng(2)
    s.step(random_actions(rng, s.N, PLAY))
    moved = s.state.copy()
    moved_out = {k: v.copy() for k, v in s.out.items()}
    mask = np.array([1, 0, 0, 1, 1, 0, 1, 0], np.uint8)
    S.restore_state(s, snap, mask)
    on, off = mask == 1, mask == 0
    assert s.state[on].tobytes() == snap[on].tobytes()
    assert s.state[off].tobytes() == moved[off].tobytes()
    h = _twin(s)
    h.state[:] = snap
    h.observe()
    for k in OUT_KEYS:
        assert s.out[k][on].tobytes() == h.out[k][on].tobytes(), k
        assert s.out[k][off].tobytes() == moved_out[k][off].tobytes(), k
    # the snapshot's own outputs came from the step's final setup launch; an observe of the snapshot repeats them
    for k in ('obs_quat', 'achieved_goal', 'desired_goal'):
        assert s.out[k][on].tobytes() == snap_out[k][on].tobytes(), k
    S.restore_state(s, snap)
    assert s.state.tobytes() == snap.tobytes()


# ------------------------------------------------------------------ invalid input, layout, the Python surface
def test_invalid_calls_are_rejected_before_any_launch():
    m, s = _stepped(PLAY, 4, seed=3, steps=1)
    Q = lib.PrbBodyQuery
    for call, word in ((Q(2, 0), 'frame'), (Q(-1, 0), 'frame'), (Q(0, 1), 'reserved')):
        with pytest.raises(ValueError, match=word):
            S.body_states(s, call=call)
    with pytest.raises(ValueError, match='at least one output'):
        S.body_states(s, outputs=())
    jq, jqd, body = _random_inputs(m, s, np.random.default_rng(0))
    st0, out0 = s.state.copy(), {k: v.copy() for k, v in s.out.items()}
    W = lib.PrbStateWrite
    for w, args, word in ((W(1 << 15, 0, 0, 0, 0), (jq, jqd, body), 'nd \\+ n_slide = 15'),
                          (W(0, 1 << 20, 0, 0, 0), (jq, jqd, body), 'nd \\+ n_slide'),
                          (W(0, 0, 4, 0, 0), (jq, jqd, body), 'n_free = 2'), (W(0, 0, 0, 1 << 31, 0), (jq, jqd, body), 'n_free'),
                          (W(0, 0, 0, 0, 0), (jq, jqd, body), 'no bit'), (W(1, 0, 0, 0, 1), (jq, jqd, body), 'reserved'),
                          (W(1, 0, 0, 0, 0), (None, jqd, body), 'joint_q_dev'), (W(0, 1, 0, 0, 0), (jq, None, body), 'joint_qd_dev'),
                          (W(0, 0, 1, 0, 0), (jq, jqd, None), 'body_dev'), (W(0, 0, 0, 2, 0), (jq, jqd, None), 'body_dev')):
        with pytest.raises(ValueError, match=word):
            S.write_state(s, w, *args)
    assert s.state.tobytes() == st0.tobytes()
    assert all(s.out[k].tobytes() == out0[k].tobytes() for k in out0)
    pick = load_model('pandaPick-v0')             # nd 9, one free body, no slide
    p = EmuSim(pick, 4)
    with pytest.raises(ValueError, match='nd \\+ n_slide = 9'):
        S.write_state(p, W(1 << 9, 0, 0, 0, 0), np.zeros((4, 9)))
    with pytest.raises(ValueError, match='n_free = 1'):
        S.write_state(p, W(0, 0, 2, 0, 0), None, None, np.zeros((4, 10, 13)))


def test_struct_layouts_match_c(tmp_path):
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "prb.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",'
           ' sizeof(prb_body_query), offsetof(prb_body_query, frame), offsetof(prb_body_query, reserved),'
           ' sizeof(prb_state_write), offsetof(prb_state_write, joint_positions), offsetof(prb_state_write, joint_velocities),'
           ' offsetof(prb_state_write, free_poses), offsetof(prb_state_write, free_velocities),'
           ' offsetof(prb_state_write, reserved));return 0;}\n')
    exe = str(tmp_path / 'prb_state_probe')
    open(exe + '.c', 'w').write(src)
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', exe, exe + '.c'])
    got = list(map(int, subprocess.check_output([exe]).split()))
    Q, W = lib.PrbBodyQuery, lib.PrbStateWrite
    assert got == [ctypes.sizeof(Q), Q.frame.offset, Q.reserved.offset, ctypes.sizeof(W), W.joint_positions.offset,
                   W.joint_velocities.offset, W.free_poses.offset, W.free_velocities.offset, W.reserved.offset]
    for name in ('prb_body_states', 'prb_write_state', 'prb_save_state', 'prb_restore_state'):
        assert name in lib.SYMBOLS
    assert emu_lib.lib().emu_max_bodies() == 17


def test_state_ids_and_python_checks():
    m = load_model(PLAY)
    bodies, joints = state_ids(m)
    urdf = [int(u) for u in np.asarray(m['arm_urdf_index'])[:12]]
    assert bodies.tolist() == [[0, u] for u in urdf] + [[1, -1], [2, -1], [3, -1], [4, -1], [5, -1]]
    assert joints.tolist() == [[0, u] for u in urdf] + [[3, 0], [4, 0], [5, 0]]
    # every row id is an id the contact report and change_dynamics know (a (body, link) that has a collider)
    nc = int(m['n_col'])
    have = set(zip(np.asarray(m['col_body'])[:nc].tolist(), np.asarray(m['col_urdf_link'])[:nc].tolist()))
    assert all((b, l) in have for b, l in bodies.tolist() if b > 0)
    pb, pj = state_ids(load_model('pandaPick-v0'))
    assert pb.shape == (10, 2) and pj.shape == (9, 2)
    assert check_frame('link') == 0 and check_frame('com') == 1
    with pytest.raises(ValueError):
        check_frame(1)
    assert check_joints(m, None) == list(range(15))
    assert check_joints(m, [(5, 0), (0, 20)]) == [14, 11]
    for bad in ([(0, 7)], [(1, 0)], [(0, 0), (0, 0)], [], [(0,)], [(True, 0)], [(0, 1.5)]):
        with pytest.raises(ValueError):
            check_joints(m, bad)
    assert check_state_value('position', None, 4, 3) is None
    assert check_state_value('position', np.zeros(3), 4, 3).shape == (3,)
    assert check_state_value('orientation', np.tile([0, 0, 0, 1.0], (4, 1)), 4, 4).dtype == np.float32
    for name, x, k in (('position', np.zeros((4, 2)), 3), ('position', np.zeros((3, 3)), 3), ('position', [np.nan, 0, 0], 3),
                       ('velocity', np.full((4, 2), np.inf), 2), ('orientation', np.zeros(4), 4),
                       ('orientation', np.array([[0, 0, 0, 1.0], [0, 0, 0, 1e-7], [0, 0, 0, 1.0], [1, 0, 0, 0]]), 4)):
        with pytest.raises(ValueError):
            check_state_value(name, x, 4, k)
