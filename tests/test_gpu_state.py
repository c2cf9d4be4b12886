"""GPU tests of the link and joint state calls (prb_body_states, prb_write_state, prb_save_state / prb_restore_state):
no side effects of reads, agreement with the numpy reference tests/np_state.py at scale on both arms, a 65 536-env
read, masked writes against the host path (edit, prb_set_state, prb_observe) and the 20 steps after them, save /
step / masked restore and its replay, env_offset, PRB_PIPELINE=fused, the Python methods and invalid calls."""
import ctypes

import numpy as np
import pytest

import np_state
from helpers import random_actions
from roboticsplayroompybullet_b200 import lib
from roboticsplayroompybullet_b200.envs import make

pytestmark = pytest.mark.gpu

PLAY = 'UR5PlayAbsRPY1Obj-v0'
PLAYS = [PLAY, 'pandaPlayAbsRPY1Obj-v0']
U32 = 2.0 ** -24
TOL = 64 * U32            # as tests/test_cpu_state.py: relative to max(1, max |ref|) per env and quantity


def _stepped(env_id, n, seed, steps=8, **kw):
    env = make(env_id, num_envs=n, seed=seed, **kw)
    env.reset()
    rng = np.random.default_rng(seed)
    for _ in range(steps):
        env.step(random_actions(rng, n, env_id))
    return env


def _outs(env):
    import torch
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in env.dev.items()}


def _check_rows(m, st, body, frame, envs):
    nd, nf = int(m['nd']), int(m['n_free'])
    worst = 0.0
    for i in envs:
        rots, vec = np_state.reference_rows(m, st[i], frame)
        got = np.concatenate([body[i, :, 0:3], body[i, :, 7:13]], 1)
        err = np.abs(got - vec).max() / max(1.0, np.abs(vec).max())
        rerr = max(np.abs(np_state.quat_mat(body[i, k, 3:7]) - rots[k]).max() for k in range(len(rots)))
        rerr = max(rerr, np.abs(np.linalg.norm(body[i, :, 3:7].astype(np.float64), axis=1) - 1.0).max())
        worst = max(worst, err, rerr)
        assert err <= TOL and rerr <= TOL, (i, frame, err / U32, rerr / U32)
        assert body[i, nd:nd + nf].tobytes() == st[i, 5 * nd:5 * nd + 13 * nf].tobytes()
    return worst / U32


def _joints(m, st):
    nd, nf, ns = int(m['nd']), int(m['n_free']), int(m['n_slide'])
    so = 5 * nd + 13 * nf
    return (np.concatenate([st[:, :nd], st[:, so:so + 2 * ns:2]], 1), np.concatenate([st[:, nd:2 * nd], st[:, so + 1:so + 2 * ns:2]], 1))


def test_reads_have_no_side_effects_and_launch_once():
    import torch
    env = _stepped(PLAY, 64, 17, record_contacts=True)
    torch.cuda.synchronize()
    st0, out0 = env.get_state().tobytes(), {k: v.tobytes() for k, v in _outs(env).items()}
    con0 = {k: v.tobytes() for k, v in env.contacts().items()}
    n0 = env.launch_count()
    env.body_states('link')
    env.body_states('com')
    env.joint_states()
    torch.cuda.synchronize()
    assert env.launch_count() - n0 == 3
    assert env.get_state().tobytes() == st0
    assert {k: v.tobytes() for k, v in _outs(env).items()} == out0
    assert {k: v.tobytes() for k, v in env.contacts().items()} == con0
    env.close()


@pytest.mark.parametrize('env_id', PLAYS)
def test_reads_match_numpy_at_scale(env_id):
    n = 8192
    env = _stepped(env_id, n, 23)
    st = env.get_state()
    m = env.model
    nd = int(m['nd'])
    # 256 envs stratified over the batch: one from each block of 32
    rng = np.random.default_rng(3)
    sample = np.arange(0, n, 32) + rng.integers(0, 32, n // 32)
    link, com = env.body_states('link'), env.body_states('com')
    for frame, d in ((0, link), (1, com)):
        body = np.concatenate([d['position'], d['orientation'], d['linear_velocity'], d['angular_velocity']], 2)
        print(env_id, 'frame', frame, 'worst', round(_check_rows(m, st, body, frame, sample), 2), 'u')
    js = env.joint_states()
    jq, jqd = _joints(m, st)
    assert js['position'].tobytes() == jq.tobytes() and js['velocity'].tobytes() == jqd.tobytes()
    # link-frame positions are calculate_jacobian's zero-offset link points, bit for bit
    pts = env._arm_dynamics([(l, -1, (0.0, 0.0, 0.0)) for l in range(nd)], None, None, None, ('position',))['position']
    assert pts.cpu().numpy().tobytes() == np.ascontiguousarray(link['position'][:, :nd]).tobytes()
    env.close()


def test_65536_env_read_of_every_output():
    import torch
    n = 65536
    env = make(PLAY, num_envs=n, seed=5)
    env.reset()
    env.step_device(torch.as_tensor(random_actions(np.random.default_rng(1), n, PLAY), device='cuda'))
    K, nj = len(env.body_state_ids), len(env.joint_state_ids)
    body = torch.full((n, K, 13), float('nan'), device='cuda')
    q, qd = (torch.full((n, nj), float('nan'), device='cuda') for _ in range(2))
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    lib.check(env.L, env._h, env.L.prb_body_states(env._h, ctypes.byref(lib.PrbBodyQuery(1, 0)), p(body), p(q), p(qd), env._stream()))
    torch.cuda.synchronize()
    st = env.get_state()
    b = body.cpu().numpy()
    assert np.isfinite(b).all()
    _check_rows(env.model, st, b, 1, [0, n // 2, n - 1])
    jq, jqd = _joints(env.model, st)
    assert q.cpu().numpy().tobytes() == jq.tobytes() and qd.cpu().numpy().tobytes() == jqd.tobytes()
    env.close()


def _groups(m):
    nd, nf, ns = int(m['nd']), int(m['n_free']), int(m['n_slide'])
    allj, allf = (1 << (nd + ns)) - 1, (1 << nf) - 1
    W = lib.PrbStateWrite
    return {'joints': W(allj, allj, 0, 0, 0), 'free_poses': W(0, 0, allf, 0, 0), 'free_velocities': W(0, 0, 0, allf, 0),
            'mixed': W(0b101100101, 0b11, 1, 2, 0)}


def test_masked_write_equals_host_path_and_the_next_20_steps():
    import torch
    n = 8192
    env = _stepped(PLAY, n, 31, record_contacts=True)
    m = env.model
    nd, K = int(m['nd']), len(env.body_state_ids)
    rng = np.random.default_rng(9)
    actions = [random_actions(rng, n, PLAY) for _ in range(20)]
    for name, w in _groups(m).items():
        s0 = env.get_state()
        mask = (rng.random(n) < 0.5).astype(np.uint8)
        jq = rng.uniform(-1.5, 1.5, (n, len(env.joint_state_ids))).astype(np.float32)
        jqd = rng.uniform(-2.0, 2.0, (n, len(env.joint_state_ids))).astype(np.float32)
        body = np.concatenate([v for v in env.body_states('link').values()], 2)
        body[:, nd:, :3] += rng.uniform(-0.03, 0.03, (n, K - nd, 3)).astype(np.float32)
        body[:, nd:, 3:7] = rng.normal(size=(n, K - nd, 4)).astype(np.float32)
        body[:, nd:, 7:] = rng.uniform(-0.3, 0.3, (n, K - nd, 6)).astype(np.float32)
        # the host path, then its 20 steps
        env.set_state(np_state.host_edit(m, s0, w, jq, jqd, body, mask))
        env.observe()
        host_state, host_out = env.get_state(), _outs(env)
        host_traj = [env.step(a)[0]['obs_quat'].copy() for a in actions]
        host_end = env.get_state()
        # the device path from the same state (the outputs before the write are those of the host path's last step)
        env.set_state(s0)
        pre_out = _outs(env)
        dev = lambda x: torch.as_tensor(x, device='cuda')
        n0 = env.launch_count()
        status = env._write_state(w, dev(jq), dev(jqd), dev(body), dev(mask)).cpu().numpy()
        torch.cuda.synchronize()
        assert env.launch_count() - n0 == 3                 # write, report clear, masked observe
        assert (status == mask).all()
        st, out = env.get_state(), _outs(env)
        on, off = mask == 1, mask == 0
        assert st[on].tobytes() == host_state[on].tobytes(), name
        assert st[off].tobytes() == s0[off].tobytes(), name
        for k in out:
            if k == 'target_poses':
                continue
            assert out[k][on].tobytes() == host_out[k][on].tobytes(), (name, k)
            assert out[k][off].tobytes() == pre_out[k][off].tobytes(), (name, k)
        assert (env.contacts()['count'][on] == 0).all()
        traj = [env.step(a)[0]['obs_quat'].copy() for a in actions]
        for t, (a, b) in enumerate(zip(traj, host_traj)):
            assert a[on].tobytes() == b[on].tobytes(), (name, t)
        assert env.get_state()[on].tobytes() == host_end[on].tobytes(), name
    env.close()


def test_save_step_restore_replays_bit_for_bit():
    import torch
    n = 8192
    env = _stepped(PLAY, n, 41, record_contacts=True)
    rng = np.random.default_rng(2)
    actions = [random_actions(rng, n, PLAY) for _ in range(20)]
    snap = env.save_state_device()
    torch.cuda.synchronize()
    saved = snap.cpu().numpy()
    first = [env.step(a)[0]['obs_quat'].copy() for a in actions]
    moved = env.save_state()
    mask = (rng.random(n) < 0.5).astype(np.uint8)
    on, off = mask == 1, mask == 0
    n0 = env.launch_count()
    env.restore_state_device(snap, torch.as_tensor(mask, device='cuda'))
    torch.cuda.synchronize()
    assert env.launch_count() - n0 == 3                     # row copy, report clear, masked observe
    now = env.save_state()
    assert now[on].tobytes() == saved[on].tobytes()
    assert now[off].tobytes() == moved[off].tobytes()
    c = env.contacts()
    assert (c['count'][on] == 0).all() and (c['collider_a'][on] == -1).all()
    assert (c['count'][off] > 0).any()
    again = [env.step(a)[0]['obs_quat'].copy() for a in actions]
    for t, (a, b) in enumerate(zip(again, first)):
        assert a[on].tobytes() == b[on].tobytes(), t
    env.close()


def test_python_methods_env_offset_and_fused_pipeline(monkeypatch):
    import torch
    n = 256
    env = _stepped(PLAY, n, 7, steps=4)
    st = env.get_state()
    ref_link, ref_com, ref_j = env.body_states('link'), env.body_states('com'), env.joint_states()
    # env_offset and a smaller handle holding a slice of the states: the same bits
    off = make(PLAY, num_envs=64, seed=7, env_offset=128)
    off.set_state(st[128:192])
    assert all(off.body_states('com')[k].tobytes() == ref_com[k][128:192].tobytes() for k in ref_com)
    off.close()
    # the fused pipeline: the same reads; a write and a restore run (their observe is the masked setup launch)
    monkeypatch.setenv('PRB_PIPELINE', 'fused')
    fz = make(PLAY, num_envs=n, seed=7)
    monkeypatch.delenv('PRB_PIPELINE')
    fz.set_state(st)
    assert all(fz.body_states('link')[k].tobytes() == ref_link[k].tobytes() for k in ref_link)
    assert all(fz.joint_states()[k].tobytes() == ref_j[k].tobytes() for k in ref_j)
    snap = fz.save_state_device()
    status = fz.reset_joint_states(np.zeros(3), joints=[(0, 0), (0, 1), (0, 2)], mask=np.arange(n) % 2)
    assert (status == np.arange(n) % 2).all()
    assert (fz.joint_states()['position'][1::2, :3] == 0).all()
    fz.restore_state_device(snap)
    torch.cuda.synchronize()
    assert fz.get_state().tobytes() == st.tobytes()
    fz.close()
    # the Python methods on the split pipeline
    u = [int(x) for x in env.arm_dof_joints]
    q = np.linspace(-0.5, 0.5, 3).astype(np.float32)
    status = env.reset_joint_states(q, velocity=[0.1, 0.2, 0.3], joints=[(0, u[1]), (0, u[4]), (5, 0)])
    assert (status == 1).all()
    js = env.joint_states()
    assert (js['position'][:, [1, 4, 14]] == q).all() and (js['velocity'][:, [1, 4, 14]] == np.float32([0.1, 0.2, 0.3])).all()
    assert js['position'][:, [0, 2, 3]].tobytes() == ref_j['position'][:, [0, 2, 3]].tobytes()
    mask = np.zeros(n, np.uint8)
    mask[:10] = 1
    status = env.reset_base_states(1, position=[0.1, 0.2, 0.3], orientation=[0.0, 0.0, 2.0, 2.0], mask=mask)
    assert list(status[:12]) == [1] * 10 + [0, 0]
    b = env.body_states('link')
    nd = int(env.model['nd'])
    assert (b['position'][:10, nd] == np.float32([0.1, 0.2, 0.3])).all()
    # (0, 0, 2, 2) comes back as (0, 0, 1/sqrt2, 1/sqrt2) to fp32 rounding
    assert np.abs(b['orientation'][:10, nd, 2:] - np.sqrt(0.5)).max() <= 4 * U32 and (b['orientation'][:10, nd, :2] == 0).all()
    assert b['linear_velocity'][:10, nd].tobytes() == ref_link['linear_velocity'][:10, nd].tobytes()
    # a CUDA input that cannot be written leaves its env unchanged, status 2
    bad = torch.zeros((n, 4), device='cuda')
    bad[:, 3] = 1.0
    bad[3] = float('nan')
    before = env.get_state()
    status = env.reset_base_states_device(2, orientation=bad).cpu().numpy()
    assert status[3] == 2 and (np.delete(status, 3) == 1).all()
    assert env.get_state()[3].tobytes() == before[3].tobytes()
    env.close()


def test_invalid_calls_launch_nothing():
    import torch
    env = _stepped(PLAY, 32, 3, steps=1)
    torch.cuda.synchronize()
    n0, st0 = env.launch_count(), env.get_state().tobytes()
    buf = torch.zeros((32, 17, 13), device='cuda')
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    L, h, s = env.L, env._h, env._stream()
    W = lib.PrbStateWrite
    calls = [L.prb_body_states(h, ctypes.byref(lib.PrbBodyQuery(2, 0)), p(buf), None, None, s),
             L.prb_body_states(h, ctypes.byref(lib.PrbBodyQuery(0, 1)), p(buf), None, None, s),
             L.prb_body_states(h, ctypes.byref(lib.PrbBodyQuery(0, 0)), None, None, None, s),
             L.prb_write_state(h, ctypes.byref(W(1 << 15, 0, 0, 0, 0)), p(buf), None, None, None, None, s),
             L.prb_write_state(h, ctypes.byref(W(0, 0, 4, 0, 0)), None, None, p(buf), None, None, s),
             L.prb_write_state(h, ctypes.byref(W(0, 0, 0, 0, 0)), None, None, None, None, None, s),
             L.prb_write_state(h, ctypes.byref(W(0, 0, 1, 0, 0)), None, None, None, None, None, s),
             L.prb_write_state(h, ctypes.byref(W(1, 0, 0, 0, 7)), p(buf), None, None, None, None, s),
             L.prb_restore_state(h, None, None, s), L.prb_save_state(h, None, s)]
    assert calls == [-1] * len(calls)
    torch.cuda.synchronize()
    assert env.launch_count() == n0 and env.get_state().tobytes() == st0
    for kw in (dict(orientation=np.zeros(4)), dict(position=[np.nan, 0, 0]), dict()):
        with pytest.raises(ValueError):
            env.reset_base_states(1, **kw)
    for args in ((np.zeros(2), None, [(0, 99), (0, 0)]), (np.zeros((31, 15)),), (np.full(15, np.inf),)):
        with pytest.raises(ValueError):
            env.reset_joint_states(*args)
    with pytest.raises(ValueError):
        env.reset_base_states(3, position=np.zeros(3))          # a slide body, not a free body
    with pytest.raises(ValueError):
        env.body_states('world')
    with pytest.raises(ValueError):
        env.restore_state_device(torch.zeros((32, 7), device='cuda'))
    assert env.launch_count() == n0
    env.close()
