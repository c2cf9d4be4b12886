"""GPU tests of the contact report (prb_enable_contacts / prb_get_contacts): no side effects on the simulation, agreement
with the fp64 oracle on a stratified sample of a large batch, invariants on every contact at 65 536 envs, determinism,
env_offset independence and the lifecycle (reset, fused pipeline)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import contacts_check as cc
from helpers import OBS_KEYS, random_actions
from oracle.oracle import Oracle
from roboticsplayroompybullet_b200.envs import make

pytestmark = pytest.mark.gpu

PLAY = 'UR5PlayAbsRPY1Obj-v0'
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')


def _steps(env, rng, n_steps):
    for _ in range(n_steps):
        env.step(random_actions(rng, env.num_envs, env.env_id))


def test_report_has_no_side_effects():
    """The same seed with the report off and on: bit-identical outputs and states over 20 scripted steps; the only extra
    launches are one report kernel per step and one emptying launch per reset."""
    n = 64
    a, b = make(PLAY, num_envs=n, seed=17), make(PLAY, num_envs=n, seed=17, record_contacts=True)
    oa, ob = a.reset(), b.reset()
    rng = np.random.default_rng(5)
    for s in range(20):
        for k in OBS_KEYS:
            assert np.array_equal(oa[k], ob[k]), (s, k)
        assert a.get_state().tobytes() == b.get_state().tobytes(), s
        act = random_actions(rng, n, PLAY)
        (oa, ra, _, ia), (ob, rb, _, ib) = a.step(act), b.step(act)
        assert np.array_equal(ra, rb) and np.array_equal(ia['target_poses'], ib['target_poses'])
    assert b.launch_count() - a.launch_count() == 21
    assert b.contacts()['count'].max() > 0
    a.close(); b.close()


def _stratified(env, k, rng):
    """k envs stratified by arm-island solver class and by whether a free body is in contact (test_gpu_parity style)."""
    u = env.debug_usage()
    cls = u[:, 0] & 0xff
    rep = env.contacts()
    body = np.asarray(env.model['col_body'])
    on = rep['collider_a'] >= 0
    free = (on & (body[np.maximum(rep['collider_a'], 0)] >= 1)).any(1)
    keys = cls * 2 + free
    groups = [np.flatnonzero(keys == g) for g in np.unique(keys)]
    per = max(1, k // len(groups))
    pick = np.concatenate([rng.choice(g, min(per, len(g)), replace=False) for g in groups])
    rest = np.setdiff1d(np.arange(env.num_envs), pick)
    pick = np.concatenate([pick, rng.choice(rest, max(0, k - len(pick)), replace=False)])
    return np.sort(pick), np.unique(cls[pick])


def test_report_matches_oracle_at_scale():
    """8 192 play envs after scripted steps; 256 envs stratified by solver class (every arm-island class and the free-body
    slots) held to the oracle: one substep from get_state() (criterion 1) and one full step (criterion 2)."""
    n = 8192
    env = make(PLAY, num_envs=n, seed=29, record_contacts=True)
    env.reset()
    rng = np.random.default_rng(8)
    _steps(env, rng, 8)
    st = env.get_state()
    env.substeps(1)
    sample, classes = _stratified(env, 256, np.random.default_rng(1))
    assert len(classes) >= 4, classes
    m = env.model
    rep = env.contacts()
    r = cc.compare(m, Oracle, rep, [(i, st[i], lambda o: o.substeps(1)) for i in sample], 1e-5)
    assert not r['bad'], r
    assert r['cond'] <= cc.COND_SHARE * len(sample), r
    assert not cc.check_invariants(m, rep, sample)
    env.set_state(st)
    act = random_actions(rng, n, PLAY)
    env.step(act)
    rep = env.contacts()
    r = cc.compare(m, Oracle, rep, [(i, st[i], (lambda a: lambda o: o.step(np.asarray(a, np.float64)))(act[i])) for i in sample],
                   1e-4, f32_probe=True)
    assert not r['bad'], r
    assert r['cond'] <= 0.16 * len(sample), r
    env.close()


def test_invariants_at_65536_envs():
    n = 65536
    env = make(PLAY, num_envs=n, seed=41, record_contacts=True)
    env.reset()
    _steps(env, np.random.default_rng(3), 4)
    rep = env.contacts()
    assert rep['count'].max() > 8 and (rep['count'] > 0).mean() > 0.9
    bad = cc.check_invariants(env.model, rep)
    assert not bad, bad
    env.close()


def test_determinism_offset_and_lifecycle():
    n = 256
    a = make(PLAY, num_envs=n, seed=9, record_contacts=True)
    b = make(PLAY, num_envs=n, seed=9, record_contacts=True)
    c = make(PLAY, num_envs=n, seed=9, env_offset=1000, record_contacts=True)
    a.reset(); b.reset()
    rng = np.random.default_rng(2)
    for _ in range(3):
        act = random_actions(rng, n, PLAY)
        a.step(act); b.step(act)
    ra, rb = a.contacts(), b.contacts()
    for k in ra:
        assert np.array_equal(ra[k], rb[k]), k
    # another env_offset given the same states reports the same
    st = a.get_state()
    c.set_state(st); a.set_state(st)
    assert (a.contacts()['count'] == 0).all()                    # set_state empties the report
    act = random_actions(rng, n, PLAY)
    a.step(act); c.step(act)
    ra, rc = a.contacts(), c.contacts()
    for k in ra:
        assert np.array_equal(ra[k], rc[k]), k
    # observe / set_goal / render leave it unchanged; reset(mask) empties the masked envs only
    a.observe(); a.render()
    a.reset_goal_pos(a.observe()['desired_goal'])
    for k, v in a.contacts().items():
        assert np.array_equal(v, ra[k]), k
    mask = np.zeros(n, np.uint8); mask[::3] = 1
    a.reset(mask=mask)
    r2 = a.contacts()
    keep = mask == 0
    assert (r2['count'][~keep] == 0).all() and (r2['collider_a'][~keep] == -1).all()
    for k in r2:
        assert np.array_equal(r2[k][keep], ra[k][keep]), k
    # toggling: off stops refreshing, on again starts empty
    a.record_contacts = False
    a.step(act)
    assert np.array_equal(a.contacts()['count'], r2['count'])
    a.record_contacts = True
    assert (a.contacts()['count'] == 0).all()
    a.substeps(1)
    assert a.contacts()['count'].max() > 0
    d = a.contacts_device()
    assert d['position_on_a'].is_cuda and tuple(d['position_on_a'].shape) == (n, 64, 3) and tuple(d['count'].shape) == (n,)
    a.close(); b.close(); c.close()


def test_fused_pipeline_rejects_the_report():
    """PRB_PIPELINE is read when the handle is created: a child process with PRB_PIPELINE=fused."""
    code = ('import sys; sys.path.insert(0, %r)\n'
            'from roboticsplayroompybullet_b200.envs import make\n'
            'from roboticsplayroompybullet_b200.lib import PrbError\n'
            'e = make(%r, num_envs=4)\n'
            'try:\n    e.record_contacts = True\nexcept PrbError:\n    print("REJECTED")\n') % (ROOT, PLAY)
    out = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, PRB_PIPELINE='fused'), capture_output=True,
                         text=True, timeout=600)
    assert 'REJECTED' in out.stdout, out.stdout + out.stderr
