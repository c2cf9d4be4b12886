"""GPU tests of the arm queries (prb_arm_dynamics): no side effects on the simulation, agreement with the independent
numpy reference tests/np_arm_dynamics.py at scale on both arms, the site-0 velocity against the step's observation, the
same bits across calls, env_offset, batch size and PRB_PIPELINE=fused, 64-bit indexing at 65 536 envs, and invalid
input."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import np_arm_dynamics as R
from helpers import random_actions
from roboticsplayroompybullet_b200 import lib
from roboticsplayroompybullet_b200.envs import make

pytestmark = pytest.mark.gpu

PLAYS = ['UR5PlayAbsRPY1Obj-v0', 'pandaPlayAbsRPY1Obj-v0']
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
OUTPUTS = ('jacobian', 'position', 'velocity', 'mass_matrix', 'tau')
U32 = 2.0 ** -24
TOL = 64 * U32            # as tests/test_cpu_arm_dynamics.py: relative to max(1, max |ref|) per env and output


def _points(nd):
    """16 points: sites 0..3, sites 0 and 2 at an offset, links 0..7 at zero offset, two links at an offset."""
    pts = [(-1, s, (0.0, 0.0, 0.0)) for s in range(4)] + [(-1, 0, (0.03, -0.02, 0.05)), (-1, 2, (0.0, 0.01, -0.02))]
    pts += [(l, -1, (0.0, 0.0, 0.0)) for l in range(8)] + [(nd - 1, -1, (0.1, 0.2, -0.1)), (2, -1, (-0.3, 0.0, 0.1))]
    return pts


def _stepped(env_id, n, seed, **kw):
    env = make(env_id, num_envs=n, seed=seed, **kw)
    env.reset()
    rng = np.random.default_rng(seed)
    for _ in range(8):
        obs, _, _, _ = env.step(random_actions(rng, n, env_id))
    return env, obs


def _all(env, q=None, qd=None, qdd=None):
    """One prb_arm_dynamics call with every output and the 16 points: dict of numpy arrays."""
    nd = int(env.model['nd'])
    return {k: v.cpu().numpy() for k, v in env._arm_dynamics(_points(nd), q, qd, qdd, OUTPUTS).items()}


def _check_env(A, nd, got, q, qd, qdd):
    ref = R.all_outputs(A, q, qd, qdd, _points(nd))
    for k in OUTPUTS:
        err = np.abs(got[k] - ref[k]).max() / max(1.0, np.abs(ref[k]).max())
        assert err <= TOL, (k, err / U32)
    assert got['mass_matrix'].tobytes() == np.ascontiguousarray(got['mass_matrix'].T).tobytes()


def test_arm_queries_have_no_side_effects():
    """A stepped handle: state, output block and contact report are byte-identical before and after the calls, and each
    call is one launch."""
    import torch
    env, _ = _stepped(PLAYS[0], 64, 17, record_contacts=True)
    nd = int(env.model['nd'])
    torch.cuda.synchronize()
    st0 = env.get_state().tobytes()
    out0 = {k: v.cpu().numpy().tobytes() for k, v in env.dev.items()}
    con0 = {k: v.tobytes() for k, v in env.contacts().items()}
    n0 = env.launch_count()
    qdd = np.random.default_rng(0).normal(size=(64, nd)).astype(np.float32)
    env.calculate_jacobian(np.zeros((4, 3)), site=0)
    env.calculate_jacobian([(0.1, 0.0, 0.0)], link=int(env.arm_dof_joints[3]), site=None, q=np.zeros((64, nd)))
    env.calculate_mass_matrix()
    env.calculate_inverse_dynamics(qdd)
    _all(env, qdd=qdd)
    torch.cuda.synchronize()
    assert env.launch_count() - n0 == 5
    assert env.get_state().tobytes() == st0
    assert {k: v.cpu().numpy().tobytes() for k, v in env.dev.items()} == out0
    assert {k: v.tobytes() for k, v in env.contacts().items()} == con0
    env.close()


@pytest.mark.parametrize('env_id', PLAYS)
def test_gpu_matches_numpy_at_scale_and_site0_velocity_is_observed(env_id):
    n = 8192
    env, obs = _stepped(env_id, n, 23)
    st = env.get_state()
    nd = int(env.model['nd'])
    A = R.arm(env.model)
    rng = np.random.default_rng(4)
    qdd = rng.uniform(-20.0, 20.0, (n, nd)).astype(np.float32)
    got = _all(env, qdd=qdd)
    sample = rng.choice(n, 256, replace=False)
    for i in sample:
        _check_env(A, nd, {k: v[i] for k, v in got.items()}, st[i, :nd], st[i, nd:2 * nd], qdd[i])
    # caller-given q and qd, beyond the limits too
    q = rng.uniform(-4.0, 4.0, (n, nd)).astype(np.float32)
    qd = rng.uniform(-5.0, 5.0, (n, nd)).astype(np.float32)
    got2 = _all(env, q, qd, qdd)
    for i in sample[:64]:
        _check_env(A, nd, {k: v[i] for k, v in got2.items()}, q[i], qd[i], qdd[i])
    # point velocity at site 0 (J qd) against the step's observed end-effector velocity, every env
    v = env.calculate_jacobian(site=0)['velocity'][:, 0]
    scale = max(1.0, np.abs(obs['velocity']).max())
    assert np.abs(v - obs['velocity']).max() <= TOL * scale, np.abs(v - obs['velocity']).max() / U32
    # the three methods agree with the all-outputs call bit for bit
    assert env.calculate_mass_matrix().tobytes() == got['mass_matrix'].tobytes()
    assert env.calculate_inverse_dynamics(qdd).tobytes() == got['tau'].tobytes()
    J = env.calculate_jacobian(np.zeros((1, 3)), site=0)
    assert np.concatenate([J['linear'], J['angular']], 2).tobytes() == got['jacobian'][:, :1].tobytes()
    env.close()


def test_same_bits_across_calls_handles_offsets_and_fused(tmp_path):
    n = 128
    a, _ = _stepped(PLAYS[0], n, 9)
    st = a.get_state()
    nd = int(a.model['nd'])
    qdd = np.random.default_rng(1).normal(size=(n, nd)).astype(np.float32)
    r1 = _all(a, qdd=qdd)
    assert all(r1[k].tobytes() == v.tobytes() for k, v in _all(a, qdd=qdd).items())
    b = make(PLAYS[0], num_envs=n, seed=9, env_offset=1000)
    b.set_state(st)
    assert all(r1[k].tobytes() == v.tobytes() for k, v in _all(b, qdd=qdd).items())
    small = make(PLAYS[0], num_envs=64, seed=3)
    small.set_state(st[32:96])
    r3 = _all(small, qdd=qdd[32:96])
    assert all(r1[k][32:96].tobytes() == r3[k].tobytes() for k in OUTPUTS)
    np.save(str(tmp_path / 'state.npy'), st)
    np.save(str(tmp_path / 'qdd.npy'), qdd)
    code = ('import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n'
            'import numpy as np, test_gpu_arm_dynamics as T\n'
            'from roboticsplayroompybullet_b200.envs import make\n'
            'e = make(%r, num_envs=%d, seed=9)\n'
            'e.set_state(np.load(%r))\n'
            'np.savez(%r, **T._all(e, qdd=np.load(%r)))\nprint("DONE")\n') % (
        ROOT, os.path.join(ROOT, 'tests'), PLAYS[0], n, str(tmp_path / 'state.npy'), str(tmp_path / 'fused.npz'),
        str(tmp_path / 'qdd.npy'))
    p = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, PRB_PIPELINE='fused'), capture_output=True,
                       text=True, timeout=900)
    assert 'DONE' in p.stdout, p.stdout + p.stderr
    fused = np.load(str(tmp_path / 'fused.npz'))
    assert all(fused[k].tobytes() == r1[k].tobytes() for k in OUTPUTS)
    a.close(); b.close(); small.close()


def test_65536_envs_every_output():
    import torch
    N = 65536
    env = make(PLAYS[0], num_envs=N, seed=31)
    env.reset()
    env.step(random_actions(np.random.default_rng(0), N, PLAYS[0]))
    nd = int(env.model['nd'])
    rng = np.random.default_rng(2)
    q, qd, qdd = (torch.as_tensor(rng.uniform(-s, s, (N, nd)).astype(np.float32), device='cuda') for s in (3.0, 2.0, 10.0))
    out = env._arm_dynamics(_points(nd), q, qd, qdd, OUTPUTS)
    A = R.arm(env.model)
    assert out['jacobian'].numel() == N * 16 * 6 * nd
    for i in (0, N // 2, N - 1):
        _check_env(A, nd, {k: v[i].cpu().numpy() for k, v in out.items()}, q[i].cpu().numpy(), qd[i].cpu().numpy(),
                   qdd[i].cpu().numpy())
    env.close()


def test_invalid_calls_launch_nothing():
    import torch
    env = make(PLAYS[0], num_envs=4, seed=2)
    env.reset()
    nd = int(env.model['nd'])
    n0 = env.launch_count()
    for kw in (dict(local_positions=np.zeros((0, 3))), dict(local_positions=np.zeros((17, 3))), dict(link=0, site=0),
               dict(link=None, site=None), dict(link=99, site=None), dict(site=4), dict(q=np.zeros((4, nd + 1))),
               dict(qd=np.full((4, nd), np.nan)), dict(local_positions=[(0.0, np.inf, 0.0)])):
        with pytest.raises(ValueError):
            env.calculate_jacobian(**kw)
    with pytest.raises(ValueError):
        env.calculate_mass_matrix(q=np.zeros((3, nd)))
    with pytest.raises(ValueError):
        env.calculate_inverse_dynamics(qdd=torch.zeros((4, nd - 1), device='cuda'))
    buf = torch.zeros(4 * 16 * 6 * 12, device='cuda')
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    P = lib.PrbArmPoint
    pt = lambda l, s, r=0: (P * 1)(P(l, s, (ctypes.c_float * 3)(0, 0, 0), r))
    cases = [(lib.PrbArmQuery(17, 0), pt(-1, 0), [p(buf)] * 5), (lib.PrbArmQuery(-1, 0), pt(-1, 0), [p(buf)] * 5),
             (lib.PrbArmQuery(1, 1), pt(-1, 0), [p(buf)] * 5), (lib.PrbArmQuery(1, 0), pt(-1, 0, 1), [p(buf)] * 5),
             (lib.PrbArmQuery(1, 0), pt(nd, -1), [p(buf)] * 5), (lib.PrbArmQuery(1, 0), pt(-1, 4), [p(buf)] * 5),
             (lib.PrbArmQuery(1, 0), pt(0, 0), [p(buf)] * 5), (lib.PrbArmQuery(1, 0), pt(-1, 0), [None] * 3 + [p(buf)] * 2),
             (lib.PrbArmQuery(0, 0), pt(-1, 0), [None] * 5), (lib.PrbArmQuery(1, 0), ctypes.POINTER(P)(), [p(buf)] * 5)]
    for c, pts, outs in cases:
        assert env.L.prb_arm_dynamics(env._h, ctypes.byref(c), pts, None, None, None, *outs, None) == -1   # PRB_ERR_INVALID
        assert env.L.prb_last_error(env._h).decode().startswith('prb_arm_dynamics: ')
    assert env.launch_count() == n0
    assert env.calculate_mass_matrix().shape == (4, nd, nd) and env.launch_count() == n0 + 1   # still usable
    env.close()
