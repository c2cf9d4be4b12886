"""GPU tests of per-env dynamics (prb_enable_dynamics / prb_get_dynamics / prb_randomize_dynamics): no side effects with
the model's values, each env equal to a handle of its patched model, a stratified sample against the fp64 oracle,
invariants at 65 536 envs, determinism and env_offset independence of the draws, reset with randomization and the
lifecycle."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import contacts_check as cc
from helpers import OBS_KEYS, compare_step, oracle_step_from, random_actions
from oracle.oracle import Oracle
from roboticsplayroompybullet_b200 import lib
from roboticsplayroompybullet_b200.envs import make
from test_cpu_dynamics import _param_sets, _patched

pytestmark = pytest.mark.gpu

PLAY = 'UR5PlayAbsRPY1Obj-v0'
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
RANDOM = {'lateral_friction': (0.5, 1.5), 'spinning_friction': (0.5, 2.0), 'mass': (0.5, 2.0), 'linear_damping': (0.5, 2.0),
          'angular_damping': (0.5, 2.0)}


def _bench_actions(env, obs, steps, seed=2):
    import torch
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench
    a = bench.synth_actions(np.random.default_rng(seed), env.num_envs, steps, env.env_id,
                            block_xyz=obs['achieved_goal'][:, :3].cpu().numpy(), ee_xyz=obs['obs_quat'][:, :3].cpu().numpy())
    return torch.as_tensor(a).cuda()


def _set_rows(env, sets):
    """Env i gets parameter set i % len(sets), written straight into the device table."""
    import torch
    d = env.dynamics_device()
    for k in d:
        rows = np.stack([sets[i % len(sets)][k] for i in range(env.num_envs)])
        d[k].copy_(torch.as_tensor(rows).reshape(d[k].shape))
    torch.cuda.synchronize()


def test_table_with_model_values_has_no_side_effects():
    """Criterion 1: 20 steps of the bench workload at 8 192 envs with the table off and on with the model's values:
    bit-identical outputs and states."""
    import torch
    n = 8192
    runs = []
    for on in (False, True):
        env = make(PLAY, num_envs=n, seed=17, per_env_dynamics=on)
        obs = env.reset_device()
        acts = _bench_actions(env, obs, 20)
        outs = []
        for t in range(20):
            o, r, _, info = env.step_device(acts[t])
            outs.append(torch.cat([o[k].reshape(n, -1) for k in OBS_KEYS] + [r[:, None], info['target_poses']], 1).cpu())
        runs.append((outs, env.get_state()))
        env.close()
    for t in range(20):
        assert torch.equal(runs[0][0][t], runs[1][0][t]), t
    assert runs[0][1].tobytes() == runs[1][1].tobytes()


def test_per_env_equals_per_model():
    """Criterion 2: 8 192 envs, env i with parameter set i % 8; each env is compared bit for bit with a handle built from
    its patched model that starts from the same state (get_state / set_state) and takes the same actions."""
    import torch
    n, steps = 8192, 6
    env = make(PLAY, num_envs=n, seed=23, per_env_dynamics=True)
    sets = _param_sets(env.model)
    K = len(sets)
    obs = env.reset_device()
    for t, a in enumerate(_bench_actions(env, obs, 8, seed=3)):
        env.step_device(a)
    _set_rows(env, sets)
    st = env.get_state()
    acts = _bench_actions(env, env.observe_device(), steps, seed=4)
    outs = []
    for t in range(steps):
        o, r, _, _ = env.step_device(acts[t])
        outs.append(torch.cat([o[k].reshape(n, -1) for k in OBS_KEYS] + [r[:, None]], 1).cpu())
    fin = env.get_state()
    env.close()
    for k in range(K):
        idx = np.arange(k, n, K)
        ref = make(PLAY, num_envs=len(idx), seed=23, model=_patched(env.model, sets[k]))
        ref.set_state(st[idx])
        for t in range(steps):
            o, r, _, _ = ref.step_device(acts[t][torch.as_tensor(idx).cuda()])
            got = torch.cat([o[key].reshape(len(idx), -1) for key in OBS_KEYS] + [r[:, None]], 1).cpu()
            assert torch.equal(got, outs[t][idx]), (k, t)
        assert ref.get_state().tobytes() == fin[idx].tobytes(), k
        ref.close()


def _stratified(env, k, rng):
    u = env.debug_usage()
    keys = u[:, 0] & 0xff
    groups = [np.flatnonzero(keys == g) for g in np.unique(keys)]
    per = max(1, k // len(groups))
    pick = np.concatenate([rng.choice(g, min(per, len(g)), replace=False) for g in groups])
    rest = np.setdiff1d(np.arange(env.num_envs), pick)
    pick = np.concatenate([pick, rng.choice(rest, max(0, k - len(pick)), replace=False)])
    return np.sort(pick), np.unique(keys[pick])


def test_randomized_sample_matches_oracle():
    """Criterion 3: 8 192 envs with randomized dynamics after scripted steps; 256 envs stratified by arm-island solver
    class against the oracle of each env's patched model, judged by helpers.compare_step."""
    n = 8192
    env = make(PLAY, num_envs=n, seed=29, randomize_dynamics=RANDOM)
    obs = env.reset_device()
    for a in _bench_actions(env, obs, 8, seed=5):
        env.step_device(a)
    st = env.get_state()
    rng = np.random.default_rng(9)
    act = random_actions(rng, n, PLAY)
    o, r, _, info = env.step(act)
    sample, classes = _stratified(env, 256, np.random.default_rng(1))
    assert len(classes) >= 3, classes
    d = env.dynamics()
    bad = {'bad_pose': 0, 'bad_vel': 0, 'bad_flags': 0, 'bad_reward': 0, 'stiff': 0}
    crng = np.random.default_rng(0)
    for i in sample:
        pm = _patched(env.model, {k: d[k][i] for k in d})
        ref = oracle_step_from(pm, st[i], act[i], Oracle)[0]
        res = compare_step(pm, {k: o[k][i:i + 1] for k in OBS_KEYS}, r[i:i + 1], {'is_success': info['is_success'][i:i + 1]},
                           [ref], st[i:i + 1], act[i:i + 1], Oracle, crng)
        for k in bad:
            bad[k] += res[k]
    env.close()
    assert bad['bad_pose'] == bad['bad_vel'] == bad['bad_flags'] == bad['bad_reward'] == 0, bad
    assert bad['stiff'] <= 0.05 * len(sample), bad


def test_invariants_at_full_size_with_randomization():
    """Criterion 4: 65 536 play envs with randomized dynamics, reset and 24 scripted steps: every key finite, unit
    quaternions, success <=> reward 0, nothing fell out of the world, and no contact was dropped."""
    import torch
    N = 65536
    env = make(PLAY, num_envs=N, seed=11, randomize_dynamics=RANDOM)
    o0 = env.reset_device()
    acts = _bench_actions(env, o0, 24)
    for t in range(24):
        o, r, _, info = env.step_device(acts[t])
    torch.cuda.synchronize()
    for k in OBS_KEYS:
        assert torch.isfinite(o[k].float()).all(), k
    oq = o['obs_quat']
    assert (oq[:, 3:7].norm(dim=1) - 1).abs().max() < 1e-5 and (oq[:, 11:15].norm(dim=1) - 1).abs().max() < 1e-5
    s = info['is_success']
    assert torch.equal((r == 0), (s > 0))
    blk = oq[:, 8:11]
    assert (blk[:, 2] > -0.2).all() and blk.abs().max() < 2.0
    assert env.overflow_count() == 0
    d = env.dynamics_device()
    assert float(d['mass'][:, 0].min()) < 0.2 and float(d['mass'][:, 0].max()) > 0.55      # the draws span the range
    env.close()


def test_draws_deterministic_and_independent_of_env_offset():
    """Criterion 5: two handles with the same seed draw the same tables and reach the same states; the draws of a handle
    at env_offset 32 equal rows 32.. of a larger handle."""
    n = 64
    a, b = make(PLAY, num_envs=n, seed=5, randomize_dynamics=RANDOM), make(PLAY, num_envs=n, seed=5, randomize_dynamics=RANDOM)
    c = make(PLAY, num_envs=16, seed=5, env_offset=32, randomize_dynamics=RANDOM)
    for e in (a, b, c):
        e.reset()
    da, db, dc = a.dynamics(), b.dynamics(), c.dynamics()
    rng = np.random.default_rng(2)
    for _ in range(3):
        act = random_actions(rng, n, PLAY)
        a.step(act); b.step(act)
    assert a.get_state().tobytes() == b.get_state().tobytes()
    for k in da:
        assert np.array_equal(da[k], db[k]), k
        assert np.array_equal(dc[k], da[k][32:48]), k
    a.reset()
    assert not np.array_equal(a.dynamics()['mass'], da['mass'])        # a new episode draws anew
    for e in (a, b, c):
        e.close()


def test_reset_settles_each_block_with_its_own_mass():
    """Criterion 6: after reset() with randomized mass every block at rest (arm clear of it) carries its own m_e g
    within 1 % (contact report)."""
    n = 64
    env = make(PLAY, num_envs=n, seed=13, record_contacts=True, randomize_dynamics={'mass': (0.3, 3.0),
                                                                                    'lateral_friction': (0.7, 1.3)})
    env.reset()
    env.substeps(1)
    rep = env.contacts()
    mass = env.dynamics()['mass'][:, 0]
    g = abs(env.model.param('gravity_z'))
    body = np.asarray(env.model['col_body'])
    checked = 0
    for i in range(n):
        k = rep['count'][i]
        ba, bb = body[rep['collider_a'][i][:k]], body[rep['collider_b'][i][:k]]
        if (((ba == 0) & (bb == 1)) | ((ba == 1) & (bb == 0))).any():
            continue
        fz = cc.block_vertical_force(env.model, rep, i, 1)
        assert abs(fz - mass[i] * g) <= 0.01 * mass[i] * g, (i, fz, mass[i] * g)
        checked += 1
    assert checked >= n - 4 and np.ptp(mass) > 0.5          # free_mass 0.3 kg x (0.3, 3.0)
    env.close()


def test_lifecycle_and_rejections():
    """Criterion 7: enable / write / disable / enable refills the model's values; randomizing needs the table and
    rejects invalid ranges before any launch; change_dynamics writes the right entries."""
    n = 8
    env = make(PLAY, num_envs=n, seed=3, per_env_dynamics=True)
    ref = env.dynamics()
    assert np.array_equal(ref['mass'][0], np.asarray(env.model['free_mass'], np.float32)[:2])
    env.change_dynamics(1, mass=np.linspace(0.1, 0.8, n), lateral_friction=0.25, mask=np.arange(n) % 2)
    d = env.dynamics()
    odd = np.arange(n) % 2 == 1
    assert np.array_equal(d['mass'][~odd], ref['mass'][~odd])
    assert np.allclose(d['mass'][odd, 0], np.linspace(0.1, 0.8, n)[odd].astype(np.float32), rtol=0, atol=0)
    ratio = d['local_inertia_diagonal'][odd, 0] / ref['local_inertia_diagonal'][odd, 0]
    assert np.allclose(ratio, (d['mass'][odd, 0] / ref['mass'][odd, 0])[:, None], rtol=1e-6)
    cols = np.nonzero(np.asarray(env.model['col_body'])[:env.model['n_col']] == 1)[0]
    assert (d['lateral_friction'][odd][:, cols] == np.float32(0.25)).all()
    assert np.array_equal(np.delete(d['lateral_friction'], cols, 1), np.delete(ref['lateral_friction'], cols, 1))
    with pytest.raises(ValueError):
        env.change_dynamics(0, 5, mass=1.0)                         # arm link: no per-env mass
    env.per_env_dynamics = False
    env.per_env_dynamics = True
    for k, v in env.dynamics().items():
        assert np.array_equal(v, ref[k]), k
    L, h = env.L, env._h
    bad = lib.PrbDynamicsRanges()
    for k in lib.DYNAMICS_RANGE_FIELDS:
        getattr(bad, k)[:] = (1.0, 1.0)
    for field, lo, hi in (('mass', 0.0, 1.0), ('lateral_friction', 2.0, 1.0), ('linear_damping', -1.0, 1.0),
                          ('angular_damping', 1.0, float('inf')), ('spinning_friction', float('nan'), 1.0)):
        r = lib.PrbDynamicsRanges.from_buffer_copy(bad)
        getattr(r, field)[:] = (lo, hi)
        before = env.launch_count()
        assert L.prb_randomize_dynamics(h, ctypes.byref(r), None, None) != 0, field
        assert env.launch_count() == before
    assert L.prb_randomize_dynamics(h, ctypes.byref(bad), None, None) == 0
    env.per_env_dynamics = False
    assert L.prb_randomize_dynamics(h, ctypes.byref(bad), None, None) != 0
    env.close()
    fresh = make(PLAY, num_envs=2, seed=3)
    assert fresh.L.prb_get_dynamics(fresh._h, ctypes.byref(lib.PrbDynamics())) != 0      # never enabled
    fresh.close()


def test_fused_pipeline_rejects_the_table():
    """PRB_PIPELINE is read when the handle is created: a child process with PRB_PIPELINE=fused."""
    code = ('import sys; sys.path.insert(0, %r)\n'
            'from roboticsplayroompybullet_b200.envs import make\n'
            'from roboticsplayroompybullet_b200.lib import PrbError\n'
            'e = make(%r, num_envs=4)\n'
            'try:\n    e.per_env_dynamics = True\nexcept PrbError:\n    print("REJECTED")\n') % (ROOT, PLAY)
    out = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, PRB_PIPELINE='fused'), capture_output=True,
                         text=True, timeout=600)
    assert 'REJECTED' in out.stdout, out.stdout + out.stderr
