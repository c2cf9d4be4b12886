"""GPU tests of closest points (prb_closest_points): no side effects on the simulation, agreement with the independent
numpy reference tests/np_closest.py at scale, the contact report's deep contacts, invariants at 65 536 envs, the same
bits across calls, env_offset, batch size and PRB_PIPELINE=fused, and invalid input."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import np_closest
from helpers import OBS_KEYS, random_actions
from roboticsplayroompybullet_b200 import lib
from roboticsplayroompybullet_b200.envs import make

pytestmark = pytest.mark.gpu

PLAY = 'UR5PlayAbsRPY1Obj-v0'
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
MAX_DISTANCES = (0.0, 0.05, 10.0)


def _calls(m):
    """(queries, max_distance) of the three query sets at the three max distances."""
    return [(qs, md) for qs in np_closest.query_sets(m).values() for md in MAX_DISTANCES]


def _stepped(n, seed, record_contacts=False):
    """n play envs after 12 random steps, the gripper closed over the last 6 (some envs grasp the block); the env and
    the last observation."""
    env = make(PLAY, num_envs=n, seed=seed, record_contacts=record_contacts)
    env.reset()
    rng = np.random.default_rng(seed)
    for k in range(12):
        a = random_actions(rng, n, PLAY)
        if k >= 6:
            a[:, -1] = -1.0
        obs, _, _, _ = env.step(a)
    return env, obs


def test_closest_points_have_no_side_effects():
    """Two handles, one running the query sets after every step: bit-identical states, outputs and contact reports, and
    the only extra launches are the closest-point calls."""
    n = 64
    a = make(PLAY, num_envs=n, seed=17, record_contacts=True)
    b = make(PLAY, num_envs=n, seed=17, record_contacts=True)
    oa, ob = a.reset(), b.reset()
    rng = np.random.default_rng(5)
    calls = 0
    for s in range(20):
        for k in OBS_KEYS:
            assert np.array_equal(oa[k], ob[k]), (s, k)
        assert a.get_state().tobytes() == b.get_state().tobytes(), s
        ca, cb = a.contacts(), b.contacts()
        assert all(np.array_equal(ca[k], cb[k]) for k in ca), s
        act = random_actions(rng, n, PLAY)
        (oa, ra, _, ia), (ob, rb, _, ib) = a.step(act), b.step(act)
        assert np.array_equal(ra, rb) and np.array_equal(ia['target_poses'], ib['target_poses'])
        for qs, md in _calls(b.model):
            b.closest_points_device(qs, md)
            calls += 1
    assert a.get_state().tobytes() == b.get_state().tobytes()
    assert b.launch_count() - a.launch_count() == calls
    a.close(); b.close()


def test_gpu_matches_numpy_and_contacts_at_scale():
    n = 8192
    env, obs = _stepped(n, 23, record_contacts=True)
    st = env.get_state()
    m = env.model
    flag = obs['gripper_proprioception']
    grasp = np.nonzero(flag == 1)[0][:64]
    assert len(grasp) > 0
    sample = np.unique(np.r_[grasp, np.random.default_rng(4).choice(n, 256 - len(grasp), replace=False)])[:256]
    tables = {int(i): np_closest.pair_table(m, st[i]) for i in sample}
    for qs, md in _calls(m):
        out = env.closest_points(qs, md)
        mk = np_closest.masks(m, qs)
        namb = 0
        for i in sample:
            a, bad = np_closest.check_env(m, st[i], mk, {k: v[i] for k, v in out.items()}, md, tables[int(i)])
            assert not bad, (qs[:3], md, i, bad[:4])
            namb += a
        assert namb <= 0.02 * len(sample) * len(mk), (md, namb)
        body = np.asarray(m['col_body'])
        c = out['collider_a']
        assert np.array_equal(out['body_a'], np.where(c >= 0, body[np.maximum(c, 0)], -1))
    # every collider pair the contact report lists below -1e-3 m is within reach in the state after the step.  The report
    # measures before the last substep's solve and integration, and a randomly driven arm link moves up to ~3 m/s, 1 cm
    # in one 1/300 s substep: 1e-2 m bounds that motion (1e-3 m does not; DESIGN.md §4.10 has the distribution)
    con = env.contacts()
    cnt = con['count']
    deep = [(e, int(con['collider_a'][e, k]), int(con['collider_b'][e, k]))
            for e in range(n) for k in np.nonzero(con['distance'][e, :cnt[e]] < -1e-3)[0]]
    assert deep
    pairs = sorted(set((a, b) for _, a, b in deep))
    got = {}
    for lo in range(0, len(pairs), 64):
        chunk = pairs[lo:lo + 64]
        d = _raw_distance(env, [(1 << a, 1 << b) for a, b in chunk], 10.0)
        for k, p in enumerate(chunk):
            got[p] = d[:, k]
    after = np.array([float(got[(a, b)][e]) for e, a, b in deep])
    print('deep contacts: %d, pairs %d, closest distance after the step: median %.3e, 99%% %.3e, max %.3e m, '
          '%d above 1e-3 m' % (len(deep), len(pairs), np.median(after), np.quantile(after, 0.99), after.max(),
                               (after > 1e-3).sum()))
    assert after.max() <= 1e-2, after.max()
    env.close()


def _raw_distance(env, masks, md):
    """prb_closest_points with collider masks (a (body, link) side can name several colliders): distance [N,Q]."""
    import torch
    N, Q = env.num_envs, len(masks)
    ca, cb = (torch.empty((N, Q), dtype=torch.int32, device='cuda') for _ in range(2))
    d = torch.empty((N, Q), dtype=torch.float32, device='cuda')
    qs = (lib.PrbClosestQuery * Q)(*[lib.PrbClosestQuery(a, b) for a, b in masks])
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    lib.check(env.L, env._h, env.L.prb_closest_points(env._h, ctypes.byref(lib.PrbClosest(Q, 0, md, 0)), qs, p(ca), p(cb),
                                                      p(d), None, None, None, None))
    return d.cpu().numpy()


def test_invariants_at_65536_envs():
    N = 65536
    env = make(PLAY, num_envs=N, seed=31)
    env.reset()
    env.step(random_actions(np.random.default_rng(0), N, PLAY))
    m = env.model
    body = np.asarray(m['col_body'])
    results = []
    for qs, md in _calls(m):
        r = env.closest_points(qs, md)
        results.append(r)
        mk = np_closest.masks(m, qs)
        ca, cb, d = r['collider_a'], r['collider_b'], r['distance']
        hit = ca >= 0
        assert (hit == (cb >= 0)).all() and (hit == np.isfinite(d)).all() and (d[hit] <= md).all()
        assert (ca[hit] != cb[hit]).all()
        for k, (ma, mb) in enumerate(mk):
            h = hit[:, k]
            assert all((ma >> int(c)) & 1 for c in np.unique(ca[h, k])) and all((mb >> int(c)) & 1 for c in np.unique(cb[h, k]))
        pa, pb, nrm = (r[k].astype(np.float64) for k in ('position_on_a', 'position_on_b', 'normal_on_b'))
        assert not pa[~hit].any() and not pb[~hit].any() and not nrm[~hit].any()
        if hit.any():
            assert np.abs(np.linalg.norm(nrm[hit], axis=-1) - 1.0).max() <= 1e-5
            assert np.abs(pa[hit] - (pb[hit] + d[hit][:, None] * nrm[hit])).max() <= 2e-5
        assert np.array_equal(r['body_b'], np.where(cb >= 0, body[np.maximum(cb, 0)], -1))
    # the witness invariants with collider poses on a sample
    st = env.get_state()
    for i in np.random.default_rng(1).choice(N, 64, replace=False):
        tab = np_closest.pair_table(m, st[i])
        for (qs, md), r in zip(_calls(m), results):
            _, bad = np_closest.check_env(m, st[i], np_closest.masks(m, qs), {k: v[i] for k, v in r.items()}, md, tab)
            assert not bad, (i, md, bad[:4])
    env.close()


def _result_bytes(r):
    return {k: np.asarray(v).tobytes() for k, v in r.items()}


def test_same_bits_across_calls_handles_offsets_and_fused(tmp_path):
    n = 128
    a, _ = _stepped(n, 9)
    st = a.get_state()
    b = make(PLAY, num_envs=n, seed=9, env_offset=1000)
    b.set_state(st)
    small = make(PLAY, num_envs=64, seed=3)
    small.set_state(np.repeat(st[77:78], 64, 0))
    np.save(str(tmp_path / 'state.npy'), st)
    results = []
    for qs, md in _calls(a.model):
        r1 = a.closest_points(qs, md)
        results.append(r1)
        for other in (a.closest_points(qs, md), b.closest_points(qs, md)):
            assert _result_bytes(r1) == _result_bytes(other)
        r3 = small.closest_points(qs, md)
        for k in r1:
            assert r1[k][77].tobytes() == r3[k][5].tobytes() == r3[k][63].tobytes(), k
    # PRB_PIPELINE=fused: a child process from the same state
    code = ('import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n'
            'import numpy as np, np_closest\n'
            'from roboticsplayroompybullet_b200.envs import make\n'
            'e = make(%r, num_envs=%d, seed=9)\n'
            'e.set_state(np.load(%r))\n'
            'out = {}\n'
            'for j, qs in enumerate(np_closest.query_sets(e.model).values()):\n'
            '    for md in %r:\n'
            '        for k, v in e.closest_points(qs, md).items():\n'
            '            out["%%d_%%r_%%s" %% (j, md, k)] = v\n'
            'np.savez(%r, **out)\nprint("DONE")\n') % (ROOT, os.path.join(ROOT, 'tests'), PLAY, n, str(tmp_path / 'state.npy'),
                                                     MAX_DISTANCES, str(tmp_path / 'fused.npz'))
    p = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, PRB_PIPELINE='fused'), capture_output=True,
                       text=True, timeout=900)
    assert 'DONE' in p.stdout, p.stdout + p.stderr
    fused = np.load(str(tmp_path / 'fused.npz'))
    i = 0
    for j, _ in enumerate(np_closest.query_sets(a.model)):
        for md in MAX_DISTANCES:
            for k, v in results[i].items():
                assert fused['%d_%r_%s' % (j, md, k)].tobytes() == v.tobytes(), (j, md, k)
            i += 1
    a.close(); b.close(); small.close()


def test_invalid_calls_launch_nothing():
    import torch
    env = make(PLAY, num_envs=4, seed=2)
    env.reset()
    n0 = env.launch_count()
    for qs, md in (([], 0.1), ([(0, 1)] * 65, 0.1), ([(99, 1)], 0.1), ([((0, 999), 1)], 0.1), ([(0, 1)], float('nan')),
                   ([(0, 1)], -1.0)):
        with pytest.raises(ValueError):
            env.closest_points(qs, md)
    buf = torch.zeros(64, device='cuda')
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    q1 = (lib.PrbClosestQuery * 1)(lib.PrbClosestQuery(1, 2))
    for c, qq, ptrs in ((lib.PrbClosest(0, 0, 0.1, 0), q1, 3), (lib.PrbClosest(65, 0, 0.1, 0), q1, 3),
                        (lib.PrbClosest(1, 1, 0.1, 0), q1, 3), (lib.PrbClosest(1, 0, 0.1, 1), q1, 3),
                        (lib.PrbClosest(1, 0, float('inf'), 0), q1, 3), (lib.PrbClosest(1, 0, -1.0, 0), q1, 3),
                        (lib.PrbClosest(1, 0, 0.1, 0), None, 3), (lib.PrbClosest(1, 0, 0.1, 0), q1, 2)):
        args = [p(buf)] * ptrs + [None] * (3 - ptrs)
        assert env.L.prb_closest_points(env._h, ctypes.byref(c), qq, *args, None, None, None, None) != 0
        assert env.L.prb_last_error(env._h).decode().startswith('prb_closest_points: ')
    assert env.launch_count() == n0
    r = env.closest_points([(0, -1)], 10.0)                      # the handle is still usable
    assert (r['collider_a'] >= 0).all() and env.launch_count() == n0 + 1
    env.close()
