"""GPU tests of ray casting (prb_ray_test): no side effects on the simulation, agreement with the independent numpy
reference tests/np_rays.py and with the step's gripper_proprioception at scale, determinism, env_offset and batch
independence, shared against per-env rays, a call past 2^31 output floats, invalid input."""
import ctypes

import numpy as np
import pytest

import np_rays
from helpers import OBS_KEYS, random_actions
from roboticsplayroompybullet_b200 import lib
from roboticsplayroompybullet_b200.envs import make

pytestmark = pytest.mark.gpu

PLAY = 'UR5PlayAbsRPY1Obj-v0'


def _sets(env, rng):
    """The three ray sets: (from, to, site) with 256 random per-env world segments, the 8 x 8 site-0 fan, the 32 x 32
    height scan."""
    st = env.get_state()
    rnd = [np_rays.random_segments(env.model, st[i], 256, rng) for i in range(env.num_envs)]
    return [(np.stack([r[0] for r in rnd]).astype(np.float32), np.stack([r[1] for r in rnd]).astype(np.float32), None),
            (*np_rays.site_fan(), 0), (*np_rays.height_scan(env.model), None)]


def test_rays_have_no_side_effects():
    """Two handles, one casting the three sets after every step: bit-identical states, outputs and contact reports, and
    the only extra launches are the ray calls."""
    n = 64
    a = make(PLAY, num_envs=n, seed=17, record_contacts=True)
    b = make(PLAY, num_envs=n, seed=17, record_contacts=True)
    oa, ob = a.reset(), b.reset()
    rng, srng = np.random.default_rng(5), np.random.default_rng(6)
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
        for frm, to, site in _sets(b, srng):
            b.ray_test_batch_device(frm, to, site=site)
            calls += 1
    assert a.get_state().tobytes() == b.get_state().tobytes()
    assert b.launch_count() - a.launch_count() == calls
    a.close(); b.close()


def test_gpu_matches_numpy_and_proprioception_at_scale():
    n = 8192
    env = make(PLAY, num_envs=n, seed=23)
    env.reset()
    rng = np.random.default_rng(2)
    for k in range(12):
        a = random_actions(rng, n, PLAY)
        if k >= 6:
            a[:, -1] = -1.0                 # close the gripper: some envs grasp the block
        obs, _, _, _ = env.step(a)
    st = env.get_state()
    # proprioception on every env: the fp64 gripper ray through the kernel, phase_observe's rule on the result
    rays = [np_rays.proprio_ray(env.model, st[i]) for i in range(n)]
    frm = np.stack([r[0] for r in rays])[:, None, :].astype(np.float32)
    to = np.stack([r[1] for r in rays])[:, None, :].astype(np.float32)
    got = env.ray_test_batch(frm, to)
    flag = obs['gripper_proprioception']
    bad = [i for i in range(n) if np_rays.proprio_flag(env.model, got['collider'][i, 0], got['fraction'][i, 0]) != flag[i]]
    for i in bad:
        assert np_rays.ray_test(env.model, st[i], frm[i], to[i])['ambiguous'][0], i
    assert flag.min() == 0 and flag.max() == 1
    # the three sets against numpy on 256 envs, those grasping the block first
    grasp = np.nonzero(flag == 1)[0][:64]
    sample = np.unique(np.r_[grasp, np.random.default_rng(4).choice(n, 256 - len(grasp), replace=False)])[:256]
    for frm, to, site in _sets(env, np.random.default_rng(8)):
        out = env.ray_test_batch(frm, to, site=site)
        amb = []
        for i in sample:
            f, t = (frm[i], to[i]) if frm.ndim == 3 else (frm, to)
            ref = np_rays.ray_test(env.model, st[i], f, t, site=site)
            amb.append(np_rays.assert_agrees((out['collider'][i], out['fraction'][i], out['position'][i], out['normal'][i]),
                                             ref, None)['ambiguous'])
        assert np.mean(amb) <= 0.02, np.mean(amb)
        body = np.asarray(env.model['col_body'])
        c = out['collider']
        assert np.array_equal(out['body'], np.where(c >= 0, body[np.maximum(c, 0)], -1))
    env.close()


def test_same_bits_across_calls_handles_and_layouts():
    n = 128
    a = make(PLAY, num_envs=n, seed=9)
    a.reset()
    rng = np.random.default_rng(1)
    for _ in range(4):
        a.step(random_actions(rng, n, PLAY))
    st = a.get_state()
    b = make(PLAY, num_envs=n, seed=9, env_offset=1000)
    b.set_state(st)
    small = make(PLAY, num_envs=64, seed=3)
    small.set_state(np.repeat(st[77:78], 64, 0))
    for frm, to, site in _sets(a, np.random.default_rng(2))[1:] + [(*np_rays.random_segments(a.model, st[0], 1500, rng), None)]:
        r1 = a.ray_test_batch(frm, to, site=site)
        for other in (a.ray_test_batch(frm, to, site=site), b.ray_test_batch(frm, to, site=site),
                      a.ray_test_batch(np.broadcast_to(frm, (n,) + frm.shape).copy(), np.broadcast_to(to, (n,) + to.shape).copy(), site=site)):
            for k in r1:
                assert r1[k].tobytes() == other[k].tobytes(), k
        r3 = small.ray_test_batch(frm, to, site=site)
        for k in r1:
            assert r1[k][77].tobytes() == r3[k][5].tobytes(), k
    a.close(); b.close(); small.close()


def test_large_call_past_2_31_and_invalid_calls():
    import torch
    N, R = 65536, 10923                      # N R 3 = 2 147 549 184 > 2^31 position floats
    env = make(PLAY, num_envs=N, seed=31)
    env.reset()
    env.step(random_actions(np.random.default_rng(0), N, PLAY))
    st = env.get_state()
    frm, to = np_rays.random_segments(env.model, st[-1], R, np.random.default_rng(3))
    f, t = (torch.as_tensor(x, dtype=torch.float32, device='cuda') for x in (frm, to))
    col = torch.empty((N, R), dtype=torch.int32, device='cuda')
    frac = torch.empty((N, R), dtype=torch.float32, device='cuda')
    pos = torch.empty((N, R, 3), dtype=torch.float32, device='cuda')
    r = lib.PrbRays(R, 0, -1, 0, 0xFFFFFFFFFFFFFFFF)
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    lib.check(env.L, env._h, env.L.prb_ray_test(env._h, ctypes.byref(r), p(f), p(t), p(col), p(frac), p(pos), None, None))
    last = {'collider': col[-1].cpu().numpy(), 'fraction': frac[-1].cpu().numpy(), 'position': pos[-1].cpu().numpy()}
    del col, frac, pos
    one = make(PLAY, num_envs=1, seed=31)
    one.set_state(st[-1:])
    ref = one.ray_test_batch(frm, to)
    for k in last:
        assert last[k].tobytes() == ref[k][0].tobytes(), k
    # invalid calls raise and launch nothing
    n0 = one.launch_count()
    good = np.zeros((4, 3), np.float32)
    for args, kw in (((np.zeros((4, 3)), np.zeros((5, 3))), {}), ((good, good), {'site': 4}), ((np.zeros((0, 3)), np.zeros((0, 3))), {}),
                     ((np.full((4, 3), np.nan), good), {}), ((np.zeros((2, 4, 3)), np.zeros((2, 4, 3))), {})):
        with pytest.raises(ValueError):
            one.ray_test_batch(*args, **kw)
    buf = torch.zeros(64, device='cuda')
    for rr, ptrs in ((lib.PrbRays(0, 0, -1, 0, 1), 4), (lib.PrbRays(16385, 0, -1, 0, 1), 4), (lib.PrbRays(4, 0, 4, 0, 1), 4),
                     (lib.PrbRays(4, 3, -1, 0, 1), 4), (lib.PrbRays(4, 0, -1, 7, 1), 4), (lib.PrbRays(4, 0, -1, 0, 1), 3)):
        q = [p(buf)] * ptrs + [None] * (4 - ptrs)
        assert one.L.prb_ray_test(one._h, ctypes.byref(rr), *q, None, None, None) != 0
        assert one.L.prb_last_error(one._h).decode().startswith('prb_ray_test: ')
    assert one.launch_count() == n0
    one.ray_test_batch(good, good + 1)                              # the handle is still usable
    env.close(); one.close()
