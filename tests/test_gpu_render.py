"""GPU tests of camera rendering (prb_render): the 'img' observation, no side effects on the simulation, agreement
with the independent numpy ray caster tests/np_render.py, determinism, cameras and sizes, invalid input."""
import ctypes

import numpy as np
import pytest

import np_render
from helpers import OBS_KEYS, random_actions
from roboticsplayroompybullet_b200.camera import Camera, default_camera, gripper_camera, projection_matrix_fov, view_matrix
from roboticsplayroompybullet_b200.envs import make
from roboticsplayroompybullet_b200.lib import PrbError

pytestmark = pytest.mark.gpu

IDS = ['UR5PlayAbsRPY1Obj-v0', 'pandaPick-v0', 'UR5Reach-v0']


def _agree(env, frames, cam, envs):
    st = env.get_state()
    # the 2 % cap on ambiguous pixels is for frames of real size: in a 16 x 8 frame one silhouette edge is 2 %
    max_amb = 0.02 if cam.width * cam.height >= 1024 else 1.0
    for i in envs:
        ref = np_render.render(env.model, st[i], cam, env.palette)
        r = np_render.compare((frames['rgb'][i], frames['depth'][i], frames['segmentation'][i]), ref)
        assert r['seg_mismatch'] == 0 and r['ambiguous'] <= max_amb and r['depth_rel'] <= 1e-5 and r['rgb'] <= 1, (i, r)


@pytest.mark.parametrize('env_id', IDS)
def test_img_layout(env_id):
    import torch
    n = 4
    env = make(env_id, num_envs=n, seed=3, record_images=True)
    for obs in (env.reset(), env.step(random_actions(np.random.default_rng(0), n, env_id))[0], env.observe()):
        assert obs['img'].shape == (n, 200, 200, 3) and obs['img'].dtype == np.uint8
        assert len(np.unique(obs['img'][0].reshape(-1, 3), axis=0)) > 4       # not a blank frame
    obs, _, _, _ = env.step_device(torch.as_tensor(random_actions(np.random.default_rng(1), n, env_id), device='cuda'))
    assert obs['img'].is_cuda and obs['img'].dtype == torch.uint8 and tuple(obs['img'].shape) == (n, 200, 200, 3)
    off = make(env_id, num_envs=n, seed=3)
    assert off.reset()['img'] is None
    env.close(); off.close()


def test_rendering_has_no_side_effects():
    """The same seed with and without record_images: bit-identical outputs and states over 20 scripted steps, and the
    only extra launches are the renders."""
    env_id, n = 'UR5PlayAbsRPY1Obj-v0', 64
    a, b = make(env_id, num_envs=n, seed=17), make(env_id, num_envs=n, seed=17, record_images=True)
    oa, ob = a.reset(), b.reset()
    rng = np.random.default_rng(5)
    for s in range(20):
        for k in OBS_KEYS:
            assert np.array_equal(oa[k], ob[k]), (s, k)
        assert a.get_state().tobytes() == b.get_state().tobytes(), s
        act = random_actions(rng, n, env_id)
        (oa, ra, _, ia), (ob, rb, _, ib) = a.step(act), b.step(act)
        assert np.array_equal(ra, rb) and np.array_equal(ia['target_poses'], ib['target_poses'])
    assert b.launch_count() - a.launch_count() == 21                    # one render per reset / step
    a.close(); b.close()


def test_gpu_matches_numpy_at_scale():
    env_id, n = 'UR5PlayAbsRPY1Obj-v0', 4096
    env = make(env_id, num_envs=n, seed=23)
    env.reset()
    rng = np.random.default_rng(2)
    for _ in range(6):
        env.step(random_actions(rng, n, env_id))
    sample = np.sort(np.random.default_rng(4).choice(n, 16, replace=False))
    for cam, envs in ((env.camera, sample), (gripper_camera(env.model), sample[:4])):
        frames = env.render(cam, depth=True, segmentation=True)
        _agree(env, frames, cam, envs)
    env.close()


def test_render_is_deterministic_and_independent_of_env_offset():
    env_id, n = 'UR5PlayAbsRPY1Obj-v0', 128
    a = make(env_id, num_envs=n, seed=9)
    a.reset()
    b = make(env_id, num_envs=n, seed=9, env_offset=1000)
    b.set_state(a.get_state())
    ra = a.render(depth=True, segmentation=True)
    for other in (a.render(depth=True, segmentation=True), b.render(depth=True, segmentation=True)):
        for k in ra:
            assert np.array_equal(ra[k], other[k]), k
    a.close(); b.close()


@pytest.mark.parametrize('n', [1, 33])
def test_cameras_and_sizes(n):
    env_id = 'pandaPick-v0'
    env = make(env_id, num_envs=n, seed=31)
    env.reset()
    custom = Camera(61, 37, view_matrix([0.6, -0.5, 0.5], [0.0, 0.0, 0.0], [0, 0, 1]), projection_matrix_fov(50.0, 61 / 37, 0.05, 3.0))
    for cam in (gripper_camera(env.model, 40, 72), custom, default_camera(env.model, 16, 8)):
        frames = env.render(cam, depth=True, segmentation=True)
        assert frames['rgb'].shape == (n, cam.height, cam.width, 3)
        assert frames['depth'].shape == frames['segmentation'].shape == (n, cam.height, cam.width)
        _agree(env, frames, cam, range(min(n, 4)))
    env.close()


def test_invalid_input_raises():
    env = make('UR5Reach-v0', num_envs=2, seed=1)
    env.reset()
    good = default_camera(env.model, 16, 16)
    bad = [Camera(0, 16, good.view, good.proj), Camera(1025, 16, good.view, good.proj),
           Camera(16, 16, np.zeros(16), good.proj), Camera(16, 16, good.view, np.zeros(16)),
           Camera(16, 16, good.view, good.proj, light_dir=(0, 0, 0))]
    for cam in bad:
        with pytest.raises(PrbError):
            env.render(cam)
    from roboticsplayroompybullet_b200.camera import camera_struct
    pal = np.ascontiguousarray(env.palette, np.float32)
    rc = env.L.prb_render(env._h, ctypes.byref(camera_struct(good)), ctypes.c_void_p(pal.ctypes.data), None, None, None, None)
    assert rc != 0                                                  # rgb_dev is required
    env.render(good)                                                # the handle is still usable
    env.close()
