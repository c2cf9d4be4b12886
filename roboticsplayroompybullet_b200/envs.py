"""Vectorised mirror of the reference's gym surface (roboticsPlayroomPybullet/envs/
environments.py:58-314 `playEnv`, envList.py:18-22, 89-99) on top of the C-ABI.

`VecPlayEnv` keeps the reference's method names, argument meaning, dict keys and per-key
layouts, with a leading [num_envs] dimension:

    reset(mask=None) -> obs dict          (playEnv.reset, :173-187)
    step(action[N,7]) -> (obs, r[N], done[N], info)   (playEnv.step, :206-214)
    reset_goal_pos(goal[N,G])             (:190-191)
    compute_reward(ag, dg[, info])        (:274-304; sparse variant bound when sparse=True, :169-170)
    _max_episode_steps, action_space / observation_space bounds as arrays

Two calling styles: numpy in / numpy out (`step`), which goes through host buffers exactly like a
reference user would (H2D of actions, D2H of the whole observation block every step), and
`step_device` for learners that keep everything on the GPU (torch tensors, zero-copy views of the
library's buffers).

With record_images=True every observation also carries 'img' (environments.py:841-845): a uint8 [N,H,W,3] frame of
`camera` (default: camera.default_camera) rendered on the GPU by prb_render after the step.  render() / render_device()
draw any other camera (e.g. camera.gripper_camera) with optional depth and segmentation.

With record_contacts=True every step also fills the contact report (PyBullet's getContactPoints after stepSimulation, for
all envs at once): contacts_device() / contacts() return each env's contact points and forces of the step's last substep.

With per_env_dynamics=True every env has its own collider friction and free-body mass, inertia and damping (PyBullet's
changeDynamics per client): change_dynamics() sets them, dynamics_device() / dynamics() return them.  With
randomize_dynamics={field: (lo, hi)} every sampled reset first draws new values for the envs it resets (domain
randomization).

ray_test_batch_device() / ray_test_batch() cast rays against every env's collision boxes (PyBullet's rayTestBatch for all
envs at once): the same rays in every env or rays per env, in the world or in a site of the arm.

closest_points_device() / closest_points() give the nearest pair of collision boxes between two bodies or links in every
env (PyBullet's getClosestPoints for all envs at once): signed distance, witness points and normal.

calculate_jacobian_device(), calculate_mass_matrix_device() and calculate_inverse_dynamics_device() (and their numpy
twins) give the arm's point Jacobians, joint-space mass matrix and inverse dynamics in every env (PyBullet's
calculateJacobian, calculateMassMatrix and calculateInverseDynamics for all envs at once); arm_dof_joints maps their
columns to PyBullet joint indices.

body_states_device() / joint_states_device() read every link, free body and slide body frame and every joint of every
env (PyBullet's getLinkStates, getBasePositionAndOrientation, getBaseVelocity, getJointStates);
reset_joint_states_device() / reset_base_states_device() write them for masked envs (resetJointState,
resetBasePositionAndOrientation, resetBaseVelocity); save_state_device() / restore_state_device() keep and restore
device-side snapshots (saveState / restoreState).  Each has a numpy twin.
"""
import math
import ctypes

import numpy as np

from . import lib as _lib
from .camera import camera_struct, default_camera, default_palette
from .model import ACTION_VARIANTS, ENV_KINDS, action_dim, load_model

OUT_KEYS = ['obs_quat', 'achieved_goal', 'desired_goal', 'controllable_achieved_goal', 'full_positional_state',
            'joints', 'velocity', 'observation', 'gripper_proprioception', 'reward', 'is_success', 'target_poses']
OBS_KEYS = OUT_KEYS[:9]


class _DevArray:
    """Exposes a library-owned device buffer through __cuda_array_interface__ (zero-copy)."""

    def __init__(self, ptr, shape, owner, typestr='<f4'):
        self.__cuda_array_interface__ = {'shape': tuple(shape), 'typestr': typestr, 'data': (int(ptr), False),
                                         'version': 2, 'strides': None}
        self._owner = owner


class VecPlayEnv:
    env_id = None

    def __init__(self, env_id=None, num_envs=1, device=0, seed=1234, env_offset=0, sparse=True, model=None,
                 record_images=False, camera=None, record_contacts=False, per_env_dynamics=False, randomize_dynamics=None):
        import torch  # device memory / streams only
        self.torch = torch
        env_id = env_id or self.env_id
        if not sparse:
            # The reference binds compute_reward once and uses it in step() AND in the reset retry loop
            # (environments.py:169-170, 185, 210); with the dense reward that loop only ends when the sampled goal
            # is >= 1 m away.  No registered id uses it; the in-kernel reward is the sparse one.
            raise NotImplementedError('sparse=False (dense reward inside step/reset) is not supported; '
                                      'use dense_reward(ag, dg) for the dense metric')
        if env_id not in ENV_KINDS and env_id not in ACTION_VARIANTS:
            raise NotImplementedError(env_id)           # environments.py:376,416,933
        self.env_id = env_id
        self.model = model if model is not None else load_model(env_id)
        m = self.model
        self.num_envs = int(num_envs)
        self.device = torch.device('cuda', device)
        self.L = _lib.load()
        self._ms = m.as_struct()
        cfg = _lib.PrbConfig(self.num_envs, int(env_offset), int(device), 0, int(seed))
        self._h = ctypes.c_void_p()
        rc = self.L.prb_create(ctypes.byref(self._ms), ctypes.byref(cfg), ctypes.byref(self._h))
        if rc != 0:
            raise _lib.PrbError('prb_create failed (%d): %s' % (rc, self.L.prb_last_error(self._h).decode()))
        b = _lib.PrbBuffers()
        _lib.check(self.L, self._h, self.L.prb_get_buffers(self._h, ctypes.byref(b)))
        self.buffers = b
        N = self.num_envs
        self.dims = {'obs_quat': b.obs_dim, 'achieved_goal': b.goal_dim, 'desired_goal': b.goal_dim,
                     'controllable_achieved_goal': 4, 'full_positional_state': b.fps_dim, 'joints': 8,
                     'velocity': 6, 'observation': b.observation_dim, 'gripper_proprioception': 1, 'reward': 1,
                     'is_success': 1, 'target_poses': b.n_ik}
        self.out_floats = int(b.out_floats)
        with torch.cuda.device(self.device):
            self.dev = {k: torch.as_tensor(_DevArray(getattr(b, k), (N, self.dims[k]), self), device=self.device)
                        for k in OUT_KEYS}
            self.state_dev = torch.as_tensor(_DevArray(b.state, (N, b.state_stride), self), device=self.device)
        # pinned host staging for the numpy path
        self.action_dim = action_dim(self.model)
        self._h_action = torch.empty((N, self.action_dim), dtype=torch.float32).pin_memory()
        self._h_out = torch.empty((self.out_floats,), dtype=torch.float32).pin_memory()
        self._h_views = {}
        self._h_slices = {}
        off = 0
        for k in OUT_KEYS:
            n = N * self.dims[k]
            self._h_views[k] = self._h_out[off:off + n].view(N, self.dims[k]).numpy()
            self._h_slices[k] = (off, off + n)
            off += n
        self._h_out_np = self._h_out.numpy()
        # gym-like metadata (environments.py:84,108-117)
        self._max_episode_steps = None if m['play'] else 250
        high = np.array([m.param('action_high_xyz')] * (self.action_dim - 1) + [m.param('action_high_grip')], np.float32)   # :88-112
        self.action_low, self.action_high = -high, high
        self.play = bool(m['play'])
        self.sparse = sparse
        self.h2d_bytes_per_step = N * self.action_dim * 4
        self.d2h_bytes_per_step = self.out_floats * 4
        # camera images (calc_state 'img'): rendered only when asked for; colours per collider, [n_col, 3] in [0, 1]
        self.record_images = bool(record_images)
        self.camera = camera if camera is not None else default_camera(m)
        self.palette = default_palette(m)
        self._img = None
        if self.record_images:
            self._img = torch.empty((N, self.camera.height, self.camera.width, 3), dtype=torch.uint8, device=self.device)
        self._col_tables = None
        # contact report: allocated by the library when first enabled
        self._record_contacts = False
        self._contact_views = None
        self.record_contacts = record_contacts
        # per-env dynamics table: allocated by the library when first enabled
        self._per_env_dynamics = False
        self._dyn_views = None
        self._dyn_ranges = None
        self.per_env_dynamics = per_env_dynamics
        self.randomize_dynamics = randomize_dynamics

    @property
    def per_env_dynamics(self):
        """True: every env runs with its own row of the dynamics table (dynamics_device, change_dynamics).  Turning it on
        fills every row with the model's values; turning it off also turns randomize_dynamics off."""
        return self._per_env_dynamics

    @per_env_dynamics.setter
    def per_env_dynamics(self, on):
        on = bool(on)
        if on != self._per_env_dynamics:
            _lib.check(self.L, self._h, self.L.prb_enable_dynamics(self._h, 1 if on else 0))
            self._per_env_dynamics = on
        if not on:
            self._dyn_ranges = None

    @property
    def randomize_dynamics(self):
        """{field: (lo, hi)} scale ranges of the model's values that every sampled reset draws from (None: no draw).
        Fields: lateral_friction, spinning_friction (one draw per body), mass, linear_damping, angular_damping (one per
        free body; the inertia follows mass); the ones not given keep (1, 1).  Setting it turns per_env_dynamics on."""
        if self._dyn_ranges is None:
            return None
        return {k: tuple(getattr(self._dyn_ranges, k)) for k in _lib.DYNAMICS_RANGE_FIELDS}

    @randomize_dynamics.setter
    def randomize_dynamics(self, spec):
        if spec is None:
            self._dyn_ranges = None
            return
        r = dynamics_ranges(spec)
        self.per_env_dynamics = True
        self._dyn_ranges = r

    @property
    def record_contacts(self):
        """True: every step / substeps call refreshes the contact report (contacts_device, contacts)."""
        return self._record_contacts

    @record_contacts.setter
    def record_contacts(self, on):
        on = bool(on)
        if on != self._record_contacts:
            _lib.check(self.L, self._h, self.L.prb_enable_contacts(self._h, 1 if on else 0))
            self._record_contacts = on

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _obs_dev(self):
        d = {k: self.dev[k] for k in OBS_KEYS}
        if self.record_images:
            d['img'] = self._render_img()
        return d

    def _render_img(self):
        """'img' of the current state into the handle's frame buffer (allocated again if self.camera changed size)."""
        cam = self.camera
        if self._img is None or self._img.shape[1:3] != (cam.height, cam.width):
            self._img = self.torch.empty((self.num_envs, cam.height, cam.width, 3), dtype=self.torch.uint8, device=self.device)
        self._render(cam, self._img)
        return self._img

    def _render(self, camera, rgb, depth=None, seg=None):
        cs = camera_struct(camera)
        pal = np.ascontiguousarray(self.palette, np.float32)
        assert pal.shape == (int(self.model['n_col']), 3), 'palette must be [n_col, 3]'
        ptr = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        _lib.check(self.L, self._h, self.L.prb_render(self._h, ctypes.byref(cs), ctypes.c_void_p(pal.ctypes.data), ptr(rgb),
                                                     ptr(depth), ptr(seg), self._stream()))

    def _body_link(self, ids):
        """(body, link) int32 CUDA tensors of collider ids (-1 stays -1): body -1 static, 0 arm, 1.. free bodies, then
        slide bodies; link the PyBullet link index (col_urdf_link)."""
        t = self.torch
        if self._col_tables is None:
            n_col = int(self.model['n_col'])
            self._col_tables = [t.as_tensor(np.asarray(self.model[key])[:n_col].astype(np.int32), device=self.device)
                                for key in ('col_body', 'col_urdf_link')]
        i = ids.clamp(min=0).long()
        return tuple(t.where(ids >= 0, tab[i], ids) for tab in self._col_tables)

    def _host_copy(self):
        """Fresh arrays for the caller (the reference returns copies, environments.py:850-855): ONE copy of the pinned result
        block, the per-key arrays are views of it."""
        buf = self._h_out_np.copy()
        return {k: buf[a:b].reshape(self.num_envs, self.dims[k]) for k, (a, b) in self._h_slices.items()}

    def _obs_host(self, c=None):
        c = c if c is not None else self._host_copy()
        d = {k: c[k] for k in OBS_KEYS}
        d['gripper_proprioception'] = d['gripper_proprioception'][:, 0].astype(np.int64)
        d['img'] = self._img.cpu().numpy() if self.record_images else None    # environments.py:841-845
        return d

    def close(self):
        if getattr(self, '_h', None) is not None and self._h:
            self.L.prb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ device-resident API
    def reset_device(self, mask=None, o=None, restore_env=True):
        """reset() of the masked envs (all when mask is None).  With `o` ([N, obs_dim] float32 CUDA tensor in the obs_quat
        layout) the envs are re-seated from that observation instead of sampled: playEnv.reset(o), trajectory replay."""
        mp = None
        if mask is not None:
            self._mask = mask.to(self.device, self.torch.uint8).contiguous()
            mp = ctypes.c_void_p(self._mask.data_ptr())
        if o is None and self._dyn_ranges is not None:      # new dynamics before the objects settle
            _lib.check(self.L, self._h, self.L.prb_randomize_dynamics(self._h, ctypes.byref(self._dyn_ranges), mp, self._stream()))
        if o is not None:
            ob = o.to(self.device, self.torch.float32).contiguous()
            assert ob.shape == (self.num_envs, self.dims['obs_quat']), 'o must be [num_envs, %d] (obs_quat layout)' % self.dims['obs_quat']
            self._o_keep = ob
            _lib.check(self.L, self._h, self.L.prb_reset_to(self._h, ctypes.c_void_p(ob.data_ptr()), mp, 1 if restore_env else 0, self._stream()))
        else:
            _lib.check(self.L, self._h, self.L.prb_reset(self._h, mp, self._stream()))
        return self._obs_dev()

    def step_device(self, action):
        """action: float32 CUDA tensor [N,7].  Returns views of the library's output buffers."""
        a = action.to(self.device, self.torch.float32).contiguous()
        assert a.shape == (self.num_envs, self.action_dim), 'action must be [num_envs, %d]' % self.action_dim   # environments.py:937,956
        self._a_keep = a
        _lib.check(self.L, self._h, self.L.prb_step(self._h, ctypes.c_void_p(a.data_ptr()), self._stream()))
        info = {'is_success': self.dev['is_success'][:, 0], 'target_poses': self.dev['target_poses']}
        return self._obs_dev(), self.dev['reward'][:, 0], None, info

    def observe_device(self):
        _lib.check(self.L, self._h, self.L.prb_observe(self._h, self._stream()))
        return self._obs_dev()

    # ------------------------------------------------------------------ reference-style (numpy) API
    def reset(self, o=None, mask=None, restore_env=True):
        """playEnv.reset(o=None) (environments.py:173-187) for every env, or for the envs of `mask`.  `o`: [N, obs_dim]
        obs_quat rows to re-seat the envs from (trajectory replay) instead of sampling."""
        mt = None
        if mask is not None:
            mt = self.torch.as_tensor(np.asarray(mask, np.uint8))
        ot = None
        if o is not None:
            ot = self.torch.as_tensor(np.ascontiguousarray(np.asarray(o, np.float32)).reshape(self.num_envs, -1))
        self.reset_device(mt, ot, restore_env)
        self.torch.cuda.current_stream(self.device).synchronize()
        self._pull()
        return self._obs_host()

    def _pull(self):
        t = self.torch
        with t.cuda.device(self.device):
            src = t.as_tensor(_DevArray(self.buffers.out_base, (self.out_floats,), self), device=self.device)
            self._h_out.copy_(src, non_blocking=True)
            t.cuda.current_stream(self.device).synchronize()

    def step(self, action):
        a = np.asarray(action, np.float32)
        assert a.shape == (self.num_envs, self.action_dim), 'action must be [num_envs, %d]' % self.action_dim
        self._h_action.numpy()[...] = a
        # the result block lands in a fresh array (the reference returns new arrays every step, environments.py:850-855):
        # prb_step_host reads it back through pinned staging in chunks and copies them out with worker threads
        buf = np.empty(self.out_floats, np.float32)
        _lib.check(self.L, self._h, self.L.prb_step_host(self._h, ctypes.c_void_p(self._h_action.data_ptr()),
                                                        ctypes.c_void_p(buf.ctypes.data), self._stream()))
        c = {k: buf[i:j].reshape(self.num_envs, self.dims[k]) for k, (i, j) in self._h_slices.items()}
        r = c['reward'][:, 0]
        info = {'is_success': c['is_success'][:, 0].astype(np.int64), 'target_poses': c['target_poses']}
        done = np.zeros(self.num_envs, dtype=bool)       # environments.py:212: always False
        if self.record_images:
            self._render_img()
        return self._obs_host(c), r, done, info

    def reset_goal_pos(self, goal):
        t = self.torch
        g = t.as_tensor(np.asarray(goal, np.float32)).reshape(self.num_envs, -1).to(self.device).contiguous()
        assert g.shape == (self.num_envs, self.dims['desired_goal']), 'goal must be [num_envs, %d]' % self.dims['desired_goal']
        self._g_keep = g
        _lib.check(self.L, self._h, self.L.prb_set_goal(self._h, ctypes.c_void_p(g.data_ptr()), None, self._stream()))

    def reset_goal_pos_device(self, goal, mask=None):
        """Device-resident reset_goal_pos (environments.py:190-191) for goal relabelling inside a rollout loop:
        goal float32 CUDA tensor [N, goal_dim], optional uint8 mask [N]."""
        t = self.torch
        g = goal.to(self.device, t.float32).reshape(self.num_envs, -1).contiguous()
        assert g.shape == (self.num_envs, self.dims['desired_goal']), 'goal must be [num_envs, %d]' % self.dims['desired_goal']
        self._g_keep = g
        mp = None
        if mask is not None:
            self._gmask = mask.to(self.device, t.uint8).contiguous()
            mp = ctypes.c_void_p(self._gmask.data_ptr())
        _lib.check(self.L, self._h, self.L.prb_set_goal(self._h, ctypes.c_void_p(g.data_ptr()), mp, self._stream()))

    def compute_reward(self, achieved_goal, desired_goal, info=None):
        """Batched compute_reward_sparse (sparse=True) or dense -||ag-dg|| (environments.py:274-304)."""
        t = self.torch
        ag = np.asarray(achieved_goal, np.float32)
        dg = np.asarray(desired_goal, np.float32)
        single = ag.ndim == 1
        G = self.dims['achieved_goal']
        assert ag.shape[-1] == G and dg.shape == ag.shape, 'goals must be [..., %d]' % G
        agd = t.as_tensor(ag.reshape(-1, G)).to(self.device).contiguous()
        dgd = t.as_tensor(dg.reshape(-1, G)).to(self.device).contiguous()
        out = t.empty(agd.shape[0], dtype=t.float32, device=self.device)
        _lib.check(self.L, self._h, self.L.prb_compute_reward(self._h, ctypes.c_void_p(agd.data_ptr()),
                                                             ctypes.c_void_p(dgd.data_ptr()), agd.shape[0],
                                                             ctypes.c_void_p(out.data_ptr()), self._stream()))
        r = out.cpu().numpy()
        return r[0] if single else r

    compute_reward_sparse = compute_reward

    def dense_reward(self, achieved_goal, desired_goal):
        """playEnv.compute_reward before the sparse rebinding (environments.py:269-275): -||ag - dg|| (host numpy)."""
        G = self.dims['achieved_goal']
        ag = np.asarray(achieved_goal, np.float32)
        d = -np.linalg.norm(ag.reshape(-1, G) - np.asarray(desired_goal, np.float32).reshape(-1, G), axis=1)
        return d[0] if ag.ndim == 1 else d

    def compute_reward_device(self, ag, dg):
        t = self.torch
        G = self.dims['achieved_goal']
        agd = ag.reshape(-1, G).to(self.device, t.float32).contiguous()
        dgd = dg.reshape(-1, G).to(self.device, t.float32).contiguous()
        out = t.empty(agd.shape[0], dtype=t.float32, device=self.device)
        _lib.check(self.L, self._h, self.L.prb_compute_reward(self._h, ctypes.c_void_p(agd.data_ptr()),
                                                             ctypes.c_void_p(dgd.data_ptr()), agd.shape[0],
                                                             ctypes.c_void_p(out.data_ptr()), self._stream()))
        return out

    # ------------------------------------------------------------------ camera images
    def render_device(self, camera=None, depth=False, segmentation=False):
        """Frame of the current state from `camera` (default: the env's camera): dict of CUDA tensors 'rgb' uint8
        [N,H,W,3] and, when asked for, 'depth' float32 [N,H,W] (eye-space depth in metres, the far plane where nothing
        is hit) and 'segmentation' int32 [N,H,W] (collider index, -1 where nothing is hit).  Asynchronous."""
        cam = camera if camera is not None else self.camera
        t, N, H, W = self.torch, self.num_envs, cam.height, cam.width
        out = {'rgb': t.empty((N, H, W, 3), dtype=t.uint8, device=self.device)}
        if depth:
            out['depth'] = t.empty((N, H, W), dtype=t.float32, device=self.device)
        if segmentation:
            out['segmentation'] = t.empty((N, H, W), dtype=t.int32, device=self.device)
        self._render(cam, out['rgb'], out.get('depth'), out.get('segmentation'))
        return out

    def render(self, camera=None, depth=False, segmentation=False):
        """render_device() as numpy arrays."""
        return {k: v.cpu().numpy() for k, v in self.render_device(camera, depth, segmentation).items()}

    def render_box_tests(self):
        """Pixel-box tests the renders of this handle have run (after tile culling)."""
        return int(self.L.prb_render_box_tests(self._h))

    # ------------------------------------------------------------------ contact report
    def contacts_device(self):
        """The contacts of the last physics substep of the most recent step (include/prb.h, prb_contacts): dict of CUDA
        tensors 'count' int32 [N]; 'collider_a', 'collider_b' int32 [N,64] (model collider indices, the ids of
        render(segmentation=True)); 'position_on_a', 'position_on_b', 'normal_on_b' float32 [N,64,3] (world, m; the normal
        points from B to A); 'distance', 'normal_force', 'lateral_friction_1', 'lateral_friction_2' float32 [N,64] (m; N);
        'lateral_friction_dir_1', 'lateral_friction_dir_2' float32 [N,64,3]; and 'body_a', 'body_b' (-1 static, 0 arm,
        1.. free bodies, then slide bodies), 'link_a', 'link_b' (PyBullet link index) int32 [N,64] looked up from the
        collider ids.  Entries past count hold -1 (ids) and 0 (floats).  All but the four looked-up arrays are zero-copy
        views of the library's buffers, overwritten by the next step."""
        t = self.torch
        if self._contact_views is None:
            c = _lib.PrbContacts()
            _lib.check(self.L, self._h, self.L.prb_get_contacts(self._h, ctypes.byref(c)))
            N, K = self.num_envs, int(c.max_contacts)
            with t.cuda.device(self.device):
                v = {'count': t.as_tensor(_DevArray(c.count, (N,), self, '<i4'), device=self.device)}
                for name, ty, k in _lib.CONTACT_FIELDS:
                    shape = (N, K) if k == 1 else (N, K, k)
                    v[name] = t.as_tensor(_DevArray(getattr(c, name), shape, self, '<' + ty), device=self.device)
            self._contact_views = v
        d = dict(self._contact_views)
        for side in ('a', 'b'):
            d['body_' + side], d['link_' + side] = self._body_link(d['collider_' + side])
        return d

    def contacts(self):
        """contacts_device() as numpy arrays."""
        return {k: v.cpu().numpy() for k, v in self.contacts_device().items()}

    # ------------------------------------------------------------------ ray casts
    def ray_test_batch_device(self, ray_from, ray_to, site=None, exclude_bodies=()):
        """PyBullet's rayTestBatch(rayFromPositions, rayToPositions) in every env at once (include/prb.h, prb_ray_test): the
        nearest collision box each segment ray_from -> ray_to hits in the current state.  ray_from, ray_to: numpy arrays or
        CUDA tensors [R,3] (the same rays in every env) or [N,R,3] (per env), R in 1..16384, in the world (site None) or
        in site 0..3 of the arm (0 the end effector, 1 the wrist, 2 and 3 the finger pads).  exclude_bodies: body ids
        whose colliders cannot be hit.  Returns a dict of CUDA tensors 'collider' int32 [N,R] (-1: no hit), 'fraction'
        float32 [N,R] (1 for no hit), 'position' and 'normal' float32 [N,R,3] (world; 0 for no hit), and 'body', 'link'
        int32 [N,R] looked up from the collider as contacts() does.  A ray that starts inside a box hits it at fraction 0.
        Asynchronous; ValueError for a bad shape, site or body, or a non-finite numpy input."""
        t = self.torch
        per_env, R, mask = check_rays(self.model, self.num_envs, ray_from, ray_to, site, exclude_bodies)
        f, g = (t.as_tensor(x).to(self.device, t.float32).contiguous() for x in (ray_from, ray_to))
        N = self.num_envs
        out = {'collider': t.empty((N, R), dtype=t.int32, device=self.device),
               'fraction': t.empty((N, R), dtype=t.float32, device=self.device),
               'position': t.empty((N, R, 3), dtype=t.float32, device=self.device),
               'normal': t.empty((N, R, 3), dtype=t.float32, device=self.device)}
        r = _lib.PrbRays(R, per_env, -1 if site is None else int(site), 0, mask)
        ptr = lambda x: ctypes.c_void_p(x.data_ptr())
        _lib.check(self.L, self._h, self.L.prb_ray_test(self._h, ctypes.byref(r), ptr(f), ptr(g), ptr(out['collider']),
                                                       ptr(out['fraction']), ptr(out['position']), ptr(out['normal']),
                                                       self._stream()))
        out['body'], out['link'] = self._body_link(out['collider'])
        return out

    def ray_test_batch(self, ray_from, ray_to, site=None, exclude_bodies=()):
        """ray_test_batch_device() as numpy arrays."""
        return {k: v.cpu().numpy() for k, v in self.ray_test_batch_device(ray_from, ray_to, site, exclude_bodies).items()}

    # ------------------------------------------------------------------ closest points
    def closest_points_device(self, queries, max_distance):
        """PyBullet's getClosestPoints(bodyA, bodyB, distance[, linkIndexA, linkIndexB]) in every env at once (include/prb.h,
        prb_closest_points).  queries: a list of Q in 1..64 pairs (side_a, side_b); a side is a body id (all its colliders)
        or a (body, link) tuple, the ids of contacts(): body -1 static scene, 0 arm, 1.. free bodies, then slide bodies;
        link the PyBullet link index.  For each query the nearest collider pair (a, b), a != b, with signed distance
        <= max_distance (m, inclusive).  Returns a dict of CUDA tensors 'collider_a', 'collider_b', 'body_a', 'body_b',
        'link_a', 'link_b' int32 [N,Q] (-1: no pair within reach), 'distance' float32 [N,Q] (< 0: penetration; inf: no
        pair), 'position_on_a', 'position_on_b', 'normal_on_b' float32 [N,Q,3] (world; the normal points from B to A;
        0 for no pair).  Asynchronous; ValueError for an unknown body or link, no or more than 64 queries, or a
        non-finite or negative max_distance."""
        t = self.torch
        qs, md = check_closest(self.model, queries, max_distance)
        N, Q = self.num_envs, len(qs)
        out = {k: t.empty((N, Q), dtype=t.int32, device=self.device) for k in ('collider_a', 'collider_b')}
        out['distance'] = t.empty((N, Q), dtype=t.float32, device=self.device)
        for k in ('position_on_a', 'position_on_b', 'normal_on_b'):
            out[k] = t.empty((N, Q, 3), dtype=t.float32, device=self.device)
        arr = (_lib.PrbClosestQuery * Q)(*[_lib.PrbClosestQuery(a, b) for a, b in qs])
        c = _lib.PrbClosest(Q, 0, md, 0)
        ptr = lambda x: ctypes.c_void_p(x.data_ptr())
        _lib.check(self.L, self._h, self.L.prb_closest_points(self._h, ctypes.byref(c), arr, *[ptr(out[k]) for k in (
            'collider_a', 'collider_b', 'distance', 'position_on_a', 'position_on_b', 'normal_on_b')], self._stream()))
        for side in ('a', 'b'):
            out['body_' + side], out['link_' + side] = self._body_link(out['collider_' + side])
        return out

    def closest_points(self, queries, max_distance):
        """closest_points_device() as numpy arrays."""
        return {k: v.cpu().numpy() for k, v in self.closest_points_device(queries, max_distance).items()}

    # ------------------------------------------------------------------ arm dynamics
    @property
    def arm_dof_joints(self):
        """PyBullet joint index of each arm DoF, i.e. of each column of the Jacobians, the mass matrix and tau (the model's
        link order; the link ids contacts() reports for body 0)."""
        return np.asarray(self.model['arm_urdf_index'])[:int(self.model['nd'])].copy()

    def _arm_dynamics(self, points, q, qd, qdd, want):
        """One prb_arm_dynamics call that asks for the outputs in `want` only: dict of CUDA tensors."""
        t = self.torch
        N, nd, P = self.num_envs, int(self.model['nd']), len(points)
        shapes = {'jacobian': (N, P, 6, nd), 'position': (N, P, 3), 'velocity': (N, P, 6), 'mass_matrix': (N, nd, nd),
                  'tau': (N, nd)}
        out = {k: t.empty(shapes[k], dtype=t.float32, device=self.device) for k in want}
        ins = [None if x is None else t.as_tensor(x).to(self.device, t.float32).contiguous() for x in (q, qd, qdd)]
        pts = (_lib.PrbArmPoint * max(P, 1))(*[_lib.PrbArmPoint(l, s, (ctypes.c_float * 3)(*o), 0) for l, s, o in points])
        ptr = lambda x: None if x is None else ctypes.c_void_p(x.data_ptr())
        _lib.check(self.L, self._h, self.L.prb_arm_dynamics(
            self._h, ctypes.byref(_lib.PrbArmQuery(P, 0)), pts, *[ptr(x) for x in ins],
            *[ptr(out.get(k)) for k in ('jacobian', 'position', 'velocity', 'mass_matrix', 'tau')], self._stream()))
        return out

    def calculate_jacobian_device(self, local_positions=((0.0, 0.0, 0.0),), link=None, site=0, q=None, qd=None):
        """PyBullet's calculateJacobian(arm, linkIndex, localPosition, q, qd, qdd) in every env at once, for P in 1..16
        points (include/prb.h, prb_arm_dynamics).  The points are local_positions [P,3] (m) in the frame of arm link
        `link` (a PyBullet link index of arm_dof_joints; pass site=None) or of site `site` (0 the end effector, 1 the
        wrist, 2 and 3 the finger pads).  q, qd: numpy arrays or CUDA tensors [N, nd]; each defaults to the env's state.
        Returns a dict of CUDA tensors 'linear' and 'angular' float32 [N,P,3,nd] (world frame; columns in arm_dof_joints
        order), 'position' [N,P,3] (world) and 'velocity' [N,P,6] (J qd: linear, angular).  Asynchronous; ValueError for
        a bad shape, an unknown link or site, both or neither of link and site, or a non-finite numpy input."""
        points = check_arm_points(self.model, local_positions, link, site)
        check_arm_inputs(self.num_envs, int(self.model['nd']), q=q, qd=qd)
        out = self._arm_dynamics(points, q, qd, None, ('jacobian', 'position', 'velocity'))
        J = out.pop('jacobian')
        out['linear'], out['angular'] = J[:, :, :3], J[:, :, 3:]
        return out

    def calculate_jacobian(self, local_positions=((0.0, 0.0, 0.0),), link=None, site=0, q=None, qd=None):
        """calculate_jacobian_device() as numpy arrays."""
        return {k: v.cpu().numpy() for k, v in self.calculate_jacobian_device(local_positions, link, site, q, qd).items()}

    def calculate_mass_matrix_device(self, q=None):
        """PyBullet's calculateMassMatrix(arm, q) in every env at once: the joint-space inertia M(q) of the arm, a CUDA
        tensor float32 [N, nd, nd] (symmetric; rows and columns in arm_dof_joints order), the matrix the step uses.
        q: numpy array or CUDA tensor [N, nd], default the env's state.  Asynchronous; ValueError for a bad shape or a
        non-finite numpy input."""
        check_arm_inputs(self.num_envs, int(self.model['nd']), q=q)
        return self._arm_dynamics([], q, None, None, ('mass_matrix',))['mass_matrix']

    def calculate_mass_matrix(self, q=None):
        """calculate_mass_matrix_device() as a numpy array."""
        return self.calculate_mass_matrix_device(q).cpu().numpy()

    def calculate_inverse_dynamics_device(self, qdd=None, q=None, qd=None):
        """PyBullet's calculateInverseDynamics(arm, q, qd, qdd) in every env at once: tau = M(q) qdd + h(q, qd), h the
        Coriolis, centrifugal and gravity term, without joint damping, motors, limits, gears or contacts; a CUDA tensor
        float32 [N, nd] (arm_dof_joints order; N m for revolute, N for prismatic DoF).  qdd default 0 (the bias h);
        q, qd default the env's state; each a numpy array or CUDA tensor [N, nd].  Asynchronous; ValueError for a bad
        shape or a non-finite numpy input."""
        check_arm_inputs(self.num_envs, int(self.model['nd']), q=q, qd=qd, qdd=qdd)
        return self._arm_dynamics([], q, qd, qdd, ('tau',))['tau']

    def calculate_inverse_dynamics(self, qdd=None, q=None, qd=None):
        """calculate_inverse_dynamics_device() as a numpy array."""
        return self.calculate_inverse_dynamics_device(qdd, q, qd).cpu().numpy()

    # ------------------------------------------------------------------ link and joint states
    @property
    def body_state_ids(self):
        """(body, link) of each row of body_states_device(), an int32 array [K, 2]: the arm's links (body 0, PyBullet link
        index, arm_dof_joints order), the free bodies (1.., link -1), then the slide bodies (door, button, dial; link -1),
        the ids of contacts() and change_dynamics()."""
        return state_ids(self.model)[0]

    @property
    def joint_state_ids(self):
        """(body, joint) of each column of joint_states_device(), an int32 array [nd + n_slide, 2]: the arm's DoF (body 0,
        PyBullet joint index, arm_dof_joints), then each slide body's one joint (joint 0 of that body)."""
        return state_ids(self.model)[1]

    def _body_states(self, frame):
        t = self.torch
        fr = check_frame(frame)
        body = t.empty((self.num_envs, len(self.body_state_ids), 13), dtype=t.float32, device=self.device)
        _lib.check(self.L, self._h, self.L.prb_body_states(self._h, ctypes.byref(_lib.PrbBodyQuery(fr, 0)),
                                                          ctypes.c_void_p(body.data_ptr()), None, None, self._stream()))
        return body

    def body_states_device(self, frame='link'):
        """PyBullet's getLinkStates(computeLinkVelocity=1), getBasePositionAndOrientation and getBaseVelocity for every body
        frame of every env at once (include/prb.h, prb_body_states): a dict of views of one float32 CUDA tensor [N,K,13],
        'position' [N,K,3], 'orientation' [N,K,4] (x, y, z, w), 'linear_velocity' and 'angular_velocity' [N,K,3], all in
        the world frame; row k is body_state_ids[k].  frame 'link': each arm link's link (joint) frame, 'com': its
        centre-of-mass frame (velocities are those of the frame's origin); free and slide bodies are the same in both.
        Asynchronous; ValueError for an unknown frame."""
        body = self._body_states(frame)
        return {'position': body[..., 0:3], 'orientation': body[..., 3:7], 'linear_velocity': body[..., 7:10],
                'angular_velocity': body[..., 10:13]}

    def body_states(self, frame='link'):
        """body_states_device() as numpy arrays."""
        return {k: v.cpu().numpy() for k, v in self.body_states_device(frame).items()}

    def joint_states_device(self):
        """PyBullet's getJointStates (positions and velocities) for every env at once: 'position' and 'velocity', float32
        CUDA tensors [N, nd + n_slide]; column j is joint_state_ids[j].  Asynchronous."""
        t = self.torch
        q, qd = (t.empty((self.num_envs, len(self.joint_state_ids)), dtype=t.float32, device=self.device) for _ in range(2))
        _lib.check(self.L, self._h, self.L.prb_body_states(self._h, ctypes.byref(_lib.PrbBodyQuery(0, 0)), None,
                                                          ctypes.c_void_p(q.data_ptr()), ctypes.c_void_p(qd.data_ptr()),
                                                          self._stream()))
        return {'position': q, 'velocity': qd}

    def joint_states(self):
        """joint_states_device() as numpy arrays."""
        return {k: v.cpu().numpy() for k, v in self.joint_states_device().items()}

    def _mask_dev(self, mask):
        if mask is None:
            return None
        t = self.torch
        m = mask if isinstance(mask, t.Tensor) else t.as_tensor(np.asarray(mask))
        if tuple(m.shape) != (self.num_envs,):
            raise ValueError('mask must be [num_envs=%d], got %s' % (self.num_envs, tuple(m.shape)))
        return m.to(self.device, t.uint8).contiguous()

    def _write_state(self, w, jq, jqd, body, mask):
        """One prb_write_state call; returns the status tensor (uint8 [N]: 0 not masked, 1 written, 2 rejected)."""
        t = self.torch
        status = t.empty(self.num_envs, dtype=t.uint8, device=self.device)
        self._w_keep = (jq, jqd, body, mask)        # the call is asynchronous: inputs live until the next write
        ptr = lambda x: None if x is None else ctypes.c_void_p(x.data_ptr())
        _lib.check(self.L, self._h, self.L.prb_write_state(self._h, ctypes.byref(w), ptr(jq), ptr(jqd), ptr(body), ptr(mask),
                                                          ptr(status), self._stream()))
        return status

    def reset_joint_states_device(self, position, velocity=None, joints=None, mask=None):
        """PyBullet's resetJointState(body, joint, targetValue, targetVelocity) for every env of `mask` (uint8 / bool [N];
        None: all) at once.  joints: a list of (body, joint) ids of joint_state_ids (None: every column); position and
        velocity: numpy arrays or CUDA tensors [N, len(joints)] or [len(joints)] (the same in every env); a missing
        velocity is 0.  Motors, goals and dynamics are left alone; the written envs' contact report is emptied and their
        observation refreshed.  Returns the status, a uint8 CUDA tensor [N] (0 not masked, 1 written, 2 rejected: a
        non-finite CUDA input leaves its env unchanged).  Asynchronous; ValueError for an unknown or repeated joint, a bad
        shape or a non-finite numpy input."""
        t = self.torch
        cols = check_joints(self.model, joints)
        N, nj = self.num_envs, len(self.joint_state_ids)
        vals = [check_state_value(name, x, N, len(cols)) for name, x in (('position', position), ('velocity', velocity))]
        jq, jqd = (t.zeros((N, nj), dtype=t.float32, device=self.device) for _ in range(2))
        ci = t.as_tensor(cols, dtype=t.long, device=self.device)
        for dst, v in zip((jq, jqd), vals):
            if v is not None:
                dst[:, ci] = t.as_tensor(v).to(self.device, t.float32).expand(N, len(cols))
        bits = sum(1 << c for c in cols)
        return self._write_state(_lib.PrbStateWrite(bits, bits, 0, 0, 0), jq, jqd, None, self._mask_dev(mask))

    def reset_joint_states(self, position, velocity=None, joints=None, mask=None):
        """reset_joint_states_device(); returns the status as a numpy array."""
        return self.reset_joint_states_device(position, velocity, joints, mask).cpu().numpy()

    def reset_base_states_device(self, body, position=None, orientation=None, linear_velocity=None, angular_velocity=None,
                                 mask=None):
        """PyBullet's resetBasePositionAndOrientation and resetBaseVelocity of free body `body` (1..n_free, the ids of
        contacts()) for every env of `mask` (None: all) at once.  Each part is a numpy array or CUDA tensor [N, k] or [k]
        (position 3, orientation 4 as x, y, z, w, normalised in fp32 by the library; velocities 3, world frame); a part
        left out keeps its current value (read with one body_states call).  The written envs' contact report is emptied
        and their observation refreshed.  Returns the status, a uint8 CUDA tensor [N] (0 not masked, 1 written, 2
        rejected: a non-finite value or a quaternion of norm < 1e-6 in a CUDA input).  Asynchronous; ValueError for a
        body that is not a free body, no part given, a bad shape, or a non-finite numpy input or zero numpy quaternion."""
        nf, nd = int(self.model['n_free']), int(self.model['nd'])
        if isinstance(body, bool) or not isinstance(body, (int, np.integer)) or not 1 <= body <= nf:
            raise ValueError('body must be a free body id 1..%d, got %r' % (nf, body))
        parts = {'position': (position, 0, 3), 'orientation': (orientation, 3, 7), 'linear_velocity': (linear_velocity, 7, 10),
                 'angular_velocity': (angular_velocity, 10, 13)}
        N = self.num_envs
        vals = {k: (check_state_value(k, x, N, b - a), a, b) for k, (x, a, b) in parts.items() if x is not None}
        if not vals:
            raise ValueError('give at least one of position, orientation, linear_velocity, angular_velocity')
        t = self.torch
        cur = self._body_states('link')
        row = nd + int(body) - 1
        for v, a, b in vals.values():
            cur[:, row, a:b] = t.as_tensor(v).to(self.device, t.float32).expand(N, b - a)
        bit = 1 << (int(body) - 1)
        pose = bit if ('position' in vals or 'orientation' in vals) else 0
        vel = bit if ('linear_velocity' in vals or 'angular_velocity' in vals) else 0
        return self._write_state(_lib.PrbStateWrite(0, 0, pose, vel, 0), None, None, cur, self._mask_dev(mask))

    def reset_base_states(self, body, position=None, orientation=None, linear_velocity=None, angular_velocity=None,
                          mask=None):
        """reset_base_states_device(); returns the status as a numpy array."""
        return self.reset_base_states_device(body, position, orientation, linear_velocity, angular_velocity, mask).cpu().numpy()

    def save_state_device(self):
        """PyBullet's saveState for every env at once: a float32 CUDA tensor [N, state_stride], a copy of the state
        (without the per-env dynamics table).  Asynchronous."""
        t = self.torch
        snap = t.empty((self.num_envs, self.buffers.state_stride), dtype=t.float32, device=self.device)
        _lib.check(self.L, self._h, self.L.prb_save_state(self._h, ctypes.c_void_p(snap.data_ptr()), self._stream()))
        return snap

    def save_state(self):
        """save_state_device() as a numpy array."""
        return self.save_state_device().cpu().numpy()

    def restore_state_device(self, saved, mask=None):
        """PyBullet's restoreState for every env of `mask` (uint8 / bool [N]; None: all) at once, from a save_state_device()
        snapshot (a CUDA tensor or numpy array [N, state_stride]): the rows come back bit for bit, the contact report of
        the restored envs is emptied and their observation refreshed.  Asynchronous; ValueError for a bad shape or a
        non-finite numpy snapshot."""
        t = self.torch
        shape = (self.num_envs, self.buffers.state_stride)
        if tuple(saved.shape) != shape:
            raise ValueError('saved must be [num_envs, state_stride] = %s, got %s' % (shape, tuple(saved.shape)))
        if not isinstance(saved, t.Tensor) and not np.isfinite(np.asarray(saved, np.float32)[:, :self.buffers.state_dim]).all():
            raise ValueError('saved must be finite')
        src = t.as_tensor(saved).to(self.device, t.float32).contiguous()
        m = self._mask_dev(mask)
        self._w_keep = (src, m)
        _lib.check(self.L, self._h, self.L.prb_restore_state(self._h, ctypes.c_void_p(src.data_ptr()),
                                                            None if m is None else ctypes.c_void_p(m.data_ptr()), self._stream()))

    def restore_state(self, saved, mask=None):
        """restore_state_device() from a numpy snapshot; synchronises the stream."""
        self.restore_state_device(saved, mask)
        self.torch.cuda.current_stream(self.device).synchronize()

    # ------------------------------------------------------------------ per-env dynamics
    def dynamics_device(self):
        """The per-env dynamics table (include/prb.h, prb_dynamics) as zero-copy CUDA tensors: 'lateral_friction',
        'spinning_friction' float32 [N, n_col]; 'mass', 'linear_damping', 'angular_damping' float32 [N, n_free];
        'local_inertia_diagonal' float32 [N, n_free, 3].  Writes take effect from the next physics substep on the same
        stream; values must be finite, mass and inertia > 0, friction and damping >= 0."""
        if self._dyn_views is None:
            if not self._per_env_dynamics:
                raise _lib.PrbError('per_env_dynamics is off')
            d = _lib.PrbDynamics()
            _lib.check(self.L, self._h, self.L.prb_get_dynamics(self._h, ctypes.byref(d)))
            N, nc, nf = self.num_envs, int(d.n_col), int(d.n_free)
            shapes = {'lateral_friction': (N, nc), 'spinning_friction': (N, nc), 'mass': (N, nf),
                      'local_inertia_diagonal': (N, nf, 3), 'linear_damping': (N, nf), 'angular_damping': (N, nf)}
            with self.torch.cuda.device(self.device):
                self._dyn_views = {k: self.torch.as_tensor(_DevArray(getattr(d, k), shapes[k], self), device=self.device)
                                   for k in _lib.DYNAMICS_FIELDS}
        return dict(self._dyn_views)

    def dynamics(self):
        """dynamics_device() as numpy arrays (copies)."""
        return {k: v.cpu().numpy() for k, v in self.dynamics_device().items()}

    def change_dynamics(self, body, link=-1, mask=None, *, lateral_friction=None, spinning_friction=None, mass=None,
                        local_inertia_diagonal=None, linear_damping=None, angular_damping=None):
        """PyBullet's changeDynamics(body, link, ...) for the envs of `mask` (uint8 / bool [N]; None: all).  body: -1 static
        scene, 0 arm, 1.. free bodies, then slide bodies (the ids of contacts()); link: the PyBullet link index.  A value
        is a scalar or one per env ([N], [N, 3] for the inertia).  Friction goes to every collider of (body, link); mass,
        inertia and damping exist for free bodies only.  mass= without local_inertia_diagonal= rescales the inertia by the
        mass ratio.  Raises ValueError for an unknown (body, link) or a bad value; needs per_env_dynamics."""
        cols, fb = dynamics_target(self.model, body, link)
        t, N = self.torch, self.num_envs
        vals = {'lateral_friction': lateral_friction, 'spinning_friction': spinning_friction, 'mass': mass,
                'local_inertia_diagonal': local_inertia_diagonal, 'linear_damping': linear_damping,
                'angular_damping': angular_damping}
        vals = {k: check_dynamics_value(k, v, N) for k, v in vals.items() if v is not None}
        if fb is None and any(k not in ('lateral_friction', 'spinning_friction') for k in vals):
            raise ValueError('mass, inertia and damping belong to free bodies only (body %d is not one)' % body)
        d = self.dynamics_device()
        sel = t.ones(N, dtype=t.bool, device=self.device) if mask is None else \
            t.as_tensor(np.asarray(mask)).to(self.device).reshape(N).bool()
        dev = lambda v: t.as_tensor(v, dtype=t.float32, device=self.device)
        for k in ('lateral_friction', 'spinning_friction'):
            if k in vals:
                ci = t.as_tensor(cols, dtype=t.long, device=self.device)
                cur = d[k][:, ci]
                d[k][:, ci] = t.where(sel[:, None], dev(vals[k])[:, None].expand_as(cur), cur)
        if 'mass' in vals and 'local_inertia_diagonal' not in vals:
            ratio = dev(vals['mass']) / d['mass'][:, fb]
            vals['local_inertia_diagonal'] = (d['local_inertia_diagonal'][:, fb] * ratio[:, None]).cpu().numpy()
        for k in ('mass', 'local_inertia_diagonal', 'linear_damping', 'angular_damping'):
            if k in vals:
                cur = d[k][:, fb]
                new = dev(vals[k])
                d[k][:, fb] = t.where(sel[:, None] if cur.dim() == 2 else sel, new, cur)

    # ------------------------------------------------------------------ raw state (tests, checkpoints)
    def get_state(self):
        out = np.zeros((self.num_envs, self.buffers.state_dim), np.float32)
        _lib.check(self.L, self._h, self.L.prb_get_state(self._h, out.ctypes.data_as(ctypes.c_void_p)))
        return out

    def set_state(self, state):
        s = np.ascontiguousarray(state, np.float32)
        assert s.shape == (self.num_envs, self.buffers.state_dim)
        _lib.check(self.L, self._h, self.L.prb_set_state(self._h, s.ctypes.data_as(ctypes.c_void_p)))

    def substeps(self, n):
        _lib.check(self.L, self._h, self.L.prb_substeps(self._h, int(n), self._stream()))

    def observe(self):
        self.observe_device()
        self._pull()
        return self._obs_host()

    def enable_kernel_timing(self, on=True):
        _lib.check(self.L, self._h, self.L.prb_enable_kernel_timing(self._h, 1 if on else 0))

    def last_kernel_ms(self):
        a, b = ctypes.c_float(), ctypes.c_float()
        _lib.check(self.L, self._h, self.L.prb_last_kernel_ms(self._h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def last_tier_ms(self):
        a, b = ctypes.c_float(), ctypes.c_float()
        _lib.check(self.L, self._h, self.L.prb_last_tier_ms(self._h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def reset_rounds(self):
        """Rounds (seat objects, settle, finish) the most recent reset needed."""
        return int(self.L.prb_reset_rounds(self._h))

    def launch_count(self):
        return int(self.L.prb_launch_count(self._h))

    def debug_usage(self):
        out = np.zeros((self.num_envs, 4), np.int32)
        _lib.check(self.L, self._h, self.L.prb_debug_usage(self._h, out.ctypes.data_as(ctypes.c_void_p)))
        return out

    def overflow_count(self):
        return int(self.L.prb_overflow_count(self._h))

    def kernel_info(self):
        a, b, c = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        self.L.prb_kernel_info(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
        return {'smem_bytes_per_block': a.value, 'envs_per_block': b.value, 'regs_per_thread': c.value}


def check_rays(model, num_envs, ray_from, ray_to, site=None, exclude_bodies=()):
    """(per_env, R, collider_mask) of a ray_test_batch call.  ValueError unless ray_from and ray_to have one shape, [R,3]
    or [num_envs,R,3] with R in 1..16384, site is None or 0..3, every excluded body exists, and numpy inputs are finite
    (CUDA tensors are not read back: a ray with a non-finite endpoint is a miss)."""
    shapes = [tuple(x.shape) for x in (ray_from, ray_to)]
    if shapes[0] != shapes[1]:
        raise ValueError('ray_from and ray_to must have the same shape, got %s and %s' % tuple(shapes))
    sh = shapes[0]
    if not ((len(sh) == 2 or (len(sh) == 3 and sh[0] == num_envs)) and sh[-1] == 3):
        raise ValueError('rays must be [R, 3] or [num_envs=%d, R, 3], got %s' % (num_envs, sh))
    R = sh[-2]
    if not 1 <= R <= 16384:
        raise ValueError('R = %d rays per env; must be in 1..16384' % R)
    if site is not None and (isinstance(site, bool) or not isinstance(site, (int, np.integer)) or not 0 <= site <= 3):
        raise ValueError('site must be None (world) or 0..3, got %r' % (site,))
    for x in (ray_from, ray_to):
        if not getattr(x, 'is_cuda', False) and not np.isfinite(np.asarray(x.cpu() if hasattr(x, 'cpu') else x, np.float64)).all():
            raise ValueError('ray endpoints must be finite')
    nc, nb = int(model['n_col']), int(model['n_free']) + int(model['n_slide'])
    body = np.asarray(model['col_body'])[:nc]
    mask = (1 << nc) - 1
    for b in exclude_bodies:
        if isinstance(b, bool) or not isinstance(b, (int, np.integer)) or not -1 <= b <= nb:
            raise ValueError('exclude_bodies: %r is not a body id (-1 static, 0 arm, 1..%d)' % (b, nb))
        for c in np.nonzero(body == b)[0]:
            mask &= ~(1 << int(c))
    return (1 if len(sh) == 3 else 0), R, mask


def check_closest(model, queries, max_distance):
    """([(mask_a, mask_b)] collider masks, max_distance) of a closest_points call.  ValueError unless there are 1..64
    queries, each a pair of sides, a side a body id or a (body, link) tuple with at least one collider, and max_distance
    is finite and >= 0."""
    queries = list(queries)
    if not 1 <= len(queries) <= 64:
        raise ValueError('closest_points needs 1..64 queries, got %d' % len(queries))
    nc = int(model['n_col'])
    body = np.asarray(model['col_body'])[:nc]

    def side_mask(side):
        if isinstance(side, tuple) and len(side) == 2:
            cols = dynamics_target(model, *side)[0]
        elif isinstance(side, (int, np.integer)) and not isinstance(side, bool):
            cols = np.nonzero(body == int(side))[0]
            if len(cols) == 0:
                raise ValueError('no collider has body %r' % (side,))
        else:
            raise ValueError('a query side is a body id or a (body, link) tuple, got %r' % (side,))
        return sum(1 << int(c) for c in cols)

    qs = []
    for q in queries:
        if not (isinstance(q, (tuple, list)) and len(q) == 2):
            raise ValueError('a query is a pair (side_a, side_b), got %r' % (q,))
        qs.append((side_mask(q[0]), side_mask(q[1])))
    md = float(max_distance)
    if not (math.isfinite(md) and md >= 0.0):
        raise ValueError('max_distance must be finite and >= 0, got %r' % (max_distance,))
    return qs, md


def check_arm_points(model, local_positions, link=None, site=0):
    """[(model link, site, (x, y, z))] prb_arm_point fields of a calculate_jacobian call.  ValueError unless exactly one of
    link (a PyBullet link index of the arm, arm_urdf_index) and site (0..3) is given and local_positions is a finite
    [P,3] with P in 1..16."""
    if (link is None) == (site is None):
        raise ValueError('give exactly one of link and site, got link=%r, site=%r' % (link, site))
    x = np.asarray(local_positions.cpu() if hasattr(local_positions, 'cpu') else local_positions, np.float64)
    if x.ndim != 2 or x.shape[1] != 3 or not 1 <= x.shape[0] <= 16:
        raise ValueError('local_positions must be [P, 3] with P in 1..16, got shape %s' % (x.shape,))
    if not np.isfinite(x).all():
        raise ValueError('local_positions must be finite')
    if site is not None:
        if isinstance(site, bool) or not isinstance(site, (int, np.integer)) or not 0 <= site <= 3:
            raise ValueError('site must be 0..3, got %r' % (site,))
        return [(-1, int(site), tuple(r)) for r in x]
    urdf = list(np.asarray(model['arm_urdf_index'])[:int(model['nd'])])
    if isinstance(link, bool) or not isinstance(link, (int, np.integer)) or int(link) not in urdf:
        raise ValueError('link must be a PyBullet link index of the arm %s, got %r' % ([int(u) for u in urdf], link))
    return [(urdf.index(int(link)), -1, tuple(r)) for r in x]


def check_arm_inputs(num_envs, nd, **arrays):
    """ValueError unless every given array (numpy or CUDA tensor; None: not given) is [num_envs, nd] and, for numpy,
    finite (CUDA tensors are not read back)."""
    for name, x in arrays.items():
        if x is None:
            continue
        shape = tuple(x.shape) if hasattr(x, 'shape') else np.shape(x)
        if shape != (num_envs, nd):
            raise ValueError('%s must be [num_envs=%d, nd=%d], got %s' % (name, num_envs, nd, shape))
        if not getattr(x, 'is_cuda', False) and not np.isfinite(np.asarray(x.cpu() if hasattr(x, 'cpu') else x, np.float64)).all():
            raise ValueError('%s must be finite' % name)


def state_ids(model):
    """(body_state_ids [K, 2], joint_state_ids [nd + n_slide, 2]) of a compiled model, int32: rows of prb_body_states are
    the arm's links (0, PyBullet link index), the free bodies (1.., -1) and the slide bodies (1 + n_free.., -1); columns of
    its joint arrays the arm's DoF (0, PyBullet joint index) and each slide body's one joint (body, 0)."""
    nd, nf, ns = int(model['nd']), int(model['n_free']), int(model['n_slide'])
    urdf = [int(u) for u in np.asarray(model['arm_urdf_index'])[:nd]]
    bodies = [(0, u) for u in urdf] + [(1 + b, -1) for b in range(nf)] + [(1 + nf + s, -1) for s in range(ns)]
    joints = [(0, u) for u in urdf] + [(1 + nf + s, 0) for s in range(ns)]
    return np.array(bodies, np.int32).reshape(-1, 2), np.array(joints, np.int32).reshape(-1, 2)


def check_frame(frame):
    """prb_body_query.frame of 'link' (0) or 'com' (1); ValueError otherwise."""
    if frame not in ('link', 'com'):
        raise ValueError("frame must be 'link' or 'com', got %r" % (frame,))
    return 0 if frame == 'link' else 1


def check_joints(model, joints):
    """Column indices of a list of (body, joint) ids of joint_state_ids (None: every column).  ValueError for an unknown
    or repeated id, or an empty list."""
    ids = [tuple(int(v) for v in r) for r in state_ids(model)[1]]
    if joints is None:
        return list(range(len(ids)))
    cols = []
    for j in joints:
        if not (isinstance(j, (tuple, list)) and len(j) == 2 and all(isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in j)):
            raise ValueError('a joint is a (body, joint) id, got %r' % (j,))
        if tuple(int(v) for v in j) not in ids:
            raise ValueError('unknown joint %r (joint_state_ids: %s)' % (tuple(j), ids))
        cols.append(ids.index(tuple(int(v) for v in j)))
    if not cols or len(set(cols)) != len(cols):
        raise ValueError('joints must be a non-empty list without repeats, got %r' % (list(joints),))
    return cols


def check_state_value(name, x, N, k):
    """A state write input (numpy array or CUDA tensor; None: not given) of shape [N, k] or [k].  ValueError for another
    shape and, for numpy, a non-finite value or an orientation of norm < 1e-6 (CUDA tensors are not read back: the
    library rejects such an env)."""
    if x is None:
        return None
    shape = tuple(x.shape) if hasattr(x, 'shape') else np.shape(x)
    if shape not in ((N, k), (k,)):
        raise ValueError('%s must be [num_envs=%d, %d] or [%d], got %s' % (name, N, k, k, shape))
    if getattr(x, 'is_cuda', False):
        return x
    a = np.asarray(x.cpu() if hasattr(x, 'cpu') else x, np.float64)
    if not np.isfinite(a).all():
        raise ValueError('%s must be finite' % name)
    if name == 'orientation' and (np.linalg.norm(a.reshape(-1, 4), axis=1) < 1e-6).any():
        raise ValueError('orientation quaternions must have a norm >= 1e-6')
    return np.ascontiguousarray(a, np.float32)


def dynamics_ranges(spec):
    """{field: (lo, hi)} -> prb_dynamics_ranges; fields not given are (1, 1).  ValueError for an unknown field or a bound
    that is not finite, lo > hi, lo < 0, or a mass lower bound of 0."""
    r = _lib.PrbDynamicsRanges()
    for k in _lib.DYNAMICS_RANGE_FIELDS:
        getattr(r, k)[:] = (1.0, 1.0)
    for k, v in dict(spec).items():
        if k not in _lib.DYNAMICS_RANGE_FIELDS:
            raise ValueError('unknown dynamics range %r (fields: %s)' % (k, ', '.join(_lib.DYNAMICS_RANGE_FIELDS)))
        lo, hi = (float(x) for x in v)
        if not (math.isfinite(lo) and math.isfinite(hi) and 0.0 <= lo <= hi) or (k == 'mass' and lo <= 0.0):
            raise ValueError('%s range (%r, %r): needs finite 0 <= lo <= hi%s' % (k, lo, hi, ', lo > 0' if k == 'mass' else ''))
        getattr(r, k)[:] = (lo, hi)
    return r


def dynamics_target(model, body, link=-1):
    """(collider indices of (body, link), free-body index or None) of a compiled model, the ids contacts() reports: body
    -1 static scene, 0 arm, 1.. free bodies, then slide bodies; link the PyBullet link index.  ValueError if (body, link)
    has no collider."""
    nc, nf = int(model['n_col']), int(model['n_free'])
    cb = np.asarray(model['col_body'])[:nc]
    cl = np.asarray(model['col_urdf_link'])[:nc]
    cols = np.nonzero((cb == int(body)) & (cl == int(link)))[0]
    if len(cols) == 0:
        raise ValueError('no collider has body %r link %r' % (body, link))
    return cols, (int(body) - 1 if 1 <= int(body) <= nf else None)


def check_dynamics_value(field, v, N):
    """A change_dynamics value as float32 [N] ([N, 3] for the inertia), broadcast from a scalar (or a 3-vector for the
    inertia).  ValueError if it is not finite, mass or inertia <= 0, or friction or damping < 0."""
    a = np.asarray(v, np.float64)
    shape = (N, 3) if field == 'local_inertia_diagonal' else (N,)
    try:
        a = np.broadcast_to(a, shape)
    except ValueError:
        raise ValueError('%s: expected a scalar or shape %s, got %s' % (field, shape, a.shape)) from None
    if not np.isfinite(a).all():
        raise ValueError('%s: values must be finite' % field)
    if field in ('mass', 'local_inertia_diagonal'):
        if not (a > 0).all():
            raise ValueError('%s: values must be > 0' % field)
    elif not (a >= 0).all():
        raise ValueError('%s: values must be >= 0' % field)
    return np.ascontiguousarray(a, np.float32)


# the three registered ids in scope (roboticsPlayroomPybullet/__init__.py:23-26,65-68,91-94)
class UR5Reach(VecPlayEnv):
    env_id = 'UR5Reach-v0'


class pandaPick(VecPlayEnv):
    env_id = 'pandaPick-v0'


class UR5PlayAbsRPY1Obj(VecPlayEnv):
    env_id = 'UR5PlayAbsRPY1Obj-v0'


# the other UR5 playroom ids: same world, other action decoder (envList.py:101-140, environments.py:915-981)
class UR5Play1Obj(VecPlayEnv):
    env_id = 'UR5Play1Obj-v0'               # absolute_quat, 8-D action


class UR5PlayRel1Obj(VecPlayEnv):
    env_id = 'UR5PlayRel1Obj-v0'            # relative_quat, 8-D action


class UR5PlayRelRPY1Obj(VecPlayEnv):
    env_id = 'UR5PlayRelRPY1Obj-v0'         # relative_rpy


class UR5PlayAbsJoints1Obj(VecPlayEnv):
    env_id = 'UR5PlayAbsJoints1Obj-v0'      # absolute_joints


class UR5PlayRelJoints1Obj(VecPlayEnv):
    env_id = 'UR5PlayRelJoints1Obj-v0'      # relative_joints


# the Panda ids (roboticsPlayroomPybullet/__init__.py:3-63, envList.py:8-86); pandaPlay-v0 / pandaPlayJoints-v0 have TWO
# objects (a second free body and 26-D observations) and are not compiled yet
class pandaReach(VecPlayEnv):
    env_id = 'pandaReach-v0'


class pandaReach2D(VecPlayEnv):
    env_id = 'pandaReach2D-v0'


class pandaPush(VecPlayEnv):
    env_id = 'pandaPush-v0'


class pandaPlayAbsRPY1Obj(VecPlayEnv):
    env_id = 'pandaPlayAbsRPY1Obj-v0'


class pandaPlay1Obj(VecPlayEnv):
    env_id = 'pandaPlay1Obj-v0'             # absolute_quat


class pandaPlayRel1Obj(VecPlayEnv):
    env_id = 'pandaPlayRel1Obj-v0'          # relative_quat


class pandaPlayRelRPY1Obj(VecPlayEnv):
    env_id = 'pandaPlayRelRPY1Obj-v0'


class pandaPlayAbsJoints1Obj(VecPlayEnv):
    env_id = 'pandaPlayAbsJoints1Obj-v0'    # 8-D: 7 joints + gripper


class pandaPlayRelJoints1Obj(VecPlayEnv):
    env_id = 'pandaPlayRelJoints1Obj-v0'


_REGISTRY = {c.env_id: c for c in (UR5Reach, pandaPick, UR5PlayAbsRPY1Obj, UR5Play1Obj, UR5PlayRel1Obj, UR5PlayRelRPY1Obj,
                                   UR5PlayAbsJoints1Obj, UR5PlayRelJoints1Obj, pandaReach, pandaReach2D, pandaPush,
                                   pandaPlayAbsRPY1Obj, pandaPlay1Obj, pandaPlayRel1Obj, pandaPlayRelRPY1Obj,
                                   pandaPlayAbsJoints1Obj, pandaPlayRelJoints1Obj)}


def make(env_id, num_envs=1, **kw):
    """gym.make analogue for the registered ids."""
    if env_id not in _REGISTRY:
        raise NotImplementedError('unknown env id %r (in scope: %s)' % (env_id, sorted(_REGISTRY)))
    return _REGISTRY[env_id](num_envs=num_envs, **kw)
