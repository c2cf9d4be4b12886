"""ctypes front-end of tests/emu/libprb_emu.so: the product's kernel source compiled with g++ against the SIMT emulator
(tests/emu/cuda_emu.h), the harness tests/emu/prb_emu.cpp.  The one build rule of the emulated kernels and the one
simulator class, EmuSim.  CPU tests only."""
import ctypes
import os
import subprocess

import numpy as np

from emu_contacts import split_report
from emu_dynamics import FIELDS as DYN_FIELDS, RANGE_FIELDS
from roboticsplayroompybullet_b200.lib import (PrbArmPoint, PrbArmQuery, PrbBodyQuery, PrbClosest, PrbClosestQuery, PrbRays,
                                               PrbStateWrite)

_TESTS = os.path.dirname(os.path.abspath(__file__))
_HERE = os.path.join(_TESTS, 'emu')
_ROOT = os.path.join(_TESTS, '..')
# every file here can reach the harness through an #include
_DEP_DIRS = [_HERE, os.path.join(_ROOT, 'roboticsplayroompybullet_b200', 'csrc'), os.path.join(_ROOT, 'include')]
_LIBS = {}

OUT_KEYS = ['obs_quat', 'achieved_goal', 'desired_goal', 'controllable_achieved_goal', 'full_positional_state',
            'joints', 'velocity', 'observation', 'gripper_proprioception', 'reward', 'is_success', 'target_poses']


class DevOut(ctypes.Structure):
    _fields_ = [(k, ctypes.c_void_p) for k in OUT_KEYS] + [('overflow', ctypes.c_void_p), ('ovf_env', ctypes.c_void_p), ('dbg', ctypes.c_void_p)]


def out_dims(m):
    return {'obs_quat': m['obs_dim'], 'achieved_goal': m['goal_dim'], 'desired_goal': m['goal_dim'],
            'controllable_achieved_goal': 4, 'full_positional_state': m['fps_dim'], 'joints': 8, 'velocity': 6,
            'observation': m['observation_dim'], 'gripper_proprioception': 1, 'reward': 1, 'is_success': 1,
            'target_poses': m['n_ik']}


def deps():
    """The sources the library is built from: every file of the harness, kernel and public header directories (the
    built libraries excepted)."""
    return sorted(os.path.realpath(os.path.join(d, f)) for d in _DEP_DIRS for f in os.listdir(d)
                  if os.path.isfile(os.path.join(d, f)) and not f.endswith('.so'))


def _declare(L):
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong
    L.emu_error.restype = ctypes.c_char_p
    for f in ('emu_report_words', 'emu_dyn_table_words', 'emu_dyn_field_offset'):
        getattr(L, f).restype = i64
    L.emu_ray_test.argtypes = [vp, i32, ctypes.POINTER(PrbRays), vp, vp, vp, vp, vp, vp, i32]
    L.emu_closest_points.argtypes = [vp, i32, ctypes.POINTER(PrbClosest), ctypes.POINTER(PrbClosestQuery), vp, vp, vp, vp, vp, vp, i32]
    L.emu_arm_dynamics.argtypes = [vp, i32, ctypes.POINTER(PrbArmQuery), ctypes.POINTER(PrbArmPoint)] + [vp] * 8
    L.emu_body_states.argtypes = [vp, i32, ctypes.POINTER(PrbBodyQuery), vp, vp, vp]
    L.emu_write_state.argtypes = [vp, vp, i32, ctypes.POINTER(PrbStateWrite), vp, vp, vp, vp, vp]
    L.emu_restore_state.argtypes = [vp, vp, i32, vp, vp]
    return L


def lib(tag='', defines=()):
    """The emulated kernels, built with g++ unless the library is newer than every file of deps().  `tag` / `defines`
    give a variant with other compile-time constants (e.g. tiny solver stages).  The library is written under a
    temporary name and renamed, so that test processes running in parallel never load a half-written file."""
    if tag not in _LIBS:
        so = os.path.join(_HERE, 'libprb_emu%s.so' % ('_' + tag if tag else ''))
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps()):
            tmp = '%s.%d.tmp.so' % (so[:-3], os.getpid())
            subprocess.check_call(['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-U_FORTIFY_SOURCE', '-Wno-unknown-pragmas'] +
                                  ['-D%s' % d for d in defines] + ['-o', tmp, os.path.join(_HERE, 'prb_emu.cpp')])
            os.replace(tmp, so)
        _LIBS[tag] = _declare(ctypes.CDLL(so))
    return _LIBS[tag]


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def rows(model, state):
    """Selects `model` in lib() and returns state ([N, state_dim] or [N, state_stride] rows) as float32 [N, state_stride]
    rows: the array itself when it already is one (read in place), else a zero-padded copy."""
    L = lib()
    ms = model.as_struct()
    if L.emu_set_model(ctypes.byref(ms)) != 0:
        raise RuntimeError(L.emu_error().decode())
    stride, sd = L.emu_state_stride(), L.emu_state_dim()
    st = np.asarray(state)
    if st.dtype != np.float32 or st.ndim != 2 or st.shape[1] != stride or not st.flags.c_contiguous:
        s2 = np.zeros((st.shape[0], stride), np.float32)
        s2[:, :sd] = st[:, :sd]
        st = s2
    return st


class EmuSim:
    """N envs stepped by the emulated kernels, like one prb_handle.  report: the contact report on
    (prb_enable_contacts); table: the per-env dynamics table on (prb_enable_dynamics) holding {field: values} (None: the
    model's dynamics); tag / defines: a variant of the library (lib())."""

    def __init__(self, model, N, seed=1234, env_offset=0, report=False, table=None, tag='', defines=()):
        self.m = model
        self.L = lib(tag, defines)
        self.ms = model.as_struct()
        if self.L.emu_set_model(ctypes.byref(self.ms)) != 0:
            raise RuntimeError(self.L.emu_error().decode())
        self.N = N
        self.stride = self.L.emu_state_stride()
        self.state_dim = self.L.emu_state_dim()
        self.state = np.zeros((N, self.stride), np.float32)
        self.seed, self.env_offset = seed, env_offset
        self.K = self.L.emu_max_contacts()
        self.rep = np.zeros(self.L.emu_report_words(N), np.float32) if report else None
        self.buf = None
        if table is not None:
            self.buf = np.zeros(self.L.emu_dyn_table_words(N), np.float32)
            self.set_table(table)
        self.out = {k: np.zeros((N, d), np.float32) for k, d in out_dims(model).items()}
        self.O = DevOut(*([self.out[k].ctypes.data for k in OUT_KEYS] + [None, None]))
        self.L.emu_init(_p(self.state), N)
        self.clear()

    def _sel(self):
        """This sim's model, report and table become the library's (the handle state of prb_capi.cu)."""
        self.L.emu_set_model(ctypes.byref(self.ms))
        self.L.emu_set_report(_p(self.rep))
        self.L.emu_set_dynamics(_p(self.buf))

    def substeps(self, n):
        self._sel()
        self.L.emu_substeps(_p(self.state), self.N, n)

    def step(self, action):
        self._sel()
        from roboticsplayroompybullet_b200.model import action_dim
        a = np.ascontiguousarray(action, np.float32).reshape(self.N, action_dim(self.m))
        self.L.emu_step(_p(self.state), _p(a), ctypes.byref(self.O), self.N)
        return {k: v.copy() for k, v in self.out.items()}

    def observe(self):
        self._sel()
        self.L.emu_observe(_p(self.state), ctypes.byref(self.O), self.N)
        return {k: v.copy() for k, v in self.out.items()}

    def reset(self, mask=None):
        self._sel()
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self.L.emu_reset(_p(self.state), ctypes.byref(self.O), _p(mk), self.N, ctypes.c_uint64(self.seed),
                         ctypes.c_uint32(self.env_offset))
        return {k: v.copy() for k, v in self.out.items()}

    def reset_to(self, obs, mask=None, restore_env=True):
        self._sel()
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        ob = np.ascontiguousarray(obs, np.float32).reshape(self.N, -1)
        self.L.emu_reset_to(_p(self.state), ctypes.byref(self.O), _p(ob), _p(mk), self.N, ctypes.c_uint64(self.seed),
                            ctypes.c_uint32(self.env_offset), 1 if restore_env else 0)
        return {k: v.copy() for k, v in self.out.items()}

    def ik(self, action):
        self._sel()
        from roboticsplayroompybullet_b200.model import action_dim
        a = np.ascontiguousarray(action, np.float32).reshape(self.N, action_dim(self.m))
        t = np.zeros((self.N, self.m['n_ik']), np.float32)
        self.L.emu_ik(_p(self.state), _p(a), _p(t), self.N)
        return t

    def set_state(self, rows):
        """prb_set_state: rows [N, <= state_stride] become the state (the rest of each row zero); the report empties."""
        self.state[:] = 0
        self.state[:, :rows.shape[1]] = rows
        self.clear()

    # ---------------------------------------------------------------- contact report
    def clear(self, mask=None):
        """The report of the masked envs (mask None: every env) becomes empty; nothing with the report off."""
        self._sel()
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self.L.emu_clear_contacts(self.N, _p(mk))

    def contacts(self):
        """The report as a dict of arrays shaped like VecPlayEnv.contacts(), with the bodies and links of the colliders."""
        d = split_report(self.rep, self.N, self.K)
        n_col = int(self.m['n_col'])
        for side in ('a', 'b'):
            ids = d['collider_' + side]
            for out, key in (('body_', 'col_body'), ('link_', 'col_urdf_link')):
                tbl = np.asarray(self.m[key])[:n_col].astype(np.int32)
                d[out + side] = np.where(ids >= 0, tbl[np.maximum(ids, 0)], ids)
        return d

    # ---------------------------------------------------------------- dynamics table
    def _views(self):
        v = {}
        for i, name in enumerate(DYN_FIELDS):
            o = self.L.emu_dyn_field_offset(self.N, i)
            end = self.L.emu_dyn_field_offset(self.N, i + 1) if i + 1 < len(DYN_FIELDS) else len(self.buf)
            v[name] = self.buf[o:end].reshape(self.N, -1)
        v['local_inertia_diagonal'] = v['local_inertia_diagonal'].reshape(self.N, -1, 3)
        return v

    def table(self):
        return {k: a.copy() for k, a in self._views().items()}

    def set_table(self, t):
        for k, a in self._views().items():
            a[...] = np.asarray(t[k], np.float32).reshape(a.shape)

    def randomize(self, ranges, mask=None):
        """prb_randomize_dynamics; ranges: {field: (lo, hi)} of RANGE_FIELDS, (1, 1) where not given."""
        self._sel()
        r = np.array([x for k in RANGE_FIELDS for x in ranges.get(k, (1.0, 1.0))], np.float32)
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self.L.emu_randomize_dynamics(_p(self.state), _p(self.buf), _p(mk), self.N, ctypes.c_uint64(self.seed),
                                      ctypes.c_uint32(self.env_offset), _p(r))


def box_box(p1, R1, h1, p2, R2, h2):
    f = lambda x: np.ascontiguousarray(x, np.float32)
    out = np.zeros(28, np.float32)
    a = [f(x) for x in (p1, R1, h1, p2, R2, h2)]
    n = lib().emu_box_box(*[x.ctypes.data_as(ctypes.c_void_p) for x in a], out.ctypes.data_as(ctypes.c_void_p))
    return out[:7 * n].reshape(n, 7)
