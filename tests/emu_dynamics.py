"""ctypes front-end of tests/emu/libdynamics_emu.so: the step pipeline with the per-env dynamics table (the `dyn` argument
of the setup kernel in csrc/prb_stream.cuh) and the randomization kernel (csrc/prb_dynamics.cuh), compiled with g++
against the SIMT emulator (tests/emu/cuda_emu.h).  CPU tests only."""
import ctypes
import os
import subprocess

import numpy as np

from emu_contacts import split_report
from emu_lib import OUT_KEYS, DevOut, out_dims

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'emu')
_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
_SRC = os.path.join(_ROOT, 'roboticsplayroompybullet_b200', 'csrc')
_LIB = None

# the table's fields in include/prb.h prb_dynamics order, with the model field each one overrides
FIELDS = ['lateral_friction', 'spinning_friction', 'mass', 'local_inertia_diagonal', 'linear_damping', 'angular_damping']
MODEL_FIELD = {'lateral_friction': 'col_friction', 'spinning_friction': 'col_spin', 'mass': 'free_mass',
               'local_inertia_diagonal': 'free_inertia', 'linear_damping': 'free_lin_damp', 'angular_damping': 'free_ang_damp'}
RANGE_FIELDS = ['lateral_friction', 'spinning_friction', 'mass', 'linear_damping', 'angular_damping']


def lib():
    """g++ build unless the library is newer than every source (written under a temporary name and renamed, so that test
    processes running in parallel never load a half-written file)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = os.path.join(_HERE, 'libdynamics_emu.so')
    deps = [os.path.join(_HERE, f) for f in ('dynamics_emu.cpp', 'cuda_emu.h')] + \
           [os.path.join(_SRC, f) for f in ('prb_dynamics.cuh', 'prb_contacts.cuh', 'prb_stream.cuh', 'prb_kernels.cuh', 'prb_device.h',
                                            'prb_convert.h')]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        tmp = '%s.%d.tmp.so' % (so[:-3], os.getpid())
        subprocess.check_call(['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-U_FORTIFY_SOURCE', '-Wno-unknown-pragmas',
                               '-o', tmp, os.path.join(_HERE, 'dynamics_emu.cpp')])
        os.replace(tmp, so)
    L = ctypes.CDLL(so)
    L.demu_error.restype = ctypes.c_char_p
    for f in ('demu_table_words', 'demu_field_offset', 'demu_report_words'):
        getattr(L, f).restype = ctypes.c_longlong
    _LIB = L
    return L


def model_table(m, N):
    """Every env's row holding the model's values, the (float) casts of csrc/prb_convert.h."""
    nc, nf = int(m['n_col']), int(m['n_free'])
    f = lambda k, n: np.asarray(m[MODEL_FIELD[k]], np.float64)[:n].astype(np.float32)
    return {'lateral_friction': np.tile(f('lateral_friction', nc), (N, 1)),
            'spinning_friction': np.tile(f('spinning_friction', nc), (N, 1)),
            'mass': np.tile(f('mass', nf), (N, 1)),
            'local_inertia_diagonal': np.tile(f('local_inertia_diagonal', 3 * nf).reshape(nf, 3), (N, 1, 1)),
            'linear_damping': np.tile(f('linear_damping', nf), (N, 1)),
            'angular_damping': np.tile(f('angular_damping', nf), (N, 1))}


class DynSim:
    """N envs stepped by the emulated kernels; table=None runs with the model's dynamics (no table)."""

    def __init__(self, model, N, table=None, report=False, seed=1234, env_offset=0):
        self.m, self.N = model, N
        self.L = lib()
        self.ms = model.as_struct()
        if self.L.demu_set_model(ctypes.byref(self.ms)) != 0:
            raise RuntimeError(self.L.demu_error().decode())
        self.seed, self.env_offset = seed, env_offset
        self.stride = self.L.demu_state_stride()
        self.state = np.zeros((N, self.stride), np.float32)
        self.buf = None
        if table is not None:
            self.buf = np.zeros(self.L.demu_table_words(N), np.float32)
            self.set_table(table)
        self.rep = None
        if report:
            self.rep = np.zeros(self.L.demu_report_words(N), np.float32)
            self.L.demu_clear_report(self._p(self.rep), N)
        self.out = {k: np.zeros((N, d), np.float32) for k, d in out_dims(model).items()}
        self.O = DevOut(*([self.out[k].ctypes.data for k in OUT_KEYS] + [None, None]))

    @staticmethod
    def _p(a):
        return None if a is None else a.ctypes.data_as(ctypes.c_void_p)

    def _views(self):
        v = {}
        for i, name in enumerate(FIELDS):
            o = self.L.demu_field_offset(self.N, i)
            end = self.L.demu_field_offset(self.N, i + 1) if i + 1 < len(FIELDS) else len(self.buf)
            v[name] = self.buf[o:end].reshape(self.N, -1)
        v['local_inertia_diagonal'] = v['local_inertia_diagonal'].reshape(self.N, -1, 3)
        return v

    def table(self):
        return {k: a.copy() for k, a in self._views().items()}

    def set_table(self, t):
        for k, a in self._views().items():
            a[...] = np.asarray(t[k], np.float32).reshape(a.shape)

    def set_state(self, rows):
        self.state[:] = 0
        self.state[:, :rows.shape[1]] = rows

    def substeps(self, n):
        self.L.demu_set_model(ctypes.byref(self.ms))
        self.L.demu_substeps(self._p(self.state), self.N, n, self._p(self.buf), self._p(self.rep))

    def step(self, action):
        from roboticsplayroompybullet_b200.model import action_dim
        self.L.demu_set_model(ctypes.byref(self.ms))
        a = np.ascontiguousarray(action, np.float32).reshape(self.N, action_dim(self.m))
        self.L.demu_step(self._p(self.state), self._p(a), ctypes.byref(self.O), self.N, self._p(self.buf), self._p(self.rep))
        return {k: v.copy() for k, v in self.out.items()}

    def randomize(self, ranges, mask=None):
        """ranges: {field: (lo, hi)} of RANGE_FIELDS, (1, 1) where not given."""
        self.L.demu_set_model(ctypes.byref(self.ms))
        r = np.array([x for k in RANGE_FIELDS for x in ranges.get(k, (1.0, 1.0))], np.float32)
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self.L.demu_randomize(self._p(self.state), self._p(self.buf), self._p(mk), self.N, ctypes.c_uint64(self.seed),
                              ctypes.c_uint32(self.env_offset), self._p(r))

    def contacts(self):
        return split_report(self.rep, self.N)
