"""ctypes front-end of tests/emu/libcontacts_emu.so: the step pipeline with the contact report (csrc/prb_contacts.cuh and
the report mode of the setup and solver kernels in csrc/prb_stream.cuh) compiled with g++ against the SIMT emulator
(tests/emu/cuda_emu.h).  CPU tests only."""
import ctypes
import os
import subprocess

import numpy as np

from emu_lib import OUT_KEYS, DevOut, out_dims

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'emu')
_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
_SRC = os.path.join(_ROOT, 'roboticsplayroompybullet_b200', 'csrc')
_LIBS = {}

# (name, numpy type, per-contact components), in the order of the report's fields (include/prb.h prb_contacts)
FIELDS = [('collider_a', np.int32, 1), ('collider_b', np.int32, 1), ('position_on_a', np.float32, 3),
          ('position_on_b', np.float32, 3), ('normal_on_b', np.float32, 3), ('distance', np.float32, 1),
          ('normal_force', np.float32, 1), ('lateral_friction_1', np.float32, 1), ('lateral_friction_2', np.float32, 1),
          ('lateral_friction_dir_1', np.float32, 3), ('lateral_friction_dir_2', np.float32, 3)]


def lib(tag='', defines=()):
    """g++ build unless the library is newer than every source (written under a temporary name and renamed, so that test
    processes running in parallel never load a half-written file).  `defines` give a variant with other compile-time
    constants, e.g. tiny solver stages."""
    if tag in _LIBS:
        return _LIBS[tag]
    so = os.path.join(_HERE, 'libcontacts_emu%s.so' % ('_' + tag if tag else ''))
    deps = [os.path.join(_HERE, f) for f in ('contacts_emu.cpp', 'cuda_emu.h')] + \
           [os.path.join(_SRC, f) for f in ('prb_contacts.cuh', 'prb_stream.cuh', 'prb_kernels.cuh', 'prb_device.h', 'prb_convert.h')]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        tmp = '%s.%d.tmp.so' % (so[:-3], os.getpid())
        subprocess.check_call(['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-U_FORTIFY_SOURCE', '-Wno-unknown-pragmas'] +
                              ['-D%s' % d for d in defines] + ['-o', tmp, os.path.join(_HERE, 'contacts_emu.cpp')])
        os.replace(tmp, so)
    L = ctypes.CDLL(so)
    L.cemu_error.restype = ctypes.c_char_p
    L.cemu_report_words.restype = ctypes.c_longlong
    _LIBS[tag] = L
    return L


def split_report(buf, N, K=64):
    """The report allocation (float32 words) as a dict of arrays shaped like VecPlayEnv.contacts()."""
    d, off = {}, 0
    for name, ty, k in FIELDS:
        n = N * K * k
        d[name] = buf[off:off + n].view(ty).reshape((N, K) if k == 1 else (N, K, k)).copy()
        off += n
    d['count'] = buf[off:off + N].view(np.int32).copy()
    return d


class ContactSim:
    """N envs stepped by the emulated kernels with the contact report on (report=False: off)."""

    def __init__(self, model, N, report=True, tag='', defines=()):
        self.m, self.N = model, N
        self.L = lib(tag, defines)
        self.ms = model.as_struct()
        if self.L.cemu_set_model(ctypes.byref(self.ms)) != 0:
            raise RuntimeError(self.L.cemu_error().decode())
        self.stride = self.L.cemu_state_stride()
        self.state = np.zeros((N, self.stride), np.float32)
        self.K = self.L.cemu_max_contacts()
        self.rep = None
        if report:
            self.rep = np.zeros(self.L.cemu_report_words(N), np.float32)
            self.L.cemu_clear(self._p(self.rep), N, None)
        self.out = {k: np.zeros((N, d), np.float32) for k, d in out_dims(model).items()}
        self.O = DevOut(*([self.out[k].ctypes.data for k in OUT_KEYS] + [None, None]))

    @staticmethod
    def _p(a):
        return None if a is None else a.ctypes.data_as(ctypes.c_void_p)

    def set_state(self, rows):
        self.state[:] = 0
        self.state[:, :rows.shape[1]] = rows

    def substeps(self, n):
        self.L.cemu_set_model(ctypes.byref(self.ms))
        self.L.cemu_substeps(self._p(self.state), self.N, n, self._p(self.rep))

    def step(self, action):
        from roboticsplayroompybullet_b200.model import action_dim
        self.L.cemu_set_model(ctypes.byref(self.ms))
        a = np.ascontiguousarray(action, np.float32).reshape(self.N, action_dim(self.m))
        self.L.cemu_step(self._p(self.state), self._p(a), ctypes.byref(self.O), self.N, self._p(self.rep))
        return {k: v.copy() for k, v in self.out.items()}

    def clear(self, mask=None):
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self.L.cemu_clear(self._p(self.rep), self.N, self._p(mk))

    def contacts(self):
        d = split_report(self.rep, self.N, self.K)
        n_col = int(self.m['n_col'])
        for side in ('a', 'b'):
            ids = d['collider_' + side]
            for out, key in (('body_', 'col_body'), ('link_', 'col_urdf_link')):
                tbl = np.asarray(self.m[key])[:n_col].astype(np.int32)
                d[out + side] = np.where(ids >= 0, tbl[np.maximum(ids, 0)], ids)
        return d
