"""ctypes front-end of tests/emu/libarm_emu.so: prb_arm_dynamics' kernel source (csrc/prb_arm.cuh) compiled with g++
against the SIMT emulator (tests/emu/cuda_emu.h).  CPU tests only."""
import ctypes
import os
import subprocess

import numpy as np

from roboticsplayroompybullet_b200.lib import PrbArmPoint, PrbArmQuery

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'emu')
_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
_SRC = os.path.join(_ROOT, 'roboticsplayroompybullet_b200', 'csrc')
_LIB = None

OUTPUTS = ('jacobian', 'position', 'velocity', 'mass_matrix', 'tau')


def lib():
    """g++ build unless the library is newer than every source; written under a temporary name and renamed, so that
    test processes running in parallel never load a half-written file."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = os.path.join(_HERE, 'libarm_emu.so')
    deps = [os.path.join(_HERE, f) for f in ('arm_emu.cpp', 'cuda_emu.h')] + \
           [os.path.join(_SRC, f) for f in ('prb_arm.cuh', 'prb_kernels.cuh', 'prb_device.h', 'prb_convert.h')] + \
           [os.path.join(_ROOT, 'include', f) for f in ('prb.h', 'prb_model.h')]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        tmp = '%s.%d.tmp.so' % (so[:-3], os.getpid())
        subprocess.check_call(['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-U_FORTIFY_SOURCE', '-Wno-unknown-pragmas',
                               '-o', tmp, os.path.join(_HERE, 'arm_emu.cpp')])
        os.replace(tmp, so)
    L = ctypes.CDLL(so)
    L.cemu_error.restype = ctypes.c_char_p
    vp = ctypes.c_void_p
    L.cemu_arm_dynamics.argtypes = [vp, ctypes.c_int, ctypes.POINTER(PrbArmQuery), ctypes.POINTER(PrbArmPoint)] + [vp] * 8
    _LIB = L
    return L


def _state(L, model, state):
    ms = model.as_struct()
    if L.cemu_set_model(ctypes.byref(ms)) != 0:
        raise RuntimeError(L.cemu_error().decode())
    stride = L.cemu_state_stride()
    st = np.asarray(state)
    if st.dtype != np.float32 or st.ndim != 2 or st.shape[1] != stride or not st.flags.c_contiguous:
        s2 = np.zeros((st.shape[0], stride), np.float32)
        s2[:, :L.cemu_state_dim()] = st[:, :L.cemu_state_dim()]
        st = s2
    return st


def point_structs(points):
    """[(link, site, (x, y, z))] -> a ctypes array of prb_arm_point (at least one element)."""
    return (PrbArmPoint * max(len(points), 1))(*[PrbArmPoint(int(l), int(s), (ctypes.c_float * 3)(*map(float, o)), 0)
                                                 for l, s, o in points])


def arm_dynamics(model, state, points, q=None, qd=None, qdd=None, outputs=OUTPUTS, call=None, structs=None):
    """prb_arm_dynamics on the emulator.  state: [N, state_dim] or [N, state_stride] rows; points: [(link, site, local)];
    q, qd, qdd: [N, nd] or None (NULL); outputs: the arrays to pass (the others are NULL); call / structs: a
    PrbArmQuery / point array to pass as is (invalid-input tests).  Returns the outputs asked for, jacobian [N,P,6,nd],
    position [N,P,3], velocity [N,P,6], mass_matrix [N,nd,nd], tau [N,nd]; ValueError with the library's message for a
    rejected call."""
    L = lib()
    st = _state(L, model, state)
    N, nd, P = st.shape[0], int(model['nd']), len(points)
    shapes = {'jacobian': (N, P, 6, nd), 'position': (N, P, 3), 'velocity': (N, P, 6), 'mass_matrix': (N, nd, nd),
              'tau': (N, nd)}
    out = {k: np.full(shapes[k], np.nan, np.float32) for k in outputs}
    ins = [None if x is None else np.ascontiguousarray(x, np.float32) for x in (q, qd, qdd)]
    call = call if call is not None else PrbArmQuery(P, 0)
    structs = structs if structs is not None else point_structs(points)
    p = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    rc = L.cemu_arm_dynamics(p(st), N, ctypes.byref(call), structs, *[p(x) for x in ins], *[p(out.get(k)) for k in OUTPUTS])
    if rc != 0:
        raise ValueError(L.cemu_error().decode())
    return out
