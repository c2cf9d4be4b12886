"""ctypes front-end of tests/emu/libclosest_emu.so: prb_closest_points' kernel source (csrc/prb_closest.cuh) compiled with
g++ against the SIMT emulator (tests/emu/cuda_emu.h).  CPU tests only."""
import ctypes
import os
import subprocess

import numpy as np

from roboticsplayroompybullet_b200.lib import PrbClosest, PrbClosestQuery

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'emu')
_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
_SRC = os.path.join(_ROOT, 'roboticsplayroompybullet_b200', 'csrc')
_LIB = None


def lib():
    """g++ build unless the library is newer than every source; written under a temporary name and renamed, so that
    test processes running in parallel never load a half-written file."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = os.path.join(_HERE, 'libclosest_emu.so')
    deps = [os.path.join(_HERE, f) for f in ('closest_emu.cpp', 'cuda_emu.h')] + \
           [os.path.join(_SRC, f) for f in ('prb_closest.cuh', 'prb_render.cuh', 'prb_kernels.cuh', 'prb_device.h', 'prb_convert.h')] + \
           [os.path.join(_ROOT, 'include', f) for f in ('prb.h', 'prb_model.h')]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        tmp = '%s.%d.tmp.so' % (so[:-3], os.getpid())
        subprocess.check_call(['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-U_FORTIFY_SOURCE', '-Wno-unknown-pragmas',
                               '-o', tmp, os.path.join(_HERE, 'closest_emu.cpp')])
        os.replace(tmp, so)
    L = ctypes.CDLL(so)
    L.cemu_error.restype = ctypes.c_char_p
    vp = ctypes.c_void_p
    L.cemu_closest_points.argtypes = [vp, ctypes.c_int, ctypes.POINTER(PrbClosest), ctypes.POINTER(PrbClosestQuery),
                                      vp, vp, vp, vp, vp, vp, ctypes.c_int]
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


FIELDS = ('collider_a', 'collider_b', 'distance', 'position_on_a', 'position_on_b', 'normal_on_b')


def closest_points(model, state, masks, max_distance, cull=True, call=None, null=()):
    """prb_closest_points on the emulator.  state: [N, state_dim] or [N, state_stride] rows; masks: [(mask_a, mask_b)];
    call: a PrbClosest to pass as is (invalid-input tests), null: names of arrays to pass as NULL ('queries' or a
    field).  Returns dict collider_a, collider_b, distance [N,Q], position_on_a, position_on_b, normal_on_b [N,Q,3];
    ValueError with the library's message for a rejected call."""
    L = lib()
    st = _state(L, model, state)
    N = st.shape[0]
    if call is None:
        call = PrbClosest(len(masks), 0, max_distance, 0)
    Q = max(len(masks), 1)
    qs = (PrbClosestQuery * Q)(*[PrbClosestQuery(a & 0xFFFFFFFFFFFFFFFF, b & 0xFFFFFFFFFFFFFFFF) for a, b in masks])
    out = {'collider_a': np.zeros((N, Q), np.int32), 'collider_b': np.zeros((N, Q), np.int32),
           'distance': np.zeros((N, Q), np.float32)}
    for k in FIELDS[3:]:
        out[k] = np.zeros((N, Q, 3), np.float32)
    p = lambda k: None if k in null else out[k].ctypes.data_as(ctypes.c_void_p)
    rc = L.cemu_closest_points(st.ctypes.data_as(ctypes.c_void_p), N, ctypes.byref(call), None if 'queries' in null else qs,
                               *[p(k) for k in FIELDS], 1 if cull else 0)
    if rc != 0:
        raise ValueError(L.cemu_error().decode())
    return out
