"""ctypes front-end of tests/emu/librays_emu.so: prb_ray_test's kernel source (csrc/prb_rays.cuh) compiled with g++
against the SIMT emulator (tests/emu/cuda_emu.h).  CPU tests only."""
import ctypes
import os
import subprocess

import numpy as np

from roboticsplayroompybullet_b200.lib import PrbRays

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
    so = os.path.join(_HERE, 'librays_emu.so')
    deps = [os.path.join(_HERE, f) for f in ('rays_emu.cpp', 'cuda_emu.h')] + \
           [os.path.join(_SRC, f) for f in ('prb_rays.cuh', 'prb_render.cuh', 'prb_kernels.cuh', 'prb_device.h', 'prb_convert.h')] + \
           [os.path.join(_ROOT, 'include', f) for f in ('prb.h', 'prb_model.h')]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        tmp = '%s.%d.tmp.so' % (so[:-3], os.getpid())
        subprocess.check_call(['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-U_FORTIFY_SOURCE', '-Wno-unknown-pragmas',
                               '-o', tmp, os.path.join(_HERE, 'rays_emu.cpp')])
        os.replace(tmp, so)
    L = ctypes.CDLL(so)
    L.yemu_error.restype = ctypes.c_char_p
    vp = ctypes.c_void_p
    L.yemu_ray_test.argtypes = [vp, ctypes.c_int, ctypes.POINTER(PrbRays), vp, vp, vp, vp, vp, vp, ctypes.c_int]
    _LIB = L
    return L


def _state(L, model, state):
    ms = model.as_struct()
    if L.yemu_set_model(ctypes.byref(ms)) != 0:
        raise RuntimeError(L.yemu_error().decode())
    stride = L.yemu_state_stride()
    st = np.asarray(state)
    if st.dtype != np.float32 or st.ndim != 2 or st.shape[1] != stride or not st.flags.c_contiguous:
        s2 = np.zeros((st.shape[0], stride), np.float32)
        s2[:, :L.yemu_state_dim()] = st[:, :L.yemu_state_dim()]
        st = s2
    return st


def ray_test(model, state, frm, to, site=None, mask=~0, force_large=False, rays=None, null=()):
    """prb_ray_test on the emulator.  state: [N, state_dim] or [N, state_stride] rows; frm, to: [R,3] (shared) or
    [N,R,3] (per env), in the world (site None) or site `site`; mask: collider_mask.  rays: a PrbRays to pass as is
    (invalid-input tests), null: names of arrays to pass as NULL.  Returns dict collider [N,R], fraction [N,R], position,
    normal [N,R,3]; ValueError with the library's message for a rejected call."""
    L = lib()
    st = _state(L, model, state)
    N = st.shape[0]
    f = np.ascontiguousarray(frm, np.float32)
    t = np.ascontiguousarray(to, np.float32)
    per_env = 1 if f.ndim == 3 else 0
    R = f.shape[-2]
    if rays is None:
        rays = PrbRays(R, per_env, -1 if site is None else site, 0, mask & 0xFFFFFFFFFFFFFFFF)
    R = rays.num_rays if 1 <= rays.num_rays <= 16384 else 1         # output size of a rejected call: any
    out = {'collider': np.zeros((N, R), np.int32), 'fraction': np.zeros((N, R), np.float32),
           'position': np.zeros((N, R, 3), np.float32), 'normal': np.zeros((N, R, 3), np.float32)}
    arrs = {'from': f, 'to': t, **out}
    p = lambda k: None if k in null else arrs[k].ctypes.data_as(ctypes.c_void_p)
    rc = L.yemu_ray_test(st.ctypes.data_as(ctypes.c_void_p), N, ctypes.byref(rays), p('from'), p('to'), p('collider'),
                         p('fraction'), p('position'), p('normal'), 1 if force_large else 0)
    if rc != 0:
        raise ValueError(L.yemu_error().decode())
    return out
