"""ctypes front-end of tests/emu/librender_emu.so: prb_render's kernel source (csrc/prb_render.cuh) compiled with g++
against the SIMT emulator (tests/emu/cuda_emu.h).  CPU tests only."""
import ctypes
import os
import subprocess

import numpy as np

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
    so = os.path.join(_HERE, 'librender_emu.so')
    deps = [os.path.join(_HERE, f) for f in ('render_emu.cpp', 'cuda_emu.h')] + \
           [os.path.join(_SRC, f) for f in ('prb_render.cuh', 'prb_kernels.cuh', 'prb_device.h', 'prb_convert.h')] + \
           [os.path.join(_ROOT, 'include', f) for f in ('prb.h', 'prb_model.h')]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        tmp = '%s.%d.tmp.so' % (so[:-3], os.getpid())
        subprocess.check_call(['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-U_FORTIFY_SOURCE', '-Wno-unknown-pragmas',
                               '-o', tmp, os.path.join(_HERE, 'render_emu.cpp')])
        os.replace(tmp, so)
    L = ctypes.CDLL(so)
    L.remu_error.restype = ctypes.c_char_p
    _LIB = L
    return L


def render(model, state, camera, palette, depth=False, segmentation=False):
    """prb_render on the emulator.  state: float32 [N, state_stride] rows (e.g. EmuSim.state), read in place, or
    [N, state_dim].  Returns dict rgb [N,H,W,3] uint8 (+ depth, segmentation) and box_tests."""
    from roboticsplayroompybullet_b200.camera import camera_struct
    L = lib()
    ms = model.as_struct()
    if L.remu_set_model(ctypes.byref(ms)) != 0:
        raise RuntimeError(L.remu_error().decode())
    stride = L.remu_state_stride()
    st = np.asarray(state)
    if st.dtype != np.float32 or st.ndim != 2 or st.shape[1] != stride or not st.flags.c_contiguous:
        s2 = np.zeros((st.shape[0], stride), np.float32)
        s2[:, :L.remu_state_dim()] = st[:, :L.remu_state_dim()]
        st = s2
    N, H, W = st.shape[0], camera.height, camera.width
    cs = camera_struct(camera)
    pal = np.ascontiguousarray(palette, np.float32).reshape(-1, 3)
    out = {'rgb': np.zeros((N, H, W, 3), np.uint8)}
    if depth:
        out['depth'] = np.zeros((N, H, W), np.float32)
    if segmentation:
        out['segmentation'] = np.zeros((N, H, W), np.int32)
    p = lambda k: out[k].ctypes.data_as(ctypes.c_void_p) if k in out else None
    tests = ctypes.c_uint64(0)
    rc = L.remu_render(st.ctypes.data_as(ctypes.c_void_p), N, ctypes.byref(cs), pal.ctypes.data_as(ctypes.c_void_p),
                       p('rgb'), p('depth'), p('segmentation'), ctypes.byref(tests))
    if rc != 0:
        raise ValueError(L.remu_error().decode())
    out['box_tests'] = int(tests.value)
    return out
