"""ctypes front-end of tests/emu/libstate_emu.so: the kernel source of prb_body_states, prb_write_state and
prb_restore_state (csrc/prb_state.cuh) compiled with g++ against the SIMT emulator (tests/emu/cuda_emu.h), together with
the step harness tests/emu/prb_emu.cpp, so that an EmuSim built on this library (sim()) is the simulator the calls read
and write.  CPU tests only."""
import ctypes
import os
import subprocess

import numpy as np

from emu_lib import EmuSim
from roboticsplayroompybullet_b200.lib import PrbBodyQuery, PrbStateWrite

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
    so = os.path.join(_HERE, 'libstate_emu.so')
    deps = [os.path.join(_HERE, f) for f in ('state_emu.cpp', 'prb_emu.cpp', 'cuda_emu.h')] + \
           [os.path.join(_SRC, f) for f in ('prb_state.cuh', 'prb_render.cuh', 'prb_kernels.cuh', 'prb_stream.cuh',
                                            'prb_reset.cuh', 'prb_device.h', 'prb_convert.h')] + \
           [os.path.join(_ROOT, 'include', f) for f in ('prb.h', 'prb_model.h')]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        tmp = '%s.%d.tmp.so' % (so[:-3], os.getpid())
        subprocess.check_call(['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-U_FORTIFY_SOURCE', '-Wno-unknown-pragmas',
                               '-o', tmp, os.path.join(_HERE, 'state_emu.cpp')])
        os.replace(tmp, so)
    L = ctypes.CDLL(so)
    L.emu_error.restype = ctypes.c_char_p
    vp = ctypes.c_void_p
    L.semu_body_states.argtypes = [vp, ctypes.c_int, ctypes.POINTER(PrbBodyQuery), vp, vp, vp]
    L.semu_write_state.argtypes = [vp, vp, ctypes.c_int, ctypes.POINTER(PrbStateWrite), vp, vp, vp, vp, vp]
    L.semu_restore_state.argtypes = [vp, vp, ctypes.c_int, vp, vp]
    _LIB = L
    return L


def sim(model, N, seed=1234):
    """An EmuSim whose kernels are this library's copy of the step harness."""
    return EmuSim(model, N, seed=seed, library=lib())


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _f32(a):
    return None if a is None else np.ascontiguousarray(a, np.float32)


def sizes(model):
    nd, nf, ns = int(model['nd']), int(model['n_free']), int(model['n_slide'])
    return nd + nf + ns, nd + ns


def body_states(s, frame=0, outputs=('body', 'q', 'qd'), call=None):
    """prb_body_states on the emulator over the rows of EmuSim s: dict 'body' [N,K,13], 'q', 'qd' [N,nd+n_slide] of the
    outputs asked for (the others are NULL); call: a PrbBodyQuery to pass as is.  ValueError for a rejected call."""
    L = lib()
    s._sel()
    K, nj = sizes(s.m)
    shapes = {'body': (s.N, K, 13), 'q': (s.N, nj), 'qd': (s.N, nj)}
    out = {k: np.full(shapes[k], np.nan, np.float32) for k in outputs}
    call = call if call is not None else PrbBodyQuery(frame, 0)
    rc = L.semu_body_states(_p(s.state), s.N, ctypes.byref(call), *[_p(out.get(k)) for k in ('body', 'q', 'qd')])
    if rc != 0:
        raise ValueError(L.emu_error().decode())
    return out


def write_state(s, w, jq=None, jqd=None, body=None, mask=None):
    """prb_write_state on the emulator over EmuSim s (state and outputs updated in place): w a PrbStateWrite; returns the
    status [N] (0 not masked, 1 written, 2 rejected).  ValueError for a rejected call."""
    L = lib()
    s._sel()
    status = np.full(s.N, 0xcd, np.uint8)
    ins = [_f32(x) for x in (jq, jqd, body)]
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    rc = L.semu_write_state(_p(s.state), ctypes.byref(s.O), s.N, ctypes.byref(w), *[_p(x) for x in ins], _p(m), _p(status))
    if rc != 0:
        raise ValueError(L.emu_error().decode())
    return status


def restore_state(s, snap, mask=None):
    """prb_restore_state on the emulator: snap [N, state_stride] rows back into EmuSim s for the masked envs."""
    L = lib()
    s._sel()
    src = np.ascontiguousarray(snap, np.float32)
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    L.semu_restore_state(_p(s.state), ctypes.byref(s.O), s.N, _p(src), _p(m))
