"""The kernel source of prb_body_states, prb_write_state and prb_restore_state (csrc/prb_state.cuh) on the emulated
kernels of emu_lib, over the rows of an EmuSim: the masked observe after a write or restore is that sim's step pipeline.
CPU tests only."""
import ctypes

import numpy as np

from roboticsplayroompybullet_b200.lib import PrbBodyQuery


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
    s._sel()
    K, nj = sizes(s.m)
    shapes = {'body': (s.N, K, 13), 'q': (s.N, nj), 'qd': (s.N, nj)}
    out = {k: np.full(shapes[k], np.nan, np.float32) for k in outputs}
    call = call if call is not None else PrbBodyQuery(frame, 0)
    rc = s.L.emu_body_states(_p(s.state), s.N, ctypes.byref(call), *[_p(out.get(k)) for k in ('body', 'q', 'qd')])
    if rc != 0:
        raise ValueError(s.L.emu_error().decode())
    return out


def write_state(s, w, jq=None, jqd=None, body=None, mask=None):
    """prb_write_state on the emulator over EmuSim s (state, outputs and report updated in place): w a PrbStateWrite;
    returns the status [N] (0 not masked, 1 written, 2 rejected).  ValueError for a rejected call."""
    s._sel()
    status = np.full(s.N, 0xcd, np.uint8)
    ins = [_f32(x) for x in (jq, jqd, body)]
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    rc = s.L.emu_write_state(_p(s.state), ctypes.byref(s.O), s.N, ctypes.byref(w), *[_p(x) for x in ins], _p(m), _p(status))
    if rc != 0:
        raise ValueError(s.L.emu_error().decode())
    return status


def restore_state(s, snap, mask=None):
    """prb_restore_state on the emulator: snap [N, state_stride] rows back into EmuSim s for the masked envs."""
    s._sel()
    src = np.ascontiguousarray(snap, np.float32)
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    s.L.emu_restore_state(_p(s.state), ctypes.byref(s.O), s.N, _p(src), _p(m))
