"""prb_closest_points' kernel source (csrc/prb_closest.cuh) on the emulated kernels of emu_lib.  CPU tests only."""
import ctypes

import numpy as np

from emu_lib import lib, rows
from roboticsplayroompybullet_b200.lib import PrbClosest, PrbClosestQuery

FIELDS = ('collider_a', 'collider_b', 'distance', 'position_on_a', 'position_on_b', 'normal_on_b')


def closest_points(model, state, masks, max_distance, cull=True, call=None, null=()):
    """prb_closest_points on the emulator.  state: [N, state_dim] or [N, state_stride] rows; masks: [(mask_a, mask_b)];
    call: a PrbClosest to pass as is (invalid-input tests), null: names of arrays to pass as NULL ('queries' or a
    field).  Returns dict collider_a, collider_b, distance [N,Q], position_on_a, position_on_b, normal_on_b [N,Q,3];
    ValueError with the library's message for a rejected call."""
    L = lib()
    st = rows(model, state)
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
    rc = L.emu_closest_points(st.ctypes.data_as(ctypes.c_void_p), N, ctypes.byref(call), None if 'queries' in null else qs,
                              *[p(k) for k in FIELDS], 1 if cull else 0)
    if rc != 0:
        raise ValueError(L.emu_error().decode())
    return out
