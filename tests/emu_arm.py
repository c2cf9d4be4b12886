"""prb_arm_dynamics' kernel source (csrc/prb_arm.cuh) on the emulated kernels of emu_lib.  CPU tests only."""
import ctypes

import numpy as np

from emu_lib import lib, rows
from roboticsplayroompybullet_b200.lib import PrbArmPoint, PrbArmQuery

OUTPUTS = ('jacobian', 'position', 'velocity', 'mass_matrix', 'tau')


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
    st = rows(model, state)
    N, nd, P = st.shape[0], int(model['nd']), len(points)
    shapes = {'jacobian': (N, P, 6, nd), 'position': (N, P, 3), 'velocity': (N, P, 6), 'mass_matrix': (N, nd, nd),
              'tau': (N, nd)}
    out = {k: np.full(shapes[k], np.nan, np.float32) for k in outputs}
    ins = [None if x is None else np.ascontiguousarray(x, np.float32) for x in (q, qd, qdd)]
    call = call if call is not None else PrbArmQuery(P, 0)
    structs = structs if structs is not None else point_structs(points)
    p = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    rc = L.emu_arm_dynamics(p(st), N, ctypes.byref(call), structs, *[p(x) for x in ins], *[p(out.get(k)) for k in OUTPUTS])
    if rc != 0:
        raise ValueError(L.emu_error().decode())
    return out
