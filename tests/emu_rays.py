"""prb_ray_test's kernel source (csrc/prb_rays.cuh) on the emulated kernels of emu_lib.  CPU tests only."""
import ctypes

import numpy as np

from emu_lib import lib, rows
from roboticsplayroompybullet_b200.lib import PrbRays


def ray_test(model, state, frm, to, site=None, mask=~0, force_large=False, rays=None, null=()):
    """prb_ray_test on the emulator.  state: [N, state_dim] or [N, state_stride] rows; frm, to: [R,3] (shared) or
    [N,R,3] (per env), in the world (site None) or site `site`; mask: collider_mask.  rays: a PrbRays to pass as is
    (invalid-input tests), null: names of arrays to pass as NULL.  Returns dict collider [N,R], fraction [N,R], position,
    normal [N,R,3]; ValueError with the library's message for a rejected call."""
    L = lib()
    st = rows(model, state)
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
    rc = L.emu_ray_test(st.ctypes.data_as(ctypes.c_void_p), N, ctypes.byref(rays), p('from'), p('to'), p('collider'),
                        p('fraction'), p('position'), p('normal'), 1 if force_large else 0)
    if rc != 0:
        raise ValueError(L.emu_error().decode())
    return out
