"""prb_render's kernel source (csrc/prb_render.cuh) on the emulated kernels of emu_lib.  CPU tests only."""
import ctypes

import numpy as np

from emu_lib import lib, rows


def render(model, state, camera, palette, depth=False, segmentation=False):
    """prb_render on the emulator.  state: float32 [N, state_stride] rows (e.g. EmuSim.state), read in place, or
    [N, state_dim].  Returns dict rgb [N,H,W,3] uint8 (+ depth, segmentation) and box_tests."""
    from roboticsplayroompybullet_b200.camera import camera_struct
    L = lib()
    st = rows(model, state)
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
    rc = L.emu_render(st.ctypes.data_as(ctypes.c_void_p), N, ctypes.byref(cs), pal.ctypes.data_as(ctypes.c_void_p),
                      p('rgb'), p('depth'), p('segmentation'), ctypes.byref(tests))
    if rc != 0:
        raise ValueError(L.emu_error().decode())
    out['box_tests'] = int(tests.value)
    return out
