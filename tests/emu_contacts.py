"""The contact report's layout (include/prb.h prb_contacts), as EmuSim(report=True) reads it from the emulated step
(csrc/prb_contacts.cuh and the report mode of the setup and solver kernels in csrc/prb_stream.cuh).  CPU tests only."""
import numpy as np

# (name, numpy type, per-contact components), in the order of the report's fields (include/prb.h prb_contacts)
FIELDS = [('collider_a', np.int32, 1), ('collider_b', np.int32, 1), ('position_on_a', np.float32, 3),
          ('position_on_b', np.float32, 3), ('normal_on_b', np.float32, 3), ('distance', np.float32, 1),
          ('normal_force', np.float32, 1), ('lateral_friction_1', np.float32, 1), ('lateral_friction_2', np.float32, 1),
          ('lateral_friction_dir_1', np.float32, 3), ('lateral_friction_dir_2', np.float32, 3)]


def split_report(buf, N, K=64):
    """The report allocation (float32 words) as a dict of arrays shaped like VecPlayEnv.contacts()."""
    d, off = {}, 0
    for name, ty, k in FIELDS:
        n = N * K * k
        d[name] = buf[off:off + n].view(ty).reshape((N, K) if k == 1 else (N, K, k)).copy()
        off += n
    d['count'] = buf[off:off + N].view(np.int32).copy()
    return d
