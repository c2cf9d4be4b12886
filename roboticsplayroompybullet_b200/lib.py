"""ctypes binding of libprb_b200.so (include/prb.h).  The library is the product's only compute
path: if it is missing or no CUDA device is present, loading/creation FAILS LOUDLY -- there is no
CPU or PyTorch fallback."""
import ctypes
import os

from .model import PrbModelStruct

_HERE = os.path.dirname(os.path.abspath(__file__))
# PRB_LIB selects another build of the same sources (A/B experiments with compile-time knobs, tools/build_variants.sh)
LIB_PATH = os.environ.get('PRB_LIB') or os.path.join(_HERE, 'libprb_b200.so')
_LIB = None


class PrbConfig(ctypes.Structure):
    _fields_ = [('num_envs', ctypes.c_int32), ('env_offset', ctypes.c_int32), ('device', ctypes.c_int32),
                ('reserved', ctypes.c_int32), ('seed', ctypes.c_uint64)]


_PTRS = ['state', 'out_base', 'obs_quat', 'achieved_goal', 'desired_goal', 'controllable_achieved_goal',
         'full_positional_state', 'joints', 'velocity', 'observation', 'gripper_proprioception', 'reward',
         'is_success', 'target_poses']
_INTS = ['num_envs', 'state_dim', 'state_stride', 'obs_dim', 'goal_dim', 'fps_dim', 'observation_dim', 'n_ik']


class PrbBuffers(ctypes.Structure):
    _fields_ = ([(n, ctypes.c_void_p) for n in _PTRS] + [('out_floats', ctypes.c_int64)] +
                [(n, ctypes.c_int32) for n in _INTS])


class PrbCamera(ctypes.Structure):
    _fields_ = [('width', ctypes.c_int32), ('height', ctypes.c_int32), ('attach', ctypes.c_int32),
                ('view', ctypes.c_float * 16), ('proj', ctypes.c_float * 16), ('light_dir', ctypes.c_float * 3),
                ('ambient', ctypes.c_float), ('diffuse', ctypes.c_float), ('background', ctypes.c_float * 3)]


class PrbRays(ctypes.Structure):
    _fields_ = [('num_rays', ctypes.c_int32), ('per_env', ctypes.c_int32), ('frame', ctypes.c_int32),
                ('reserved', ctypes.c_int32), ('collider_mask', ctypes.c_uint64)]


class PrbClosestQuery(ctypes.Structure):
    _fields_ = [('mask_a', ctypes.c_uint64), ('mask_b', ctypes.c_uint64)]


class PrbClosest(ctypes.Structure):
    _fields_ = [('num_queries', ctypes.c_int32), ('reserved', ctypes.c_int32), ('max_distance', ctypes.c_float),
                ('reserved2', ctypes.c_int32)]


class PrbArmPoint(ctypes.Structure):
    _fields_ = [('link', ctypes.c_int32), ('site', ctypes.c_int32), ('local_position', ctypes.c_float * 3),
                ('reserved', ctypes.c_int32)]


class PrbArmQuery(ctypes.Structure):
    _fields_ = [('num_points', ctypes.c_int32), ('reserved', ctypes.c_int32)]


class PrbBodyQuery(ctypes.Structure):
    _fields_ = [('frame', ctypes.c_int32), ('reserved', ctypes.c_int32)]


class PrbStateWrite(ctypes.Structure):
    _fields_ = [('joint_positions', ctypes.c_uint32), ('joint_velocities', ctypes.c_uint32), ('free_poses', ctypes.c_uint32),
                ('free_velocities', ctypes.c_uint32), ('reserved', ctypes.c_int32)]


# prb_contacts: the contact report's device arrays; (name, element type, per-contact components) in struct order
CONTACT_FIELDS = [('collider_a', 'i4', 1), ('collider_b', 'i4', 1), ('position_on_a', 'f4', 3), ('position_on_b', 'f4', 3),
                  ('normal_on_b', 'f4', 3), ('distance', 'f4', 1), ('normal_force', 'f4', 1), ('lateral_friction_1', 'f4', 1),
                  ('lateral_friction_2', 'f4', 1), ('lateral_friction_dir_1', 'f4', 3), ('lateral_friction_dir_2', 'f4', 3)]


class PrbContacts(ctypes.Structure):
    _fields_ = ([('count', ctypes.c_void_p)] + [(n, ctypes.c_void_p) for n, _, _ in CONTACT_FIELDS] +
                [('num_envs', ctypes.c_int32), ('max_contacts', ctypes.c_int32)])


# prb_dynamics: the per-env dynamics table's device arrays, in struct order
DYNAMICS_FIELDS = ['lateral_friction', 'spinning_friction', 'mass', 'local_inertia_diagonal', 'linear_damping', 'angular_damping']
# prb_dynamics_ranges, in struct order
DYNAMICS_RANGE_FIELDS = ['lateral_friction', 'spinning_friction', 'mass', 'linear_damping', 'angular_damping']


class PrbDynamics(ctypes.Structure):
    _fields_ = ([(n, ctypes.c_void_p) for n in DYNAMICS_FIELDS] +
                [('num_envs', ctypes.c_int32), ('n_col', ctypes.c_int32), ('n_free', ctypes.c_int32)])


class PrbDynamicsRanges(ctypes.Structure):
    _fields_ = [(n, ctypes.c_float * 2) for n in DYNAMICS_RANGE_FIELDS]


# every symbol include/prb.h declares (a CPU test checks the built library exports them all)
SYMBOLS = ['prb_create', 'prb_destroy', 'prb_reset', 'prb_reset_rounds', 'prb_reset_to', 'prb_set_goal', 'prb_step', 'prb_observe', 'prb_substeps',
           'prb_get_buffers', 'prb_compute_reward', 'prb_get_state', 'prb_set_state', 'prb_step_host',
           'prb_enable_kernel_timing', 'prb_last_kernel_ms', 'prb_last_tier_ms', 'prb_launch_count', 'prb_overflow_count', 'prb_debug_usage', 'prb_kernel_info', 'prb_render', 'prb_render_box_tests',
           'prb_ray_test', 'prb_closest_points', 'prb_arm_dynamics',
           'prb_body_states', 'prb_write_state', 'prb_save_state', 'prb_restore_state',
           'prb_enable_contacts', 'prb_get_contacts', 'prb_enable_dynamics', 'prb_get_dynamics', 'prb_randomize_dynamics',
           'prb_last_error',
           'prb_version']


class PrbError(RuntimeError):
    pass


def load():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise PrbError('%s not built: run `python -c "import __graft_entry__ as g; g.build()"` '
                       '(nvcc, sm_100a). There is no CPU fallback.' % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    L.prb_create.argtypes = [ctypes.POINTER(PrbModelStruct), ctypes.POINTER(PrbConfig), ctypes.POINTER(vp)]
    L.prb_destroy.argtypes = [vp]
    L.prb_reset.argtypes = [vp, vp, vp]
    L.prb_reset_rounds.argtypes = [vp]
    L.prb_reset_to.argtypes = [vp, vp, vp, i32, vp]
    L.prb_set_goal.argtypes = [vp, vp, vp, vp]
    L.prb_step.argtypes = [vp, vp, vp]
    L.prb_observe.argtypes = [vp, vp]
    L.prb_substeps.argtypes = [vp, i32, vp]
    L.prb_get_buffers.argtypes = [vp, ctypes.POINTER(PrbBuffers)]
    L.prb_compute_reward.argtypes = [vp, vp, vp, i64, vp, vp]
    L.prb_get_state.argtypes = [vp, vp]
    L.prb_set_state.argtypes = [vp, vp]
    L.prb_step_host.argtypes = [vp, vp, vp, vp]
    L.prb_enable_kernel_timing.argtypes = [vp, i32]
    L.prb_last_kernel_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    L.prb_last_tier_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    L.prb_launch_count.argtypes = [vp]
    L.prb_launch_count.restype = i64
    L.prb_overflow_count.argtypes = [vp]
    L.prb_debug_usage.argtypes = [vp, vp]
    L.prb_overflow_count.restype = i64
    L.prb_kernel_info.argtypes = [vp, ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(i32)]
    L.prb_render.argtypes = [vp, ctypes.POINTER(PrbCamera), vp, vp, vp, vp, vp]
    L.prb_render_box_tests.argtypes = [vp]
    L.prb_render_box_tests.restype = i64
    L.prb_ray_test.argtypes = [vp, ctypes.POINTER(PrbRays), vp, vp, vp, vp, vp, vp, vp]
    L.prb_closest_points.argtypes = [vp, ctypes.POINTER(PrbClosest), ctypes.POINTER(PrbClosestQuery), vp, vp, vp, vp, vp, vp, vp]
    L.prb_arm_dynamics.argtypes = [vp, ctypes.POINTER(PrbArmQuery), ctypes.POINTER(PrbArmPoint), vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.prb_body_states.argtypes = [vp, ctypes.POINTER(PrbBodyQuery), vp, vp, vp, vp]
    L.prb_write_state.argtypes = [vp, ctypes.POINTER(PrbStateWrite), vp, vp, vp, vp, vp, vp]
    L.prb_save_state.argtypes = [vp, vp, vp]
    L.prb_restore_state.argtypes = [vp, vp, vp, vp]
    L.prb_enable_contacts.argtypes = [vp, i32]
    L.prb_get_contacts.argtypes = [vp, ctypes.POINTER(PrbContacts)]
    L.prb_enable_dynamics.argtypes = [vp, i32]
    L.prb_get_dynamics.argtypes = [vp, ctypes.POINTER(PrbDynamics)]
    L.prb_randomize_dynamics.argtypes = [vp, ctypes.POINTER(PrbDynamicsRanges), vp, vp]
    L.prb_last_error.argtypes = [vp]
    L.prb_last_error.restype = ctypes.c_char_p
    L.prb_version.restype = ctypes.c_char_p
    _LIB = L
    return L


def check(L, handle, rc):
    if rc != 0:
        raise PrbError('libprb_b200: status %d: %s' % (rc, L.prb_last_error(handle).decode()))
