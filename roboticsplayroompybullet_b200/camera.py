"""Cameras for prb_render (include/prb.h): the OpenGL look-at / perspective matrices PyBullet's computeViewMatrix,
computeViewMatrixFromYawPitchRoll and computeProjectionMatrixFOV return (column-major, flattened to 16 floats),
the default world and gripper cameras, and the default colour of every collider.

The reference fills calc_state's 'img' from a fixed world camera (environments.py:841-845) and also has a camera on
the gripper (:33-49).  Their constants are not in this tree, so the cameras and colours here are this project's own
(INTEGRATION.md §5)."""

import numpy as np


def _normalize(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v)


def view_matrix(eye, target, up):
    """computeViewMatrix(cameraEyePosition, cameraTargetPosition, cameraUpVector): world -> eye, column-major [16]."""
    eye = np.asarray(eye, np.float64)
    f = _normalize(np.asarray(target, np.float64) - eye)
    s = _normalize(np.cross(f, _normalize(up)))
    u = np.cross(s, f)
    M = np.eye(4)
    M[0, :3], M[1, :3], M[2, :3] = s, u, -f
    M[:3, 3] = [-s @ eye, -u @ eye, f @ eye]
    return M.T.reshape(16).astype(np.float32)


def _rot(axis, a):
    c, s = np.cos(a), np.sin(a)
    if axis == 0:
        return np.array([[1, 0, 0], [0, c, -s], [0, s, c]])
    if axis == 1:
        return np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])
    return np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]])


def yaw_pitch_eye(target, dist, yaw, pitch, up_axis=2):
    """Eye position and up vector of computeViewMatrixFromYawPitchRoll (degrees; PyBullet ignores the roll)."""
    y, p = np.radians(yaw), np.radians(pitch)
    if up_axis == 2:
        R = _rot(2, y) @ _rot(0, p)                 # setEulerZYX(yaw, roll = 0, pitch)
        eye, up = np.array([0.0, -dist, 0.0]), np.array([0.0, 0.0, 1.0])
    elif up_axis == 1:
        R = _rot(1, y) @ _rot(0, -p)                # setEulerZYX(roll = 0, yaw, -pitch)
        eye, up = np.array([0.0, 0.0, -dist]), np.array([0.0, 1.0, 0.0])
    else:
        raise ValueError('up_axis must be 1 or 2')
    return np.asarray(target, np.float64) + R @ eye, R @ up


def view_matrix_from_yaw_pitch_roll(target, dist, yaw, pitch, roll, up_axis=2):
    """computeViewMatrixFromYawPitchRoll: the camera circles `target` at `dist`; angles in degrees.  The roll argument
    is accepted and ignored, as PyBullet does."""
    eye, up = yaw_pitch_eye(target, dist, yaw, pitch, up_axis)
    return view_matrix(eye, target, up)


def projection_matrix_fov(fov, aspect, near, far):
    """computeProjectionMatrixFOV: vertical field of view in degrees, aspect = width / height; column-major [16]."""
    ys = 1.0 / np.tan(np.radians(fov) / 2)
    M = np.zeros((4, 4))
    M[0, 0], M[1, 1] = ys / aspect, ys
    M[2, 2], M[2, 3] = (far + near) / (near - far), 2 * far * near / (near - far)
    M[3, 2] = -1.0
    return M.T.reshape(16).astype(np.float32)


class Camera:
    """A pinhole camera: `view` maps the world (attach=False) or the end-effector site frame (attach=True, a camera
    carried by the gripper) to eye coordinates; `proj` is a perspective projection.  Both are column-major [16], as
    the functions above and PyBullet return them.  Shading: colour * (ambient + diffuse * max(0, n . light_dir))."""

    def __init__(self, width, height, view, proj, attach=False, light_dir=(0.3, -0.5, 1.0), ambient=0.45, diffuse=0.55,
                 background=(0.78, 0.86, 0.96)):
        self.width, self.height, self.attach = int(width), int(height), bool(attach)
        self.view = np.asarray(view, np.float32).reshape(16)
        self.proj = np.asarray(proj, np.float32).reshape(16)
        self.light_dir = np.asarray(light_dir, np.float32).reshape(3)
        self.ambient, self.diffuse = float(ambient), float(diffuse)
        self.background = np.asarray(background, np.float32).reshape(3)


def camera_struct(cam):
    """ctypes prb_camera of a Camera."""
    from .lib import PrbCamera
    s = PrbCamera()
    s.width, s.height, s.attach = cam.width, cam.height, 1 if cam.attach else 0
    s.view[:] = [float(x) for x in cam.view]
    s.proj[:] = [float(x) for x in cam.proj]
    s.light_dir[:] = [float(x) for x in cam.light_dir]
    s.ambient, s.diffuse = cam.ambient, cam.diffuse
    s.background[:] = [float(x) for x in cam.background]
    return s


def default_camera(model, width=200, height=200):
    """World camera in front of the workspace (the desk side of the playroom), looking at the centre of the goal box."""
    lo, hi = np.asarray(model['goal_lo'][:3]), np.asarray(model['goal_hi'][:3])
    target = 0.5 * (lo + hi)
    if model['play']:
        view = view_matrix_from_yaw_pitch_roll(target + [0.0, 0.05, 0.0], 1.25, 0.0, -32.0, 0.0)
    else:
        view = view_matrix_from_yaw_pitch_roll(target, 1.0, 0.0, -40.0, 0.0)
    return Camera(width, height, view, projection_matrix_fov(60.0, width / height, 0.05, 5.0))


def gripper_camera(model, width=200, height=200):
    """Camera carried by the gripper: in the end-effector site frame the approach axis is -z (the grasp point lies
    beyond the pads) and the pads sit on the x axis; the eye is beside the fingers and looks down the approach axis."""
    view = view_matrix([0.0, 0.06, 0.08], [0.0, 0.0, -0.2], [0.0, 1.0, 0.0])
    return Camera(width, height, view, projection_matrix_fov(75.0, width / height, 0.01, 3.0), attach=True)


# colours by role
ARM_RGB = (0.72, 0.72, 0.76)
SCENE_RGB = (0.80, 0.68, 0.52)       # static scene: desk, shelves, tray
GROUND_RGB = (0.45, 0.47, 0.50)      # static colliders larger than 1 m (ground plane)
FREE_RGB = [(0.85, 0.18, 0.16), (0.55, 0.33, 0.18)]                     # block / cube, drawer
SLIDE_RGB = [(0.22, 0.48, 0.82), (0.95, 0.78, 0.10), (0.20, 0.68, 0.30)]   # door, button, dial


def default_palette(model):
    """[n_col, 3] float32 colours from col_body: arm, each free body, each slide body, static scene."""
    n = int(model['n_col'])
    body = np.asarray(model['col_body'])
    half = np.asarray(model['col_half'], np.float64).reshape(n, 3)
    nf = int(model['n_free'])
    out = np.zeros((n, 3), np.float32)
    for c in range(n):
        b = int(body[c])
        if b == 0:
            out[c] = ARM_RGB
        elif b < 0:
            out[c] = GROUND_RGB if half[c].max() > 1.0 else SCENE_RGB
        elif b <= nf:
            out[c] = FREE_RGB[(b - 1) % len(FREE_RGB)]
        else:
            out[c] = SLIDE_RGB[(b - 1 - nf) % len(SLIDE_RGB)]
    return out
