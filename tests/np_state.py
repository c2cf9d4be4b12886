"""fp64 numpy reference of prb_body_states: every body row of one state row (arm links in the link or COM frame from
tests/np_arm_dynamics.py's forward kinematics, link twists by an outward pass, free bodies from the state, slide bodies
from the model's joint frames), and the host edit prb_write_state must reproduce."""
import numpy as np

import np_arm_dynamics as R


def quat_mat(x):
    x, y, z, w = np.asarray(x, np.float64) / np.linalg.norm(np.asarray(x, np.float64))
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def twists(A, q, qd):
    """Angular velocity w and linear velocity v of every link frame origin (world), fp64."""
    nd = A['nd']
    _, p, a, _ = R.fk(A, q)
    w, v = np.zeros((nd, 3)), np.zeros((nd, 3))
    for i in range(nd):
        par = A['parent'][i]
        wp, vp, pp = (np.zeros(3), np.zeros(3), A['base_pos']) if par < 0 else (w[par], v[par], p[par])
        v[i] = vp + np.cross(wp, p[i] - pp)
        if A['jtype'][i] == 0:
            w[i] = wp + a[i] * qd[i]
        else:
            w[i] = wp
            v[i] = v[i] + a[i] * qd[i]
    return w, v


def reference_rows(m, row, frame):
    """[K, 3, 3] rotations and [K, 12] (pos, linear velocity, angular velocity) of one state row, fp64."""
    A = R.arm(m)
    nd, nf, ns = int(m['nd']), int(m['n_free']), int(m['n_slide'])
    st = np.asarray(row, np.float64)
    q, qd = st[:nd], st[nd:2 * nd]
    Rl, p, _, c = R.fk(A, q)
    w, v = twists(A, q, qd)
    rots, vec = [], []
    for l in range(nd):
        o = c[l] if frame else p[l]
        rots.append(Rl[l])
        vec.append(np.concatenate([o, v[l] + np.cross(w[l], o - p[l]), w[l]]))
    for b in range(nf):
        r = st[5 * nd + 13 * b:5 * nd + 13 * b + 13]
        rots.append(quat_mat(r[3:7]))
        vec.append(np.concatenate([r[:3], r[7:13]]))
    so = 5 * nd + 13 * nf
    for s in range(ns):
        sq, sqd = st[so + 2 * s], st[so + 2 * s + 1]
        R0 = np.asarray(m['slide_rot'], np.float64).reshape(-1, 3, 3)[s]
        ax = np.asarray(m['slide_axis'], np.float64).reshape(-1, 3)[s]
        p0 = np.asarray(m['slide_pos'], np.float64).reshape(-1, 3)[s]
        aw = R0 @ ax
        if int(np.asarray(m['slide_jtype'])[s]) == 0:
            rots.append(R0 @ R._axis_angle(ax, sq))
            vec.append(np.concatenate([p0, np.zeros(3), aw * sqd]))
        else:
            rots.append(R0)
            vec.append(np.concatenate([p0 + aw * sq, aw * sqd, np.zeros(3)]))
    return np.array(rots), np.array(vec)


def normalised(qs):
    """The library's fp32 normalisation: n = sqrt(((x x + y y) + z z) + w w), q / n, each step rounded to fp32."""
    q = np.asarray(qs, np.float32)
    x, y, z, w = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    n = np.sqrt(((x * x + y * y) + z * z) + w * w)
    return q / n[..., None]


def host_edit(m, st, w, jq, jqd, body, mask):
    """The host path: the selected words of the masked rows edited in numpy (quaternions normalised as the library does)."""
    nd, nf, ns = int(m['nd']), int(m['n_free']), int(m['n_slide'])
    so = 5 * nd + 13 * nf
    st = st.copy()
    for e in np.nonzero(mask)[0]:
        for j in range(nd + ns):
            iq = j if j < nd else so + 2 * (j - nd)
            iqd = nd + j if j < nd else iq + 1
            if (w.joint_positions >> j) & 1:
                st[e, iq] = jq[e, j]
            if (w.joint_velocities >> j) & 1:
                st[e, iqd] = jqd[e, j]
        for b in range(nf):
            o = 5 * nd + 13 * b
            if (w.free_poses >> b) & 1:
                st[e, o:o + 3] = body[e, nd + b, 0:3]
                st[e, o + 3:o + 7] = normalised(body[e, nd + b, 3:7])
            if (w.free_velocities >> b) & 1:
                st[e, o + 7:o + 13] = body[e, nd + b, 7:13]
    return st
