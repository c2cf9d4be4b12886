"""fp64 numpy reference of the arm queries (prb_arm_dynamics): forward kinematics, point Jacobians from their definition,
the mass matrix from a recursive Newton-Euler pass (column i = RNEA(q, 0, e_i) - RNEA(q, 0, 0) with gravity off) and
the bias h = RNEA(q, qd, 0).  Built from the compiled model alone; it shares no code with the kernel (which sums over
subtrees, composite-rigid-body style) nor with the oracle (articulated-body algorithm)."""
import numpy as np


def _axis_angle(a, q):
    K = np.array([[0.0, -a[2], a[1]], [a[2], 0.0, -a[0]], [-a[1], a[0], 0.0]])
    return np.eye(3) + np.sin(q) * K + (1.0 - np.cos(q)) * (K @ K)


def arm(m):
    """The arm's constants from the model, fp64."""
    nd = int(m['nd'])
    g = lambda k, *s: np.asarray(m[k], np.float64).reshape(*s)
    return {'nd': nd, 'parent': np.asarray(m['arm_parent'])[:nd], 'jtype': np.asarray(m['arm_jtype'])[:nd],
            'jpos': g('arm_jpos', -1, 3)[:nd], 'jrot': g('arm_jrot', -1, 3, 3)[:nd], 'axis': g('arm_axis', -1, 3)[:nd],
            'com': g('arm_com', -1, 3)[:nd], 'mass': g('arm_mass', -1)[:nd], 'inertia': g('arm_inertia', -1, 3, 3)[:nd],
            'base_pos': g('arm_base_pos', 3), 'base_rot': g('arm_base_rot', 3, 3), 'site_link': np.asarray(m['site_link'])[:4],
            'site_pos': g('site_pos', -1, 3)[:4], 'site_rot': g('site_rot', -1, 3, 3)[:4], 'jdamp': g('arm_jdamp', -1)[:nd],
            'gravity_z': m.param('gravity_z')}


def fk(A, q):
    """Link frames (R [nd,3,3], p [nd,3]), world joint axes a [nd,3] and COMs c [nd,3]."""
    nd = A['nd']
    R, p, a, c = np.zeros((nd, 3, 3)), np.zeros((nd, 3)), np.zeros((nd, 3)), np.zeros((nd, 3))
    for i in range(nd):
        par = A['parent'][i]
        pR, pp = (A['base_rot'], A['base_pos']) if par < 0 else (R[par], p[par])
        R0 = pR @ A['jrot'][i]
        ax = A['axis'][i]
        p[i] = pp + pR @ A['jpos'][i]
        if A['jtype'][i] == 0:
            R[i] = R0 @ _axis_angle(ax, q[i])
        else:
            R[i] = R0
            p[i] = p[i] + (R0 @ ax) * q[i]
        a[i] = R0 @ ax
        c[i] = p[i] + R[i] @ A['com'][i]
    return R, p, a, c


def ancestors(A, l):
    out = set()
    while l >= 0:
        out.add(int(l))
        l = A['parent'][l]
    return out


def point(A, q, link, site, local):
    """(model link, world position) of a point: local in the frame of `link` (site -1) or of site `site`."""
    R, p, _, _ = fk(A, q)
    local = np.asarray(local, np.float64)
    if site >= 0:
        link = int(A['site_link'][site])
        local = A['site_pos'][site] + A['site_rot'][site] @ local
    return link, p[link] + R[link] @ local


def jacobian(A, q, link, site, local):
    """J [6, nd] (linear rows, angular rows) of a point, from its definition, and the point's world position."""
    _, p, a, _ = fk(A, q)
    l, x = point(A, q, link, site, local)
    J = np.zeros((6, A['nd']))
    for j in ancestors(A, l):
        if A['jtype'][j] == 0:
            J[:3, j], J[3:, j] = np.cross(a[j], x - p[j]), a[j]
        else:
            J[:3, j] = a[j]
    return J, x


def rnea(A, q, qd, qdd, gravity=True):
    """Joint forces tau = M qdd + h(q, qd) (gravity off: no gravity term) by a recursive Newton-Euler pass in the world
    frame: link velocities and accelerations outwards, link wrenches inwards."""
    nd = A['nd']
    R, p, a, c = fk(A, q)
    w, al, acc = np.zeros((nd, 3)), np.zeros((nd, 3)), np.zeros((nd, 3))    # angular vel / acc, acceleration of p_i
    a0 = np.array([0.0, 0.0, -A['gravity_z'] if gravity else 0.0])          # gravity as an upward base acceleration
    f, n = np.zeros((nd, 3)), np.zeros((nd, 3))
    for i in range(nd):
        par = A['parent'][i]
        wp, alp, ap, pp = (np.zeros(3), np.zeros(3), a0, A['base_pos']) if par < 0 else (w[par], al[par], acc[par], p[par])
        r = p[i] - pp
        acc[i] = ap + np.cross(alp, r) + np.cross(wp, np.cross(wp, r))
        if A['jtype'][i] == 0:
            w[i] = wp + a[i] * qd[i]
            al[i] = alp + np.cross(wp, a[i] * qd[i]) + a[i] * qdd[i]
        else:
            w[i], al[i] = wp, alp
            acc[i] = acc[i] + 2.0 * np.cross(wp, a[i] * qd[i]) + a[i] * qdd[i]
        rc = c[i] - p[i]
        ac = acc[i] + np.cross(al[i], rc) + np.cross(w[i], np.cross(w[i], rc))
        Iw = R[i] @ A['inertia'][i] @ R[i].T
        f[i] = A['mass'][i] * ac
        n[i] = Iw @ al[i] + np.cross(w[i], Iw @ w[i]) + np.cross(rc, f[i])   # about p_i
    F, N = f.copy(), n.copy()
    tau = np.zeros(nd)
    for i in range(nd - 1, -1, -1):
        tau[i] = a[i] @ N[i] if A['jtype'][i] == 0 else a[i] @ F[i]
        par = A['parent'][i]
        if par >= 0:
            F[par] += F[i]
            N[par] += N[i] + np.cross(p[i] - p[par], F[i])
    return tau


def mass_matrix(A, q):
    nd = A['nd']
    z = np.zeros(nd)
    base = rnea(A, q, z, z, gravity=False)
    return np.stack([rnea(A, q, z, np.eye(nd)[i], gravity=False) - base for i in range(nd)], 1)


def bias(A, q, qd):
    return rnea(A, q, qd, np.zeros(A['nd']))


def kinetic_energy(A, q, qd):
    """sum over links of 1/2 m |v_c|^2 + 1/2 w^T I w, from the link twists of the forward pass."""
    nd = A['nd']
    R, p, a, c = fk(A, q)
    w, v = np.zeros((nd, 3)), np.zeros((nd, 3))
    T = 0.0
    for i in range(nd):
        par = A['parent'][i]
        wp, vp, pp = (np.zeros(3), np.zeros(3), A['base_pos']) if par < 0 else (w[par], v[par], p[par])
        v[i] = vp + np.cross(wp, p[i] - pp)
        if A['jtype'][i] == 0:
            w[i] = wp + a[i] * qd[i]
        else:
            w[i] = wp
            v[i] = v[i] + a[i] * qd[i]
        vc = v[i] + np.cross(w[i], c[i] - p[i])
        Iw = R[i] @ A['inertia'][i] @ R[i].T
        T += 0.5 * A['mass'][i] * vc @ vc + 0.5 * w[i] @ Iw @ w[i]
    return T


def all_outputs(A, q, qd, qdd, points):
    """Every output of one env: points [(link, site, local)] -> jacobian [P,6,nd], position [P,3], velocity [P,6],
    mass_matrix [nd,nd], tau [nd]."""
    q, qd, qdd = (np.asarray(x, np.float64) for x in (q, qd, qdd))
    Js, xs = zip(*[jacobian(A, q, l, s, o) for l, s, o in points]) if points else ((), ())
    J = np.array(Js).reshape(len(points), 6, A['nd'])
    M = mass_matrix(A, q)
    return {'jacobian': J, 'position': np.array(xs).reshape(len(points), 3), 'velocity': J @ qd,
            'mass_matrix': M, 'tau': M @ qdd + bias(A, q, qd)}
