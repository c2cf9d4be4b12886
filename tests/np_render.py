"""Independent numpy fp64 ray caster of the box worlds, the reference prb_render is compared against.

Collider poses come from np_dynamics.fk (arm), the free-body quaternions and the slide coordinates of the state row.
A pixel's ray is the segment between the unprojections of its NDC point on the near and the far plane through
inverse(proj . view); the nearest slab entry on it wins (first collider on a tie), its eye depth is -z of the hit in
eye coordinates.  It shares no code with the kernel, which casts from the eye with a direction of unit eye depth.

A pixel is AMBIGUOUS when the collider it sees is decided by rounding: four sub-pixel jitters of +-0.01 px do not all
see the same collider as the centre, or the two nearest distinct colliders of the centre ray lie within 1e-5 relative
depth of each other."""
import numpy as np

from np_dynamics import _rot, fk

JITTER = 0.01
TIE_REL = 1e-5


def _quat_mat(q):
    x, y, z, w = np.asarray(q, np.float64) / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def poses(m, st):
    """World pose (R [n,3,3], p [n,3]) of every collider, site-0 pose (R, p) of the end effector."""
    st = np.asarray(st, np.float64)
    nd, nf, ns, n = m['nd'], m['n_free'], m['n_slide'], m['n_col']
    R, P, _, _ = fk(m, st[:nd])
    bodies = {}
    for b in range(nf):
        o = 5 * nd + 13 * b
        bodies[1 + b] = (_quat_mat(st[o + 3:o + 7]), st[o:o + 3])
    for s in range(ns):
        q = st[5 * nd + 13 * nf + 2 * s]
        R0 = m['slide_rot'].reshape(-1, 3, 3)[s]
        p0 = m['slide_pos'].reshape(-1, 3)[s]
        ax = m['slide_axis'].reshape(-1, 3)[s]
        bodies[1 + nf + s] = (R0 @ _rot(ax, q), p0) if m['slide_jtype'][s] == 0 else (R0, p0 + R0 @ ax * q)
    cR, cp = np.zeros((n, 3, 3)), np.zeros((n, 3))
    for c in range(n):
        b, l = m['col_body'][c], m['col_link'][c]
        if b < 0:
            Rb, pb = np.eye(3), np.zeros(3)
        elif b == 0:
            Rb, pb = (m['arm_base_rot'].reshape(3, 3), m['arm_base_pos']) if l < 0 else (R[l], P[l])
        else:
            Rb, pb = bodies[b]
        cR[c] = Rb @ m['col_rot'].reshape(-1, 3, 3)[c]
        cp[c] = pb + Rb @ m['col_pos'].reshape(-1, 3)[c]
    l0 = m['site_link'][0]
    sR = R[l0] @ m['site_rot'].reshape(-1, 3, 3)[0]
    sp = P[l0] + R[l0] @ m['site_pos'].reshape(-1, 3)[0]
    return cR, cp, sR, sp


def _mat(col_major):
    return np.asarray(col_major, np.float64).reshape(4, 4).T


def world_view(cam, sR, sp):
    V = _mat(cam.view)
    if cam.attach:                       # view is given in the site frame: world -> site -> eye
        T = np.eye(4)
        T[:3, :3], T[:3, 3] = sR.T, -sR.T @ sp
        V = V @ T
    return V


def _cast(m, cR, cp, Minv, V, xn, yn):
    """Nearest hit of the rays of NDC points (xn, yn) [k]: collider [k] (-1: none), depth [k], entry [k,n] (inf: miss),
    normal axis info for shading."""
    k = xn.shape[0]
    a = np.stack([xn, yn, -np.ones(k), np.ones(k)], 1) @ Minv.T
    b = np.stack([xn, yn, np.ones(k), np.ones(k)], 1) @ Minv.T
    a = a[:, :3] / a[:, 3:]
    b = b[:, :3] / b[:, 3:]
    d = b - a
    h = m['col_half'].reshape(-1, 3)
    # box coordinates: o [k,n,3], dl [k,n,3]
    o = np.einsum('nji,knj->kni', cR, a[:, None, :] - cp[None])
    dl = np.einsum('nji,kj->kni', cR, d)
    par = np.abs(dl) < 1e-12
    with np.errstate(divide='ignore', invalid='ignore'):
        ta = (-h[None] - o) / dl
        tb = (h[None] - o) / dl
    lo, hi = np.minimum(ta, tb), np.maximum(ta, tb)
    inside = (o >= -h[None]) & (o <= h[None])
    lo = np.where(par, np.where(inside, -np.inf, np.inf), lo)
    hi = np.where(par, np.where(inside, np.inf, -np.inf), hi)
    s0 = np.maximum(0.0, lo.max(2))
    s1 = np.minimum(1.0, hi.min(2))
    hit = (s0 <= s1) & (s0 < 1.0)
    s = np.where(hit, s0, np.inf)
    c = np.argmin(s, 1)
    sc = s[np.arange(k), c]
    c = np.where(np.isfinite(sc), c, -1)
    p = a + d * np.where(np.isfinite(sc), sc, 1.0)[:, None]
    depth = -(np.c_[p, np.ones(k)] @ V.T)[:, 2]
    return c, depth, s, lo, dl, d


def render(m, st, cam, palette):
    """rgb uint8 [H,W,3], depth float64 [H,W], seg int [H,W], ambiguous bool [H,W] of one env."""
    cR, cp, sR, sp = poses(m, st)
    V = world_view(cam, sR, sp)
    Pm = _mat(cam.proj)
    Minv = np.linalg.inv(Pm @ V)
    far = Pm[2, 3] / (Pm[2, 2] + 1.0)
    H, W = cam.height, cam.width
    ii, jj = np.meshgrid(np.arange(H), np.arange(W), indexing='ij')
    ii, jj = ii.ravel().astype(np.float64), jj.ravel().astype(np.float64)
    ndc = lambda j, i: (2 * (j + 0.5) / W - 1, 1 - 2 * (i + 0.5) / H)
    c, depth, s, lo, dl, d = _cast(m, cR, cp, Minv, V, *ndc(jj, ii))
    k = len(c)
    amb = np.zeros(k, bool)
    for dj, di in ((JITTER, JITTER), (JITTER, -JITTER), (-JITTER, JITTER), (-JITTER, -JITTER)):
        amb |= _cast(m, cR, cp, Minv, V, *ndc(jj + dj, ii + di))[0] != c
    # two nearest distinct colliders within TIE_REL relative eye depth (depth is affine in s: near at 0, far at 1)
    near = Pm[2, 3] / (Pm[2, 2] - 1.0)
    with np.errstate(invalid='ignore'):
        ds = near + np.sort(s, 1)[:, :2] * (far - near)
        amb |= np.isfinite(ds[:, 1]) & (ds[:, 1] - ds[:, 0] <= TIE_REL * ds[:, 0])
    # shading: face of the entry (the slab that set lo), or -ray direction where the near plane cuts the box
    light = np.asarray(cam.light_dir, np.float64)
    light = light / np.linalg.norm(light)
    rgb = np.tile(np.floor(255 * np.clip(np.asarray(cam.background, np.float64), 0, 1) + 0.5), (k, 1))
    h_ = c >= 0
    idx = np.nonzero(h_)[0]
    cc = c[idx]
    lo_c = lo[idx, cc]                     # [h,3]
    ax = np.argmax(lo_c, 1)
    sgn = -np.sign(dl[idx, cc, ax])
    n = cR[cc, :, ax] * sgn[:, None]       # world axis `ax` of the box
    clipped = lo_c.max(1) < 0.0
    dn = d[idx] / np.linalg.norm(d[idx], axis=1, keepdims=True)
    n = np.where(clipped[:, None], -dn, n)
    shade = cam.ambient + cam.diffuse * np.maximum(0.0, n @ light)
    col = np.asarray(palette, np.float64).reshape(-1, 3)[cc] * shade[:, None]
    rgb[idx] = np.floor(255 * np.clip(col, 0, 1) + 0.5)
    depth = np.where(h_, depth, far)
    return (rgb.reshape(H, W, 3).astype(np.uint8), depth.reshape(H, W), c.reshape(H, W), amb.reshape(H, W))


DEPTH_FLOOR = 1.0     # m


def compare(got, ref):
    """Acceptance rule of a rendered frame against render(): dict with the ambiguous fraction, the count of
    non-ambiguous pixels whose collider differs, and over pixels whose collider agrees the worst depth error relative
    to max(depth, DEPTH_FLOOR) and the worst RGB difference.  The floor (1e-5 m absolute below 1 m): the kernel's poses
    are fp32 (spacing 1.2e-7 m near 1 m from the origin) through up to 12 chained joint transforms, ~1e-6 m, and a
    face seen at grazing incidence amplifies that; a hit 1 cm from a gripper camera cannot be placed to 1e-7 m."""
    rgb, depth, seg = got
    rrgb, rdepth, rseg, amb = ref
    same = seg == rseg
    rel = np.abs(depth.astype(np.float64) - rdepth) / np.maximum(np.abs(rdepth), DEPTH_FLOOR)
    drgb = np.abs(rgb.astype(np.int32) - rrgb.astype(np.int32)).max(-1)
    return {'ambiguous': float(amb.mean()), 'seg_mismatch': int((~same & ~amb).sum()),
            'depth_rel': float(rel[same].max()) if same.any() else 0.0,
            'rgb': int(drgb[same].max()) if same.any() else 0}
