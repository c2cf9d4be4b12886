"""Independent numpy fp64 reference of prb_ray_test: world endpoints from the fp64 site poses (collider poses from
np_render.poses), a segment caster with the slab rule of phase_observe, nearest hit, entry-face normal.

A ray is AMBIGUOUS when its collider is decided by rounding: shifting both endpoints by +-TOL along two directions
perpendicular to the ray, or moving either endpoint TOL outwards along the ray, changes the collider; or the two
nearest distinct colliders enter within TOL of each other; or a hit lies within TOL of the ray's start (a box entered
within TOL, or the start inside a box within TOL of its entry face) or of its end.  Its
NORMAL is ambiguous when the two largest slab entries of the hit box lie within TOL.  TOL is in metres along the ray."""
import numpy as np

from np_dynamics import fk
from np_render import poses

TOL = 1e-5


def cast_segments(m, cR, cp, a, b, mask=None):
    """Nearest box hit of the segments a -> b [k,3] (world): collider [k] (-1: none), fraction s [k,n] of every collider
    (inf: miss), unclipped slab entries lo [k,n,3] (-inf / inf on parallel axes inside / outside the slab), dl [k,n,3]
    (segment in box coordinates) and d [k,3].  The slab rule of phase_observe: t in [0, 1], |dl_k| < 1e-12 parallel, a
    hit when t0 <= t1 and t0 < 1, the nearest wins, the lower collider on a tie.  mask [n] bool: colliders that can be hit.
    (np_render._cast applies the same rule to camera rays given as NDC points.)"""
    k = a.shape[0]
    d = b - a
    h = m['col_half'].reshape(-1, 3)
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
    if mask is not None:
        hit &= np.asarray(mask, bool)[None]
    s = np.where(hit, s0, np.inf)
    c = np.argmin(s, 1)
    c = np.where(np.isfinite(s[np.arange(k), c]), c, -1)
    return c, s, lo, dl, d


def site_pose(m, st, s):
    """World pose (R [3,3], p [3]) of site s of the arm."""
    nd = m['nd']
    R, P, _, _ = fk(m, np.asarray(st, np.float64)[:nd])
    l = m['site_link'][s]
    return R[l] @ m['site_rot'].reshape(-1, 3, 3)[s], P[l] + R[l] @ m['site_pos'].reshape(-1, 3)[s]


def world_endpoints(m, st, frm, to, site=None):
    frm, to = np.asarray(frm, np.float64).reshape(-1, 3), np.asarray(to, np.float64).reshape(-1, 3)
    if site is None:
        return frm, to
    R, p = site_pose(m, st, site)
    return p + frm @ R.T, p + to @ R.T


def _perp(d):
    """Two unit directions perpendicular to each row of d (zero rows: the x and y axes)."""
    n = np.linalg.norm(d, axis=1, keepdims=True)
    u = np.where(n > 0, d / np.where(n > 0, n, 1.0), [[0.0, 0.0, 1.0]])
    ref = np.where(np.abs(u[:, :1]) < 0.9, [[1.0, 0.0, 0.0]], [[0.0, 1.0, 0.0]])
    e1 = np.cross(u, ref)
    e1 /= np.linalg.norm(e1, axis=1, keepdims=True)
    return e1, np.cross(u, e1)


def ray_test(m, st, frm, to, site=None, mask=None):
    """One env: rays frm -> to [R,3] in the world (site None) or site `site`.  mask: bool [n_col] (None: all).
    Returns dict collider [R], fraction [R], position [R,3], normal [R,3] (the kernel's miss values), ambiguous [R],
    normal_ambiguous [R]."""
    cR, cp, _, _ = poses(m, st)
    a, b = world_endpoints(m, st, frm, to, site)
    k = a.shape[0]
    fin = np.isfinite(a).all(1) & np.isfinite(b).all(1)
    a0, b0 = np.where(fin[:, None], a, 0.0), np.where(fin[:, None], b, 0.0)
    c, s, lo, dl, d = cast_segments(m, cR, cp, a0, b0, mask)
    c = np.where(fin, c, -1)
    hit = c >= 0
    ci = np.maximum(c, 0)
    sc = np.where(hit, s[np.arange(k), ci], 1.0)
    pos = np.where(hit[:, None], a0 + d * sc[:, None], 0.0)
    # normal: the slab whose entry set t0 (> 0), against the ray; -dir when the ray starts inside; 0 for zero length
    lo_c = lo[np.arange(k), ci]                                   # [k,3]
    ax = np.argmax(lo_c, 1)
    entered = lo_c.max(1) > 0.0
    sgn = -np.sign(dl[np.arange(k), ci, ax])
    n_face = cR[ci, :, ax] * sgn[:, None]
    L = np.linalg.norm(d, axis=1)
    n_in = np.where(L[:, None] > 0, -d / np.where(L > 0, L, 1.0)[:, None], 0.0)
    nrm = np.where(hit[:, None], np.where(entered[:, None], n_face, n_in), 0.0)
    # ambiguity
    amb = np.zeros(k, bool)
    u = d / np.where(L > 0, L, 1.0)[:, None]
    e1, e2 = _perp(d)
    for da, db in ((TOL * e1, TOL * e1), (-TOL * e1, -TOL * e1), (TOL * e2, TOL * e2), (-TOL * e2, -TOL * e2),
                   (0.0 * u, TOL * u), (-TOL * u, 0.0 * u)):
        amb |= cast_segments(m, cR, cp, a0 + da, b0 + db, mask)[0] != c
    with np.errstate(invalid='ignore'):
        ss = np.sort(s, 1)[:, :2] * L[:, None]
        # two boxes entered within TOL (two boxes that both contain the start tie at 0 by index in both casters)
        amb |= np.isfinite(ss[:, 1]) & (ss[:, 1] - ss[:, 0] <= TOL) & (ss[:, 1] > 0)
        # a box entered within TOL after the start, or containing the start within TOL of its entry face
        lmax = lo.max(2) * L[:, None]
        amb |= (np.isfinite(s) & (((s > 0) & (s * L[:, None] <= TOL)) | ((s == 0) & (lmax >= -TOL)))).any(1)
    amb |= hit & ((1.0 - sc) * L <= TOL)
    amb &= fin
    top = np.sort(np.where(np.isfinite(lo_c), lo_c, -1e300), 1)
    namb = hit & entered & ((top[:, 2] - top[:, 1]) * L <= TOL)
    return {'collider': c, 'fraction': sc, 'position': pos, 'normal': nrm, 'ambiguous': amb, 'normal_ambiguous': namb,
            'length': L}


def compare(got, ref):
    """Acceptance rule of one env's kernel results against ray_test(): dict with the ambiguous fraction, the count of
    unambiguous rays whose collider differs, and over rays whose collider agrees the worst |d(fraction L)| relative to
    max(fraction L, 1 m), the worst position error beyond that bound (m) and the worst normal error (unambiguous normals)."""
    col, frac, pos, nrm = got
    amb = ref['ambiguous']
    same = col == ref['collider']
    L = ref['length']
    dist = ref['fraction'] * L
    bound = 1e-5 * np.maximum(dist, 1.0)
    dfrac = np.abs(frac.astype(np.float64) * L - dist) / np.maximum(dist, 1.0)
    dpos = np.abs(pos.astype(np.float64) - ref['position']).max(1) - bound
    nok = same & ~amb & ~ref['normal_ambiguous']
    dn = np.abs(nrm.astype(np.float64) - ref['normal']).max(1)
    return {'ambiguous': float(amb.mean()), 'mismatch': int((~same & ~amb).sum()),
            'frac_rel': float(dfrac[same].max()) if same.any() else 0.0,
            'pos_excess': float(dpos[same].max()) if same.any() else -1.0,
            'normal': float(dn[nok].max()) if nok.any() else 0.0}


def assert_agrees(got, ref, max_amb=0.02):
    """compare() within the bounds; max_amb None leaves the ambiguous share to the caller (a cap over a whole ray set)."""
    r = compare(got, ref)
    assert r['mismatch'] == 0 and (max_amb is None or r['ambiguous'] <= max_amb) and r['frac_rel'] <= 1e-5 \
        and r['pos_excess'] <= 1e-6 and r['normal'] <= 1e-5, r
    return r


# ------------------------------------------------------------------ the three ray sets of the tests and tools/bench_rays.py
def random_segments(m, st, n, rng):
    """n random world segments with both endpoints in the colliders' world AABB grown by 0.1 m."""
    cR, cp, _, _ = poses(m, st)
    h = m['col_half'].reshape(-1, 3)
    ext = np.abs(cR) @ h[:, :, None]
    lo, hi = (cp - ext[..., 0]).min(0) - 0.1, (cp + ext[..., 0]).max(0) + 0.1
    return rng.uniform(lo, hi, (n, 3)), rng.uniform(lo, hi, (n, 3))


def site_fan(n=8, length=1.0):
    """n x n rays in the end-effector site frame from beside the fingers (the gripper camera's eye) down the approach
    axis -z, spread +-40 degrees."""
    ang = np.radians(np.linspace(-40.0, 40.0, n))
    ax, ay = np.meshgrid(ang, ang, indexing='ij')
    d = np.stack([np.tan(ax.ravel()), np.tan(ay.ravel()), -np.ones(n * n)], 1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    frm = np.tile([0.0, 0.06, 0.08], (n * n, 1))
    return frm, frm + length * d


def height_scan(m, n=32):
    """n x n vertical world rays from 1.5 m above the top of the largest static thin box (the table or the ground) down to
    0.3 m below it, over the cells of an n x n grid on that box."""
    nc = int(m['n_col'])
    body, half, pos = np.asarray(m['col_body'])[:nc], m['col_half'].reshape(-1, 3)[:nc], m['col_pos'].reshape(-1, 3)[:nc]
    static = [c for c in range(nc) if body[c] < 0]
    top = max(static, key=lambda c: half[c][0] * half[c][1] if half[c][2] < 0.05 and half[c].max() < 2.0 else 0)
    cx, cy, cz = pos[top]
    hx, hy, hz = min(half[top][0], 1.0), min(half[top][1], 1.0), half[top][2]
    g = (np.arange(n) + 0.5) / n * 2 - 1                  # cell centres: no ray grazes the box's edges
    x, y = np.meshgrid(cx + hx * g, cy + hy * g, indexing='ij')
    xy = np.stack([x.ravel(), y.ravel()], 1)
    z = cz + hz
    return np.c_[xy, np.full(n * n, z + 1.5)], np.c_[xy, np.full(n * n, z - 0.3)]


def proprio_ray(m, st):
    """gripper_proprioception's ray (phase_observe) in fp64 from sites 0..3: (from, to) in the world."""
    R0, ep = site_pose(m, st, 0)
    _, wr = site_pose(m, st, 1)
    _, g1 = site_pose(m, st, 2)
    _, g2 = site_pose(m, st, 3)
    ew = ep - wr
    return ep - ew * 0.5, (g1 + g2) * 0.5 + ew * 0.2


def proprio_flag(m, col, frac):
    """phase_observe's flag from a ray result: a hit at fraction < 1 on a link other than 18 and 20."""
    if col < 0 or not frac < 1.0:
        return 0.0
    li = int(np.asarray(m['col_urdf_link'])[col])
    return 0.0 if li in (18, 20) else 1.0
