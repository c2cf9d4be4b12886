"""Independent numpy fp64 reference of prb_closest_points: collider poses from np_render.poses, the signed distance of
every ordered collider pair of an env (its own separating-axis test and feature enumeration), the nearest pair per query.

Box pair (A, B), computed in A's frame:
  * overlap along a unit axis n: hA.|RA^T n| + hB.|RB^T n| - |n.(pB - pA)|, over A's 3 face axes, B's 3, the 9 edge
    crosses a_i x b_j (skipped when |a_i x b_j|^2 < 1e-10); no negative overlap: d = -min overlap, the normal that axis
    turned towards A (the axis as it is when n.(pA - pB) = 0), the lowest axis on a tie;
  * separated: d = min over A's vertices against box B, B's vertices against box A, and the 12 x 12 edge-edge segment
    distances.

A query is AMBIGUOUS when rounding can decide its pair: the best and second-best pair lie within TOL of each other, or
the best within TOL of max_distance.  It is a TIE when they lie within TIE (coplanar faces of several colliders): then any
of the tied pairs is the right answer.  A penetration NORMAL is ambiguous when the two smallest overlaps lie within TOL or
|n.(pA - pB)| <= TOL (its orientation)."""
import numpy as np

from np_render import poses

TOL = 2e-5
TIE = 1e-9
EDGE_EPS2 = 1e-10


def _seg_closest(p, u, hp, q, v, hq):
    """Closest points of segments p + s u (|s| <= hp) and q + t v (|t| <= hq), u, v unit; broadcast over leading axes."""
    r = p - q
    b = (u * v).sum(-1)
    c = (u * r).sum(-1)
    f = (v * r).sum(-1)
    den = 1.0 - b * b
    with np.errstate(divide='ignore', invalid='ignore'):
        s = np.where(den > 1e-15, np.clip((b * f - c) / np.where(den > 1e-15, den, 1.0), -hp, hp), 0.0)
    t = b * s + f
    tc = np.clip(t, -hq, hq)
    s = np.where(t != tc, np.clip(b * tc - c, -hp, hp), s)
    return p + u * s[..., None], q + v * tc[..., None]


def _edges(h):
    """12 edges of the box |x_k| <= h_k [..., 3]: centres [..., 12, 3], axis index [12], half lengths [..., 12]."""
    cs, ax = [], []
    for i in range(3):
        o = [k for k in range(3) if k != i]
        for s1 in (1.0, -1.0):
            for s2 in (1.0, -1.0):
                sg = np.zeros(3)
                sg[o[0]], sg[o[1]] = s1, s2
                cs.append(sg)
                ax.append(i)
    cs, ax = np.array(cs), np.array(ax)
    return cs * h[..., None, :], ax, h[..., ax]


def box_pairs(RA, pA, hA, RB, pB, hB):
    """Signed distance of K box pairs (R [K,3,3], p [K,3], h [K,3]).  Returns dict d [K], normal [K,3] (B -> A, world),
    pa, pb [K,3] (world witness: for separated pairs the closest points; for overlapping ones the deepest vertex of A
    along -normal and pb = pa - d normal, not the kernel's choice: the kernel's witness is checked by its invariants), axis [K] (0..14, -1 separated), ov_gap [K] (second-smallest minus smallest
    overlap), axis_dot [K] (|n.(pA - pB)|)."""
    K = len(pA)
    B = np.einsum('kji,kjl->kil', RA, RB)                       # RA^T RB: column j is b_j in A's frame
    t = np.einsum('kji,kj->ki', RA, pB - pA)
    E = np.broadcast_to(np.eye(3), (K, 3, 3))
    axes = [E[:, k] for k in range(3)] + [B[:, :, j] for j in range(3)]
    valid = [np.ones(K, bool)] * 6
    for i in range(3):
        for j in range(3):
            c = np.cross(E[:, i], B[:, :, j])
            l2 = (c * c).sum(1)
            valid.append(l2 >= EDGE_EPS2)
            axes.append(c / np.sqrt(np.where(l2 > 0, l2, 1.0))[:, None])
    N = np.stack(axes, 1)                                        # [K,15,3]
    ok = np.stack(valid, 1)
    ov = (np.abs(N) * hA[:, None]).sum(2) + (np.abs(np.einsum('kji,kaj->kai', B, N)) * hB[:, None]).sum(2) \
        - np.abs((N * t[:, None]).sum(2))
    ov = np.where(ok, ov, np.inf)
    k = np.argmin(ov, 1)
    srt = np.sort(ov, 1)
    n = N[np.arange(K), k]
    nt = (n * t).sum(1)
    n = np.where((nt > 0)[:, None], -n, n)
    sep = srt[:, 0] < 0
    # overlapping: A's support along -n (sign(0) = +)
    pa_o = np.where(n <= 0, hA, -hA)
    d_o = -srt[:, 0]
    pb_o = pa_o - d_o[:, None] * n
    # separated: vertices against boxes, edges against edges
    sg = np.array([[sx, sy, sz] for sz in (1, -1) for sy in (1, -1) for sx in (1, -1)], float)
    va = sg[None] * hA[:, None]                                  # [K,8,3] A's vertices
    qa = np.einsum('kji,kvj->kvi', B, va - t[:, None])           # in B's frame
    qc = np.clip(qa, -hB[:, None], hB[:, None])
    da = ((qa - qc) ** 2).sum(2)
    pb_va = t[:, None] + np.einsum('kij,kvj->kvi', B, qc)
    vb = t[:, None] + np.einsum('kij,kvj->kvi', B, sg[None] * hB[:, None])
    vbc = np.clip(vb, -hA[:, None], hA[:, None])
    db = ((vb - vbc) ** 2).sum(2)
    ca, axa, la = _edges(hA)                                     # [K,12,3], [12], [K,12]
    cb_l, axb, lb = _edges(hB)
    cb = t[:, None] + np.einsum('kij,kej->kei', B, cb_l)
    ua = np.eye(3)[axa][None].repeat(K, 0)                       # [K,12,3]
    ub = np.transpose(B, (0, 2, 1))[:, axb]                      # [K,12,3]: b_j rows
    xa, xb = _seg_closest(ca[:, :, None], ua[:, :, None], la[:, :, None], cb[:, None], ub[:, None], lb[:, None])
    de = ((xa - xb) ** 2).sum(3).reshape(K, 144)
    cand = np.concatenate([da, db, de], 1)
    j = np.argmin(cand, 1)
    d_s = np.sqrt(cand[np.arange(K), j])
    pa_all = np.concatenate([va, vbc, xa.reshape(K, 144, 3)], 1)
    pb_all = np.concatenate([pb_va, vb, xb.reshape(K, 144, 3)], 1)
    pa_s, pb_s = pa_all[np.arange(K), j], pb_all[np.arange(K), j]
    with np.errstate(divide='ignore', invalid='ignore'):
        n_s = np.where((d_s > 0)[:, None], (pa_s - pb_s) / d_s[:, None], n)
    d = np.where(sep, d_s, d_o)
    pa = np.where(sep[:, None], pa_s, pa_o)
    pb = np.where(sep[:, None], pb_s, pb_o)
    nn = np.where(sep[:, None], n_s, n)
    w = lambda x: np.einsum('kij,kj->ki', RA, x)
    return {'d': d, 'normal': w(nn), 'pa': pA + w(pa), 'pb': pA + w(pb), 'axis': np.where(sep, -1, k),
            'ov_gap': srt[:, 1] - srt[:, 0], 'axis_dot': np.abs(nt)}


def pair_table(m, st):
    """box_pairs of every ordered collider pair (a, b) of one env: dict of [n, n] / [n, n, 3] arrays."""
    cR, cp, _, _ = poses(m, st)
    n = int(m['n_col'])
    h = m['col_half'].reshape(-1, 3)[:n].astype(np.float64)
    a, b = np.meshgrid(np.arange(n), np.arange(n), indexing='ij')
    a, b = a.ravel(), b.ravel()
    r = box_pairs(cR[a], cp[a], h[a], cR[b], cp[b], h[b])
    return {k: v.reshape((n, n) + v.shape[1:]) for k, v in r.items()}, (cR, cp, h)


def closest(table, mask_a, mask_b, max_distance):
    """One query of one env: (a, b, d, ambiguous, tie); a = b = -1, d = inf when no pair lies within max_distance."""
    D = table['d']
    n = D.shape[0]
    sel = np.zeros((n, n), bool)
    ia = [c for c in range(n) if (mask_a >> c) & 1]
    ib = [c for c in range(n) if (mask_b >> c) & 1]
    sel[np.ix_(ia, ib)] = True
    np.fill_diagonal(sel, False)
    v = np.where(sel, D, np.inf).ravel()
    o = np.argsort(v, kind='stable')
    best, second = v[o[0]], v[o[1]] if len(o) > 1 else np.inf
    amb = bool(abs(best - max_distance) <= TOL or (np.isfinite(second) and second - best <= TOL and second <= max_distance + TOL))
    tie = bool(np.isfinite(second) and second - best <= TIE)
    if not best <= max_distance:
        return -1, -1, np.inf, amb, tie
    return int(o[0] // n), int(o[0] % n), float(best), amb, tie


def witness_errors(geom, a, b, d, pa, pb, nrm):
    """The invariants of a reported result (world, m): | |pa - pb| - |d| |, pa's distance outside A, pb's outside B, and
    for d <= 0 |n.pa - min_A n.x| and |n.pb - max_B n.x| (0 otherwise).  geom: (cR, cp, h) of pair_table."""
    cR, cp, h = geom
    pa, pb, nrm = (np.asarray(x, np.float64) for x in (pa, pb, nrm))

    def outside(c, x):
        q = np.abs(cR[c].T @ (x - cp[c])) - h[c]
        return max(np.linalg.norm(np.maximum(q, 0.0)), 0.0)

    e = [abs(np.linalg.norm(pa - pb) - abs(d)), outside(a, pa), outside(b, pb), 0.0, 0.0]
    if d <= 0:
        sup = lambda c: float(np.abs(cR[c].T @ nrm) @ h[c])
        e[3] = abs(nrm @ pa - (nrm @ cp[a] - sup(a)))
        e[4] = abs(nrm @ pb - (nrm @ cp[b] + sup(b)))
    return e


def check_env(m, st, queries, got, max_distance, table=None):
    """Acceptance rule for one env's kernel results (got: dict of [Q] / [Q,3] arrays) against the reference: returns
    (number of ambiguous queries whose pair differs from the reference's, ties aside, list of failures).  Unambiguous
    queries: the same pair and |dd| <= 1e-5 max(1, |d|); a differing pair of an ambiguous query: its reference distance
    within TOL of the best; any reported pair: its reference distance within 1e-5 max(1, |d|), the witness invariants within TOL, and for a penetration
    whose normal is unambiguous the reference's normal within 1e-5."""
    if table is None:
        table = pair_table(m, st)
    tab, geom = table
    namb, bad = 0, []
    for k, (ma, mb) in enumerate(queries):
        a, b, d, amb, tie = closest(tab, ma, mb, max_distance)
        ga, gb, gd = int(got['collider_a'][k]), int(got['collider_b'][k]), float(got['distance'][k])
        if (ga, gb) != (a, b):
            if not amb or (ga >= 0 and a >= 0 and tab['d'][ga, gb] - d > TOL):
                bad.append((k, 'pair', (ga, gb), (a, b), gd, d))
                continue
            namb += not tie
        if ga < 0:
            if not (gb == -1 and gd == np.inf and not np.any(got['position_on_a'][k]) and not np.any(got['normal_on_b'][k])):
                bad.append((k, 'miss values'))
            continue
        rd = tab['d'][ga, gb]
        if abs(gd - rd) > 1e-5 * max(1.0, abs(rd)) or not gd <= max_distance:
            bad.append((k, 'distance', gd, rd))
        e = witness_errors(geom, ga, gb, gd, got['position_on_a'][k], got['position_on_b'][k], got['normal_on_b'][k])
        if max(e) > TOL:
            bad.append((k, 'witness', e))
        if rd <= -TOL and tab['ov_gap'][ga, gb] > TOL and tab['axis_dot'][ga, gb] > TOL:
            if np.abs(np.asarray(got['normal_on_b'][k], np.float64) - tab['normal'][ga, gb]).max() > 1e-5:
                bad.append((k, 'normal', got['normal_on_b'][k], tab['normal'][ga, gb]))
    return namb, bad


# ------------------------------------------------------------------ the query sets of the tests and tools/bench_closest.py
def body_mask(m, body, link=None):
    nc = int(m['n_col'])
    cb = np.asarray(m['col_body'])[:nc]
    sel = cb == body
    if link is not None:
        sel &= np.asarray(m['col_urdf_link'])[:nc] == link
    return sum(1 << int(c) for c in np.nonzero(sel)[0])


def bodies(m):
    nc = int(m['n_col'])
    return sorted(set(int(b) for b in np.asarray(m['col_body'])[:nc]))


def pad_links(m):
    """PyBullet link indices of the arm's finger pads (the links of sites 2 and 3)."""
    nc = int(m['n_col'])
    cl, cu, cb = (np.asarray(m[k])[:nc] for k in ('col_link', 'col_urdf_link', 'col_body'))
    out = []
    for s in (2, 3):
        li = int(m['site_link'][s])
        c = np.nonzero((cb == 0) & (cl == li))[0]
        if len(c):
            out.append(int(cu[c[0]]))
    return sorted(set(out))


def query_sets(m):
    """name -> list of (side_a, side_b) in closest_points form: every ordered pair of distinct bodies, each finger-pad
    link against the block (body 1), the arm against the static scene."""
    bs = bodies(m)
    sets = {'bodies': [(a, b) for a in bs for b in bs if a != b],
            'arm_static': [(0, -1)]}
    if 1 in bs:
        sets['pads_block'] = [((0, l), 1) for l in pad_links(m)]
    return sets


def masks(m, queries):
    def side(s):
        return body_mask(m, *s) if isinstance(s, tuple) else body_mask(m, s)
    return [(side(a), side(b)) for a, b in queries]
