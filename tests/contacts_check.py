"""Checks of the contact report (include/prb.h prb_contacts) shared by the CPU and GPU tests: the oracle's contacts and
impulses of its last substep, the comparison rule (same contacts in the same order, geometry, per-object-pair force
totals, conditioning), and the invariants that need no oracle."""
import ctypes

import numpy as np

from helpers import COND_K

PAIR_REL, PAIR_ABS = 0.01, 1e-3       # per-object-pair force totals: 1 % or 1e-3 N, whichever is larger
COND_SHARE = 0.02                     # at most 2 % of the envs may need the conditioning rule


def plane_space(n):
    """Bullet's btPlaneSpace1 in fp64 (the oracle's friction directions)."""
    if abs(n[2]) > 0.7071067811865476:
        a = n[1] ** 2 + n[2] ** 2
        k = 1.0 / np.sqrt(a)
        p = np.array([0.0, -n[2] * k, n[1] * k])
        return p, np.array([a * k, -n[0] * p[2], n[0] * p[1]])
    a = n[0] ** 2 + n[1] ** 2
    k = 1.0 / np.sqrt(a)
    p = np.array([-n[1] * k, n[0] * k, 0.0])
    return p, np.array([-n[2] * p[1], n[2] * p[0], a * k])


def oracle_report(o):
    """Contacts of the oracle's most recent substep with their forces: dict like one env of VecPlayEnv.contacts()."""
    L = o.L
    nc = L.orc_last_contacts()
    pairs = np.zeros(2 * max(nc, 1), np.int32)
    data = np.zeros(10 * max(nc, 1), o.dtype)
    L.orc_last_contact_pairs(pairs.ctypes.data_as(ctypes.c_void_p))
    L.orc_last_contact_data(data.ctypes.data_as(ctypes.c_void_p))
    data = data[:10 * nc].reshape(nc, 10)
    _, _, sc, _ = o.last_rows()
    dt = o.model.param('dt')
    fric = sc[len(sc) - 2 * nc:]                        # the friction rows come last, two per contact in contact order
    normal_of = fric[0::2, 7].astype(int) if nc else np.zeros(0, int)
    r = {'count': nc, 'collider_a': pairs[0:2 * nc:2].copy(), 'collider_b': pairs[1:2 * nc:2].copy(),
         'position_on_a': data[:, 0:3], 'position_on_b': data[:, 3:6], 'normal_on_b': data[:, 6:9], 'distance': data[:, 9],
         'normal_force': sc[normal_of, 5] / dt if nc else np.zeros(0),
         'lateral_friction_1': fric[0::2, 5] / dt, 'lateral_friction_2': fric[1::2, 5] / dt}
    tt = [plane_space(n) for n in data[:, 6:9]]
    r['lateral_friction_dir_1'] = np.array([t[0] for t in tt]).reshape(nc, 3)
    r['lateral_friction_dir_2'] = np.array([t[1] for t in tt]).reshape(nc, 3)
    return r


def env_report(rep, i):
    """Env i of a batched report, cut to its count."""
    n = int(rep['count'][i])
    return {k: (n if k == 'count' else np.asarray(v[i][:n], np.float64 if v.dtype.kind == 'f' else v.dtype)) for k, v in rep.items()}


def pair_totals(model, r):
    """{(col_obj of A, col_obj of B): [sum normal_force, sum friction force vector on A (3)]}."""
    obj = np.asarray(model['col_obj'])
    out = {}
    for k in range(int(r['count'])):
        key = (int(obj[r['collider_a'][k]]), int(obj[r['collider_b'][k]]))
        f = np.concatenate([[r['normal_force'][k]], r['lateral_friction_1'][k] * r['lateral_friction_dir_1'][k] +
                            r['lateral_friction_2'][k] * r['lateral_friction_dir_2'][k]])
        out[key] = out.get(key, 0.0) + f
    return out


def totals_error(a, b):
    """Worst excess of per-pair total differences over the tolerance (<= 1 passes) and the worst absolute difference."""
    worst, diff = 0.0, 0.0
    for key in set(a) | set(b):
        x, y = a.get(key, np.zeros(4)), b.get(key, np.zeros(4))
        for d, ref in ((abs(x[0] - y[0]), abs(y[0])), (np.linalg.norm(x[1:] - y[1:]), np.linalg.norm(y[1:]))):
            worst = max(worst, d / max(PAIR_REL * ref, PAIR_ABS))
            diff = max(diff, d)
    return worst, diff


def same_contacts(got, ref):
    return got['count'] == ref['count'] and np.array_equal(got['collider_a'], ref['collider_a']) and \
        np.array_equal(got['collider_b'], ref['collider_b'])


def geometry_error(got, ref):
    if got['count'] == 0:
        return 0.0
    return max(float(np.abs(got[k] - ref[k]).max()) for k in ('position_on_a', 'position_on_b', 'normal_on_b', 'distance'))


def perturbed(state_row, model, rng):
    """The state with every non-zero entry moved by one fp32 ulp in a random direction (goal / bookkeeping untouched), as
    helpers.ulp_spread does."""
    x = np.asarray(state_row, np.float32)
    tail = int(model['goal_dim']) + 10
    sgn = np.sign(rng.standard_normal(len(x))).astype(np.float32)
    y = np.nextafter(x, x + sgn * np.float32(1e9)).astype(np.float32)
    y[x == 0] = 0
    y[-tail:] = x[-tail:]
    return y


def _as64(r):
    return {k: (v if k in ('count', 'collider_a', 'collider_b') else np.asarray(v, np.float64)) for k, v in r.items()}


def compare(model, Oracle, rep, states, geom_tol, rng=None, n_pert=8, f32_probe=False):
    """Compares envs of a batched report with the oracle run from the same states.  states: (env, state row, advance)
    with advance(o) moving the oracle like the batch was moved (o.substeps(1) or o.step(action)).  An env beyond a criterion is accepted only when the oracle itself
    moves by a comparable amount (1 / COND_K of it) when its input state is perturbed by one fp32 ulp.  With f32_probe,
    also when the oracle's fp32 restatement (Oracle(f32=True)) deviates from the fp64 oracle by 1 / COND_K of it: over
    the 12 substeps of a full step the rounding of the whole computation, not only of the input, sets the spread.  Returns
    {n, cond (envs accepted by these rules), cond_envs (which), bad (list of (env, reason)), worst_geom, worst_force}."""
    rng = rng if rng is not None else np.random.default_rng(0)
    res = {'n': len(states), 'cond': 0, 'cond_envs': [], 'bad': [], 'worst_geom': 0.0, 'worst_force': 0.0}
    for j, (i, row, adv) in enumerate(states):
        o = Oracle(model)
        o.state[:] = np.asarray(row, np.float64)
        adv(o)
        ref = oracle_report(o)
        got = env_report(rep, i)
        reason, err_geom, err_force = None, 0.0, 0.0
        if not same_contacts(got, ref):
            reason = 'contacts %d vs %d' % (got['count'], ref['count'])
        else:
            err_geom = geometry_error(got, ref)
            err_force, diff = totals_error(pair_totals(model, got), pair_totals(model, ref))
            res['worst_geom'] = max(res['worst_geom'], err_geom)
            res['worst_force'] = max(res['worst_force'], diff)
            if err_geom > geom_tol:
                reason = 'geometry %.2e' % err_geom
            elif err_force > 1.0:
                reason = 'forces %.2f x tolerance' % err_force
        if reason is None:
            continue
        # conditioning: the oracle's own spread under 1-ulp input perturbations
        tot_ref = pair_totals(model, ref)
        spread_geom, spread_force, set_changes = 0.0, 0.0, False
        for _ in range(n_pert):
            p = Oracle(model)
            p.state[:] = perturbed(row, model, rng).astype(np.float64)
            adv(p)
            rp = oracle_report(p)
            if not same_contacts(rp, ref):
                set_changes = True
                continue
            spread_geom = max(spread_geom, geometry_error(rp, ref))
            spread_force = max(spread_force, totals_error(pair_totals(model, rp), tot_ref)[1])
        if f32_probe:
            p = Oracle(model, f32=True)
            p.state[:] = np.asarray(row, np.float32)
            adv(p)
            rp = _as64(oracle_report(p))
            if not same_contacts(rp, ref):
                set_changes = True
            else:
                spread_geom = max(spread_geom, geometry_error(rp, ref))
                spread_force = max(spread_force, totals_error(pair_totals(model, rp), tot_ref)[1])
        if reason.startswith('contacts'):
            ok = set_changes
        elif reason.startswith('geometry'):
            ok = set_changes or (err_geom <= COND_K * spread_geom and spread_geom > geom_tol / COND_K)
        else:
            diff = totals_error(pair_totals(model, got), tot_ref)[1]
            ok = set_changes or diff <= COND_K * spread_force
        if ok:
            res['cond'] += 1
            res['cond_envs'].append(i)
        else:
            res['bad'].append((i, reason))
    return res


def check_invariants(model, rep, envs=None):
    """Physics every report must satisfy, for every contact of the given envs (all when None): normal_force >= 0, unit and
    mutually orthogonal normal and friction directions, position_on_a = position_on_b + distance * normal_on_b,
    |lateral_friction_k| <= mu normal_force with mu = clamp(friction_a friction_b, +-10) (the per-direction bound of the
    cone solver; 1e-6 N plus fp32 rounding of the clamp), collider pairs from the model's pair list, and the padding.
    Returns a list of violations (empty: all hold)."""
    cnt = np.asarray(rep['count'])
    N, K = rep['collider_a'].shape
    envs = np.arange(N) if envs is None else np.asarray(envs)
    bad = []
    if cnt.min() < 0 or cnt.max() > K:
        bad.append('count out of range')
    valid = np.arange(K)[None, :] < cnt[envs][:, None]
    ca, cb = rep['collider_a'][envs], rep['collider_b'][envs]
    pad = ~valid
    if (ca[pad] != -1).any() or (cb[pad] != -1).any():
        bad.append('padding of the collider ids')
    for k in ('position_on_a', 'position_on_b', 'normal_on_b', 'distance', 'normal_force', 'lateral_friction_1',
              'lateral_friction_2', 'lateral_friction_dir_1', 'lateral_friction_dir_2'):
        if np.any(rep[k][envs][pad] != 0):
            bad.append('padding of ' + k)
    if 'body_a' in rep and ((rep['body_a'][envs][pad] != -1).any() or (rep['link_b'][envs][pad] != -1).any()):
        bad.append('padding of the looked-up ids')
    g = lambda k: np.asarray(rep[k][envs][valid], np.float64)
    n, t1, t2 = g('normal_on_b'), g('lateral_friction_dir_1'), g('lateral_friction_dir_2')
    fn, f1, f2 = g('normal_force'), g('lateral_friction_1'), g('lateral_friction_2')
    a, b = ca[valid], cb[valid]
    if len(a) == 0:
        return bad
    if fn.min() < 0:
        bad.append('negative normal force %g' % fn.min())
    for name, v in (('normal', n), ('dir 1', t1), ('dir 2', t2)):
        e = np.abs(np.linalg.norm(v, axis=1) - 1).max()
        if e > 1e-5:
            bad.append('%s not unit (%.2e)' % (name, e))
    o = max(np.abs((n * t1).sum(1)).max(), np.abs((n * t2).sum(1)).max(), np.abs((t1 * t2).sum(1)).max())
    if o > 1e-5:
        bad.append('directions not orthogonal (%.2e)' % o)
    rel = np.abs(g('position_on_a') - (g('position_on_b') + g('distance')[:, None] * n)).max()
    if rel > 1e-6:
        bad.append('position relation (%.2e)' % rel)
    fr = np.asarray(model['col_friction'], np.float64)
    mu = np.clip(fr[a] * fr[b], -10, 10)
    lim = mu * fn * (1 + 1e-6) + 1e-6
    over = max((np.abs(f1) - lim).max(), (np.abs(f2) - lim).max())
    if over > 0:
        bad.append('friction beyond mu * normal force by %.2e N' % over)
    pairs = set(zip(np.asarray(model['pair_a'])[:int(model['n_pair'])].tolist(), np.asarray(model['pair_b'])[:int(model['n_pair'])].tolist()))
    if any((int(x), int(y)) not in pairs for x, y in zip(a, b)):
        bad.append('collider pair not in the model pair list')
    return bad


def block_vertical_force(model, rep, i, body):
    """Vertical component of the total contact force on free body `body` (1-based body index) in env i."""
    cb_ = np.asarray(model['col_body'])
    f = 0.0
    for k in range(int(rep['count'][i])):
        a, b = rep['collider_a'][i][k], rep['collider_b'][i][k]
        F = rep['normal_force'][i][k] * np.asarray(rep['normal_on_b'][i][k], np.float64) + \
            rep['lateral_friction_1'][i][k] * np.asarray(rep['lateral_friction_dir_1'][i][k], np.float64) + \
            rep['lateral_friction_2'][i][k] * np.asarray(rep['lateral_friction_dir_2'][i][k], np.float64)
        if cb_[a] == body:
            f += F[2]
        if cb_[b] == body:
            f -= F[2]
    return f
