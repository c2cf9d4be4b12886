"""Shared helpers for the parity tests: seeded synthetic actions (SURVEY.md §8d) and comparison of a batched
result against per-env oracle runs started from identical states.

Every key of the reference's calc_state dict (environments.py:849-861) is compared, in four groups:
  pose    obs_quat (non-velocity entries), achieved_goal, desired_goal, controllable_achieved_goal,
          full_positional_state, joints, observation (its Euler entries modulo 2 pi): 1e-4 m / 1e-3 rad
          (BASELINE.json north_star; quaternion components and joint angles are held to the tighter 1e-4)
  vel     velocity (end-effector twist) and the velocity entries of obs_quat in the Reach / Pick layouts:
          |dv| <= VEL_ABS + VEL_REL |v| with VEL_ABS = 3e-2 m/s: the pose tolerance seen as a speed (1e-4 m per 1/300 s
          substep); north_star states no velocity tolerance of its own
  flags   gripper_proprioception, reward, is_success: identical away from thresholds
  target  target_poses (IK + clipping): 1e-5 relative in the bulk (fp32 vs the oracle's fp64)

Conditioning.  A stiff state (fingers closed on the block: soft-contact CFM rows against motor rows with 240 N
limits) amplifies rounding.  `ulp_spread` measures that amplification on the ORACLE itself: its input state is
perturbed by one fp32 ulp per entry and the fp64 step repeated; an env whose CUDA result is further than the pose
tolerance from the oracle is accepted only if it is within COND_K x that spread.
"""
import numpy as np

OBS_KEYS = ['obs_quat', 'achieved_goal', 'desired_goal', 'controllable_achieved_goal', 'full_positional_state',
            'joints', 'velocity', 'observation', 'gripper_proprioception']

POS_TOL = 1e-4        # m (and quaternion components / joint angles)
ANG_TOL = 1e-3        # rad (Euler entries of 'observation')
VEL_ABS, VEL_REL = 3e-2, 1e-2   # the pose tolerance seen as a speed: 1e-4 m per 1/300 s substep = 3e-2 m/s (rad/s)
COND_K = 8.0          # |cuda - oracle| <= COND_K x (spread of the oracle under 1-ulp input perturbations)
DIAL_PERIOD = 2.0 / 2.2   # scenes.py:342-343: (q mod 2) / 2.2 wraps at q = 0 -> compare modulo the period
# compile-time defines of the small-stage build (csrc/prb_stream.cuh): arm-island classes of 104-120 q and a free-body stage
# of 16 q, so that most arm records are read from the class buffer in place; emulated and nvcc builds use the same list
SMALL_STAGE = ['ARM_CAPQ0=104', 'ARM_CAPQ1=108', 'ARM_CAPQ2=112', 'ARM_CAPQ3=116', 'ARM_CAPQ4=120', 'PGS_STAGE_F=16']


def random_actions(rng, n, env_id):
    if 'Play' in env_id:
        lo, hi = [-0.30, -0.05, 0.0], [0.30, 0.50, 0.35]
    else:
        lo, hi = [-0.18, -0.18, -0.05], [0.18, 0.18, 0.2]
    a = np.concatenate([rng.uniform(lo, hi, (n, 3)), rng.uniform(-0.5, 0.5, (n, 3)), rng.uniform(-1, 1, (n, 1))], 1)
    tail = rng.random(n) < 0.05                      # 5% from the full clip box: exercises the +-inc clamp
    a[tail, :6] = rng.uniform(-6, 6, (int(tail.sum()), 6))
    return a.astype(np.float32)


def oracle_step_from(model, state_row, action, Oracle):
    o = Oracle(model)
    o.state[:] = state_row.astype(np.float64)
    d = o.step(action.astype(np.float64))
    return d, o.state.copy()


def _layout(model):
    """Index sets inside obs_quat / observation for this env kind."""
    od = int(model['obs_dim'])
    vel_idx = {7: [3, 4, 5], 13: [3, 4, 5, 10, 11, 12]}.get(od, [])
    dial_obs = [18] if od == 19 else []              # dial reading: periodic
    return od, vel_idx, dial_obs


def _wrap(d, period):
    return np.abs((d + 0.5 * period) % period - 0.5 * period)


def key_errors(model, got, ref):
    """Per-group worst errors of one env: dict(pose, ang, vel (scaled: <= 1 passes), flags (count of mismatches))."""
    od, vel_idx, dial_obs = _layout(model)
    play = od == 19
    pose, ang, vel, flags = 0.0, 0.0, 0.0, 0
    g = {k: np.asarray(got[k], np.float64).ravel() for k in OBS_KEYS}
    r = {k: np.asarray(ref[k], np.float64).ravel() for k in OBS_KEYS}
    # ---- obs_quat
    d = np.abs(g['obs_quat'] - r['obs_quat'])
    if dial_obs:
        d[dial_obs] = _wrap(g['obs_quat'][dial_obs] - r['obs_quat'][dial_obs], DIAL_PERIOD)
    mask = np.ones(od, bool)
    mask[vel_idx] = False
    pose = max(pose, float(d[mask].max()))
    for i in vel_idx:
        vel = max(vel, d[i] / (VEL_ABS + VEL_REL * abs(r['obs_quat'][i])))
    # ---- goals / positional state (play: last entry is the dial reading)
    for k in ['achieved_goal', 'desired_goal', 'full_positional_state']:
        d = np.abs(g[k] - r[k])
        if play:
            d[-1] = _wrap(g[k][-1:] - r[k][-1:], DIAL_PERIOD)[0]
        pose = max(pose, float(d.max()))
    for k in ['controllable_achieved_goal', 'joints']:
        pose = max(pose, float(np.abs(g[k] - r[k]).max()))
    # ---- velocity: end-effector twist
    d = np.abs(g['velocity'] - r['velocity'])
    vel = max(vel, float((d / (VEL_ABS + VEL_REL * np.abs(r['velocity']))).max()))
    # ---- observation: [xyz, euler(state[3:7]), state[7:]] (environments.py:859; in the non-play layouts the "euler" is
    #      of (velocity, gripper) — a dimension quirk: compared as plain numbers with the angle tolerance there)
    d = np.abs(g['observation'] - r['observation'])
    d[3:6] = _wrap(g['observation'][3:6] - r['observation'][3:6], 2 * np.pi)
    if play:
        d[-1] = _wrap(g['observation'][-1:] - r['observation'][-1:], DIAL_PERIOD)[0]
        ang = max(ang, float(d[3:6].max()))
        pose = max(pose, float(np.delete(d, [3, 4, 5]).max()))
    else:
        pose = max(pose, float(d[0:3].max()))
        # entries 3:6 are euler(quat = (v_x, v_y, v_z, grip)), un-normalised: a velocity error dv turns the "quaternion" by
        # ~dv / |quat|, and the angles are undefined when it vanishes (arm at rest, gripper reading 0)
        fq = r['obs_quat'][3:7]
        nq = float(np.linalg.norm(fq))
        if nq > 0.05:
            tol = ANG_TOL + 4.0 * (VEL_ABS + VEL_REL * float(np.abs(fq[:3]).max())) / nq
            vel = max(vel, float(d[3:6].max()) / tol)
        rest = d[6:]                                 # Pick: block xyz (pose), block velocity (vel)
        if len(rest):
            pose = max(pose, float(rest[:3].max()))
            rv = r['observation'][9:12]
            vel = max(vel, float((rest[3:6] / (VEL_ABS + VEL_REL * np.abs(rv))).max()))
    # ---- flags
    flags += int(g['gripper_proprioception'][0] != r['gripper_proprioception'][0])
    return {'pose': pose, 'ang': ang, 'vel': vel, 'flags': flags}


def ulp_spread(model, state_row, action, Oracle, ref, rng, n_pert=8):
    """Worst pose-group and velocity-group deviation of the oracle's own fp64 step when every non-zero entry of its (fp32)
    input state moves by one ulp in a random direction (goal / bookkeeping entries untouched)."""
    x = np.asarray(state_row, np.float32)
    G = int(model['goal_dim'])
    tail = G + 10
    worst = {'pose': 0.0, 'vel': 0.0}
    for _ in range(n_pert):
        sgn = np.sign(rng.standard_normal(len(x))).astype(np.float32)
        y = np.nextafter(x, x + sgn * np.float32(1e9)).astype(np.float32)
        y[x == 0] = 0
        y[-tail:] = x[-tail:]
        o = Oracle(model)
        o.state[:] = y.astype(np.float64)
        d = o.step(np.asarray(action, np.float64))
        e = key_errors(model, d, ref)
        worst['pose'] = max(worst['pose'], e['pose'], e['ang'] * POS_TOL / ANG_TOL)
        worst['vel'] = max(worst['vel'], e['vel'])
    return worst


def compare_step(model, obs, r, info, oracle_outs, states=None, actions=None, Oracle=None, rng=None):
    """Compares every key of a batched step with the per-env oracle results.  Returns a dict:
    n, bad_pose (envs beyond the pose tolerance and not explained by conditioning), stiff (envs beyond a tolerance
    but within COND_K x their ulp spread), bad_vel, bad_flags, bad_reward, worst_pose, worst_unexplained, worst_vel."""
    n = len(oracle_outs)
    out = {'n': n, 'bad_pose': 0, 'stiff': 0, 'bad_vel': 0, 'bad_flags': 0, 'bad_reward': 0, 'worst_pose': 0.0,
           'worst_unexplained': 0.0, 'worst_vel': 0.0}
    rng = rng if rng is not None else np.random.default_rng(0)
    for i in range(n):
        ref = oracle_outs[i]
        got = {k: np.asarray(obs[k][i]) for k in OBS_KEYS}
        e = key_errors(model, got, ref)
        pose = max(e['pose'], e['ang'] * POS_TOL / ANG_TOL)          # angles on the pose scale
        out['worst_pose'] = max(out['worst_pose'], pose)
        out['worst_vel'] = max(out['worst_vel'], e['vel'])
        rr = float(ref['reward'][0])
        rew_bad = not (r[i] == rr or abs(r[i] - rr) < 1e-4) or int(info['is_success'][i]) != int(ref['is_success'][0])
        over_pose, over_vel = pose > POS_TOL, e['vel'] > 1.0
        ex_pose = ex_vel = False
        if (over_pose or over_vel or e['flags'] or rew_bad) and states is not None:
            sp = ulp_spread(model, states[i], actions[i], Oracle, ref, rng)
            ex_pose = pose <= COND_K * sp['pose'] and sp['pose'] > POS_TOL / COND_K
            ex_vel = e['vel'] <= COND_K * sp['vel'] and sp['vel'] > 1.0 / COND_K
        if over_pose:
            if ex_pose:
                out['stiff'] += 1
            else:
                out['bad_pose'] += 1
                out['worst_unexplained'] = max(out['worst_unexplained'], pose)
        if over_vel:
            if ex_vel or ex_pose:
                out['stiff'] += 0 if over_pose else 1
            else:
                out['bad_vel'] += 1
        if e['flags'] and not (ex_pose or ex_vel):
            out['bad_flags'] += 1
        if rew_bad and not (ex_pose or ex_vel):
            out['bad_reward'] += 1
    return out
