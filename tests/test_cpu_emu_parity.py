"""The product's kernel source (csrc/prb_kernels.cuh) compiled for the CPU SIMT emulator
(tests/emu) against the fp64 oracle: same tolerances as the GPU parity tests, tiny sizes.
This exercises the warp-collective code paths (shuffles, ballots, scans) without a GPU; it is a
test harness, not a product path."""
import numpy as np
import pytest

from roboticsplayroompybullet_b200.model import load_model
from oracle.oracle import Oracle
from emu_lib import EmuSim, box_box as emu_box_box
from oracle.oracle import box_box as orc_box_box


def _sync(sim, o, i=0):
    o.state[:] = o.state.astype(np.float32).astype(np.float64)
    sim.state[i, :o.state_dim] = o.state.astype(np.float32)


@pytest.mark.parametrize('env_id', ['UR5Reach-v0', 'pandaPick-v0', 'pandaReach-v0', 'pandaReach2D-v0', 'pandaPush-v0'])
def test_emu_step_matches_oracle_arm_envs(env_id):
    m = load_model(env_id)
    sim, o = EmuSim(m, 1, seed=4), Oracle(m, seed=4)
    de, do = sim.reset(), o.reset()
    assert np.abs(de['desired_goal'][0] - do['desired_goal']).max() < 1e-6
    rng = np.random.default_rng(0)
    for _ in range(3):
        a = np.concatenate([rng.uniform(-0.15, 0.15, 3), rng.uniform(-0.3, 0.3, 3), rng.uniform(-1, 1, 1)])
        _sync(sim, o)
        de, do = sim.step(a[None]), o.step(a)
        nd = m['nd']
        assert np.abs(sim.state[0, :nd] - o.state[:nd]).max() < 2e-6                  # joint positions
        assert np.abs(de['target_poses'][0] - do['target_poses']).max() < 2e-6        # IK + clipping
        assert np.abs(de['obs_quat'][0][:3] - do['obs_quat'][:3]).max() < 1e-5
        assert de['reward'][0, 0] == do['reward'][0]


def test_emu_play_step_with_contacts():
    m = load_model('UR5PlayAbsRPY1Obj-v0')
    sim, o = EmuSim(m, 1, seed=3), Oracle(m, seed=3)
    o.reset()
    blk = o.state[60:63].copy()
    for a in [[blk[0], blk[1], 0.15, 0, 0, 0, -1], [blk[0], blk[1], 0.10, 0.1, 0, 0, 1]]:
        _sync(sim, o)
        de, do = sim.step(np.array([a])), o.step(a)
        sd = o.state_dim
        d = np.abs(sim.state[0, :sd - 1] - o.state[:sd - 1])
        assert d[:12].max() < 2e-6 and d[60:67].max() < 1e-5 and d[73:80].max() < 1e-5
        for k in ['obs_quat', 'achieved_goal', 'full_positional_state', 'observation']:
            assert np.abs(de[k][0] - do[k]).max() < 2e-5, k
        assert o.L.orc_last_contacts() >= 8            # block on table + drawer on its blockers


def test_emu_box_box_matches_oracle():
    rng = np.random.default_rng(5)
    from scipy.spatial.transform import Rotation
    n_hit = 0
    for _ in range(60):
        R1 = Rotation.random(random_state=rng.integers(1 << 30)).as_matrix()
        R2 = Rotation.random(random_state=rng.integers(1 << 30)).as_matrix()
        h1, h2 = rng.uniform(0.02, 0.1, 3), rng.uniform(0.02, 0.1, 3)
        p2 = rng.uniform(-0.08, 0.08, 3)
        a = orc_box_box([0, 0, 0], R1.reshape(-1), h1, p2, R2.reshape(-1), h2)
        b = emu_box_box([0, 0, 0], R1.reshape(-1), h1, p2, R2.reshape(-1), h2)
        assert len(a) == len(b)
        if len(a):
            n_hit += 1
            assert np.abs(a - b).max() < 5e-5
    assert n_hit > 20


def _stream_headers(env=0):
    """Decode the three header float4 of one env's record stream (csrc/prb_stream.cuh, Q_HDR)."""
    import ctypes
    from emu_lib import lib
    L = lib()
    L.emu_sbuf.restype = ctypes.POINTER(ctypes.c_float)
    sbq = L.emu_sbuf_q()
    buf = np.ctypeslib.as_array(L.emu_sbuf(), shape=(sbq, 32, 4))
    h = [buf[i, env].view(np.int32).copy() for i in range(3)]
    return {'njr': int(h[0][0] & 0xff), 'nc0': int((h[0][0] >> 8) & 0xff), 'canon': int((h[0][0] >> 24) & 1), 'cls': int((h[0][0] >> 25) & 7),
            'nc1': int(h[1][0] & 0xff), 'nc2': int(h[2][0] & 0xff),
            'slot_free0': int((h[1][0] >> 16) & 3), 'slot_free1': int((h[1][0] >> 18) & 3)}


def test_emu_grasp_sequence_islands_and_arm_solver():
    """Scripted reach-close-lift of the block, every env step started from the oracle's state.  While the
    gripper is away the block and the drawer are their own constraint islands (slots 1, 2: free-body
    solver) and the arm island has joint rows only; once the fingers touch the block its island merges
    into slot 0 and is solved by the arm-island kernel from its size class's heavy buffer.  Both paths must match the
    fp64 oracle to the one-step pose tolerance."""
    m = load_model('UR5PlayAbsRPY1Obj-v0')
    sim, o = EmuSim(m, 1, seed=3), Oracle(m, seed=3)
    o.reset()
    blk = o.state[60:63].copy()
    act = lambda z, g: np.array([blk[0], blk[1], z, 0, 0, 0, g])
    seq = [act(0.15, -1)] * 3 + [act(-0.01, -1)] * 12 + [act(-0.01, 1)] * 10 + [act(0.2, 1)] * 8
    errs, merged, separate = [], 0, 0
    for a in seq:
        _sync(sim, o)
        sim.step(a[None]); o.step(a)
        sd = o.state_dim
        d = np.abs(sim.state[0, :sd - 1] - o.state[:sd - 1])
        errs.append(max(d[:12].max(), d[60:63].max(), d[73:76].max()))
        h = _stream_headers()
        assert h['njr'] >= 12                                    # 12 motors (+ gear, limits)
        if h['slot_free0'] == 0:
            merged += 1
            assert h['nc0'] > 0 and h['nc1'] == 0                # block contacts moved to the arm island
            assert h['cls'] >= 1 and h['canon'] == 1             # heavy: solved from a class buffer; all 12 + 3 motors present
        else:
            separate += 1
            assert h['slot_free0'] == 1 and h['nc1'] >= 1
        assert h['slot_free1'] == 2 and h['nc2'] >= 4            # drawer rests on its blockers throughout
    assert merged >= 8 and separate >= 8
    errs = np.array(errs)
    assert np.median(errs) < 1e-6
    assert (errs < 1e-4).sum() >= len(errs) - 2                  # contact onset may flip by one substep (fp32 vs fp64)
    assert o.state[62] > 0.1                                     # lifted


@pytest.mark.parametrize('env_id', ['UR5Play1Obj-v0', 'UR5PlayRel1Obj-v0', 'UR5PlayRelRPY1Obj-v0',
                                    'UR5PlayAbsJoints1Obj-v0', 'UR5PlayRelJoints1Obj-v0',
                                    'pandaPlayAbsRPY1Obj-v0', 'pandaPlay1Obj-v0', 'pandaPlayRel1Obj-v0', 'pandaPlayRelRPY1Obj-v0',
                                    'pandaPlayAbsJoints1Obj-v0', 'pandaPlayRelJoints1Obj-v0'])
def test_emu_action_decoders_match_oracle(env_id):
    """The other UR5 playroom ids differ from UR5PlayAbsRPY1Obj-v0 only by the action decoder
    (environments.py:915-981): kernel vs oracle on the decoded motor targets and the resulting step."""
    from roboticsplayroompybullet_b200.model import action_dim
    m = load_model(env_id)
    A = action_dim(m)
    nd, nik = m['nd'], m['n_ik']
    sim, o = EmuSim(m, 1, seed=5), Oracle(m, seed=5)
    o.reset()
    rng = np.random.default_rng(7)
    ee = o.fk_sites(o.state[:nd])[0]
    for _ in range(3):
        if 'Joints' in env_id:
            assert A == nik + 1                                                       # 7 (UR5) / 8 (Panda): environments.py:98-107
            a = np.concatenate([rng.uniform(-0.05, 0.05, nik) + (o.state[:nik] if 'Abs' in env_id else 0), rng.uniform(-1, 1, 1)])
        elif A == 8:
            q = ee[3:7] if 'Rel' not in env_id else np.zeros(4)
            a = np.concatenate([(ee[:3] if 'Rel' not in env_id else 0) + rng.uniform(-0.03, 0.03, 3),
                                q + rng.uniform(-0.05, 0.05, 4), rng.uniform(-1, 1, 1)])
        elif 'Rel' in env_id:
            a = np.concatenate([rng.uniform(-0.03, 0.03, 3), rng.uniform(-0.1, 0.1, 3), rng.uniform(-1, 1, 1)])
        else:                                                                         # absolute rpy: around the current pose
            from oracle.oracle import euler_from_quat
            a = np.concatenate([ee[:3] + rng.uniform(-0.03, 0.03, 3), euler_from_quat(ee[3:7]) + rng.uniform(-0.1, 0.1, 3), rng.uniform(-1, 1, 1)])
        assert len(a) == A
        _sync(sim, o)
        de, do = sim.step(a[None]), o.step(a)
        assert np.abs(de['target_poses'][0] - do['target_poses']).max() < 5e-6
        assert np.abs(sim.state[0, :nd] - o.state[:nd]).max() < 5e-6
        assert np.abs(de['obs_quat'][0][:7] - do['obs_quat'][:7]).max() < 2e-5
        # the command moved the arm the way its decoder says
        assert np.abs(do['target_poses'] - o.state[:nik]).max() < 0.3


def test_emu_records_read_in_place_when_stage_is_small():
    """Capacity only costs speed, never contacts: with tiny solver stages (arm-island classes of 104-120 q, free-body
    stage of 16 q) every grasp lands in the last class and most of its records are read from the class buffer in
    place; the grasp sequence must give the SAME states as the normal build, bit for bit."""
    from helpers import SMALL_STAGE
    m = load_model('UR5PlayAbsRPY1Obj-v0')
    a_sim, b_sim, o = EmuSim(m, 1, seed=3), EmuSim(m, 1, seed=3, tag='smallstage', defines=SMALL_STAGE), Oracle(m, seed=3)
    o.reset()
    blk = o.state[60:63].copy()
    act = lambda z, g: np.array([blk[0], blk[1], z, 0, 0, 0, g])
    seq = [act(-0.01, -1)] * 14 + [act(-0.01, 1)] * 8 + [act(0.15, 1)] * 4
    a_sim.state[0, :o.state_dim] = o.state.astype(np.float32)
    b_sim.state[0, :o.state_dim] = o.state.astype(np.float32)
    for a in seq:
        da, db = a_sim.step(a[None]), b_sim.step(a[None])
        assert np.array_equal(a_sim.state, b_sim.state)
        for k in da:
            assert np.array_equal(da[k], db[k]), k
    assert a_sim.state[0, 62] > 0.05            # the block was grasped and lifted on the way


def test_emu_reset_rounds_match_oracle():
    """reset() as rounds on the masked step pipeline (prb_reset.cuh): same counter-based draws as the oracle's
    orc_reset, including the envs that need a second attempt because the sampled goal is already satisfied
    (environments.py:180-185), and a masked reset that leaves the other envs untouched."""
    m = load_model('UR5PlayAbsRPY1Obj-v0')
    n = 6
    sim = EmuSim(m, n, seed=21)
    sd = Oracle(m).state_dim
    d = sim.reset()
    rounds = sim.L.emu_reset_rounds()
    attempts = sim.state[:, sd - 1].copy()
    assert rounds >= 2 and attempts.max() >= 2, (rounds, attempts)      # seed chosen so that a retry happens
    for i in range(n):
        o = Oracle(m, seed=21, env_id=i)
        do = o.reset()
        assert o.state[-1] == attempts[i]
        for k in ['achieved_goal', 'desired_goal']:
            assert np.abs(d[k][i] - do[k]).max() < 2e-3, (i, k)
        assert np.abs(d['obs_quat'][i][:7] - do['obs_quat'][:7]).max() < 1e-5       # end-effector pose after reset_arm
        assert abs(d['obs_quat'][i][7] - do['obs_quat'][7]) < 1e-3                  # gripper reading (23 x the pad joint)
    before = sim.state.copy()
    mask = np.zeros(n, np.uint8); mask[2] = 1
    sim.reset(mask)
    keep = np.arange(n) != 2
    assert np.array_equal(sim.state[keep], before[keep])
    assert sim.state[2, sd - 1] > before[2, sd - 1]


@pytest.mark.parametrize('env_id', ['UR5Reach-v0', 'pandaPick-v0', 'UR5PlayAbsRPY1Obj-v0'])
def test_emu_every_key_matches_oracle(env_id):
    """The all-key comparison the GPU parity tests use (tests/helpers.py: pose / velocity / flag groups, dial and Euler
    wrap, conditioning rule) run on the emulated kernels: no env may need the conditioning allowance here."""
    from helpers import compare_step, random_actions, oracle_step_from, OBS_KEYS
    m = load_model(env_id)
    n = 4
    sim = EmuSim(m, n, seed=7)
    sim.reset()
    rng = np.random.default_rng(3)
    sd = Oracle(m).state_dim
    for step in range(2):
        st = sim.state[:, :sd].copy()
        a = random_actions(rng, n, env_id)
        de = sim.step(a)
        outs = [oracle_step_from(m, st[i], a[i], Oracle)[0] for i in range(n)]
        res = compare_step(m, {k: de[k] for k in OBS_KEYS}, de['reward'][:, 0], {'is_success': de['is_success'][:, 0]}, outs,
                           st, a, Oracle)
        assert res['bad_pose'] == res['bad_vel'] == res['bad_flags'] == res['bad_reward'] == res['stiff'] == 0, res
        assert res['worst_pose'] < 2e-5 and res['worst_vel'] < 0.1, res


def test_emu_solver_regression_bit_identical():
    """48 heavy states sampled on the B200 from the scripted bench workload (arm islands of 150-770 stream q: every size
    class of the arm-island solver), stepped once.  The fixture (tools/make_solver_golden.py) holds the states the ROUND-1
    solver produced (four lanes per env, quad-shuffle reductions); the thread-per-env solver that replaced it keeps the
    arithmetic of every row visit, so the results must be the same bits — and match the oracle by the all-key rule."""
    import os
    from helpers import compare_step, oracle_step_from, OBS_KEYS
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'heavy_step_r1.npz'))
    m = load_model('UR5PlayAbsRPY1Obj-v0')
    n = len(g['state'])
    sim = EmuSim(m, n, seed=1)
    sd = Oracle(m).state_dim
    sim.state[:, :sd] = g['state']
    import ctypes
    cc = (ctypes.c_longlong * 8)()
    sim.L.emu_class_counts(cc, 1)
    de = sim.step(g['action'])
    sim.L.emu_class_counts(cc, 1)
    assert all(c > 0 for c in list(cc)[:5]), list(cc)[:5]          # every size class (incl. read-in-place) solved something
    assert np.array_equal(sim.state[:, :sd], g['state_after'])
    assert np.array_equal(de['obs_quat'], g['obs_quat']) and np.array_equal(de['reward'], g['reward'])
    outs = [oracle_step_from(m, g['state'][i], g['action'][i], Oracle)[0] for i in range(n)]
    res = compare_step(m, {k: de[k] for k in OBS_KEYS}, de['reward'][:, 0], {'is_success': de['is_success'][:, 0]}, outs,
                       g['state'], g['action'], Oracle)
    assert res['bad_pose'] <= 2 and res['bad_reward'] <= 1, res       # these are the stiffest 0.1 % of the workload


@pytest.mark.parametrize('env_id', ['UR5PlayAbsRPY1Obj-v0', 'pandaPick-v0', 'UR5Reach-v0'])
def test_emu_reset_from_observation(env_id):
    """playEnv.reset(o) (environments.py:173-187, 541-556, 582-596): re-seating from an observation of a rollout puts the
    object and the end effector back where the observation says (trajectory replay), with the oracle's reset_to as the
    reference; in the play env the drawer / door / button / dial are restored as well (restore_env, a documented
    extension) or left at their defaults like the reference does."""
    m = load_model(env_id)
    sim, o = EmuSim(m, 2, seed=9), Oracle(m, seed=9, env_id=0)
    o.reset()
    rng = np.random.default_rng(1)
    play = env_id.startswith('UR5Play')
    blk = o.state[60:63].copy() if play else None
    for k in range(6):                                    # a short rollout; in the play env push the door a little
        a = np.concatenate([rng.uniform(-0.1, 0.1, 3) + (np.array([0.0, 0.3, 0.12]) if play else 0), rng.uniform(-0.2, 0.2, 3), [1.0]])
        d = o.step(a)
    if play:
        o.state[86] = 0.05; o.state[88] = 0.02; o.state[90] = 0.7   # door, button, dial away from their defaults
        o.state[74] = -0.04                                          # drawer pulled
        d = o.calc_state()
    obs = d['obs_quat'].astype(np.float32)
    o2 = Oracle(m, seed=9, env_id=0)
    o2.state[:] = o.state
    sim.state[0, :o.state_dim] = o.state.astype(np.float32)
    sim.state[1, :o.state_dim] = o.state.astype(np.float32)
    before1 = sim.state[1].copy()
    de = sim.reset_to(np.stack([obs, obs]), mask=np.array([1, 0], np.uint8))
    do = o2.reset_to(obs)
    assert np.array_equal(sim.state[1], before1)                                     # masked out: untouched
    assert np.abs(de['obs_quat'][0] - do['obs_quat']).max() < 2e-5
    assert np.abs(de['desired_goal'][0] - do['desired_goal']).max() < 2e-5
    assert sim.state[0, o.state_dim - 1] == o2.state[-1]                             # same number of goal draws
    # replay property: object pose exactly as observed, end effector at the observed pose up to the IK tolerance
    od = m['obs_dim']
    o_obj = {7: None, 13: 7, 19: 8}[od]
    if o_obj is not None:
        assert np.abs(de['obs_quat'][0][o_obj:o_obj + 3] - obs[o_obj:o_obj + 3]).max() < 1e-6
    assert np.abs(de['obs_quat'][0][:3] - obs[:3]).max() < 2.5e-2             # one 20-iteration IK call from the rest pose (:593)
    if play:
        assert np.abs(de['obs_quat'][0][15:19] - obs[15:19]).max() < 1e-5              # drawer, door, button, dial restored
        d_ref = sim.reset_to(np.stack([obs, obs]), mask=np.array([1, 0], np.uint8), restore_env=False)
        assert np.abs(d_ref['obs_quat'][0][16:19] - [0, 0, 0]).max() < 1e-6           # reference behaviour: defaults


def test_emu_more_than_32_contacts():
    """17 states with 33-45 contacts after manifold reduction, four of them with more than 32 overlapping collider pairs in the
    broad phase (found by oracle rollouts with 25 % random jumps: the arm rammed into the drawer and the cabinet;
    tests/golden/many_contacts.npz holds the INPUT states and actions only).  The narrow phase and the row writer give a
    lane two pairs / two contacts there and the largest arm islands are read partly in place: no pair or contact may be
    dropped and the step must match the oracle like any other (one of the states is ill-conditioned and covered by the
    ulp rule; another one has a four-way tie in the manifold reduction between coincident candidates of two collider pairs,
    which only the absolute 2 um tie rule resolves the same way in fp32 and fp64)."""
    import os
    from helpers import compare_step, oracle_step_from, OBS_KEYS
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'many_contacts.npz'))
    m = load_model('UR5PlayAbsRPY1Obj-v0')
    n = len(g['state'])
    assert n >= 10 and g['nc'].min() > 32
    sim = EmuSim(m, n, seed=1)
    sd = Oracle(m).state_dim
    sim.state[:, :sd] = g['state']
    ov0 = sim.L.emu_overflow()
    de = sim.step(g['action'])
    assert sim.L.emu_overflow() == ov0                                   # nothing dropped
    outs = [oracle_step_from(m, g['state'][i], g['action'][i], Oracle)[0] for i in range(n)]
    res = compare_step(m, {k: de[k] for k in OBS_KEYS}, de['reward'][:, 0], {'is_success': de['is_success'][:, 0]}, outs,
                       g['state'], g['action'], Oracle)
    assert res['bad_pose'] == 0 and res['bad_vel'] == 0 and res['bad_reward'] == 0 and res['stiff'] <= 2, res


def test_emu_fused_pipeline_counts_each_overflowing_env_once():
    """The fused A/B kernel holds 32 overlapping pairs and 32 contacts per env (prb_kernels.cuh, CfgL): every one of the 17
    many-contact states exceeds that in some substep of its step, and the capacity counter goes up by exactly one per env
    step, however many substeps dropped something.  The split pipeline drops nothing on the same states."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'many_contacts.npz'))
    m = load_model('UR5PlayAbsRPY1Obj-v0')
    n = len(g['state'])
    sd = Oracle(m).state_dim
    deltas = {}
    for fused in (1, 0):
        sim = EmuSim(m, n, seed=1)
        sim.state[:, :sd] = g['state']
        ov0 = sim.L.emu_overflow()
        sim.L.emu_set_fused(fused)
        try:
            de = sim.step(g['action'])
        finally:
            sim.L.emu_set_fused(0)
        deltas[fused] = sim.L.emu_overflow() - ov0
        assert all(np.isfinite(v).all() for v in de.values()) and np.isfinite(sim.state).all()
    assert deltas == {1: n, 0: 0}, deltas
