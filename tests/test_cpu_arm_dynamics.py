"""CPU tests of the arm queries (prb_arm_dynamics): the numpy reference tests/np_arm_dynamics.py against the oracle's
kinematics and articulated-body dynamics, the kernel source (csrc/prb_arm.cuh, under the SIMT emulator) against that
reference, the end-effector velocity the step observes, invalid input, the struct layout and the Python surface's
checks."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import emu_arm
import np_arm_dynamics as R
from emu_lib import EmuSim
from helpers import random_actions
from oracle.oracle import Oracle
from roboticsplayroompybullet_b200 import lib
from roboticsplayroompybullet_b200.envs import check_arm_inputs, check_arm_points
from roboticsplayroompybullet_b200.model import load_model

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
PLAY = 'UR5PlayAbsRPY1Obj-v0'
ARMS = [PLAY, 'pandaPlayAbsRPY1Obj-v0']
U32 = 2.0 ** -24          # fp32 unit roundoff
# Kernel against the fp64 reference: |got - ref| <= TOL * max(1, max |ref|) per env and output.  Every output is a short
# chain of fp32 products and sums (frames composed over <= 8 links, subtree sums over <= 12 links, dot products over
# <= 12 columns), each step a few ulps of the running magnitude; measured worst 12u (Panda tau with q beyond the
# limits), so 64u leaves a 5x margin.
TOL = 64 * U32


def _quat_mat(x):
    x, y, z, w = x
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _limits(m):
    nd = int(m['nd'])
    lo, hi = np.asarray(m['arm_lo'])[:nd], np.asarray(m['arm_hi'])[:nd]
    return np.maximum(lo, -np.pi), np.minimum(hi, np.pi)


def _points(m):
    """Sites 0..3 at zero offset and at an offset, and every link at zero offset and at an offset."""
    nd = int(m['nd'])
    pts = [(-1, s, (0.0, 0.0, 0.0)) for s in range(4)] + [(-1, 0, (0.03, -0.02, 0.05)), (-1, 2, (0.0, 0.01, -0.02))]
    pts += [(l, -1, (0.0, 0.0, 0.0)) for l in range(nd)][:8] + [(nd - 1, -1, (0.1, 0.2, -0.1)), (2, -1, (-0.3, 0.0, 0.1))]
    return pts[:16]


# ------------------------------------------------------------------ the reference against the oracle
@pytest.mark.parametrize('env_id', ARMS)
def test_reference_matches_oracle(env_id):
    m = load_model(env_id)
    A, o, nd = R.arm(m), Oracle(m), int(m['nd'])
    # the oracle's arm link damping is zero in every compiled model, so its free motion has M qdd + h = -jdamp qd
    assert m.param('arm_lin_damp') == 0.0 and m.param('arm_ang_damp') == 0.0
    lo, hi = _limits(m)
    rng = np.random.default_rng(7)
    for _ in range(6):
        q, qd = rng.uniform(lo, hi), rng.uniform(-2.0, 2.0, nd)
        # Jacobian columns against central differences of the oracle's site poses (position and orientation)
        h = 1e-6
        for s in range(4):
            J, x = R.jacobian(A, q, -1, s, (0.0, 0.0, 0.0))
            assert np.abs(x - o.fk_sites(q)[s, :3]).max() <= 1e-12
            Rm = _quat_mat(o.fk_sites(q)[s, 3:])
            for j in range(nd):
                dq = np.zeros(nd)
                dq[j] = h
                fp, fm = o.fk_sites(q + dq)[s], o.fk_sites(q - dq)[s]
                assert np.abs((fp[:3] - fm[:3]) / (2 * h) - J[:3, j]).max() <= 1e-8, (s, j)
                W = (_quat_mat(fp[3:]) - _quat_mat(fm[3:])) / (2 * h) @ Rm.T
                assert np.abs(np.array([W[2, 1], W[0, 2], W[1, 0]]) - J[3:, j]).max() <= 1e-8, (s, j)
        # M times the oracle's M^-1 (unit-impulse responses of its articulated-body pass) is I, up to the conditioning:
        # kappa(M) reaches ~2e4 on the UR5, whose light gripper links sit next to its heavy shoulder
        M = R.mass_matrix(A, q)
        kappa = np.linalg.cond(M)
        assert np.abs(M @ o.minv(q) - np.eye(nd)).max() <= 1e-14 * kappa * nd, kappa
        assert np.abs(M - M.T).max() <= 1e-12 * np.abs(M).max()
        # tau at the oracle's free-motion acceleration is the joint damping it applies
        hb = R.bias(A, q, qd)
        tau = M @ o.qdd(q, qd) + hb
        assert np.abs(tau + A['jdamp'] * qd).max() <= 1e-14 * kappa * max(1.0, np.abs(hb).max()), np.abs(tau).max()
        # kinetic energy of the links
        assert abs(0.5 * qd @ M @ qd - R.kinetic_energy(A, q, qd)) <= 1e-12 * max(1.0, R.kinetic_energy(A, q, qd))


# ------------------------------------------------------------------ the kernel against the reference
def _check(m, states, q=None, qd=None, qdd=None):
    """Every output of the emulated kernel on these states against np_arm_dynamics; M symmetric bit for bit.  Returns
    the worst error per output in units of TOL."""
    nd, pts = int(m['nd']), _points(m)
    out = emu_arm.arm_dynamics(m, states, pts, q, qd, qdd)
    A = R.arm(m)
    worst = {k: 0.0 for k in out}
    for i in range(len(states)):
        qi = states[i, :nd] if q is None else q[i]
        qdi = states[i, nd:2 * nd] if qd is None else qd[i]
        qddi = np.zeros(nd) if qdd is None else qdd[i]
        ref = R.all_outputs(A, np.float32(qi), np.float32(qdi), np.float32(qddi), pts)
        for k, v in out.items():
            err = np.abs(v[i] - ref[k]).max() / max(1.0, np.abs(ref[k]).max())
            worst[k] = max(worst[k], err / TOL)
            assert err <= TOL, (k, i, err / U32)
        Mi = out['mass_matrix'][i]
        assert Mi.tobytes() == np.ascontiguousarray(Mi.T).tobytes(), i
    return worst


def _reset_states(env_id, n, seed):
    m = load_model(env_id)
    out = []
    for i in range(n):
        o = Oracle(m, seed=seed + i)
        o.reset()
        out.append(np.asarray(o.state, np.float32))
    return m, np.stack(out)


@pytest.mark.parametrize('env_id', ['UR5Reach-v0'] + ARMS)
def test_emu_matches_reference_reset_states(env_id):
    m, states = _reset_states(env_id, 4, seed=11)
    _check(m, states)


@pytest.mark.parametrize('golden', ['heavy_step_r1.npz', 'many_contacts.npz'])
def test_emu_matches_reference_golden_states(golden):
    _check(load_model(PLAY), np.load(os.path.join(GOLDEN, golden))['state'][:6])


def _stepped(env_id, n, seed):
    m = load_model(env_id)
    sim = EmuSim(m, n, seed=seed)
    sim.reset()
    rng = np.random.default_rng(seed)
    for _ in range(8):
        sim.step(random_actions(rng, n, env_id))
    return m, sim


@pytest.mark.parametrize('env_id', ARMS)
def test_emu_matches_reference_stepped_states_and_caller_inputs(env_id):
    m, sim = _stepped(env_id, 16, seed=5)
    st = sim.state[:, :sim.state_dim].copy()
    print(env_id, 'stepped', _check(m, st))
    nd = int(m['nd'])
    lo, hi = _limits(m)
    rng = np.random.default_rng(3)
    n = len(st)
    inside = (rng.uniform(lo, hi, (n, nd)), rng.uniform(-3.0, 3.0, (n, nd)), rng.uniform(-20.0, 20.0, (n, nd)))
    beyond = (rng.uniform(lo - 2.0, hi + 2.0, (n, nd)), rng.uniform(-10.0, 10.0, (n, nd)), rng.uniform(-100.0, 100.0, (n, nd)))
    for q, qd, qdd in (inside, beyond):
        q, qd, qdd = (x.astype(np.float32) for x in (q, qd, qdd))
        print(env_id, 'caller', _check(m, st, q, qd, qdd))
        _check(m, st, q, None, qdd)          # q given, qd from the state
        _check(m, st, None, qd, None)        # qd given, q from the state


def test_caller_inputs_equal_to_the_state_give_the_same_bits_and_outputs_are_independent():
    for env_id in ARMS:
        m, sim = _stepped(env_id, 8, seed=9)
        st = sim.state[:, :sim.state_dim].copy()
        nd, pts = int(m['nd']), _points(m)
        ref = emu_arm.arm_dynamics(m, st, pts)
        same = emu_arm.arm_dynamics(m, st, pts, q=st[:, :nd], qd=st[:, nd:2 * nd])
        assert all(ref[k].tobytes() == same[k].tobytes() for k in ref)
        # zero qdd is the bias: the same bits as no qdd
        assert emu_arm.arm_dynamics(m, st, pts, qdd=np.zeros((8, nd), np.float32))['tau'].tobytes() == ref['tau'].tobytes()
        # each output alone (what each Python method asks for) gives the same bits as all of them
        for k in emu_arm.OUTPUTS:
            one = emu_arm.arm_dynamics(m, st, pts if k in ('jacobian', 'position', 'velocity') else [], outputs=(k,))
            assert one[k].tobytes() == ref[k].tobytes(), k


@pytest.mark.parametrize('env_id', ARMS)
def test_site0_velocity_is_the_observed_velocity_and_points_sit_on_frames(env_id):
    """point_velocity at site 0 (J qd, summed over columns) against the step's observed end-effector velocity (the
    forward pass's link twist moved to the site): two code paths, equal within fp32 rounding."""
    m, sim = _stepped(env_id, 16, seed=13)
    obs = sim.observe()
    st = sim.state[:, :sim.state_dim].copy()
    nd = int(m['nd'])
    out = emu_arm.arm_dynamics(m, st, [(-1, 0, (0.0, 0.0, 0.0))] + [(l, -1, (0.0, 0.0, 0.0)) for l in range(min(nd, 15))])
    v = out['velocity'][:, 0]
    scale = max(1.0, np.abs(obs['velocity']).max())
    assert np.abs(v - obs['velocity']).max() <= TOL * scale, np.abs(v - obs['velocity']).max() / U32
    A = R.arm(m)
    for i in range(len(st)):
        q = st[i, :nd].astype(np.float64)
        _, p, _, _ = R.fk(A, q)
        assert np.abs(out['position'][i, 1:] - p[:15]).max() <= TOL * max(1.0, np.abs(p).max())
        sites = Oracle(m).fk_sites(q)
        assert np.abs(out['position'][i, 0] - sites[0, :3]).max() <= TOL * max(1.0, np.abs(sites[:, :3]).max())


# ------------------------------------------------------------------ invalid input, layout, the Python surface
def test_invalid_calls_are_rejected_and_write_nothing():
    m, states = _reset_states(PLAY, 1, seed=1)
    P = lib.PrbArmPoint
    pt = lambda l, s, r=0: (P * 1)(P(l, s, (ctypes.c_float * 3)(0, 0, 0), r))
    good = [(-1, 0, (0.0, 0.0, 0.0))]
    bad = [(dict(call=lib.PrbArmQuery(-1, 0)), 'num_points'), (dict(call=lib.PrbArmQuery(17, 0)), 'num_points'),
           (dict(call=lib.PrbArmQuery(1, 1)), 'reserved'), (dict(structs=pt(-1, 0, 5)), 'reserved'),
           (dict(structs=pt(12, -1)), 'link'), (dict(structs=pt(-2, -1)), 'link'),
           (dict(structs=pt(-1, 4)), 'site'), (dict(structs=pt(-1, -2)), 'site'), (dict(structs=pt(3, 0)), 'link -1'),
           (dict(structs=ctypes.POINTER(P)()), 'points_host'),
           (dict(outputs=('mass_matrix', 'tau')), 'points need'), (dict(outputs=()), 'at least one output')]
    for kw, word in bad:
        with pytest.raises(ValueError, match=word):
            emu_arm.arm_dynamics(m, states, good, **kw)
    with pytest.raises(ValueError, match='num_points >= 1'):
        emu_arm.arm_dynamics(m, states, [], outputs=('jacobian',))
    # the emulated launch happens after the checks only: a valid call writes every output, and a rejected one none
    assert all(np.isfinite(v).all() for v in emu_arm.arm_dynamics(m, states, good).values())


def test_struct_layout_matches_c(tmp_path):
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "prb.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n",'
           ' sizeof(prb_arm_point), offsetof(prb_arm_point, link), offsetof(prb_arm_point, site),'
           ' offsetof(prb_arm_point, local_position), offsetof(prb_arm_point, reserved), sizeof(prb_arm_query),'
           ' offsetof(prb_arm_query, num_points), offsetof(prb_arm_query, reserved));return 0;}\n')
    exe = str(tmp_path / 'prb_arm_probe')
    open(exe + '.c', 'w').write(src)
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', exe, exe + '.c'])
    got = list(map(int, subprocess.check_output([exe]).split()))
    P_, Q_ = lib.PrbArmPoint, lib.PrbArmQuery
    assert got == [ctypes.sizeof(P_), P_.link.offset, P_.site.offset, P_.local_position.offset, P_.reserved.offset,
                   ctypes.sizeof(Q_), Q_.num_points.offset, Q_.reserved.offset]
    assert 'prb_arm_dynamics' in lib.SYMBOLS


def test_check_arm_points_and_inputs():
    m = load_model(PLAY)
    urdf = list(np.asarray(m['arm_urdf_index'])[:12])
    assert check_arm_points(m, [(0, 0, 0)]) == [(-1, 0, (0.0, 0.0, 0.0))]
    assert check_arm_points(m, [(1, 2, 3), (0, 0, 0)], link=18, site=None) == [(urdf.index(18), -1, (1.0, 2.0, 3.0)),
                                                                              (urdf.index(18), -1, (0.0, 0.0, 0.0))]
    assert len(check_arm_points(m, np.zeros((16, 3)), site=3)) == 16
    for lp, link, site in (([(0, 0, 0)], 18, 0), ([(0, 0, 0)], None, None), (np.zeros((0, 3)), None, 0),
                           (np.zeros((17, 3)), None, 0), (np.zeros(3), None, 0), ([(0, 0, np.nan)], None, 0),
                           ([(0, 0, 0)], 6, None), ([(0, 0, 0)], 99, None), ([(0, 0, 0)], None, 4),
                           ([(0, 0, 0)], None, -1), ([(0, 0, 0)], None, True)):
        with pytest.raises(ValueError):
            check_arm_points(m, lp, link, site)
    check_arm_inputs(4, 12, q=np.zeros((4, 12)), qd=None)
    for kw in (dict(q=np.zeros((4, 9))), dict(qd=np.zeros((3, 12))), dict(qdd=np.zeros(12)),
               dict(q=np.full((4, 12), np.inf))):
        with pytest.raises(ValueError):
            check_arm_inputs(4, 12, **kw)
