"""CPU tests of closest points (prb_closest_points): the numpy reference tests/np_closest.py against scipy's bounded least
squares and support functions, the kernel source (csrc/prb_closest.cuh, under the SIMT emulator) against that reference,
known answers on two boxes, culling, invalid input and the Python surface's checks."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from scipy.optimize import lsq_linear
from scipy.spatial.transform import Rotation

import emu_closest
import np_closest
from emu_lib import EmuSim
from helpers import random_actions
from oracle.oracle import Oracle
from roboticsplayroompybullet_b200 import lib
from roboticsplayroompybullet_b200.envs import check_closest
from roboticsplayroompybullet_b200.model import load_model

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
PLAY = 'UR5PlayAbsRPY1Obj-v0'
MAX_DISTANCES = (0.0, 0.05, 10.0)


def _states(env_id, n, seed):
    m = load_model(env_id)
    out = []
    for i in range(n):
        o = Oracle(m, seed=seed + i)
        o.reset()
        out.append(np.asarray(o.state, np.float32))
    return m, np.stack(out)


# ------------------------------------------------------------------ the reference against code it shares nothing with
def _lsq_distance(RA, pA, hA, RB, pB, hB):
    """min |RA u - RB v + (pA - pB)| over |u| <= hA, |v| <= hB (scipy's bounded least squares)."""
    r = lsq_linear(np.hstack([RA, -RB]), pB - pA, bounds=(np.r_[-hA, -hB], np.r_[hA, hB]), method='bvls', tol=1e-14)
    return float(np.linalg.norm(r.fun))


def test_reference_matches_least_squares_and_support_functions():
    rng = np.random.default_rng(0)
    K = 2000
    hA, hB = rng.uniform(0.02, 0.5, (K, 3)), rng.uniform(0.02, 0.5, (K, 3))
    RA, RB = Rotation.random(K, random_state=1).as_matrix(), Rotation.random(K, random_state=2).as_matrix()
    pA = rng.uniform(-1, 1, (K, 3))
    pB = pA + rng.normal(size=(K, 3)) * rng.uniform(0.1, 0.9, (K, 1))
    r = np_closest.box_pairs(RA, pA, hA, RB, pB, hB)
    sep = r['d'] > 0
    assert 0.2 < sep.mean() < 0.8, sep.mean()
    dirs = Rotation.random(1000, random_state=3).apply([1.0, 0.0, 0.0])
    for k in range(K):
        if sep[k]:
            assert abs(_lsq_distance(RA[k], pA[k], hA[k], RB[k], pB[k], hB[k]) - r['d'][k]) <= 1e-9, k
            continue
        depth, n = -r['d'][k], r['normal'][k]
        out = _lsq_distance(RA[k], pA[k] + (depth + 1e-4) * n, hA[k], RB[k], pB[k], hB[k])
        assert abs(out - 1e-4) <= 1e-8, (k, out)
        assert _lsq_distance(RA[k], pA[k] + (depth - 1e-4) * n, hA[k], RB[k], pB[k], hB[k]) <= 1e-10, k
        # overlap of the projections on every sampled direction: support(A) + support(B) - |u.(pA - pB)|
        ov = np.abs(dirs @ RA[k]) @ hA[k] + np.abs(dirs @ RB[k]) @ hB[k] - np.abs(dirs @ (pA[k] - pB[k]))
        assert ov.min() >= depth - 1e-9, k


# ------------------------------------------------------------------ the kernel against the reference
def _check(m, states, culled_too=True):
    """Every query set at every max distance on every state: the emulated kernel against np_closest.  A query whose pair
    rounding can decide may report another pair than the reference (its distance is still checked); at most 2 % of each
    set's queries over all states do.  (Ambiguous queries that agree are not capped: two colliders of one body resting
    on coplanar faces tie exactly in every reset state.)  Culling on and off give the same bits."""
    tables = [np_closest.pair_table(m, st) for st in states]
    for name, qs in np_closest.query_sets(m).items():
        mk = np_closest.masks(m, qs)
        for md in MAX_DISTANCES:
            out = emu_closest.closest_points(m, states, mk, md)
            if culled_too:
                off = emu_closest.closest_points(m, states, mk, md, cull=False)
                assert all(out[k].tobytes() == off[k].tobytes() for k in out), (name, md)
            namb = 0
            for i, st in enumerate(states):
                a, bad = np_closest.check_env(m, st, mk, {k: v[i] for k, v in out.items()}, md, tables[i])
                assert not bad, (name, md, i, bad[:4])
                namb += a
            assert namb <= 0.02 * len(states) * len(mk), (name, md, namb)


@pytest.mark.parametrize('env_id', [PLAY, 'pandaPlayAbsRPY1Obj-v0', 'pandaPick-v0'])
def test_emu_closest_match_numpy_reset_states(env_id):
    m, states = _states(env_id, 3, seed=41)
    _check(m, states)


@pytest.mark.parametrize('golden', ['heavy_step_r1.npz', 'many_contacts.npz'])
def test_emu_closest_match_numpy_golden_states(golden):
    _check(load_model(PLAY), np.load(os.path.join(GOLDEN, golden))['state'][:6])


def test_emu_closest_match_numpy_stepped_states():
    """After 12 steps, the gripper closed over the last 6: blocks resting on pads in part, tilted on an edge, in the
    fingers -- the witness cases a reset state does not show."""
    m = load_model(PLAY)
    sim = EmuSim(m, 32, seed=23)
    sim.reset()
    rng = np.random.default_rng(23)
    for k in range(12):
        a = random_actions(rng, 32, PLAY)
        if k >= 6:
            a[:, -1] = -1.0
        sim.step(a)
    _check(m, sim.state[:, :sim.state_dim].copy())


# ------------------------------------------------------------------ known answers on two boxes
C = np.array([0.25, -0.5, 1.0])
S2 = np.sqrt(0.5)


def _two_boxes(poses):
    """The play world with two of its static colliders replaced by boxes (pos relative to C, rot, half extents): model,
    state, [(pose of A, pose of B)] in closest_points' mask form, the two indices."""
    m0 = load_model(PLAY)
    n = int(m0['n_col'])
    ia, ib = [c for c in range(n) if m0['col_body'][c] < 0][:2]
    out = []
    for pa, pb in poses:
        m = load_model(PLAY)
        for k in ('col_pos', 'col_half', 'col_rot'):
            m.d[k] = m[k].copy()
        for c, (p, R, h) in ((ia, pa), (ib, pb)):
            m.d['col_pos'].reshape(n, 3)[c] = C + np.asarray(p, float)
            m.d['col_rot'].reshape(n, 3, 3)[c] = R
            m.d['col_half'].reshape(n, 3)[c] = h
        out.append(m)
    _, st = _states(PLAY, 1, seed=3)
    return out, st, ia, ib


def _rx(a):
    return Rotation.from_euler('x', a, degrees=True).as_matrix()


def _ry(a):
    return Rotation.from_euler('y', a, degrees=True).as_matrix()


def test_known_answers_two_boxes():
    I = np.eye(3)
    cube = np.array([0.5, 0.5, 0.5])
    small = np.array([0.25, 0.25, 0.25])
    zA, hB = 0.5 * np.sqrt(2.0), 0.25 * np.sqrt(2.0)          # heights of the top edge of A and bottom edge of B
    # (A pose, B pose, max_distance, expected d (None: miss), normal, pa, pb (None: check the invariants only))
    cases = [
        (((0, 0, 0), I, cube), ((1.0, 0, 0), I, small), 1.0, 0.25, (-1, 0, 0), None, None),          # axis-aligned gap
        (((0, 0, 0), I, cube), ((1.0, 1.0, 1.0), I, small), 1.0, 0.25 * np.sqrt(3.0), -np.ones(3) / np.sqrt(3.0),
         (0.5, 0.5, 0.5), (0.75, 0.75, 0.75)),                                                        # corner to corner
        (((0, 0, 0), _rx(45), cube), ((0, 0, zA + hB + 0.1), _ry(45), small), 1.0, 0.1, (0, 0, -1),
         (0, 0, zA), (0, 0, zA + 0.1)),                                                               # skewed edges
        (((0, 0, 0), I, cube), ((0.3, 0.1, 1.0), I, small), 1.0, 0.25, (0, 0, -1), None, None),       # parallel faces
        (((0, 0, 0), I, cube), ((0.1, -0.05, 0.6875), I, small), 1.0, -0.0625, (0, 0, -1), None, None),   # face overlap
        (((0, 0, 0), _rx(45), cube), ((0, 0, zA + hB - 0.01), _ry(45), small), 1.0, -0.01, (0, 0, -1),
         (0, 0, zA), (0, 0, zA - 0.01)),                                                              # edge-cross overlap
        (((0, 0, 0), I, (0.5, 0.375, 0.25)), ((0, 0, 0), I, (0.5, 0.375, 0.25)), 1.0, -0.5, (0, 0, 1), None, None),  # coincident
        (((0, 0, 0), I, cube), ((1.0, 0, 0), I, small), 0.25, 0.25, (-1, 0, 0), None, None),          # exactly at max
        (((0, 0, 0), I, cube), ((1.0, 0, 0), I, small), 0.2499, None, None, None, None),               # just beyond it
    ]
    models, st, ia, ib = _two_boxes([(c[0], c[1]) for c in cases])
    for k, (m, (_, _, md, d, n, pa, pb)) in enumerate(zip(models, cases)):
        out = emu_closest.closest_points(m, st, [(1 << ia, 1 << ib)], md)
        got = {f: v[0, 0] for f, v in out.items()}
        if d is None:
            assert got['collider_a'] == -1 and got['collider_b'] == -1 and got['distance'] == np.inf, k
            assert not got['position_on_a'].any() and not got['normal_on_b'].any(), k
            continue
        assert (got['collider_a'], got['collider_b']) == (ia, ib), k
        assert abs(got['distance'] - d) <= 1e-6, (k, got['distance'], d)
        assert np.abs(got['normal_on_b'] - np.asarray(n, float)).max() <= 1e-6, (k, got['normal_on_b'])
        if pa is not None:
            assert np.abs(got['position_on_a'] - C - pa).max() <= 1e-6, (k, got['position_on_a'] - C)
            assert np.abs(got['position_on_b'] - C - pb).max() <= 1e-6, (k, got['position_on_b'] - C)
        tab, geom = np_closest.pair_table(m, st[0])
        assert max(np_closest.witness_errors(geom, ia, ib, float(got['distance']), got['position_on_a'],
                                             got['position_on_b'], got['normal_on_b'])) <= 1e-6, k
        assert abs(tab['d'][ia, ib] - d) <= 1e-9, k
    # the edge-cross overlap's minimum axis is an edge cross in the reference
    tab, _ = np_closest.pair_table(models[5], st[0])
    assert tab['axis'][ia, ib] >= 6
    # the small box resting into the big one: its own deepest vertex, A's top face above it
    out = emu_closest.closest_points(models[4], st, [(1 << ia, 1 << ib)], 1.0)
    assert abs(out['position_on_a'][0, 0, 2] - C[2] - 0.5) <= 1e-6 and abs(out['position_on_b'][0, 0, 2] - C[2] - 0.4375) <= 1e-6
    # masks whose only pair is a == b
    out = emu_closest.closest_points(models[0], st, [(1 << ia, 1 << ia), (1 << ib, 1 << ib)], 10.0)
    assert (out['collider_a'] == -1).all() and (out['distance'] == np.inf).all()
    # swapping A and B: the same distance, the normal reversed
    out = emu_closest.closest_points(models[1], st, [(1 << ia, 1 << ib), (1 << ib, 1 << ia)], 10.0)
    assert out['distance'][0, 0] == out['distance'][0, 1]
    assert np.abs(out['normal_on_b'][0, 0] + out['normal_on_b'][0, 1]).max() <= 1e-6


# ------------------------------------------------------------------ invalid input, layout, the Python surface
def test_invalid_calls_are_rejected():
    m, states = _states(PLAY, 1, seed=1)
    q = [(1, 2)]
    nan = float('nan')
    bad = [(lib.PrbClosest(0, 0, 0.1, 0), 'num_queries'), (lib.PrbClosest(65, 0, 0.1, 0), 'num_queries'),
           (lib.PrbClosest(1, 1, 0.1, 0), 'reserved'), (lib.PrbClosest(1, 0, 0.1, 3), 'reserved'),
           (lib.PrbClosest(1, 0, nan, 0), 'max_distance'), (lib.PrbClosest(1, 0, float('inf'), 0), 'max_distance'),
           (lib.PrbClosest(1, 0, -0.01, 0), 'max_distance')]
    for c, word in bad:
        with pytest.raises(ValueError, match=word):
            emu_closest.closest_points(m, states, q, 0.1, call=c)
    for name in ('queries', 'collider_a', 'collider_b', 'distance'):
        with pytest.raises(ValueError, match='required'):
            emu_closest.closest_points(m, states, q, 0.1, null=(name,))
    out = emu_closest.closest_points(m, states, q, 0.1, null=('position_on_a', 'position_on_b', 'normal_on_b'))
    ref = emu_closest.closest_points(m, states, q, 0.1)
    assert all(out[k].tobytes() == ref[k].tobytes() for k in ('collider_a', 'collider_b', 'distance'))
    # bits >= n_col are ignored
    full = emu_closest.closest_points(m, states, [(~0, ~0)], 10.0)
    nc = int(m['n_col'])
    assert full['distance'].tobytes() == emu_closest.closest_points(m, states, [((1 << nc) - 1,) * 2], 10.0)['distance'].tobytes()


def test_struct_layout_matches_c(tmp_path):
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "prb.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu\\n",'
           ' sizeof(prb_closest), offsetof(prb_closest, reserved), offsetof(prb_closest, max_distance),'
           ' offsetof(prb_closest, reserved2), sizeof(prb_closest_query), offsetof(prb_closest_query, mask_a),'
           ' offsetof(prb_closest_query, mask_b));return 0;}\n')
    exe = str(tmp_path / 'prb_closest_probe')
    open(exe + '.c', 'w').write(src)
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', exe, exe + '.c'])
    got = list(map(int, subprocess.check_output([exe]).split()))
    C_, Q_ = lib.PrbClosest, lib.PrbClosestQuery
    assert got == [ctypes.sizeof(C_), C_.reserved.offset, C_.max_distance.offset, C_.reserved2.offset, ctypes.sizeof(Q_),
                   Q_.mask_a.offset, Q_.mask_b.offset]
    assert 'prb_closest_points' in lib.SYMBOLS


def test_check_closest():
    m = load_model(PLAY)
    nc = int(m['n_col'])
    body, link = np.asarray(m['col_body'])[:nc], np.asarray(m['col_urdf_link'])[:nc]
    qs, md = check_closest(m, [(0, -1), ((0, 18), 1)], 0.05)
    assert md == pytest.approx(0.05)
    assert qs[0] == (sum(1 << c for c in range(nc) if body[c] == 0), sum(1 << c for c in range(nc) if body[c] == -1))
    assert qs[1] == (sum(1 << c for c in range(nc) if body[c] == 0 and link[c] == 18), sum(1 << c for c in range(nc) if body[c] == 1))
    assert check_closest(m, [(0, 0)] * 64, 0)[1] == 0.0
    for queries, d in (([], 0.1), ([(0, 1)] * 65, 0.1), ([(99, 1)], 0.1), ([((0, 999), 1)], 0.1), ([('x', 1)], 0.1),
                       ([(True, 1)], 0.1), ([(0,)], 0.1), ([(0, 1)], float('nan')), ([(0, 1)], -1.0), ([(0, 1)], float('inf'))):
        with pytest.raises(ValueError):
            check_closest(m, queries, d)
