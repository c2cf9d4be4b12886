"""The two fixtures that reach the rarest paths of the step, run through the library built for the B200:

  tests/golden/heavy_step_r1.npz   48 states whose arm islands fill every size class of the arm-island solver
                                   (prb_pgs_arm_kernel, classes 0-4; class 4 reads the records beyond its stage in place);
  tests/golden/many_contacts.npz   17 states with 33-45 contacts after manifold reduction, four of them with more than 32
                                   overlapping collider pairs (the second narrow-phase pass, a lane writing two contact
                                   rows, the write-back of the second contact's impulses into the report).

The emulator runs these paths one fiber at a time, replaces the bulk-copy staging of the arm-island kernel with a loop and
does not contract FMAs; here they run with real races possible: against the fp64 oracle, tiled over 65 535 envs against a
65-env handle bit for bit, in the small-stage build (most records read in place) against the default build, and in the fused
A/B pipeline, whose 32-pair / 32-contact capacity they exceed, for its capacity counter."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import contacts_check as cc
from helpers import OBS_KEYS, SMALL_STAGE, compare_step, oracle_step_from
from oracle.oracle import Oracle
from roboticsplayroompybullet_b200.model import load_model
from test_gpu_parity import _record

pytestmark = pytest.mark.gpu

PLAY = 'UR5PlayAbsRPY1Obj-v0'
TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
FIXTURES = ['heavy_step_r1', 'many_contacts']
OUT_KEYS = OBS_KEYS + ['reward', 'is_success', 'target_poses']
N_TILED = 65535          # not a multiple of 32, of 8, or of any class's envs per bundle


def _golden(name):
    g = np.load(os.path.join(TESTS, 'golden', name + '.npz'))
    return g['state'], g['action']


def _all_states():
    """The 48 heavy states followed by the 17 many-contact states, with their actions."""
    sa = [_golden(f) for f in FIXTURES]
    return np.concatenate([s for s, _ in sa]), np.concatenate([a for _, a in sa])


def _tiling(n, seed=12):
    """Source state (0..64) of each of n envs: every state about n / 65 times, scattered by a seeded permutation so that
    copies land in different warps, blocks, bundles and list positions."""
    return np.random.default_rng(seed).permutation(n) % 65


def _outputs(obs, r, info):
    d = {k: np.asarray(obs[k]) for k in OBS_KEYS}
    d['reward'], d['is_success'], d['target_poses'] = np.asarray(r), np.asarray(info['is_success']), np.asarray(info['target_poses'])
    return d


def _step(env, act):
    obs, r, _, info = env.step(act)
    return _outputs(obs, r, info)


def _finite(out):
    return all(np.isfinite(np.asarray(v, np.float64)).all() for v in out.values())


def _make(n, **kw):
    from roboticsplayroompybullet_b200.envs import make
    return make(PLAY, num_envs=n, seed=1, **kw)


def _classes(use):
    """Per env: 0 light (no arm-island contact), k + 1 arm-island class k, in the last substep's setup launch."""
    return use[:, 0] & 0x7f


# ---------------------------------------------------------------------------------------------------------------- (a)
@pytest.mark.parametrize('name', FIXTURES)
def test_fixture_matches_oracle(name):
    """One env step of each fixture in a handle of exactly its size against the fp64 oracle from the same states, all keys,
    at the limits the emulator meets (tests/test_cpu_emu_parity.py: test_emu_solver_regression_bit_identical,
    test_emu_more_than_32_contacts); nothing dropped, everything finite.  The size classes of one substep must be the ones
    the emulator sees: heavy_step_r1 7 / 4 / 25 / 7 / 4 envs in arm classes 0..4, many_contacts 0 / 1 / 0 / 1 / 12."""
    st, act = _golden(name)
    n = len(st)
    m = load_model(PLAY)
    env = _make(n)
    env.set_state(st)
    env.substeps(1)
    per_class = np.bincount(_classes(env.debug_usage()), minlength=6)[1:6]
    env.set_state(st)
    obs, r, _, info = env.step(act)
    finite = _finite(_outputs(obs, r, info)) and np.isfinite(env.get_state()).all()
    overflow = env.overflow_count()
    env.close()
    outs = [oracle_step_from(m, st[i], act[i], Oracle)[0] for i in range(n)]
    res = compare_step(m, obs, r, info, outs, st, act, Oracle)
    _record('heavy_states_oracle[%s]' % name, dict(res, overflow=overflow, **{'class%d' % k: int(c) for k, c in enumerate(per_class)}))
    assert finite
    assert overflow == 0
    if name == 'heavy_step_r1':
        assert list(per_class) == [7, 4, 25, 7, 4], per_class
        assert res['bad_pose'] <= 2 and res['bad_reward'] <= 1, res       # the stiffest 0.1 % of the scripted workload
    else:
        assert list(per_class) == [0, 1, 0, 1, 12], per_class
        assert res['bad_pose'] == 0 and res['bad_vel'] == 0 and res['bad_reward'] == 0 and res['stiff'] <= 2, res


# ---------------------------------------------------------------------------------------------------------------- (b)
def _check_beyond_32(m, rep, states, advance, tol, skip=()):
    """For every env (but those in `skip`) where the oracle has more than 32 contacts: the report's contacts 33 and beyond
    are the oracle's, in order, within `tol` in geometry.  Returns the number of such envs."""
    many = 0
    for i, (row, adv) in enumerate(zip(states, advance)):
        if i in skip:
            continue
        o = Oracle(m)
        o.state[:] = np.asarray(row, np.float64)
        adv(o)
        ref, got = cc.oracle_report(o), cc.env_report(rep, i)
        if ref['count'] <= 32:
            continue
        many += 1
        assert cc.same_contacts(got, ref), (i, got['count'], ref['count'])
        tail, tail_ref = ({k: (v - 32 if k == 'count' else v[32:]) for k, v in r.items()} for r in (got, ref))
        assert cc.geometry_error(tail, tail_ref) <= tol, (i, cc.geometry_error(tail, tail_ref))
    return many


def test_many_contact_report_matches_oracle():
    """The contact report of the 17 many-contact states against the oracle, after one substep (geometry 1e-5) and after a
    full step (1e-4, with the fp32 probe), by the rules of test_cpu_contacts.test_report_matches_oracle.  After one substep
    five states have more than 32 contacts (the oracle's counts are 16 46 12 31 18 32 26 39 26 20 34 30 31 34 32 11 33), after
    the step all 17 do: contacts 33 and beyond come from the second row a lane writes and from its impulse write-back, and
    must be the oracle's in order and geometry, except in an env the conditioning rule accepts (none on the B200; under the
    emulator, after the step, state 11 reports one contact more than the oracle, which gains or loses it itself when its
    input moves by one fp32 ulp)."""
    st, act = _golden('many_contacts')
    n = len(st)
    m = load_model(PLAY)
    env = _make(n, record_contacts=True)
    stats = {}
    for full in (False, True):
        env.set_state(st)
        if full:
            env.step(act)
            adv = lambda a: (lambda o: o.step(np.asarray(a, np.float64)))
        else:
            env.substeps(1)
            adv = lambda a: (lambda o: o.substeps(1))
        rep = env.contacts()
        tol = 1e-4 if full else 1e-5
        bad = cc.check_invariants(m, rep)
        assert not bad, bad
        res = cc.compare(m, Oracle, rep, [(i, st[i], adv(act[i])) for i in range(n)], tol, f32_probe=full)
        assert not res['bad'], res
        assert res['cond'] <= (0.16 if full else cc.COND_SHARE) * n, res
        many = _check_beyond_32(m, rep, st, [adv(a) for a in act], tol, skip=res['cond_envs'])
        assert many >= (n - res['cond'] if full else 5), many
        assert (rep['count'] > 32).sum() >= (n if full else 5), rep['count']
        stats['step' if full else 'substep'] = {k: res[k] for k in ('n', 'cond', 'worst_geom', 'worst_force')}
        stats['step' if full else 'substep']['more_than_32'] = int((rep['count'] > 32).sum())
    assert env.overflow_count() == 0
    env.close()
    for k, v in stats.items():
        _record('heavy_states_report[%s]' % k, v)


# ---------------------------------------------------------------------------------------------------------------- (c)
@pytest.fixture(scope='module')
def ref65():
    """The 65 fixture states stepped once in a 65-env handle, report off and on; the same bits as the 48- and 17-env
    handles of test_fixture_matches_oracle give."""
    import torch
    st, act = _all_states()
    env = _make(65)
    env.set_state(st)
    off = _step(env, act)
    ref = {'out': off, 'state': env.get_state(), 'use': env.debug_usage()}
    env.record_contacts = True
    env.set_state(st)
    on = _step(env, act)
    for k in OUT_KEYS:
        assert np.array_equal(on[k], off[k]), k
    assert np.array_equal(env.get_state(), ref['state'])
    ref['rep'] = {k: v.clone() for k, v in env.contacts_device().items()}
    torch.cuda.synchronize()
    assert env.overflow_count() == 0
    env.close()
    lo = 0
    for name in FIXTURES:
        s, a = _golden(name)
        e = _make(len(s))
        e.set_state(s)
        o = _step(e, a)
        for k in OUT_KEYS:
            assert np.array_equal(o[k], off[k][lo:lo + len(s)]), (name, k)
        assert np.array_equal(e.get_state(), ref['state'][lo:lo + len(s)]), name
        e.close()
        lo += len(s)
    return ref


def test_tiled_heavy_batch_bit_identical(ref65):
    """65 535 envs, every one a copy of one of the 65 fixture states (about 1 008 copies each, scattered): every heavy-class
    queue and staging buffer runs full.  One step must give each env the bits its source state gets in the 65-env handle
    (outputs, state, debug_usage), with the report off and on, and the report must be the source's; three more steps
    keep the copies of one state bit-identical to each other.  Catches work-counter, bundle-staging, in-place read and
    write-back races that a sampled comparison cannot."""
    import torch
    st, act = _all_states()
    src = _tiling(N_TILED)
    assert np.bincount(src, minlength=65).min() >= 1008
    env = _make(N_TILED)
    # report off
    env.set_state(st[src])
    out = _step(env, act[src])
    state = env.get_state()
    use = env.debug_usage()
    for k in OUT_KEYS:
        assert np.array_equal(out[k], ref65['out'][k][src]), k
    assert np.array_equal(state, ref65['state'][src])
    assert np.array_equal(use, ref65['use'][src])
    assert env.overflow_count() == 0
    cls = _classes(use)
    assert (np.bincount(cls, minlength=6)[1:] > 0).all(), np.bincount(cls, minlength=6)
    # report on: the same bits, and each env reports what its source reports
    env.record_contacts = True
    env.set_state(st[src])
    out2 = _step(env, act[src])
    for k in OUT_KEYS:
        assert np.array_equal(out2[k], out[k]), k
    assert np.array_equal(env.get_state(), state)
    src_t = torch.as_tensor(src, device='cuda')
    rep = env.contacts_device()
    for k, v in rep.items():
        assert torch.equal(v, ref65['rep'][k][src_t]), k
    assert env.overflow_count() == 0
    # three more steps: copies of one state stay identical
    first = np.array([np.flatnonzero(src == s)[0] for s in range(65)])
    for _ in range(3):
        out3 = _step(env, act[src])
    state3 = env.get_state()
    assert np.isfinite(state3).all() and _finite(out3)
    assert np.array_equal(state3, state3[first[src]])
    for k in OUT_KEYS:
        assert np.array_equal(out3[k], out3[k][first[src]]), k
    rep = env.contacts_device()
    pick = torch.as_tensor(first[src], device='cuda')
    for k, v in rep.items():
        assert torch.equal(v, v[pick]), k
    assert env.overflow_count() == 0
    _record('heavy_states_tiled', {'n': N_TILED, **{'class%d' % k: int(c) for k, c in enumerate(np.bincount(cls, minlength=6)[1:])}})
    env.close()


# ---------------------------------------------------------------------------------------------------------------- (d)
def tiled_run(out_path, n):
    """One step of the 65 fixture states tiled to n envs with the report on, in this process's library (PRB_LIB): writes
    the outputs, the state after the step, the report and debug_usage after one substep and after the step."""
    st, act = _all_states()
    src = _tiling(n)
    env = _make(n, record_contacts=True)
    env.set_state(st[src])
    env.substeps(1)
    use1 = env.debug_usage()
    env.set_state(st[src])
    out = _step(env, act[src])
    rep = env.contacts()
    np.savez(out_path, src=src, state=env.get_state(), use1=use1, use=env.debug_usage(), overflow=env.overflow_count(),
             **{'out_' + k: v for k, v in out.items()}, **{'rep_' + k: v for k, v in rep.items()})
    env.close()


def _child(code, **env):
    e = dict(os.environ)
    for k, v in env.items():
        if v is None:
            e.pop(k, None)
        else:
            e[k] = v
    p = subprocess.run([sys.executable, '-c', 'import sys; sys.path[:0] = [%r, %r]\n' % (ROOT, TESTS) + code], env=e,
                       capture_output=True, text=True, timeout=1200)
    assert p.returncode == 0, p.stdout + p.stderr
    return p.stdout


def test_small_stage_build_bit_identical(tmp_path):
    """The small-stage build (tests/helpers.py SMALL_STAGE: arm-island classes of 104-120 q, free-body stage of 16 q), built
    with nvcc for sm_100a: nearly every heavy state lands in the last class and has most of its records read in place
    (45 of the 48 heavy states under the emulator, 4 in the default build).  The 65 fixture states tiled to 4 096 envs, so
    that every class has several bundles, must step to the same bits as in the default build: outputs, state, report."""
    sys.path.insert(0, ROOT)
    import __graft_entry__
    so = str(tmp_path / 'libprb_smallstage.so')
    __graft_entry__.compile_library(so, SMALL_STAGE)
    n = 4096
    runs = {}
    for tag, lib in (('default', None), ('small', so)):
        path = str(tmp_path / (tag + '.npz'))
        _child('from test_gpu_heavy_states import tiled_run\ntiled_run(%r, %d)\n' % (path, n), PRB_LIB=lib)
        runs[tag] = np.load(path)
    a, b = runs['default'], runs['small']
    for k in a.files:
        if k.startswith('use'):
            continue
        assert np.array_equal(a[k], b[k]), k
    assert int(a['overflow']) == 0 and int(b['overflow']) == 0
    src = a['src']
    heavy_copy = np.array([np.flatnonzero(src == s)[0] for s in range(48)])     # one copy of each heavy state
    c4 = {t: int((_classes(r['use1'])[heavy_copy] == 5).sum()) for t, r in runs.items()}
    _record('heavy_states_small_stage', {'n': n, 'class4_default': c4['default'], 'class4_small': c4['small']})
    assert c4['small'] >= 40 and c4['default'] <= 8, c4


# ---------------------------------------------------------------------------------------------------------------- (e)
def test_fused_pipeline_counts_overflow_once_per_env_step():
    """PRB_PIPELINE=fused (read when the handle is created: a child process).  The fused kernel holds 32 overlapping pairs
    and 32 contacts per env; each of the 17 many-contact states exceeds that in some substep of its step, so the capacity
    counter goes up by exactly 17 (once per env step, not per substep), a second step adds at most 17, and every output
    stays finite.  test_fixture_matches_oracle asserts 0 for the split pipeline on the same states."""
    code = ('import json, numpy as np\n'
            'from test_gpu_heavy_states import _golden, _make, _outputs, _finite\n'
            'from roboticsplayroompybullet_b200.lib import PrbError\n'
            'st, act = _golden("many_contacts")\n'
            'env = _make(len(st))\n'
            'try:\n    env.record_contacts = True\n    fused = False\nexcept PrbError:\n    fused = True\n'
            'env.set_state(st)\n'
            'counts, finite = [env.overflow_count()], True\n'
            'for _ in range(2):\n'
            '    obs, r, _, info = env.step(act)\n'
            '    counts.append(env.overflow_count())\n'
            '    finite = finite and _finite(_outputs(obs, r, info)) and bool(np.isfinite(env.get_state()).all())\n'
            'print("RESULT " + json.dumps({"fused": fused, "counts": counts, "finite": finite}))\n')
    out = _child(code, PRB_PIPELINE='fused')
    res = json.loads([l for l in out.splitlines() if l.startswith('RESULT ')][0][7:])
    _record('heavy_states_fused_overflow', {'step1': res['counts'][1] - res['counts'][0], 'step2': res['counts'][2] - res['counts'][1]})
    assert res['fused'], res                          # the child really ran the fused pipeline
    c = res['counts']
    assert c[0] == 0 and c[1] == 17 and c[2] - c[1] <= 17, c
    assert res['finite'], res
