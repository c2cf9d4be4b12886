"""Per-env dynamics (include/prb.h prb_dynamics) on the CPU SIMT emulator: the setup kernel with the table
(EmuSim(table=...), tests/emu/prb_emu.cpp) against itself without it, against emulator runs and oracle runs of models
patched to each env's values, against physics that shares no code with the kernels, and the randomization kernel."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import contacts_check as cc
from emu_dynamics import FIELDS, MODEL_FIELD, model_table
from emu_lib import EmuSim
from helpers import OBS_KEYS, compare_step, oracle_step_from, random_actions
from oracle.oracle import Oracle
from roboticsplayroompybullet_b200 import envs, lib
from roboticsplayroompybullet_b200.model import CompiledModel, load_model

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
PLAY = 'UR5PlayAbsRPY1Obj-v0'


def _rollout_states(env_id, n=4, steps=2, seed=5):
    m = load_model(env_id)
    sim = EmuSim(m, n, seed=seed)
    sim.reset()
    sd = sim.state_dim
    rng = np.random.default_rng(seed)
    st, act = [], []
    for _ in range(steps):
        sim.step(random_actions(rng, n, env_id))
        st.append(sim.state[:, :sd].copy()); act.append(random_actions(rng, n, env_id))
    return m, np.concatenate(st), np.concatenate(act)


def _inputs():
    sets = []
    for f in ('heavy_step_r1.npz', 'many_contacts.npz'):
        g = np.load(os.path.join(GOLDEN, f))
        sets.append((load_model(PLAY), g['state'], g['action']))
    for env_id in (PLAY, 'pandaPick-v0'):
        sets.append(_rollout_states(env_id))
    return sets


def _param_sets(m):
    """K = 8 rows: each field changed alone, all of them together, and the model's own values."""
    base = model_table(m, 1)
    row = lambda: {k: v[0].copy() for k, v in base.items()}
    out = []
    s = row(); s['lateral_friction'] *= np.float32(0.6); s['lateral_friction'][np.asarray(m['col_body'])[:m['n_col']] == 1] = 1.3; out.append(s)
    s = row(); s['spinning_friction'] += np.float32(0.02); out.append(s)
    s = row(); s['mass'] *= np.float32(2.5); out.append(s)
    s = row(); s['local_inertia_diagonal'] *= np.float32(0.4); out.append(s)
    s = row(); s['linear_damping'][:] = 0.7; out.append(s)
    s = row(); s['angular_damping'][:] = 0.9; out.append(s)
    s = {k: out[i][k] for i, k in enumerate(FIELDS)}; out.append({k: v.copy() for k, v in s.items()})
    out.append(row())
    return out


def _patched(m, s):
    """The model with the fp32 values of row s stored as float64 (the same fp32 after prb_convert.h's casts)."""
    d = dict(m.d)
    d.update(m.meta)
    for k, mk in MODEL_FIELD.items():
        a = np.array(m[mk], np.float64)
        v = np.asarray(s[k], np.float32).astype(np.float64).reshape(-1)
        a[:len(v)] = v
        d[mk] = a
    return CompiledModel(d)


def _table(sets, N):
    return {k: np.stack([sets[i % len(sets)][k] for i in range(N)]) for k in FIELDS}


def test_table_with_model_values_is_bit_identical():
    """Criterion 1: every output key and the state are the same bits with the table holding the model's values and with
    no table, over full steps of every input set."""
    for m, states, actions in _inputs():
        N = len(states)
        off, on = EmuSim(m, N), EmuSim(m, N, table=model_table(m, N))
        for s in (off, on):
            s.set_state(states)
        for _ in range(2):
            a, b = off.step(actions), on.step(actions)
            assert np.array_equal(off.state, on.state)
            for k in a:
                assert np.array_equal(a[k], b[k]), k


def test_per_env_equals_per_model():
    """Criterion 2: env i runs parameter set i % 8; it matches, bit for bit, a run of the model patched to that set."""
    for m, states, actions in _inputs():
        sets = _param_sets(m)
        K, N = len(sets), len(states)
        sim = EmuSim(m, N, table=_table(sets, N))
        sim.set_state(states)
        out = sim.step(actions)
        for k in range(K):
            idx = np.arange(k, N, K)
            if len(idx) == 0:
                continue
            ref = EmuSim(_patched(m, sets[k]), len(idx))
            ref.set_state(states[idx])
            ro = ref.step(actions[idx])
            assert np.array_equal(sim.state[idx], ref.state), k
            for key in ro:
                assert np.array_equal(out[key][idx], ro[key]), (k, key)


def _oracle_check(m, sets, states, actions, out, rng):
    K = len(sets)
    outs = [oracle_step_from(_patched(m, sets[i % K]), states[i], actions[i], Oracle)[0] for i in range(len(states))]
    # the conditioning rule perturbs the oracle of each env's own patched model
    res = {'n': 0, 'bad_pose': 0, 'bad_vel': 0, 'bad_flags': 0, 'bad_reward': 0, 'stiff': 0}
    for i in range(len(states)):
        pm = _patched(m, sets[i % K])
        r = compare_step(pm, {k: out[k][i:i + 1] for k in OBS_KEYS}, out['reward'][i:i + 1, 0],
                         {'is_success': out['is_success'][i:i + 1, 0]}, [outs[i]], states[i:i + 1], actions[i:i + 1], Oracle, rng)
        for k in res:
            res[k] += r[k]
    return res


def test_oracle_parity_one_step():
    """Criterion 3: one step of every input set with the 8 parameter sets against the oracle of each env's patched
    model, judged by helpers.compare_step (tolerances and the ulp_spread conditioning rule)."""
    rng = np.random.default_rng(0)
    for m, states, actions in _inputs():
        sets = _param_sets(m)
        N = len(states)
        sim = EmuSim(m, N, table=_table(sets, N))
        sim.set_state(states)
        out = sim.step(actions)
        res = _oracle_check(m, sets, states, actions, out, rng)
        assert res['bad_pose'] == res['bad_vel'] == res['bad_flags'] == res['bad_reward'] == 0, res


def test_oracle_parity_rollout():
    """Criterion 3: a 30-step open-loop rollout of the play world, 8 envs with the 8 parameter sets; every step is
    compared with the patched oracle from the same state."""
    m = load_model(PLAY)
    sets = _param_sets(m)
    N = len(sets)
    base = EmuSim(m, N, seed=21)
    base.reset()
    sd = base.state_dim
    sim = EmuSim(m, N, table=_table(sets, N))
    sim.set_state(base.state[:, :sd])
    rng, crng = np.random.default_rng(4), np.random.default_rng(1)
    stiff = 0
    for _ in range(30):
        st = sim.state[:, :sd].copy()
        a = random_actions(rng, N, PLAY)
        out = sim.step(a)
        res = _oracle_check(m, sets, st, a, out, crng)
        assert res['bad_pose'] == res['bad_vel'] == res['bad_flags'] == res['bad_reward'] == 0, res
        stiff += res['stiff']
    assert stiff <= 0.05 * 30 * N, stiff


def _block_on_table(m, N, table, report=False):
    """N copies of a play env with the block parked at rest on the table top, far from the arm, settled with `table`."""
    base = EmuSim(m, 1, seed=2)
    base.reset()
    f0 = 5 * m['nd']
    st = np.repeat(base.state[:, :base.state_dim], N, 0)
    st[:, f0:f0 + 3] = [0.0, 0.18, st[0, f0 + 2]]
    st[:, f0 + 3:f0 + 7] = [0, 0, 0, 1]
    st[:, f0 + 7:f0 + 13] = 0
    sim = EmuSim(m, N, report=report, table=table)
    sim.set_state(st)
    sim.substeps(60)
    return sim, f0


def test_sliding_block_decelerates_at_its_own_friction():
    """Criterion 4: a block sliding on the table decelerates at mu_block mu_table g within 2 %, for five per-env block
    frictions (linear damping 0 in the table, so that friction alone acts)."""
    m = load_model(PLAY)
    mus = np.array([0.3, 0.5, 0.8, 1.0, 1.4], np.float32)
    N = len(mus)
    t = model_table(m, N)
    body = np.asarray(m['col_body'])[:m['n_col']]
    t['lateral_friction'][:, body == 1] = mus[:, None]
    t['linear_damping'][:] = 0
    sim, f0 = _block_on_table(m, N, t)
    table_mu = np.float32(m['col_friction'][int(np.nonzero(body == -1)[0][0])])
    sim.state[:, f0 + 7] = 0.8
    v0 = sim.state[:, f0 + 7].astype(np.float64)
    n, dt, g = 12, m.param('dt'), -m.param('gravity_z')
    sim.substeps(1)                     # the first substep also absorbs the settle residual
    v1 = sim.state[:, f0 + 7].astype(np.float64)
    sim.substeps(n)
    v = sim.state[:, f0 + 7].astype(np.float64)
    dec = (v1 - v) / (n * dt)
    ref = np.minimum(mus * table_mu, 10.0) * g
    assert (v > 0.1).all() and (v0 > v1).all()
    assert np.abs(dec - ref).max() <= 0.02 * ref.max(), (dec, ref)
    assert (np.abs(dec - ref) <= 0.02 * ref).all(), (dec, ref)


def test_resting_block_carries_its_own_weight():
    """Criterion 4: with the contact report on, a block at rest on the table carries m_e g within 1 % for five per-env
    masses (inertia scaled with the mass)."""
    m = load_model(PLAY)
    scale = np.array([0.3, 0.7, 1.0, 2.0, 4.0], np.float32)
    N = len(scale)
    t = model_table(m, N)
    t['mass'][:, 0] *= scale
    t['local_inertia_diagonal'][:, 0] *= scale[:, None]
    sim, _ = _block_on_table(m, N, t, report=True)
    sim.substeps(1)
    rep = sim.contacts()
    g = abs(m.param('gravity_z'))
    for i in range(N):
        mg = float(t['mass'][i, 0]) * g
        fz = cc.block_vertical_force(m, rep, i, 1)
        assert abs(fz - mg) <= 0.01 * mg, (i, fz, mg)


def test_free_flight_with_per_env_damping():
    """Criterion 4: free flight of the block with per-env linear and angular damping follows the fp64 semi-implicit
    recurrence v' = v + dt (g - (k + k |v|) v), p' = p + dt v' (linear) and the same for a spin about a principal axis,
    where the gyroscopic term vanishes."""
    m = load_model(PLAY)
    damp = np.array([[0.0, 0.0], [0.04, 0.1], [0.5, 0.3], [2.0, 1.0]], np.float32)
    N = len(damp)
    base = EmuSim(m, 1, seed=1)
    base.reset()
    f0 = 5 * m['nd']
    st = np.repeat(base.state[:, :base.state_dim], N, 0)
    st[:, f0:f0 + 3] = [0.0, 0.2, 1.0]
    st[:, f0 + 3:f0 + 7] = [0, 0, 0, 1]
    st[:, f0 + 7:f0 + 13] = [0.3, -0.1, 0.5, 0.0, 0.0, 6.0]
    t = model_table(m, N)
    t['linear_damping'][:, 0] = damp[:, 0]
    t['angular_damping'][:, 0] = damp[:, 1]
    sim = EmuSim(m, N, table=t)
    sim.set_state(st)
    dt, g = m.param('dt'), np.array([0, 0, m.param('gravity_z')])
    v = st[:, f0 + 7:f0 + 10].astype(np.float64)
    p = st[:, f0:f0 + 3].astype(np.float64)
    w = st[:, f0 + 12].astype(np.float64)
    kl, ka = damp[:, 0].astype(np.float64), damp[:, 1].astype(np.float64)
    for _ in range(60):
        sim.substeps(1)
        v = v + dt * (g - (kl + kl * np.linalg.norm(v, axis=1))[:, None] * v)
        p = p + dt * v
        w = w + dt * (-(ka + ka * np.abs(w)) * w)
        s = sim.state[:, :sim.state.shape[1]].astype(np.float64)
        assert np.abs(s[:, f0 + 7:f0 + 10] - v).max() < 2e-5
        assert np.abs(s[:, f0:f0 + 3] - p).max() < 2e-4
        assert np.abs(s[:, f0 + 12] - w).max() < 2e-4 * 6
    assert sim.state[3, f0 + 12] < 0.9 * sim.state[0, f0 + 12]          # the damping acted


# ------------------------------------------------------------------ randomization kernel
def _rsim(m, N, counters, seed=77, env_offset=0):
    sim = EmuSim(m, N, table=model_table(m, N), seed=seed, env_offset=env_offset)
    o_cnt = Oracle(m).state_dim - 1
    sim.state[:, o_cnt] = counters
    return sim


RANGES = {'lateral_friction': (0.5, 1.5), 'spinning_friction': (0.2, 3.0), 'mass': (0.5, 2.0), 'linear_damping': (0.0, 4.0),
          'angular_damping': (0.9, 1.1)}


@pytest.mark.parametrize('env_id', [PLAY, 'pandaPick-v0'])
def test_randomize_ranges_and_sharing(env_id):
    """Values lie in fl(model lo)..fl(model hi); friction shares one draw per body, mass / damping one per free body, and
    the inertia takes its mass's draw."""
    m = load_model(env_id)
    N = 64
    sim = _rsim(m, N, np.arange(N) % 5)
    sim.randomize(RANGES)
    t, base = sim.table(), model_table(m, N)
    for k, mk in MODEL_FIELD.items():
        lo, hi = RANGES['mass' if k == 'local_inertia_diagonal' else k]
        b = base[k]
        assert (t[k] >= b * np.float32(lo)).all() and (t[k] <= b * np.float32(hi)).all(), k
    body = np.asarray(m['col_body'])[:m['n_col']]
    for k in ('lateral_friction', 'spinning_friction'):
        nz = base[k][0] > 0
        s = np.where(nz, t[k] / np.where(nz, base[k], 1), np.nan)
        for bd in np.unique(body):
            sel = (body == bd) & nz
            if sel.sum() > 1:
                assert (np.nanmax(s[:, sel], 1) - np.nanmin(s[:, sel], 1)).max() < 1e-6, (k, bd)
        assert np.unique(np.round(s[:, nz], 5)).size >= N            # draws differ between envs
    ratio = (t['local_inertia_diagonal'] / base['local_inertia_diagonal']) / (t['mass'] / base['mass'])[:, :, None]
    assert np.abs(ratio - 1).max() < 1e-6


def test_randomize_unit_range_mask_determinism():
    """(1, 1) gives the model's values exactly; masked-out envs are untouched; the same (seed, env_offset + e, reset
    counter) gives the same draw whatever the batch size and offset; another reset counter gives another draw."""
    m = load_model(PLAY)
    N = 12
    cnt = np.arange(N) % 4 + 3
    sim = _rsim(m, N, cnt)
    sim.randomize(RANGES)
    sim.randomize({})
    for k, v in model_table(m, N).items():
        assert np.array_equal(sim.table()[k], v), k
    sim.randomize(RANGES)
    full = sim.table()
    # a shard: rows 5..9 at env_offset 5 in a batch of 5
    shard = _rsim(m, 5, cnt[5:10], env_offset=5)
    shard.randomize(RANGES)
    for k in FIELDS:
        assert np.array_equal(shard.table()[k], full[k][5:10]), k
    # mask: only the odd envs draw again, with a new reset counter
    mask = (np.arange(N) % 2).astype(np.uint8)
    o_cnt = Oracle(m).state_dim - 1
    sim.state[:, o_cnt] += 1
    sim.randomize(RANGES, mask)
    t = sim.table()
    for k in FIELDS:
        assert np.array_equal(t[k][mask == 0], full[k][mask == 0]), k
    assert not np.array_equal(t['mass'][mask == 1], full['mass'][mask == 1])
    assert (t['mass'][mask == 1] != full['mass'][mask == 1]).all()
    # and a different seed draws differently
    other = _rsim(m, N, cnt, seed=78)
    other.randomize(RANGES)
    assert (other.table()['mass'] != full['mass']).all()


# ------------------------------------------------------------------ Python surface (no GPU)
def test_struct_layout_matches_c(tmp_path):
    """ctypes mirrors of prb_dynamics and prb_dynamics_ranges == what a C compiler lays out."""
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "prb.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu\\n",'
           ' sizeof(prb_dynamics), offsetof(prb_dynamics, angular_damping), offsetof(prb_dynamics, num_envs),'
           ' offsetof(prb_dynamics, n_free), sizeof(prb_dynamics_ranges), offsetof(prb_dynamics_ranges, mass),'
           ' offsetof(prb_dynamics_ranges, angular_damping));return 0;}\n')
    exe = str(tmp_path / 'prb_dynamics_probe')
    open(exe + '.c', 'w').write(src)
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', exe, exe + '.c'])
    got = list(map(int, subprocess.check_output([exe]).split()))
    D, R = lib.PrbDynamics, lib.PrbDynamicsRanges
    assert got == [ctypes.sizeof(D), D.angular_damping.offset, D.num_envs.offset, D.n_free.offset, ctypes.sizeof(R),
                   R.mass.offset, R.angular_damping.offset]
    assert [f for f, _ in D._fields_[:6]] == FIELDS


def test_change_dynamics_targets():
    """(body, link) -> colliders and free body, as contacts() reports them, and the ValueErrors."""
    m = load_model(PLAY)
    nc = m['n_col']
    body, link = np.asarray(m['col_body'])[:nc], np.asarray(m['col_urdf_link'])[:nc]
    for b in np.unique(body):
        for l in np.unique(link[body == b]):
            cols, fb = envs.dynamics_target(m, int(b), int(l))
            assert set(cols) == set(np.nonzero((body == b) & (link == l))[0])
            assert fb == (b - 1 if 1 <= b <= m['n_free'] else None)
    cols, fb = envs.dynamics_target(m, 1)
    assert fb == 0 and (body[cols] == 1).all()
    cols, fb = envs.dynamics_target(m, 0, 17)
    assert len(cols) == 2 and fb is None
    for b, l in ((0, 7), (9, -1), (1, 0), (-1, 3)):
        with pytest.raises(ValueError):
            envs.dynamics_target(m, b, l)
    N = 4
    assert envs.check_dynamics_value('mass', 0.5, N).shape == (N,)
    assert envs.check_dynamics_value('local_inertia_diagonal', [1e-4, 2e-4, 3e-4], N).shape == (N, 3)
    assert envs.check_dynamics_value('lateral_friction', np.arange(N), N).dtype == np.float32
    for f, v in (('mass', 0.0), ('mass', -1.0), ('local_inertia_diagonal', [1, 0, 1]), ('lateral_friction', -0.1),
                 ('linear_damping', -1e-3), ('angular_damping', np.nan), ('spinning_friction', np.inf), ('mass', [1.0, 2.0])):
        with pytest.raises(ValueError):
            envs.check_dynamics_value(f, v, N)


def test_randomize_ranges_validation():
    r = envs.dynamics_ranges({'mass': (0.5, 2.0)})
    assert tuple(r.mass) == (0.5, 2.0) and tuple(r.lateral_friction) == (1.0, 1.0)
    for bad in ({'mass': (0.0, 1.0)}, {'mass': (2.0, 1.0)}, {'lateral_friction': (-0.1, 1.0)}, {'linear_damping': (0, np.inf)},
                {'angular_damping': (np.nan, 1.0)}, {'gravity': (1, 1)}):
        with pytest.raises(ValueError):
            envs.dynamics_ranges(bad)
    assert tuple(envs.dynamics_ranges({'linear_damping': (0.0, 0.0)}).linear_damping) == (0.0, 0.0)
