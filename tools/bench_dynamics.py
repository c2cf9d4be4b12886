"""Cost of the per-env dynamics table (per_env_dynamics) on one GPU; prints one JSON line and appends it to
profiles/r3_bench_dynamics.jsonl (--out).

    python tools/bench_dynamics.py [--sizes 8192,65536] [--steps 20] [--rounds 5]

For each batch size one play handle runs the device-resident step (step_device, scripted actions) in three modes,
alternating in rounds of --steps steps timed with CUDA events, so that all see the same machine state:
  off         no table (the model's dynamics)
  defaults    table on, every row the model's values: against `off` this is the cost of the lookups
  randomized  table on after a draw with lateral friction (0.5, 1.5) and mass (0.5, 2.0): different physics, so a
              workload of its own rather than an overhead
Reports the median ms per env step of each mode, the spread of the rounds, launches per step, the table's device
memory, and the device name and power limit read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

MODES = ('off', 'defaults', 'randomized')
RANGES = {'lateral_friction': (0.5, 1.5), 'mass': (0.5, 2.0)}


def device_info(index):
    out = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = [x.strip() for x in out.split(',')]
    return name, power


def set_mode(env, mode, ranges):
    env.per_env_dynamics = False
    if mode != 'off':
        env.per_env_dynamics = True              # off -> on: the model's values
    if mode == 'randomized':
        from roboticsplayroompybullet_b200 import lib
        lib.check(env.L, env._h, env.L.prb_randomize_dynamics(env._h, ctypes.byref(ranges), None, env._stream()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--env', default='UR5PlayAbsRPY1Obj-v0')
    ap.add_argument('--sizes', default='8192,65536')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=4)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r3_bench_dynamics.jsonl'))
    args = ap.parse_args()
    import torch
    import bench
    from roboticsplayroompybullet_b200.envs import dynamics_ranges, make
    assert torch.cuda.is_available(), 'bench_dynamics needs a GPU'
    ranges = dynamics_ranges(RANGES)
    res = {'env': args.env, 'steps': args.steps, 'rounds': args.rounds, 'ranges': RANGES}
    for n in [int(x) for x in args.sizes.split(',')]:
        env = make(args.env, num_envs=n, seed=1234)
        o0 = env.reset_device()
        acts = torch.as_tensor(bench.synth_actions(np.random.default_rng(0), n, args.steps, args.env,
                                                   block_xyz=o0['achieved_goal'][:, :3].cpu().numpy(),
                                                   ee_xyz=o0['obs_quat'][:, :3].cpu().numpy())).cuda()
        for mode in MODES:
            set_mode(env, mode, ranges)
            for k in range(args.warmup):
                env.step_device(acts[k])
        torch.cuda.synchronize()
        ms = {m: [] for m in MODES}
        launches = {}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):
            for mode in MODES:
                set_mode(env, mode, ranges)
                torch.cuda.synchronize()
                l0 = env.launch_count()
                e0.record()
                for k in range(args.steps):
                    env.step_device(acts[k])
                e1.record()
                e1.synchronize()
                ms[mode].append(e0.elapsed_time(e1) / args.steps)
                launches[mode] = (env.launch_count() - l0) / args.steps
        med = {m: float(np.median(ms[m])) for m in MODES}
        nc, nf = int(env.model['n_col']), int(env.model['n_free'])
        r = {'step_ms_' + m: round(med[m], 3) for m in MODES}
        r.update({'step_ms_%s_all' % m: [round(x, 3) for x in ms[m]] for m in MODES})
        r['defaults_vs_off_pct'] = round(100 * (med['defaults'] / med['off'] - 1), 2)
        r['randomized_vs_off_pct'] = round(100 * (med['randomized'] / med['off'] - 1), 2)
        r.update({'launches_per_step_' + m: launches[m] for m in MODES})
        r['table_mb'] = round(n * (2 * nc + 6 * nf) * 4 / 1e6, 1)
        res[str(n)] = r
        env.close()
        del env
        torch.cuda.empty_cache()
    res['device'], res['power_limit'] = device_info(torch.cuda.current_device())
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'a') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
