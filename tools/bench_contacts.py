"""Cost of the contact report (record_contacts) on one GPU; prints one JSON line.

    python tools/bench_contacts.py [--sizes 8192,65536] [--steps 20] [--rounds 5]

For each batch size one play handle runs the device-resident step (step_device, scripted actions) with the report off
and on, alternating in rounds of --steps steps timed with CUDA events, so that both see the same machine state.  Reports
the median ms per env step of each, the overhead, kernel launches per step of each, the report's device memory, and
the device name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def device_info(index):
    out = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = [x.strip() for x in out.split(',')]
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--env', default='UR5PlayAbsRPY1Obj-v0')
    ap.add_argument('--sizes', default='8192,65536')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=4)
    args = ap.parse_args()
    import torch
    from helpers import random_actions
    from roboticsplayroompybullet_b200.envs import make
    assert torch.cuda.is_available(), 'bench_contacts needs a GPU'
    res = {'env': args.env, 'steps': args.steps, 'rounds': args.rounds}
    for n in [int(x) for x in args.sizes.split(',')]:
        env = make(args.env, num_envs=n, seed=1234)
        env.reset()
        rng = np.random.default_rng(0)
        acts = [torch.as_tensor(random_actions(rng, n, args.env), device='cuda') for _ in range(8)]
        for on in (False, True):
            env.record_contacts = on
            for k in range(args.warmup):
                env.step_device(acts[k % len(acts)])
        torch.cuda.synchronize()
        ms = {False: [], True: []}
        launches = {}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):
            for on in (False, True):
                env.record_contacts = on
                l0 = env.launch_count()
                e0.record()
                for k in range(args.steps):
                    env.step_device(acts[k % len(acts)])
                e1.record()
                e1.synchronize()
                ms[on].append(e0.elapsed_time(e1) / args.steps)
                launches[on] = (env.launch_count() - l0) / args.steps
        off, on = float(np.median(ms[False])), float(np.median(ms[True]))
        res[str(n)] = {'step_ms_off': round(off, 3), 'step_ms_on': round(on, 3), 'overhead_pct': round(100 * (on / off - 1), 2),
                       'step_ms_off_all': [round(x, 3) for x in ms[False]], 'step_ms_on_all': [round(x, 3) for x in ms[True]],
                       'launches_per_step_off': launches[False], 'launches_per_step_on': launches[True],
                       'report_mb': round(n * (21 * 64 + 1) * 4 / 1e6, 1)}
        env.close()
        del env
        torch.cuda.empty_cache()
    res['device'], res['power_limit'] = device_info(torch.cuda.current_device())
    print(json.dumps(res))


if __name__ == '__main__':
    main()
