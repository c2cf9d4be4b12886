"""Ray casting throughput (prb_ray_test) on one GPU; prints one JSON line per workload.

    python tools/bench_rays.py [--calls 60] [--warmup 5]

Workloads (UR5PlayAbsRPY1Obj-v0 after scripted steps, so the arm is not at its reset pose):
  a  65 536 envs x 1 per-env world ray (the gripper ray of every env)   warp-per-env launch shape
  b  65 536 envs x 64 shared rays in site 0 (the 8 x 8 fan)             block-per-env launch shape
  c  8 192 envs x 1 024 shared world rays (the 32 x 32 height scan)     block-per-env, one chunk
Each call is timed by its own pair of CUDA events with L2 flushed (a 256 MB fill) before it, outside the pair; the
median and the spread (min, max) over --calls calls after --warmup untimed calls.  rays/s is N R / median; box tests per
ray is the number of colliders the mask lets through (the kernel tests every one).  The device name and power limit
are read in the same run."""
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
    ap.add_argument('--calls', type=int, default=60)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--envs', type=int, default=65536)
    ap.add_argument('--envs-c', type=int, default=8192)
    args = ap.parse_args()
    import torch
    import np_rays
    from helpers import random_actions
    from roboticsplayroompybullet_b200.envs import make
    assert torch.cuda.is_available(), 'bench_rays needs a GPU'
    env_id = 'UR5PlayAbsRPY1Obj-v0'
    name, power = device_info(torch.cuda.current_device())
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device='cuda')    # > 126 MB L2

    def bench(env, frm, to, site, tag):
        f, t = (torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float32, device='cuda') for x in (frm, to))
        for _ in range(args.warmup):
            env.ray_test_batch_device(f, t, site=site)
        ms = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for k in range(args.calls):
            flush.fill_(float(k))
            e0.record()
            out = env.ray_test_batch_device(f, t, site=site)
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = float(np.median(ms))
        N, R = env.num_envs, frm.shape[-2]
        hit = float((out['collider'] >= 0).float().mean())
        line = {'workload': tag, 'env': env_id, 'num_envs': N, 'rays_per_env': R, 'per_env': frm.ndim == 3,
                'frame': 'world' if site is None else 'site %d' % site, 'median_ms': round(med, 4),
                'min_ms': round(min(ms), 4), 'max_ms': round(max(ms), 4), 'rays_per_s': N * R / (med * 1e-3),
                'box_tests_per_ray': int(env.model['n_col']), 'hit_fraction': round(hit, 4), 'calls': args.calls,
                'l2_flushed': True, 'device': name, 'power_limit': power}
        print(json.dumps(line), flush=True)

    rng = np.random.default_rng(0)
    for n, shapes in ((args.envs, 'ab'), (args.envs_c, 'c')):
        env = make(env_id, num_envs=n, seed=1234)
        env.reset()
        for k in range(4):
            env.step_device(torch.as_tensor(random_actions(rng, n, env_id), device='cuda'))
        torch.cuda.synchronize()
        st = env.get_state()
        if 'a' in shapes:
            rays = [np_rays.proprio_ray(env.model, st[i]) for i in range(0, n, max(1, n // 1024))]
            idx = np.arange(n) % len(rays)                      # gripper rays of a sample of envs, tiled
            frm = np.stack([rays[i][0] for i in idx])[:, None, :]
            to = np.stack([rays[i][1] for i in idx])[:, None, :]
            bench(env, frm, to, None, 'a')
        if 'b' in shapes:
            bench(env, *np_rays.site_fan(), 0, 'b')
        if 'c' in shapes:
            bench(env, *np_rays.height_scan(env.model), None, 'c')
        env.close()
        del env
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
