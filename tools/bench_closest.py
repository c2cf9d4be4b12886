"""Closest-points throughput (prb_closest_points) on one GPU; prints one JSON line per workload.

    python tools/bench_closest.py [--calls 60] [--warmup 5]

Workloads (UR5PlayAbsRPY1Obj-v0 after scripted steps, so the arm is not at its reset pose; bodies: -1 static scene,
0 arm, 1 block, 2 drawer, 3 door, 4 button, 5 dial):
  a  65 536 envs x 1 query: arm vs block, max 0.2 m
  b  65 536 envs x 8 queries: arm vs static, arm vs each of the 5 movable bodies, block vs static, drawer vs static,
     max 0.05 m
  c  8 192 envs x 42 queries: every ordered pair of distinct bodies, max 10 m (culling by max_distance removes nothing)
Each call is timed by its own pair of CUDA events with L2 flushed (a 256 MB fill) before it, outside the pair; the
median and the spread (min, max) over --calls calls after --warmup untimed calls.  pairs_per_query is the number of
(a, b) pairs the masks give; exact_per_query the number the kernel's culling keeps for the exact test, recomputed here
in fp64 from the same bounds on a sample of envs (the kernel does not count).  The device name and power limit are read
in the same run."""
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


def kept_pairs(m, st, masks, max_distance):
    """Pairs per query that prb_closest.cuh's culling keeps (closest_bounds, in fp64): mean over the envs of st."""
    from np_render import poses
    n = int(m['n_col'])
    h = m['col_half'].reshape(-1, 3)[:n].astype(np.float64)
    r = np.linalg.norm(h, axis=1)
    kept = np.zeros(len(masks))
    for s in st:
        R, p, _, _ = poses(m, s)

        def sd(c, x):                                     # signed distance of points x [k,3] to boxes c [k]
            q = np.abs(np.einsum('kji,kj->ki', R[c], x - p[c])) - h[c]
            return np.linalg.norm(np.maximum(q, 0), axis=1) + np.minimum(q.max(1), 0)

        for k, (ma, mb) in enumerate(masks):
            A = [c for c in range(n) if (ma >> c) & 1]
            B = [c for c in range(n) if (mb >> c) & 1]
            a, b = (np.array(x) for x in zip(*[(x, y) for x in A for y in B if x != y]))
            sb, sa = sd(a, p[b]), sd(b, p[a])
            L = np.maximum(sb - r[b], sa - r[a])
            U = np.minimum(np.maximum(sb, 0), np.maximum(sa, 0))
            mg = 1e-4 + 1e-4 * (np.linalg.norm(p[b] - p[a], axis=1) + r[a] + r[b])
            kept[k] += (L - mg <= min((U + mg).min(), max_distance)).sum()
    return kept / len(st)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--calls', type=int, default=60)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--envs', type=int, default=65536)
    ap.add_argument('--envs-c', type=int, default=8192)
    args = ap.parse_args()
    import torch
    import np_closest
    from helpers import random_actions
    from roboticsplayroompybullet_b200.envs import check_closest, make
    assert torch.cuda.is_available(), 'bench_closest needs a GPU'
    env_id = 'UR5PlayAbsRPY1Obj-v0'
    name, power = device_info(torch.cuda.current_device())
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device='cuda')    # > 126 MB L2

    def bench(env, queries, md, tag):
        for _ in range(args.warmup):
            env.closest_points_device(queries, md)
        ms = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for k in range(args.calls):
            flush.fill_(float(k))
            e0.record()
            out = env.closest_points_device(queries, md)
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = float(np.median(ms))
        N, Q = env.num_envs, len(queries)
        masks, _ = check_closest(env.model, queries, md)
        st = env.get_state()[np.linspace(0, N - 1, 32).astype(int)]
        pairs = [bin(a).count('1') * bin(b).count('1') - bin(a & b).count('1') for a, b in masks]
        line = {'workload': tag, 'env': env_id, 'num_envs': N, 'queries': Q, 'max_distance': md, 'median_ms': round(med, 4),
                'min_ms': round(min(ms), 4), 'max_ms': round(max(ms), 4), 'queries_per_s': N * Q / (med * 1e-3),
                'pairs_per_query': round(float(np.mean(pairs)), 2),
                'exact_per_query': round(float(kept_pairs(env.model, st, masks, md).mean()), 2),
                'found_fraction': round(float((out['collider_a'] >= 0).float().mean()), 4), 'calls': args.calls,
                'l2_flushed': True, 'device': name, 'power_limit': power}
        print(json.dumps(line), flush=True)

    rng = np.random.default_rng(0)
    for n, shapes in ((args.envs, 'ab'), (args.envs_c, 'c')):
        env = make(env_id, num_envs=n, seed=1234)
        env.reset()
        for k in range(4):
            env.step_device(torch.as_tensor(random_actions(rng, n, env_id), device='cuda'))
        torch.cuda.synchronize()
        if 'a' in shapes:
            bench(env, [(0, 1)], 0.2, 'a')
        if 'b' in shapes:
            bench(env, [(0, -1)] + [(0, b) for b in range(1, 6)] + [(1, -1), (2, -1)], 0.05, 'b')
        if 'c' in shapes:
            bench(env, np_closest.query_sets(env.model)['bodies'], 10.0, 'c')
        env.close()
        del env
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
