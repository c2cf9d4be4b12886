"""Arm-query throughput (prb_arm_dynamics) on one GPU; prints one JSON line per workload.

    python tools/bench_arm_dynamics.py [--envs 65536] [--calls 50] [--repeats 7] [--warmup 10]

Workloads (UR5PlayAbsRPY1Obj-v0, nd = 12, after 4 random steps so the arm is away from its reset pose):
  mass_matrix     M only (calculate_mass_matrix_device's call): [N,12,12]
  jacobian_site0  the site-0 Jacobian, P = 1 (calculate_jacobian_device's call): J [N,1,6,12], position, velocity
  all_p16         every output with P = 16 and caller-given q, qd, qdd: J [N,16,6,12], position, velocity, M, tau
Each call goes straight to the C ABI with preallocated outputs.  A repeat times --calls back-to-back calls with one pair
of CUDA events and divides, so the launch gaps of one call hide behind the previous kernel; the median and the spread
(min, max) over --repeats repeats after --warmup untimed calls.  The same output buffers are rewritten every call; the
all_p16 outputs (~0.38 GB at 65 536 envs) exceed the 126 MB L2, the smaller ones fit it.  bytes_written counts the
outputs, bytes_read the state rows' q, qd and the caller's arrays; hbm_share is (read + written) / time over 7.7 TB/s.
The device name and power limit are read in the same run."""
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

HBM_BYTES_PER_S = 7.7e12


def device_info(index):
    out = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = [x.strip() for x in out.split(',')]
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=65536)
    ap.add_argument('--calls', type=int, default=50)
    ap.add_argument('--repeats', type=int, default=7)
    ap.add_argument('--warmup', type=int, default=10)
    args = ap.parse_args()
    import torch
    from helpers import random_actions
    from roboticsplayroompybullet_b200 import lib
    from roboticsplayroompybullet_b200.envs import make
    assert torch.cuda.is_available(), 'bench_arm_dynamics needs a GPU'
    env_id = 'UR5PlayAbsRPY1Obj-v0'
    name, power = device_info(torch.cuda.current_device())
    N = args.envs
    env = make(env_id, num_envs=N, seed=1234)
    env.reset()
    rng = np.random.default_rng(0)
    for _ in range(4):
        env.step_device(torch.as_tensor(random_actions(rng, N, env_id), device='cuda'))
    nd = int(env.model['nd'])
    f32 = lambda *s: torch.empty(s, dtype=torch.float32, device='cuda')
    q, qd, qdd = (torch.as_tensor(rng.uniform(-s, s, (N, nd)).astype(np.float32), device='cuda') for s in (3.0, 2.0, 10.0))
    P16 = [(-1, s, (0.0, 0.0, 0.0)) for s in range(4)] + [(l, -1, (0.01 * l, 0.0, 0.02)) for l in range(12)]
    workloads = [
        ('mass_matrix', [], (None, None, None), {'mass_matrix': f32(N, nd, nd)}),
        ('jacobian_site0', [(-1, 0, (0.0, 0.0, 0.0))], (None, None, None),
         {'jacobian': f32(N, 1, 6, nd), 'position': f32(N, 1, 3), 'velocity': f32(N, 1, 6)}),
        ('all_p16', P16, (q, qd, qdd), {'jacobian': f32(N, 16, 6, nd), 'position': f32(N, 16, 3), 'velocity': f32(N, 16, 6),
                                        'mass_matrix': f32(N, nd, nd), 'tau': f32(N, nd)}),
    ]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    ptr = lambda x: None if x is None else ctypes.c_void_p(x.data_ptr())
    for tag, pts, ins, outs in workloads:
        P = len(pts)
        arr = (lib.PrbArmPoint * max(P, 1))(*[lib.PrbArmPoint(l, s, (ctypes.c_float * 3)(*o), 0) for l, s, o in pts])
        query = lib.PrbArmQuery(P, 0)
        args_c = [env._h, ctypes.byref(query), arr] + [ptr(x) for x in ins] + \
                 [ptr(outs.get(k)) for k in ('jacobian', 'position', 'velocity', 'mass_matrix', 'tau')] + [stream]
        call = lambda: lib.check(env.L, env._h, env.L.prb_arm_dynamics(*args_c))
        for _ in range(args.warmup):
            call()
        torch.cuda.synchronize()
        ms = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.repeats):
            e0.record()
            for _ in range(args.calls):
                call()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1) / args.calls)
        med = float(np.median(ms))
        written = sum(x.numel() * 4 for x in outs.values())
        read = N * nd * 4 * (2 if ins[0] is None else 3)
        bps = (written + read) / (med * 1e-3)
        print(json.dumps({'workload': tag, 'env': env_id, 'num_envs': N, 'points': P, 'outputs': sorted(outs),
                          'median_ms': round(med, 4), 'min_ms': round(min(ms), 4), 'max_ms': round(max(ms), 4),
                          'bytes_written': written, 'bytes_read': read, 'bytes_per_s': bps,
                          'hbm_share': round(bps / HBM_BYTES_PER_S, 4), 'calls_per_repeat': args.calls,
                          'repeats': args.repeats, 'device': name, 'power_limit': power}), flush=True)
    env.close()


if __name__ == '__main__':
    main()
