"""Link and joint state throughput (prb_body_states, prb_write_state, prb_save_state / prb_restore_state) on one GPU,
against the host round trip it replaces; prints one JSON line per workload.

    python tools/bench_state.py [--envs 65536] [--calls 50] [--repeats 7] [--warmup 10]

Workloads (UR5PlayAbsRPY1Obj-v0, K = 17 body rows, 15 joint columns, after 4 random steps):
  body_states_link   every body row in link frames, [N,17,13] (body_states_device('link')'s call)
  body_states_com    the same in COM frames
  write_half         a masked write of the block's pose and every joint position on half the envs (a fixed random
                     mask), including the report clear and the masked observe the call launches
  save_restore       prb_save_state, then prb_restore_state of the same half of the envs
  host_roundtrip     prb_get_state + prb_set_state of the whole batch (VecPlayEnv.get_state / set_state), the host path
                     the device calls replace
The device calls go straight to the C ABI with preallocated buffers: a repeat times --calls back-to-back calls with one
pair of CUDA events and divides; host_roundtrip is timed with the host clock around synchronous calls.  Median and
spread (min, max) over --repeats repeats after --warmup untimed calls.  The body block (58 MB at 65 536 envs) and the
snapshot (33 MB) fit the 126 MB L2, so repeated calls read the state and rewrite their outputs from L2.  bytes counts
each call's outputs and inputs once.  The device name and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from bench_arm_dynamics import device_info  # noqa: E402


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
    assert torch.cuda.is_available(), 'bench_state needs a GPU'
    env_id = 'UR5PlayAbsRPY1Obj-v0'
    name, power = device_info(torch.cuda.current_device())
    N = args.envs
    env = make(env_id, num_envs=N, seed=1234)
    env.reset()
    rng = np.random.default_rng(0)
    for _ in range(4):
        env.step_device(torch.as_tensor(random_actions(rng, N, env_id), device='cuda'))
    K, nj = len(env.body_state_ids), len(env.joint_state_ids)
    stride = env.buffers.state_stride
    f32 = lambda *s: torch.empty(s, dtype=torch.float32, device='cuda')
    body, snap = f32(N, K, 13), f32(N, stride)
    jq = env.joint_states_device()['position'].clone()
    src = env._body_states('link').clone()
    mask = torch.as_tensor(rng.random(N) < 0.5, device='cuda').to(torch.uint8)
    status = torch.empty(N, dtype=torch.uint8, device='cuda')
    half = int(mask.sum().item())
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    L, h = env.L, env._h
    q_link, q_com = lib.PrbBodyQuery(0, 0), lib.PrbBodyQuery(1, 0)
    w = lib.PrbStateWrite((1 << nj) - 1, 0, 1, 0, 0)
    out_bytes = N * (env.out_floats // N) * 4
    workloads = [
        ('body_states_link', lambda: lib.check(L, h, L.prb_body_states(h, ctypes.byref(q_link), p(body), None, None, stream)),
         N * K * 13 * 4 + N * stride * 4),
        ('body_states_com', lambda: lib.check(L, h, L.prb_body_states(h, ctypes.byref(q_com), p(body), None, None, stream)),
         N * K * 13 * 4 + N * stride * 4),
        ('write_half', lambda: lib.check(L, h, L.prb_write_state(h, ctypes.byref(w), p(jq), None, p(src), p(mask), p(status), stream)),
         half * (nj + 7) * 4 * 2 + half * out_bytes // N),
        ('save_restore', lambda: (lib.check(L, h, L.prb_save_state(h, p(snap), stream)),
                                  lib.check(L, h, L.prb_restore_state(h, p(snap), p(mask), stream))),
         N * stride * 4 * 2 + half * stride * 4 * 2 + half * out_bytes // N),
    ]
    for tag, call, nbytes in workloads:
        for _ in range(args.warmup):
            call()
        torch.cuda.synchronize()
        c0 = env.launch_count()
        call()
        torch.cuda.synchronize()
        launches = env.launch_count() - c0
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
        print(json.dumps({'workload': tag, 'env': env_id, 'num_envs': N, 'masked_envs': half if 'half' in tag or 'restore' in tag else N,
                          'launches_per_call': launches, 'median_ms': round(med, 4), 'min_ms': round(min(ms), 4),
                          'max_ms': round(max(ms), 4), 'bytes': nbytes, 'bytes_per_s': nbytes / (med * 1e-3),
                          'calls_per_repeat': args.calls, 'repeats': args.repeats, 'device': name, 'power_limit': power}),
              flush=True)
    # the host path: whole-batch copies through pageable host memory, synchronous
    st = env.get_state()
    for _ in range(3):
        env.set_state(env.get_state())
    ms = []
    for _ in range(args.repeats):
        t0 = time.perf_counter()
        env.set_state(env.get_state())
        torch.cuda.synchronize()
        ms.append(1e3 * (time.perf_counter() - t0))
    med = float(np.median(ms))
    print(json.dumps({'workload': 'host_roundtrip', 'env': env_id, 'num_envs': N, 'masked_envs': N, 'launches_per_call': 0,
                      'median_ms': round(med, 4), 'min_ms': round(min(ms), 4), 'max_ms': round(max(ms), 4),
                      'bytes': 2 * st.nbytes, 'bytes_per_s': 2 * st.nbytes / (med * 1e-3), 'calls_per_repeat': 1,
                      'repeats': args.repeats, 'device': name, 'power_limit': power}), flush=True)
    env.close()


if __name__ == '__main__':
    main()
