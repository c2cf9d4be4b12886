"""Camera rendering throughput (prb_render) on one GPU; prints one JSON line.

    python tools/bench_render.py --envs 8192 --size 200 [--renders 50] [--steps 20]

ms per render and pixels/s from CUDA events over --renders renders of the default world camera after warm-up;
the step alone and step + render end to end (device-resident step_device with record_images, CUDA events around
--steps steps); the mean number of boxes tested per pixel after tile culling; the device name and power limit read in the
same run.  The play envs are stepped with scripted actions first, so the arm is not at its reset pose."""
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
    ap.add_argument('--envs', type=int, default=8192)
    ap.add_argument('--size', type=int, default=200)
    ap.add_argument('--renders', type=int, default=50)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    import torch
    from helpers import random_actions
    from roboticsplayroompybullet_b200.camera import default_camera
    from roboticsplayroompybullet_b200.envs import make
    from roboticsplayroompybullet_b200.model import load_model
    assert torch.cuda.is_available(), 'bench_render needs a GPU'
    cam = default_camera(load_model(args.env), args.size, args.size)
    n = args.envs
    env = make(args.env, num_envs=n, seed=1234, camera=cam, record_images=True)
    env.reset()
    rng = np.random.default_rng(0)
    acts = [torch.as_tensor(random_actions(rng, n, args.env), device='cuda') for _ in range(8)]
    for k in range(args.warmup + 4):
        env.step_device(acts[k % len(acts)])
    torch.cuda.synchronize()
    # renders only
    rgb = torch.empty((n, cam.height, cam.width, 3), dtype=torch.uint8, device='cuda')
    for _ in range(args.warmup):
        env._render(cam, rgb)
    t0 = env.render_box_tests()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.renders):
        env._render(cam, rgb)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / args.renders
    tests = (env.render_box_tests() - t0) / args.renders
    pixels = n * cam.width * cam.height
    # steps alone, then step + render (record_images: step_device renders 'img' after every step)
    env.record_images = False
    e0.record()
    for k in range(args.steps):
        env.step_device(acts[k % len(acts)])
    e1.record()
    e1.synchronize()
    ms_step = e0.elapsed_time(e1) / args.steps
    env.record_images = True
    e0.record()
    for k in range(args.steps):
        env.step_device(acts[k % len(acts)])
    e1.record()
    e1.synchronize()
    ms_step_render = e0.elapsed_time(e1) / args.steps
    name, power = device_info(torch.cuda.current_device())
    print(json.dumps({'env': args.env, 'num_envs': n, 'width': cam.width, 'height': cam.height,
                      'render_ms': round(ms, 4), 'pixels_per_s': pixels / (ms * 1e-3),
                      'step_ms': round(ms_step, 3), 'step_render_ms': round(ms_step_render, 3), 'step_render_env_steps_per_s': n / (ms_step_render * 1e-3),
                      'boxes_tested_per_pixel': round(tests / pixels, 3), 'renders': args.renders, 'steps': args.steps,
                      'device': name, 'power_limit': power}))
    env.close()


if __name__ == '__main__':
    main()
