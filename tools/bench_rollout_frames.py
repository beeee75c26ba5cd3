#!/usr/bin/env python
"""Rollout(store='zone_obs') against Rollout(store='frames') on one GPU, alternating the two in the same process.

Per configuration (env id, envs, T = 128):
  collection  device time per Rollout.step (CUDA events around T steps with a fixed action tensor, no policy) and host
              time per Rollout.step (the enqueue: the frames store adds the capture launch);
  update      FusedZoneEnvModel forward + backward on a T B / 10 minibatch gathered from the rollout, gather included;
  memory      the rollout's device bytes, from the shapes (Rollout.storage_bytes).
Prints one JSON line per (configuration, store) and a header line with the GPU name and power limit.

    python tools/bench_rollout_frames.py [--reps 3] [--out profiles/r04_rollout_frames.jsonl] [--small]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import combinatorial_rl_tasks_b200 as crl  # noqa: E402
from combinatorial_rl_tasks_b200.rollout import Rollout  # noqa: E402

CONFIGS = [('PointTSP-v0', 65536), ('ColourMatch-v0', 262144), ('PointTTSP-v0', 262144)]


def gpu_header():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'gpu': torch.cuda.get_device_name(0), 'nvidia_smi': q.stdout.strip().splitlines()[:1]}


def collect(ro, actions):
    """One rollout: returns (device ms per step, host ms per step)."""
    ro.begin()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    h0 = time.perf_counter()
    for t in range(ro.T):
        ro.step(t, actions)
    h1 = time.perf_counter()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / ro.T, 1e3 * (h1 - h0) / ro.T


def update(ro, model, idx):
    """Gather a minibatch from the rollout and run the fused forward + backward: device ms."""
    T, B = ro.T, ro.env.num_envs
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    o = ro.obs[:T].reshape(T * B, 8)[idx]
    if ro.store == 'frames':
        batch = {'obs': o, 'zone_frames': ro._frames_view(slice(0, T)).reshape(T * B)[idx]}
    else:
        batch = {'obs': o, 'zone_obs': ro.zone_obs[:T].reshape((T * B,) + tuple(ro.zone_obs.shape[2:]))[idx]}
    model(batch).sum().backward()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--T', type=int, default=128)
    ap.add_argument('--out', default=None)
    ap.add_argument('--small', action='store_true', help='B / 64: a quick end-to-end check, not a measurement')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_rollout_frames.py measures on a GPU; none found')
    lines = [dict(gpu_header(), T=args.T, reps=args.reps)]
    print(json.dumps(lines[0]), flush=True)
    for env_id, B in CONFIGS:
        B = B // 64 if args.small else B
        ros = {}
        for store in ('zone_obs', 'frames'):
            env = crl.ZoneVecEnv(env_id, B, seed_mode='fixed_range', min_seed=1, max_seed=100)
            ros[store] = Rollout(env, args.T, store=store)
        spec = ros['frames'].env.spec
        model = crl.FusedZoneEnvModel(8, spec.zone_dim, spec.num_zones, hidden=185)
        g = torch.Generator(device='cuda').manual_seed(0)
        actions = torch.rand(B, 2, device='cuda', generator=g) * 2 - 1
        idx = torch.randint(0, args.T * B, (args.T * B // 10,), device='cuda', generator=g)
        res = {s: {'step_device_ms': [], 'step_host_ms': [], 'update_ms': []} for s in ros}
        for store in ros:                                        # warm-up: modules, workspaces
            collect(ros[store], actions)
            update(ros[store], model, idx)
        for _ in range(args.reps):
            for store in ('zone_obs', 'frames'):                 # alternate the two stores
                d, h = collect(ros[store], actions)
                res[store]['step_device_ms'].append(d)
                res[store]['step_host_ms'].append(h)
                if store == 'frames':
                    ros[store].finish(torch.zeros(B, device='cuda'))    # raises if the layout table overflowed
                res[store]['update_ms'].append(update(ros[store], model, idx))
        for store, ro in ros.items():
            sb = ro.storage_bytes()
            zone = sum(v for k, v in sb.items() if k in ('zone_obs', 'frames', 'layout_xy', 'layout_tmax'))
            r = res[store]
            line = {'env': env_id, 'envs': B, 'T': args.T, 'store': store,
                    'step_device_us': [round(1e3 * x, 2) for x in r['step_device_ms']],
                    'step_host_us': [round(1e3 * x, 2) for x in r['step_host_ms']],
                    'update_ms': [round(x, 3) for x in r['update_ms']],
                    'update_rows': args.T * B // 10,
                    'storage_bytes': sum(sb.values()), 'zone_state_bytes': zone,
                    'layout_capacity': getattr(ro, 'layout_capacity', None)}
            lines.append(line)
            print(json.dumps(line), flush=True)
        del ros, model
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write('\n'.join(json.dumps(x) for x in lines) + '\n')


if __name__ == '__main__':
    main()
