#!/usr/bin/env python
"""crl_copy_envs (copy_envs_kernel) on one GPU: branching and restoring, against a plain device-to-device copy.

Per task (PointTSP-v0, PointTTSP-v0, ColourMatch-v0):
  branch   B = 65,536 envs, each copied onto K consecutive envs of a B K env (K = 4, 16; src ids given, dst ids NULL):
           the planner's branch, 1,048,576 dst envs at K = 16;
  restore  a B-env snapshot onto all envs of a B-env ZoneVecEnv (both ids NULL); four snapshot / env pairs taken in
           turn, so that one pass (4 x about 80 MB) does not fit the 126 MB L2.
Bytes per copied env come from crl_plane_bytes (num_envs = 1) for the planes the copy touches: read = the state and
output planes plus the 4-byte src id, written = the same planes plus the two next_ready slots.  The reference is
torch's copy_ between two device buffers of (read + written) / 2 bytes per copied env, timed in the same process,
alternating with the kernel (in turn over four buffer pairs for the restore); both with CUDA events over `--iters`
launches after warm-up, median of `--reps`.
Branch reads gather each src env K times in a row: DRAM sees it about once (the other K - 1 come from L2), which
`dram_bytes` counts.  Writes a JSON file with the GPU name and power limit read in the same run.

    python tools/bench_copy_envs.py [--out profiles/r06_copy_envs.json] [--small]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import combinatorial_rl_tasks_b200 as crl  # noqa: E402
from combinatorial_rl_tasks_b200 import _lib  # noqa: E402
from combinatorial_rl_tasks_b200.vec_env import _copy_out  # noqa: E402

TASKS = ('PointTSP-v0', 'PointTTSP-v0', 'ColourMatch-v0')
# crl_plane_bytes entries a copy reads and writes: pose, aux, zone_xy, zone_tmax, cooldown, seed, episode, origin,
# obs, zone_obs, result, goal, shaped_reward; next_ready (13) is written only
COPIED = (0, 1, 2, 3, 4, 5, 6, 7, 14, 15, 16, 20, 21)


def gpu_header():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return {'gpu': torch.cuda.get_device_name(0), 'nvidia_smi': q.stdout.strip()}


def env_bytes(env, src_ids):
    cfg = _lib.CrlConfig.from_buffer_copy(env.cfg)
    cfg.num_envs = 1
    b = (ctypes.c_int64 * _lib.NUM_PLANES)()
    _lib.check(env.lib.crl_plane_bytes(cfg, b, _lib.NUM_PLANES))
    planes = sum(b[i] for i in COPIED)
    return planes + (4 if src_ids else 0), planes + b[13]


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters          # us per launch


def measure(launch, n, rd, wr, iters, reps, rotate=1):
    """Alternate the kernel and the reference copy; medians of `reps` windows of `iters` launches each.  The copy takes
    `rotate` buffer pairs in turn, as the kernel does its src / dst pairs."""
    half = (rd + wr) * n // 2
    bufs = [(torch.empty(half, dtype=torch.uint8, device='cuda'), torch.empty(half, dtype=torch.uint8, device='cuda'))
            for _ in range(rotate)]
    copy = lambda i: bufs[i % rotate][1].copy_(bufs[i % rotate][0])
    for _ in range(3):
        launch(0)
        copy(0)
    torch.cuda.synchronize()
    k, c = [], []
    for _ in range(reps):
        k.append(timed(launch, iters))
        c.append(timed(copy, iters))
    k_us, c_us = sorted(k)[reps // 2], sorted(c)[reps // 2]
    return {'kernel_us': round(k_us, 2), 'kernel_GBps': round((rd + wr) * n / k_us / 1e3, 1),
            'copy_us': round(c_us, 2), 'copy_GBps': round(2 * half / c_us / 1e3, 1), 'ratio_to_copy': round(c_us / k_us, 3),
            'kernel_us_all': [round(x, 2) for x in k], 'copy_us_all': [round(x, 2) for x in c]}


def raw_launch(dst, src, n, src_ids, dst_ids=None):
    """crl_copy_envs with everything resolved once: what a captured or tight planning loop issues."""
    both = True
    args = (dst.cfg, dst.state, _copy_out(dst, both), None if dst_ids is None else dst_ids.data_ptr(), src.cfg, src.state,
            _copy_out(src, both), None if src_ids is None else src_ids.data_ptr(), n, dst.copy_rejects.data_ptr())
    fn = dst.lib.crl_copy_envs

    def launch(_):
        rc = fn(*args, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        if rc:
            _lib.check(rc)
    return launch


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join('profiles', 'r06_copy_envs.json'))
    ap.add_argument('--envs', type=int, default=65536)
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--small', action='store_true', help='a quick run at 4,096 envs')
    a = ap.parse_args(argv)
    B = 4096 if a.small else a.envs
    out = {'tool': 'tools/bench_copy_envs.py', **gpu_header(), 'envs': B, 'iters': a.iters, 'reps': a.reps, 'results': []}
    for env_id in TASKS:
        src = crl.ZoneVecEnv(env_id, B, prefetch_every=0)
        src.seed(1)
        src.reset()
        for _ in range(8):
            src.step_random(action_seed=2)
        for K in (4, 16):
            dst = crl.ZoneVecEnv(env_id, B * K, prefetch_every=0)
            sid = torch.arange(B, dtype=torch.int32, device='cuda').repeat_interleave(K)
            dst.copy_envs_from(src, sid)                # through the public call once, and check it
            r = sid.long()
            for k in ('pose', 'aux', 'seeds', 'obs', 'zone_obs', 'result'):
                assert torch.equal(getattr(dst, k), getattr(src, k)[r]), (env_id, K, k)
            assert torch.equal(dst.zone_xy, src.zone_xy[:, r])
            rd, wr = env_bytes(src, True)
            n = B * K
            res = {'task': env_id, 'mode': 'branch', 'src_envs': B, 'K': K, 'copied_envs': n,
                   'bytes_read_per_env': rd, 'bytes_written_per_env': wr,
                   'dram_bytes': (rd - 4) * B + 4 * n + wr * n}
            res.update(measure(raw_launch(dst, src, n, sid), n, rd, wr, a.iters, a.reps))
            res['dram_GBps'] = round(res['dram_bytes'] / res['kernel_us'] / 1e3, 1)
            print(json.dumps({k: v for k, v in res.items() if not k.endswith('_all')}), flush=True)
            out['results'].append(res)
            del dst, sid
            torch.cuda.empty_cache()
        snaps = [src.snapshot() for _ in range(4)]
        dsts = [crl.ZoneVecEnv(env_id, B, prefetch_every=0) for _ in range(4)]
        dsts[0].copy_envs_from(snaps[0])
        for k in ('pose', 'aux', 'seeds', 'obs', 'zone_obs', 'result'):
            assert torch.equal(getattr(dsts[0], k), getattr(src, k)), (env_id, 'restore', k)
        launches = [raw_launch(d, s, B, None) for d, s in zip(dsts, snaps)]
        rd, wr = env_bytes(src, False)
        res = {'task': env_id, 'mode': 'restore', 'src_envs': B, 'K': 1, 'copied_envs': B,
               'bytes_read_per_env': rd, 'bytes_written_per_env': wr, 'dram_bytes': (rd + wr) * B}
        res.update(measure(lambda i: launches[i % 4](i), B, rd, wr, a.iters, a.reps, rotate=4))
        res['dram_GBps'] = round(res['dram_bytes'] / res['kernel_us'] / 1e3, 1)
        print(json.dumps({k: v for k, v in res.items() if not k.endswith('_all')}), flush=True)
        out['results'].append(res)
        del snaps, dsts, src
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print('wrote', a.out)
    return out


if __name__ == '__main__':
    main()
