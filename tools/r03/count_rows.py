#!/usr/bin/env python
"""zone_obs rows a CRL_STEP_ZONE_OBS_DELTA step writes, per env-step, on one replica of bench.py's ring: the same
seeds, in-kernel actions (action_seed 1234, device step counter), auto-reset and sampler cadence, with
CRL_STEP_TRACK_ROWS added so that the kernel counts the rows it writes.  Prints one JSON line per workload.
Usage: python tools/r03/count_rows.py ENV_ID:B[:STEPS] ..."""
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def count(env_id, B, steps):
    import torch
    import combinatorial_rl_tasks_b200 as crl
    from combinatorial_rl_tasks_b200 import _lib
    env = crl.ZoneVecEnv(env_id, B, prefetch_every=32)
    env.seed(1)
    env.reset()
    rd, wr = ctypes.c_int64(), ctypes.c_int64()
    env.lib.crl_step_bytes(env.cfg, ctypes.byref(rd), ctypes.byref(wr))
    row_bytes = 4 * env.spec.num_zones * env.spec.zone_dim
    flags = _lib.STEP_AUTO_RESET | _lib.STEP_ACTION_COUNTER | _lib.STEP_ZONE_OBS_DELTA | _lib.STEP_TRACK_ROWS
    rows = torch.zeros((), dtype=torch.int64, device=env.device)
    env._row_list[:4].zero_()
    for _ in range(steps):
        _lib.check(env.lib.crl_step(env.cfg, env.state, None, env.out, flags, 1234, 0, env._stream()))
        rows += env._row_list[0]                     # word 0 counts this step's rows
        env._row_list[:1].zero_()
        env.tick()
    per = int(rows.item()) / (steps * B)
    full = rd.value + wr.value - 8                   # bench.py's figure: no action plane with in-kernel actions
    return {'env': env_id, 'envs': B, 'steps': steps, 'rows_per_env_step': per, 'full_bytes_per_env_step': full,
            'row_bytes': row_bytes, 'bytes_per_env_step': full - row_bytes + per * row_bytes,
            'episodes': env.counters()['episodes']}


if __name__ == '__main__':
    for arg in sys.argv[1:]:
        parts = arg.split(':')
        print(json.dumps(count(parts[0], int(parts[1]), int(parts[2]) if len(parts) > 2 else 6000)), flush=True)
