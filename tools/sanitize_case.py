"""Small all-paths case for compute-sanitizer (memcheck / racecheck): every kernel, ragged
batch, fused auto-reset, host-supplied layouts, qpos/qvel import/export, host-buffer step."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import combinatorial_rl_tasks_b200 as crl  # noqa: E402

for env_id in ('PointTSP-v0', 'PointTTSP-v0', 'ColourMatch-v0', 'PointTSP-v1'):
    B = 301
    env = crl.ZoneVecEnv(env_id, B)
    env.seed(11)
    env.reset()
    bits = env.aux[:, 3].view(torch.int32)
    bits.copy_((bits & ~0xffff) | (env.spec.num_steps - 6))
    for t in range(12):                      # every env finishes and is rebuilt in-kernel
        env.step_random(action_seed=5)
    env.step(torch.zeros(B, 2, device='cuda'))
    env.step_no_reset(torch.ones(B, 2, device='cuda'))
    env.step_host(np.zeros((B, 2), np.float32))
    env.reset(mask=torch.arange(B) % 3 == 0)
    N = env.spec.num_zones
    rs = np.random.RandomState(0)
    lay = {'xy0': rs.uniform(-2, 2, (5, 2)), 'rot0': rs.uniform(0, 6, 5), 'zone_xy': rs.uniform(-2, 2, (5, N, 2)),
           'zone_max_steps': rs.randint(100, 900, (5, N)), 'colours': rs.randint(0, 3, (5, N))}
    env.reset(layout=lay, env_ids=[0, 7, 33, 299, 300])
    env.set_qpos_qvel(rs.uniform(-1, 1, (5, 3)), rs.uniform(-1, 1, (5, 3)), env_ids=[0, 7, 33, 299, 300])
    qp, qv = env.get_qpos_qvel()
    env.physics_substeps(torch.zeros(B, 2, device='cuda'), 3)
    for t in range(6):                       # chained back-to-back steps (per-warp ticket / stamp ordering)
        env.step_random(action_seed=9, chained=True)
    env.step_host(np.zeros((B, 2), np.float32))                       # full copy: the host mirror becomes valid
    env.step_host(np.zeros((B, 2), np.float32))                       # delta rows + zero-copy obs / result
    torch.cuda.synchronize()
    print(env_id, 'ok', env.counters())

# goal-conditioned variant + WaitWrapper + rollout slots + GAE
from combinatorial_rl_tasks_b200.rollout import Rollout  # noqa: E402
env = crl.ZoneVecEnv('PointTTSP-v3', 300, wait=True)
env.seed(3)
env.cfg.num_steps = 9
ro = Rollout(env, 6)
ro.begin()
for t in range(6):
    env.set_goal(torch.where(env.needs_goal(), torch.full((300,), t % 15, dtype=torch.int32, device='cuda'),
                             torch.full((300,), -1, dtype=torch.int32, device='cuda')))
    ro.step(t, torch.zeros(300, 2, device='cuda'), torch.zeros(300, device='cuda'))
ro.finish(torch.zeros(300, device='cuda'))
env.get_goal(); env.available_goals()
for t in range(8):
    env.step_no_reset(torch.zeros(300, 2, device='cuda'))            # envs park as they finish
torch.cuda.synchronize()
print('PointTTSP-v3 ok', env.counters())
