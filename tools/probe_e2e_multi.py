"""Diagnostic (not a bench line): how does a step_host call scale when k of the N ranks of one box run it at once?
torchrun --nproc-per-node N tools/probe_e2e_multi.py   -> one JSON line per (mode, active ranks) from rank 0.
Modes: zero_copy (one kernel, posted writes to pinned memory), d2h (the copy engine alone moving the same 2.6 MB),
d2h_big (26 MB per call)."""
import os, sys, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
import combinatorial_rl_tasks_b200 as crl

rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
local = int(os.environ.get('LOCAL_RANK', 0))
torch.cuda.set_device(local)
dev = torch.device('cuda', local)
if world > 1:
    dist.init_process_group('nccl', device_id=dev)
B = 65536
env = crl.ZoneVecEnv('PointTSP-v0', B, device=dev, env_offset=rank * B); env.seed(1 + rank * B); env.reset()
acts = env.pinned_actions(4)
rs = np.random.RandomState(rank)
for a in acts:
    np.copyto(a, rs.uniform(-1, 1, a.shape).astype(np.float32))
h = env._host_buffers()
big_src = torch.empty(26 * 1024 * 1024, dtype=torch.uint8, device=dev)
big_dst = torch.empty(26 * 1024 * 1024, dtype=torch.uint8).pin_memory()
s = torch.cuda.current_stream()
n_call = [0]
def zero_copy():
    env.step_host(acts[n_call[0] % 4]); n_call[0] += 1
def d2h():
    h['obs'].copy_(env.obs, non_blocking=True); h['result'].copy_(env.result, non_blocking=True); s.synchronize()
def d2h_big():
    big_dst.copy_(big_src, non_blocking=True); s.synchronize()
def dev_step():
    env.step(env._actions_dev); s.synchronize()

def barrier():
    if world > 1:
        dist.barrier()

def timed(fn, active, seconds=0.25, group=10):
    for _ in range(3):
        if active: fn()
    torch.cuda.synchronize(); barrier()
    per = []
    t_start = time.perf_counter()
    while active:
        t0 = time.perf_counter()
        for _ in range(group): fn()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        per.append((t1 - t0) / group)
        if t1 - t_start >= seconds: break
    torch.cuda.synchronize(); barrier()
    med = sorted(per)[len(per) // 2] if per else 0.0
    t = torch.tensor([med], device=dev, dtype=torch.float64)
    if world > 1:
        g = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        return [float(x) for x in g]
    return [med]

sets = {'all': list(range(world)), 'rank0': [0]}
if world >= 2: sets['0,1'] = [0, 1]
if world >= 4: sets['0,2'] = [0, 2]; sets['0-3'] = [0, 1, 2, 3]; sets['even'] = list(range(0, world, 2))
if world >= 8: sets['0,4'] = [0, 4]; sets['0,1,4,5'] = [0, 1, 4, 5]
for mode, fn in (('zero_copy', zero_copy), ('d2h', d2h), ('d2h_big', d2h_big), ('dev_step', dev_step)):
    for name, ranks in sets.items():
        if mode in ('d2h_big', 'dev_step') and name not in ('all', 'rank0', '0,1', '0,4'):
            continue
        us = timed(fn, rank in ranks, seconds=0.2 if mode != 'd2h_big' else 0.3, group=10 if mode != 'd2h_big' else 3)
        if rank == 0:
            act = [u * 1e6 for i, u in enumerate(us) if i in ranks]
            print(json.dumps({'mode': mode, 'active': name, 'n_active': len(ranks), 'us_per_call_max': round(max(act), 1),
                              'us_per_call_min': round(min(act), 1), 'us': [round(a, 1) for a in act]}), flush=True)
if world > 1:
    dist.destroy_process_group()
