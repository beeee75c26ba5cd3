"""Diagnostic (not a bench line): where does a step_host call spend its time?"""
import os, sys, time, ctypes
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import combinatorial_rl_tasks_b200 as crl
from combinatorial_rl_tasks_b200 import _lib

B = 65536
env = crl.ZoneVecEnv('PointTSP-v0', B); env.seed(1); env.reset()
a = np.random.RandomState(0).uniform(-1, 1, (B, 2)).astype(np.float32)
for _ in range(5): env.step_host(a)
def t(f, n=200):
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(n): f()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / n * 1e6
h = env._host_buffers()
print('step_host(full)             %.1f us' % t(lambda: env.step_host(a, delta=False), 50))
env.step_host(a)
print('np.copyto actions           %.1f us' % t(lambda: np.copyto(h['np']['actions'], a)))
s = torch.cuda.current_stream()
def h2d(): env._actions_dev.copy_(h['actions'], non_blocking=True); s.synchronize()
print('H2D actions + sync          %.1f us' % t(h2d))
def d2h_obs(): h['obs'].copy_(env.obs, non_blocking=True); s.synchronize()
print('D2H obs (2 MB) + sync       %.1f us' % t(d2h_obs))
def d2h_res(): h['result'].copy_(env.result, non_blocking=True); s.synchronize()
print('D2H result (0.5 MB) + sync  %.1f us' % t(d2h_res))
def both(): h['obs'].copy_(env.obs, non_blocking=True); h['result'].copy_(env.result, non_blocking=True); s.synchronize()
print('D2H obs+result + sync       %.1f us' % t(both))
def kern(): env.step(env._actions_dev); s.synchronize()
print('device step + sync          %.1f us' % t(kern))
print('empty sync                  %.1f us' % t(lambda: s.synchronize()))
env.step_host(a)
print('step_host(delta, zero-copy)           %.1f us' % t(lambda: env.step_host(a)))
print('step_host(delta, zero-copy, pinned in)%.1f us' % t(lambda: env.step_host(h['np']['actions'])))
pa = env.pinned_actions(1)[0]; np.copyto(pa, a)
print('  ... pinned_actions() array           %.1f us' % t(lambda: env.step_host(pa)))
ref = crl.ZoneVecEnv('PointTSP-v0', B); ref.seed(1); ref.reset()
env2 = crl.ZoneVecEnv('PointTSP-v0', B); env2.seed(1); env2.reset()
rs = np.random.RandomState(3)
for k in range(60):
    aa = rs.uniform(-1, 1, (B, 2)).astype(np.float32)
    o1, r1, d1, i1 = ref.step_host(aa, delta=False)
    o2, r2, d2, i2 = env2.step_host(aa)
    assert np.array_equal(o1['obs'], o2['obs']) and np.array_equal(o1['zone_obs'], o2['zone_obs']) and np.array_equal(r1, r2) and np.array_equal(d1, d2), k
print('zero-copy host buffers identical to full copy over 60 steps')
