"""CRL_STEP_ZONE_OBS_DELTA is refused on the host, before anything is launched, where the step would not write
the device zone_obs rows it changes: with CRL_STEP_NO_ZONE_OBS and in the goal-conditioned / WaitWrapper / walled
kernels.  Needs no GPU."""
import ctypes


def test_zone_obs_delta_is_refused_where_it_does_not_apply():
    from combinatorial_rl_tasks_b200 import _lib
    lib = _lib.load()
    cfg = _lib.CrlConfig(task=0, num_envs=64, num_zones=15, num_steps=2000, frameskip=10, max_cooldown=150,
                         zone_size=0.2)
    buf = (ctypes.c_char * 4096)()
    a16 = (ctypes.addressof(buf) + 15) & ~15
    st = _lib.CrlState(pose=a16, aux=a16, zone_xy=a16, seed=a16, episode=a16, origin=a16, counters=a16, goal=a16)
    out = _lib.CrlOut(obs=a16, zone_obs=a16, result=a16, shaped_reward=a16)
    delta = _lib.STEP_ZONE_OBS_DELTA
    assert lib.crl_step(cfg, st, None, out, delta | _lib.STEP_NO_ZONE_OBS, 0, 0, None) == -2
    assert lib.crl_step(cfg, st, None, out, delta | _lib.STEP_GOALS, 0, 0, None) == -2
    assert lib.crl_step(cfg, st, None, out, delta | _lib.STEP_WAIT, 0, 0, None) == -2
    cfg.walled = 1
    assert lib.crl_step(cfg, st, None, out, delta, 0, 0, None) == -2
