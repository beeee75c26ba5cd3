"""crl_copy_envs refuses bad arguments on the host, before anything is launched, and ZoneVecEnv.copy_envs_from refuses
bad sources and host ids before touching the device.  Needs no GPU."""
import ctypes

import pytest


@pytest.fixture(scope='module')
def lib():
    from combinatorial_rl_tasks_b200 import _lib
    return _lib.load()


def _cfg(task=0, n=15, **kw):
    from combinatorial_rl_tasks_b200 import _lib
    args = dict(task=task, num_envs=64, num_zones=n, num_steps=2000, frameskip=10, max_cooldown=150, zone_size=0.2)
    args.update(kw)
    return _lib.CrlConfig(**args)


BUF = (ctypes.c_char * 4096)()
A16 = (ctypes.addressof(BUF) + 15) & ~15


def _state(**kw):
    from combinatorial_rl_tasks_b200 import _lib
    args = dict(pose=A16, aux=A16, zone_xy=A16, zone_tmax=A16, cooldown=A16, seed=A16, episode=A16, origin=A16)
    args.update(kw)
    return _lib.CrlState(**args)


def _out(**kw):
    from combinatorial_rl_tasks_b200 import _lib
    args = dict(obs=A16, zone_obs=A16, result=A16, shaped_reward=A16)
    args.update(kw)
    return _lib.CrlOut(**args)


def _copy(lib, dcfg=None, dst=None, dout=None, scfg=None, src=None, sout=None, n=0, dst_ids=None, src_ids=None,
          rejected=None):
    return lib.crl_copy_envs(dcfg if dcfg is not None else _cfg(), dst if dst is not None else _state(), dout, dst_ids,
                             scfg if scfg is not None else _cfg(), src if src is not None else _state(), sout, src_ids,
                             n, rejected, None)


def test_n_zero_is_a_no_op(lib):
    assert _copy(lib) == 0
    assert _copy(lib, dout=_out(), sout=_out()) == 0
    # the batch's size, offset and seed range may differ
    assert _copy(lib, dcfg=_cfg(num_envs=1000, env_offset=64, seed_mode=1, min_seed=5, max_seed=9)) == 0
    assert _copy(lib, dcfg=_cfg(task=1), scfg=_cfg(task=1)) == 0
    assert _copy(lib, dcfg=_cfg(task=2, n=6), scfg=_cfg(task=2, n=6)) == 0


def test_mismatched_configs(lib):
    assert _copy(lib, dcfg=_cfg(num_steps=24)) == -2
    assert _copy(lib, dcfg=_cfg(task=1)) == -2
    assert _copy(lib, dcfg=_cfg(frameskip=5)) == -2
    assert _copy(lib, dcfg=_cfg(zone_size=0.3)) == -2
    assert _copy(lib, dcfg=_cfg(time_saved_reward=0.5)) == -2
    assert _copy(lib, dcfg=_cfg(initial_visited=1)) == -2
    assert _copy(lib, dcfg=_cfg(walled=1, robot_keepout=0.4, zone_keepout=0.55),
                 scfg=_cfg(robot_keepout=0.4, zone_keepout=0.55)) == -2
    assert _copy(lib, dcfg=_cfg(n=5), scfg=_cfg()) == -2
    assert _copy(lib, scfg=_cfg(num_steps=0)) == -2                     # each config on its own, too


def test_negative_n(lib):
    assert _copy(lib, n=-1) == -2


def test_null_planes(lib):
    assert lib.crl_copy_envs(None, _state(), None, None, _cfg(), _state(), None, None, 1, None, None) == -1
    assert lib.crl_copy_envs(_cfg(), None, None, None, _cfg(), _state(), None, None, 1, None, None) == -1
    assert lib.crl_copy_envs(_cfg(), _state(), None, None, _cfg(), None, None, None, 1, None, None) == -1
    for plane in ('pose', 'aux', 'zone_xy', 'seed', 'episode', 'origin'):
        assert _copy(lib, dst=_state(**{plane: None}), n=1) == -1, plane
        assert _copy(lib, src=_state(**{plane: None}), n=1) == -1, plane
    tt, cm = _cfg(task=1), _cfg(task=2, n=6)
    assert _copy(lib, dcfg=tt, scfg=tt, src=_state(zone_tmax=None), n=1) == -1
    assert _copy(lib, dcfg=cm, scfg=cm, dst=_state(cooldown=None), n=1) == -1


def test_output_on_one_side_only(lib):
    assert _copy(lib, dout=_out(), n=1) == -1
    assert _copy(lib, sout=_out(), n=1) == -1
    for field in ('obs', 'zone_obs', 'result', 'shaped_reward'):
        assert _copy(lib, dout=_out(**{field: None}), sout=_out(), n=1) == -1, field
        assert _copy(lib, dout=_out(), sout=_out(**{field: None}), n=1) == -1, field


def test_misaligned_planes(lib):
    for plane in ('pose', 'aux', 'zone_xy', 'origin'):
        assert _copy(lib, dst=_state(**{plane: A16 + 4}), n=1) == -3, plane
        assert _copy(lib, src=_state(**{plane: A16 + 8}), n=1) == -3, plane
    assert _copy(lib, dout=_out(obs=A16 + 8), sout=_out(), n=1) == -3
    assert _copy(lib, dout=_out(), sout=_out(result=A16 + 4), n=1) == -3


def test_unsupported_num_zones(lib):
    assert _copy(lib, dcfg=_cfg(n=7), scfg=_cfg(n=7), n=1) == -4
    assert _copy(lib, dcfg=_cfg(task=2, n=5), scfg=_cfg(task=2, n=5)) == -4


def _fake_env(env_id, num_envs, num_steps=None, device='cuda:0'):
    """A ZoneVecEnv shell with what copy_envs_from checks before it touches the device (the constructor needs one)."""
    import torch
    from combinatorial_rl_tasks_b200 import ZoneVecEnv, _lib
    from combinatorial_rl_tasks_b200.config import ENV_SPECS
    env = ZoneVecEnv.__new__(ZoneVecEnv)
    spec = ENV_SPECS[env_id]
    env.env_id, env.spec, env.num_envs = env_id, spec, num_envs
    env.device = torch.device(device)
    env._dev_index = env.device.index
    env.cfg = _lib.CrlConfig(task=spec.task, num_envs=num_envs, num_zones=spec.num_zones,
                             num_steps=num_steps or spec.num_steps, frameskip=spec.frameskip,
                             max_cooldown=spec.max_cooldown, zone_size=spec.zone_size)
    return env


def test_copy_envs_from_refusals():
    dst = _fake_env('PointTSP-v0', 8)
    with pytest.raises(TypeError):
        dst.copy_envs_from(object())
    with pytest.raises(ValueError, match='PointTTSP'):
        dst.copy_envs_from(_fake_env('PointTTSP-v0', 8))
    with pytest.raises(ValueError, match='config'):
        dst.copy_envs_from(_fake_env('PointTSP-v0', 8, num_steps=24))
    with pytest.raises(ValueError, match='lives on'):
        dst.copy_envs_from(_fake_env('PointTSP-v0', 8, device='cuda:1'))
    src = _fake_env('PointTSP-v0', 4)
    with pytest.raises(ValueError, match=r'\[0, 4\)'):
        dst.copy_envs_from(src, [0, 4])
    with pytest.raises(ValueError, match=r'\[0, 8\)'):
        dst.copy_envs_from(src, [0, 1], [7, 8])
    with pytest.raises(ValueError, match=r'\[0, 8\)'):
        dst.copy_envs_from(src, [0, 1], [-1, 2])
    with pytest.raises(ValueError, match='distinct'):
        dst.copy_envs_from(src, [0, 1], [3, 3])
    with pytest.raises(ValueError, match='2 src ids but 3 dst ids'):
        dst.copy_envs_from(src, [0, 1], [1, 2, 3])
    with pytest.raises(ValueError, match='integers'):
        dst.copy_envs_from(src, [0.5])
    with pytest.raises(ValueError, match='from a src of 4'):
        dst.copy_envs_from(src, None, [0, 1, 2, 3, 4])            # None src ids: 0..n-1 must fit the src
    with pytest.raises(ValueError, match='into an env of 4'):
        src.copy_envs_from(dst)                                      # all 8 envs of dst do not fit
    with pytest.raises(ValueError, match='no envs'):
        dst.snapshot([])
