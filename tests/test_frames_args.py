"""The rollout-frames entries (crl_frame_capture, crl_zone_encode_frames, crl_zone_encode_backward_frames,
crl_frames_zone_obs) refuse bad arguments on the host, before anything is launched.  Needs no GPU."""
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


def _shape(obs_dim=8, zone_dim=6, hidden=64, num_zones=15):
    from combinatorial_rl_tasks_b200 import _lib
    return _lib.CrlEncoderShape(obs_dim=obs_dim, zone_dim=zone_dim, hidden=hidden, num_zones=num_zones)


BUF = (ctypes.c_char * 4096)()
A16 = (ctypes.addressof(BUF) + 15) & ~15


def _state():
    from combinatorial_rl_tasks_b200 import _lib
    return _lib.CrlState(pose=A16, aux=A16, zone_xy=A16, zone_tmax=A16, cooldown=A16, seed=A16, episode=A16,
                         origin=A16, counters=A16)


def test_frame_capture_refusals(lib):
    cap = lambda cfg=None, st=None, result=A16, initial=0, frames=A16, xy=A16, tmax=A16, capacity=64, fill=A16: \
        lib.crl_frame_capture(cfg if cfg is not None else _cfg(), st if st is not None else _state(), result, initial,
                              frames, xy, tmax, capacity, fill, None)
    assert lib.crl_frame_capture(None, _state(), A16, 0, A16, A16, A16, 64, A16, None) == -1
    assert lib.crl_frame_capture(_cfg(), None, A16, 0, A16, A16, A16, 64, A16, None) == -1
    from combinatorial_rl_tasks_b200 import _lib
    assert cap(st=_lib.CrlState(zone_xy=A16)) == -1                      # no aux plane
    assert cap(frames=None) == -1
    assert cap(xy=None) == -1
    assert cap(fill=None) == -1
    assert cap(result=None) == -1                                        # a step's capture needs its done flags
    assert cap(cfg=_cfg(task=1), tmax=None) == -1                        # TimedTSP: the timeouts go into the table
    assert cap(capacity=0) == -2
    assert cap(cfg=_cfg(n=0)) == -2
    assert cap(cfg=_cfg(task=2, n=8)) == -2                              # ColourMatch holds at most 7 zones
    assert cap(frames=A16 + 4) == -3                                     # records are 16-byte vectors
    assert cap(xy=A16 + 4) == -3


def test_zone_encode_frames_refusals(lib):
    enc = lambda shape=None, cfg=None, m=64, obs=A16, frames=A16, xy=A16, tmax=None, packed=A16, pooled=A16: \
        lib.crl_zone_encode_frames(shape or _shape(), cfg if cfg is not None else _cfg(), m, obs, frames, xy, tmax,
                                   packed, pooled, None, None)
    assert enc(shape=_shape(obs_dim=9)) == -4                            # the rows are [obs (8), zone features]
    assert enc(shape=_shape(num_zones=14)) == -2                         # the task's num_zones
    assert enc(shape=_shape(zone_dim=7)) == -2                           # and zone_dim
    assert enc(cfg=_cfg(task=1), shape=_shape(zone_dim=7)) == -1         # TimedTSP without the timeout table
    assert enc(frames=None) == -1
    assert enc(xy=None) == -1
    assert enc(obs=None) == -1
    assert enc(m=0) == -2
    assert enc(frames=A16 + 8) == -3
    assert lib.crl_zone_encode_frames(_shape(), None, 64, A16, A16, A16, None, A16, A16, None, None) == -1


def test_zone_encode_backward_frames_refusals(lib):
    bwd = lambda shape=None, cfg=None, m=64, frames=A16, g=A16, ws=A16: \
        lib.crl_zone_encode_backward_frames(shape or _shape(), cfg if cfg is not None else _cfg(), m, A16, frames, A16,
                                            None, A16, g, ws, A16, A16, A16, A16, None, None)
    assert bwd(shape=_shape(obs_dim=9)) == -4
    assert bwd(shape=_shape(num_zones=5)) == -2
    assert bwd(frames=None) == -1
    assert bwd(g=None) == -1
    assert bwd(ws=None) == -1
    assert bwd(m=0) == -2
    assert lib.crl_zone_encode_backward_frames(_shape(), None, 64, A16, A16, A16, None, A16, A16, A16, A16, A16, A16,
                                               A16, None, None) == -1


def test_frames_zone_obs_refusals(lib):
    assert lib.crl_frames_zone_obs(None, 64, A16, A16, None, A16, None) == -1
    assert lib.crl_frames_zone_obs(_cfg(), 64, A16, A16, None, None, None) == -1
    assert lib.crl_frames_zone_obs(_cfg(), 64, None, A16, None, A16, None) == -1
    assert lib.crl_frames_zone_obs(_cfg(task=1), 64, A16, A16, None, A16, None) == -1
    assert lib.crl_frames_zone_obs(_cfg(), 0, A16, A16, None, A16, None) == -2
    assert lib.crl_frames_zone_obs(_cfg(num_steps=0), 64, A16, A16, None, A16, None) == -2
