"""Rollout(store='frames'): a 16-byte record per env and frame plus one layout per episode instead of zone_obs.

Twin envs with the same seeds take the same actions, one stored as zone_obs and one as frames.  Everything the frames
rollout hands out must equal the twin's bit for bit: obs and result of every slot, the rows rebuilt from the records,
the advantages, and the encoder's forward and backward run straight from the records."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

B = 4 * 33                    # ragged against 32
T = 64


@pytest.fixture(scope='module')
def crl():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    import combinatorial_rl_tasks_b200 as m
    return m


def _bits(x):
    return x.contiguous().view(torch.int32)


def _state_dict(obs_dim, zone_dim, h, seed=0):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s, sc: (torch.randn(*s, generator=g) * sc)
    return {'zone_net_.0.weight': r(h, obs_dim + zone_dim, sc=0.4), 'zone_net_.0.bias': r(h, sc=0.2),
            'zone_net_.2.weight': r(h, h, sc=0.1), 'zone_net_.2.bias': r(h, sc=0.2),
            'zone_net_.4.weight': r(h, h, sc=0.1), 'zone_net_.4.bias': r(h, sc=0.2),
            'combine_net_.weight': r(h, obs_dim + h, sc=0.1), 'combine_net_.bias': r(h, sc=0.1)}


def _twins(crl, env_id, num_steps, capacity=None):
    """Two envs with the same seeds and short episodes, one Rollout of each store."""
    from combinatorial_rl_tasks_b200.rollout import Rollout
    env, twin = crl.ZoneVecEnv(env_id, B), crl.ZoneVecEnv(env_id, B)
    for e in (env, twin):
        e.seed(4242)
        e.cfg.num_steps = num_steps
    return (Rollout(env, T, store='frames', layout_capacity=capacity), Rollout(twin, T, store='zone_obs'))


def _collect(ro, tw, rs, check=True):
    """One rollout of both twins with the same actions; returns (next value, the frames rollout's exps)."""
    env, twin = ro.env, tw.env
    o, o2 = ro.begin(), tw.begin()
    for t in range(T):
        a = torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda()
        v = torch.from_numpy(rs.normal(0, 2, B).astype(np.float32)).cuda()
        if env.spec.goals:
            for e in (env, twin):
                need = e.needs_goal()
                e.set_goal(torch.where(need, torch.full((B,), t % env.spec.num_zones, dtype=torch.int32, device='cuda'),
                                       torch.full((B,), -1, dtype=torch.int32, device='cuda')))
        o, r, d, info = ro.step(t, a, v, torch.zeros(B, 2, device='cuda'))
        o2, r2, d2, i2 = tw.step(t, a, v, torch.zeros(B, 2, device='cuda'))
        if check:
            assert torch.equal(r, r2) and torch.equal(d, d2), t
    return torch.from_numpy(rs.normal(0, 2, B).astype(np.float32)).cuda()


@pytest.mark.parametrize('env_id', ['PointTSP-v0', 'PointTTSP-v0', 'ColourMatch-v0', 'PointTSP-v5', 'walled/PointTSP-v0',
                                    'PointTSP-v3'])
def test_frames_rebuild_the_twins_rows(crl, env_id):
    # a TimedTSP episode ends at the first zone that times out, a few steps in when num_steps is 24: room for a reset
    # of every env at every step, so that no frame here is an overflowed one
    ro, tw = _twins(crl, env_id, 24, capacity=B * (T + 1))
    rs = np.random.RandomState(5)
    for k in range(2):                                    # the second rollout carries slot T over
        nv = _collect(ro, tw, rs)
        for t in range(T + 1):
            assert torch.equal(_bits(ro.obs[t]), _bits(tw.obs[t])), (k, t)
            assert torch.equal(ro.result[t], tw.result[t]), (k, t)
            assert (ro.frames[t, :, 1] != -1).all(), (k, t)                 # every record has its layout entry
            rows = ro.obs_at(t)['zone_frames'].zone_obs()
            assert torch.equal(_bits(rows), _bits(tw.zone_obs[t])), (k, t)
        if ro.shaped is not None:
            assert torch.equal(_bits(ro.shaped), _bits(tw.shaped))
        # envs that reset at least twice inside this rollout, so a layout entry is taken more than once per env
        assert (ro.dones.sum(0) >= 2).any(), k
        exps, exps2 = ro.finish(nv), tw.finish(nv)
        assert torch.equal(_bits(exps['advantage']), _bits(exps2['advantage'])), k
        assert torch.equal(_bits(exps['returnn']), _bits(exps2['returnn'])), k
        flat, flat2 = ro.finish(nv, flatten=True), tw.finish(nv, flatten=True)
        assert torch.equal(_bits(flat['obs']['zone_frames'].zone_obs()), _bits(flat2['obs']['zone_obs'])), k
        assert torch.equal(_bits(flat['obs']['obs']), _bits(flat2['obs']['obs'])), k
    sb, sb2 = ro.storage_bytes(), tw.storage_bytes()
    assert 'zone_obs' not in sb and sb2['zone_obs'] == (T + 1) * B * env_spec_row_bytes(ro.env)
    assert sb['frames'] == (T + 1) * B * 16


def env_spec_row_bytes(env):
    return 4 * env.spec.num_zones * env.spec.zone_dim


@pytest.fixture(scope='module')
def pointtsp_rollout(crl):
    """A PointTSP pair after two rollouts (the second carried over)."""
    ro, tw = _twins(crl, 'PointTSP-v0', 24, capacity=B * (2 + T // 24 + 1))
    rs = np.random.RandomState(9)
    for _ in range(2):
        nv = _collect(ro, tw, rs, check=False)
    ro.finish(nv)
    return ro, tw


def test_forward_from_frames_equals_forward_on_rows(crl, pointtsp_rollout):
    from combinatorial_rl_tasks_b200.rollout import ZoneFrames
    ro, tw = pointtsp_rollout
    enc = crl.ZoneEncoder(_state_dict(8, 6, 185), num_zones=15)
    obs = ro.obs.reshape(-1, 8)
    frames = ZoneFrames(ro.frames.reshape(-1, 4), ro.layout_xy, ro.layout_tmax, ro.env.cfg)
    rows = frames.zone_obs()
    assert torch.equal(_bits(rows), _bits(tw.zone_obs.reshape(-1, 15, 6)))
    g = torch.Generator(device='cuda').manual_seed(1)
    for idx in (None, torch.randint(0, (T + 1) * B, (T * B // 10,), device='cuda', generator=g),
                torch.tensor([77], device='cuda')):
        o = obs if idx is None else obs[idx].contiguous()
        f = frames if idx is None else frames[idx]
        z = rows if idx is None else rows[idx].contiguous()
        a, b = enc.pooled_from_frames(o, f), enc.pooled(o, z)
        assert torch.isfinite(a).all()
        assert torch.equal(_bits(a), _bits(b)), None if idx is None else idx.numel()
        # the whole ZoneEnvModel forward through __call__: the frames dict and the rows dict agree
        y, y2 = enc({'obs': o, 'zone_frames': f}), enc._head(enc.packed_head, o, b)
        assert torch.equal(_bits(y), _bits(y2))
    assert enc.healthy()


def test_backward_from_frames_equals_backward_on_rows(crl, pointtsp_rollout):
    ro, tw = pointtsp_rollout
    exps, exps2 = ro.finish(torch.zeros(B, device='cuda')), tw.finish(torch.zeros(B, device='cuda'))
    flat = lambda x: x.reshape((T * B,) + tuple(x.shape[2:]))
    idx = torch.randint(0, T * B, (T * B // 10,), device='cuda', generator=torch.Generator(device='cuda').manual_seed(3))
    o = flat(exps['obs']['obs'])[idx]
    fr = flat(exps['obs']['zone_frames'])[idx]
    z = flat(exps2['obs']['zone_obs'])[idx]
    assert torch.equal(_bits(fr.zone_obs()), _bits(z))
    # the library entries: dW1, db1, dW2, db2 bit for bit
    model = crl.FusedZoneEnvModel(8, 6, 15, hidden=185)
    model.load_state_dict(_state_dict(8, 6, 185, seed=2))
    core = model._core
    l1, l2 = model.zone_net_[0], model.zone_net_[2]
    core.pack(l1.weight.detach().contiguous(), l1.bias.detach().contiguous(), l2.weight.detach().contiguous(),
              l2.bias.detach().contiguous())
    gp = torch.randn(o.shape[0], 185, device='cuda', generator=torch.Generator(device='cuda').manual_seed(4))
    got = core.backward_frames(o.contiguous(), fr.flat_records(), fr, gp)
    want = core.backward(o.contiguous(), z.contiguous(), gp)
    for a, b, name in zip(got, want, ('dw1', 'db1', 'dw2', 'db2')):
        assert torch.equal(_bits(a), _bits(b)), name
    # FusedZoneEnvModel: every parameter's .grad after one loss.backward(), zone_frames input vs zone_obs input
    grads = []
    for batch in ({'obs': o, 'zone_frames': fr}, {'obs': o, 'zone_obs': z}):
        model.zero_grad(set_to_none=True)
        y = model(batch)
        (y.square().mean() + y[:, :3].sum()).backward()
        grads.append({k: p.grad.clone() for k, p in model.named_parameters()})
    assert grads[0].keys() == grads[1].keys()
    for k in grads[0]:
        assert torch.equal(_bits(grads[0][k]), _bits(grads[1][k])), k
    assert model.healthy()


def test_overflow_raises_and_poisons_only_its_frames(crl):
    ro, tw = _twins(crl, 'PointTSP-v0', 8, capacity=B + 2)
    rs = np.random.RandomState(11)
    nv = _collect(ro, tw, rs)
    with pytest.raises(RuntimeError, match='needed'):
        ro.finish(nv)
    enc = crl.ZoneEncoder(_state_dict(8, 6, 64), num_zones=15)
    from combinatorial_rl_tasks_b200.rollout import ZoneFrames
    frames = ZoneFrames(ro.frames.reshape(-1, 4), ro.layout_xy, ro.layout_tmax, ro.env.cfg)
    obs = ro.obs.reshape(-1, 8)
    a = enc.pooled_from_frames(obs, frames)
    b = enc.pooled(obs, tw.zone_obs.reshape(-1, 15, 6))
    lost = ro.frames.reshape(-1, 4)[:, 1] == -1                    # CRL_FRAME_NO_LAYOUT
    assert lost.any() and not lost.all()
    assert torch.isnan(a[lost]).all()
    assert torch.equal(_bits(a[~lost]), _bits(b[~lost]))
    rows = frames.zone_obs()
    assert torch.isnan(rows[lost]).all()
    assert torch.equal(_bits(rows[~lost]), _bits(tw.zone_obs.reshape(-1, 15, 6)[~lost]))


def test_refusals(crl):
    from combinatorial_rl_tasks_b200 import _lib
    from combinatorial_rl_tasks_b200.rollout import Rollout
    with pytest.raises(ValueError, match='wait'):
        Rollout(crl.ZoneVecEnv('PointTSP-v0', 64, wait=True), 8, store='frames')
    ro = Rollout(crl.ZoneVecEnv('PointTSP-v0', 64), 8, store='frames')
    ro.begin()
    lib = _lib.load()
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    h = 64
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device='cuda')
    out = torch.zeros(64, h, device='cuda')
    call = lambda shape: lib.crl_zone_encode_frames(shape, ro.env.cfg, 64, ro.obs[0].data_ptr(), ro.frames[0].data_ptr(),
                                                    ro.layout_xy.data_ptr(), None, buf.data_ptr(), out.data_ptr(), None, s)
    assert call(_lib.CrlEncoderShape(obs_dim=9, zone_dim=6, hidden=h, num_zones=15)) == -4
    assert call(_lib.CrlEncoderShape(obs_dim=8, zone_dim=6, hidden=h, num_zones=14)) == -2
    enc = crl.ZoneEncoder(_state_dict(8, 6, h), num_zones=14)
    with pytest.raises(AssertionError):
        enc.pooled_from_frames(ro.obs[0], ro.obs_at(0)['zone_frames'])
    model = crl.FusedZoneEnvModel(8, 6, 14, hidden=h)
    with pytest.raises(AssertionError):
        model(ro.obs_at(0))


@pytest.mark.parametrize('extra', [['--fused-train'], ['--fused-encoder'], []], ids=['fused-train', 'fused-encoder', 'torch'])
def test_example_collect_loop_runs_on_frames(crl, extra):
    """examples/collect_ppo.py --store frames: three updates, with the fused training model, the fused collection
    encoder and the plain torch policy (which materialises the rows)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'examples', 'collect_ppo.py'), '--envs', '2048', '--frames', '16',
                          '--updates', '3', '--env', 'PointTTSP-v0', '--store', 'frames'] + extra,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = out.stdout.splitlines()
    assert sum(l.startswith('update ') for l in lines) == 3 and 'nan' not in out.stdout and 'storage (frames)' in out.stdout
