"""crl_copy_envs / ZoneVecEnv.copy_envs_from / snapshot: an env copied from another takes the same actions to the same
outputs and state, bit for bit, through auto-resets; a snapshot restores that state on any envs."""
import importlib.util
import os
import zlib

import numpy as np
import pytest

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

B = 4 * 33                    # ragged against 32
BD = 4 * 50                   # the larger dst
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLANES = ('pose', 'aux', 'zone_tmax', 'cooldown', 'seeds', 'episode', 'origin', 'goal')
OUTPUTS = ('obs', 'zone_obs', 'result', 'shaped_reward')


@pytest.fixture(scope='module')
def crl():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    import combinatorial_rl_tasks_b200 as m
    return m


def _bits(x):
    x = x.contiguous()
    return x.view(torch.int32) if x.element_size() == 4 else x.view(torch.uint8)


def _make(crl, env_id, n, seed, num_steps, **kw):
    env = crl.ZoneVecEnv(env_id, n, **kw)
    env.seed(seed)
    env.cfg.num_steps = num_steps
    env.reset()
    return env


def _rows(env, name, ids):
    """Rows ``ids`` of a per-env plane or output of an env (or snapshot), as raw bits."""
    t = getattr(env, name)
    if t is None:
        return None
    if name == 'zone_xy':
        return _bits(t[:, ids])
    if name == 'zone_tmax':
        return t[:, ids].contiguous()
    return _bits(t[ids])


def _assert_same(dst, did, src, sid, names, where):
    for k in names:
        a, b = _rows(dst, k, did), _rows(src, k, sid)
        assert (a is None) == (b is None), (k, where)
        if a is not None:
            assert torch.equal(a, b), (k, where)


def _goals(env, rs):
    return torch.from_numpy(rs.randint(-1, env.spec.num_zones, env.num_envs).astype(np.int32)).cuda()


CASES = [('PointTSP-v0', {}), ('PointTTSP-v0', {}), ('ColourMatch-v0', {}), ('PointTSP-v1', {}), ('PointTSP-v5', {}),
         ('PointTSP-v3', {}), ('walled/PointTSP-v0', {}), ('PointTSP-v0', {'wait': True})]


@pytest.mark.parametrize('rows', ['current', 'stale'])
@pytest.mark.parametrize('env_id,kw', CASES, ids=[c[0] + ('-wait' if c[1] else '') for c in CASES])
def test_continuation_is_bit_identical(crl, env_id, kw, rows):
    num_steps = 24
    rs = np.random.RandomState(zlib.crc32(f'{env_id} {rows} {kw}'.encode()))
    src = _make(crl, env_id, B, 4242, num_steps, **kw)
    dst = _make(crl, env_id, BD, 77, num_steps, **kw)
    wait = kw.get('wait', False)
    step = (lambda e, a: e.step_no_reset(a)) if wait else (lambda e, a: e.step(a))
    goals = src.spec.goals
    if rows == 'stale':
        src.write_zone_obs = False                                   # the src's rows fall behind its state
    for _ in range(rs.randint(5, 40)):
        if goals:
            src.set_goal(_goals(src, rs))
        step(src, torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda())
    if rows == 'stale':
        src.write_zone_obs = True
    n = BD - 9                                                       # 9 dst envs stay as they are
    sid = np.concatenate([rs.permutation(B), rs.randint(0, B, n - B)])
    did = rs.permutation(BD)[:n]
    dst.copy_envs_from(src, sid, did)
    assert dst._zone_obs_ok == (rows == 'current')
    sid_t, did_t = torch.from_numpy(sid).cuda(), torch.from_numpy(did).cuda()
    _assert_same(dst, did_t, src, sid_t, PLANES + ('zone_xy', 'obs', 'result', 'shaped_reward'), 'copy')
    if rows == 'current':
        _assert_same(dst, did_t, src, sid_t, ('zone_obs',), 'copy')
    done_any = 0
    for t in range(3 * num_steps + 5):
        a = torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda()
        ad = torch.zeros(BD, 2, device='cuda')
        ad[did_t] = a[sid_t.long()]
        if goals:
            g = _goals(src, rs)
            gd = torch.full((BD,), -1, dtype=torch.int32, device='cuda')
            gd[did_t] = g[sid_t.long()]
            src.set_goal(g)
            dst.set_goal(gd)
        step(src, a)
        step(dst, ad)
        _assert_same(dst, did_t, src, sid_t, OUTPUTS, t)
        done_any += int(src.done.sum())
    assert done_any > 0
    _assert_same(dst, did_t, src, sid_t, PLANES + ('zone_xy',), 'end')
    assert dst.check_state() == [0] * 8


@pytest.mark.parametrize('env_id', ['PointTSP-v0', 'PointTTSP-v0', 'ColourMatch-v0'])
def test_planes_equal_an_indexed_copy(crl, env_id):
    rs = np.random.RandomState(3)
    src, dst = _make(crl, env_id, B, 11, 30), _make(crl, env_id, BD, 12, 30)
    for e in (src, dst):
        for _ in range(17):
            e.step(torch.from_numpy(rs.uniform(-1, 1, (e.num_envs, 2)).astype(np.float32)).cuda())
    dst.prefetch(torch.cuda.current_stream())                        # every slot of dst parked and ready
    sd_src, sd_dst = src.state_dict(), dst.state_dict()
    assert (dst.next_ready != 0).any()
    n = 70
    sid, did = rs.randint(0, B, n), rs.permutation(BD)[:n]
    dst.copy_envs_from(src, sid, did)
    after = dst.state_dict()
    rest = np.setdiff1d(np.arange(BD), did)
    for k in ('pose', 'aux', 'zone_xy', 'zone_tmax', 'cooldown', 'seeds', 'episode', 'origin', 'goal') + OUTPUTS:
        if sd_src.get(k) is None:
            continue
        if k in ('zone_xy', 'zone_tmax'):
            assert torch.equal(after[k][:, did], sd_src[k][:, sid]), k
            assert torch.equal(after[k][:, rest], sd_dst[k][:, rest]), k
        else:
            assert torch.equal(after[k][did], sd_src[k][sid]), k
            assert torch.equal(after[k][rest], sd_dst[k][rest]), k
    assert (dst.next_ready[:, did] == 0).all()
    assert torch.equal(after['counters_dev'], sd_dst['counters_dev'])
    assert torch.equal(src.state_dict()['counters_dev'], sd_src['counters_dev'])
    assert int(dst.copy_rejects.item()) == 0


@pytest.mark.parametrize('env_id', ['PointTSP-v0', 'PointTTSP-v0', 'ColourMatch-v0'])
def test_snapshot_and_restore(crl, env_id):
    rs = np.random.RandomState(8)
    env = _make(crl, env_id, B, 99, 40)
    for _ in range(9):
        env.step(torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda())
    ids = rs.permutation(B)[:40]
    others = np.setdiff1d(np.arange(B), ids)[:40]
    snap = env.snapshot(ids)
    assert snap.num_envs == 40 and snap.zone_obs_ok and snap.nbytes() > 0
    acts, first = [], []
    for _ in range(200):
        a = torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda()
        env.step(a)
        acts.append(a[ids])
        first.append({k: _rows(env, k, ids).clone() for k in OUTPUTS})
    env.copy_envs_from(snap, None, ids)
    env.copy_envs_from(snap, None, others)
    assert env._zone_obs_ok                                          # the restored rows are current
    for t in range(200):
        a = torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda()
        a[ids], a[others] = acts[t], acts[t]
        env.step(a)
        for k in OUTPUTS:
            assert torch.equal(_rows(env, k, ids), first[t][k]), (k, t)
            assert torch.equal(_rows(env, k, others), first[t][k]), (k, t)
    assert env.check_state() == [0] * 8


def test_in_place_permutation(crl):
    rs = np.random.RandomState(4)
    env = _make(crl, 'ColourMatch-v0', B, 5, 50)
    for _ in range(23):
        env.step(torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda())
    sd = env.state_dict()
    perm = rs.permutation(B)
    env.copy_envs_from(env, perm, np.arange(B))
    after = env.state_dict()
    for k in ('pose', 'aux', 'zone_xy', 'cooldown', 'seeds', 'episode', 'origin', 'goal') + OUTPUTS:
        if k == 'zone_xy':
            assert torch.equal(after[k], sd[k][:, perm]), k
        else:
            assert torch.equal(after[k], sd[k][perm]), k


def test_device_ids_out_of_range_are_skipped_and_counted(crl):
    rs = np.random.RandomState(6)
    src, dst = _make(crl, 'PointTTSP-v0', B, 21, 40), _make(crl, 'PointTTSP-v0', BD, 22, 40)
    for _ in range(5):
        src.step(torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda())
    sid = torch.tensor([0, 5, -1, B, 7, 9, 3], dtype=torch.int32, device='cuda')
    did = torch.tensor([10, BD, 11, 12, -4, 13, 14], dtype=torch.int32, device='cuda')
    before = dst.state_dict()
    dst.copy_envs_from(src, sid, did)
    assert int(dst.copy_rejects.item()) == 4
    after = dst.state_dict()
    for k in ('pose', 'aux', 'seeds', 'obs', 'zone_obs', 'result'):
        assert torch.equal(after[k][[11, 12]], before[k][[11, 12]]), k           # their src id was out of range
        assert torch.equal(after[k][[10, 13, 14]], src.state_dict()[k][[0, 9, 3]]), k
    # within one env, through the snapshot: a rejected src id still leaves its dst alone, and is counted once
    sd = dst.state_dict()
    dst.copy_envs_from(dst, torch.tensor([1, BD + 1, 2], dtype=torch.int64, device='cuda'),
                       torch.tensor([20, 21, 22], dtype=torch.int64, device='cuda'))
    assert int(dst.copy_rejects.item()) == 5
    after = dst.state_dict()
    for k in ('pose', 'aux', 'seeds', 'zone_obs'):
        assert torch.equal(after[k][21], sd[k][21]), k
        assert torch.equal(after[k][[20, 22]], sd[k][[1, 2]]), k


def test_fixed_range_matches_until_the_episode_ends(crl):
    rs = np.random.RandomState(10)
    kw = dict(seed_mode='fixed_range', min_seed=1, max_seed=50)
    src = _make(crl, 'PointTSP-v0', B, 1, 20, **kw)
    dst = _make(crl, 'PointTSP-v0', BD, 1, 20, env_offset=1000, **kw)
    for _ in range(7):
        src.step(torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda())
    sid, did = np.arange(B), rs.permutation(BD)[:B]
    dst.copy_envs_from(src, sid, did)
    did_t = torch.from_numpy(did).cuda()
    live = torch.ones(B, dtype=torch.bool, device='cuda')
    for t in range(30):
        a = torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda()
        ad = torch.zeros(BD, 2, device='cuda')
        ad[did_t] = a
        src.step(a)
        dst.step(ad)
        same = (_bits(dst.result[did_t]) == _bits(src.result)).all(1)
        assert bool((same | ~live).all()), t
        done = src.done.clone()
        same_obs = (_bits(dst.obs[did_t]) == _bits(src.obs)).all(1)
        assert bool((same_obs | ~live | done).all()), t
        live &= ~done
    assert not bool(live.any())                                      # every episode ended within the window


def test_step_host_after_a_copy(crl):
    rs = np.random.RandomState(12)
    for env_id in ('PointTSP-v0', 'PointTTSP-v0'):
        src, dst = _make(crl, env_id, B, 31, 30), _make(crl, env_id, BD, 32, 30)
        for _ in range(6):
            src.step(torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda())
        dst.step_host(rs.uniform(-1, 1, (BD, 2)).astype(np.float32))  # the host mirror is live before the copy
        sid, did = rs.randint(0, B, 100), rs.permutation(BD)[:100]
        dst.copy_envs_from(src, sid, did)
        for t in range(40):
            a = rs.uniform(-1, 1, (B, 2)).astype(np.float32)
            ad = rs.uniform(-1, 1, (BD, 2)).astype(np.float32)
            ad[did] = a[sid]
            src.step(torch.from_numpy(a).cuda())
            obs, reward, done, _ = dst.step_host(ad)
            torch.cuda.synchronize()
            assert np.array_equal(obs['obs'][did].view(np.int32), src.obs[sid].cpu().numpy().view(np.int32)), t
            assert np.array_equal(np.ascontiguousarray(obs['zone_obs'][did]).view(np.int32),
                                  src.zone_obs[sid].cpu().numpy().view(np.int32)), t
            assert np.array_equal(reward[did].view(np.int32), src.reward[sid].cpu().numpy().view(np.int32)), t
            assert np.array_equal(done[did], src.done[sid].cpu().numpy()), t


def test_frames_rollout_refuses_a_copied_env(crl):
    from combinatorial_rl_tasks_b200.rollout import Rollout
    env = _make(crl, 'PointTSP-v0', B, 41, 30)
    ro = Rollout(env, 8, store='frames')
    ro.begin()
    a = torch.zeros(B, 2, device='cuda')
    ro.step(0, a)
    snap = env.snapshot([1, 2])
    env.copy_envs_from(snap, None, [5, 6])
    with pytest.raises(RuntimeError, match='copied'):
        ro.step(1, a)
    ro.begin()                                                       # a new rollout starts from the copied state
    ro.step(0, a)


def test_lookahead_example_runs(crl, capsys):
    spec = importlib.util.spec_from_file_location('lookahead', os.path.join(ROOT, 'examples', 'lookahead.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    res = mod.main(['--envs', '8', '--branches', '4', '--horizon', '5', '--steps', '12'])
    assert set(res) >= {'mpc_return', 'random_return'}
    assert 'random' in capsys.readouterr().out
