"""Device reset (Philox), auto-reset, ragged batches, sharding independence and
size-independent properties at the BASELINE.json sizes.  All through the C ABI."""
import numpy as np
import pytest

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

from oracle import c_oracle as co  # noqa: E402

TASKS = ['PointTSP-v0', 'PointTTSP-v0', 'ColourMatch-v0']


@pytest.fixture(scope='module')
def crl():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    import combinatorial_rl_tasks_b200 as m
    return m


def bits_of(env):
    return env.aux[:, 3].view(torch.int32).cpu().numpy().astype(np.int64) & 0xffffffff


def tmax_of(env):
    w = env.zone_tmax.cpu().numpy().astype(np.int64) & 0xffffffff          # (ceil(N/2), B)
    N = env.spec.num_zones
    return np.stack([w & 0xffff, w >> 16], 1).reshape(-1, w.shape[1])[:N].T  # (B, N)


def cooldown_of(env):
    return env.cooldown.cpu().numpy().view(np.uint8).reshape(env.num_envs, 8)[:, :env.spec.num_zones]


def snapshot(env):
    keys = ['pose', 'aux', 'zone_xy', 'zone_tmax', 'cooldown', 'seeds', 'episode', 'origin', 'obs', 'zone_obs', 'result']
    return {k: getattr(env, k).clone() for k in keys if getattr(env, k) is not None}


@pytest.mark.parametrize('env_id', TASKS)
def test_device_reset_matches_design_twin(crl, env_id):
    """crl_reset (Philox on the device, one warp per env) against the sequential twin in
    oracle/crl_oracle.c: layouts, headings, colours bit-exact; timeouts (fp64 log/cos on
    both sides) equal."""
    B = 500                                      # ragged: last warp holds 20 envs
    env = crl.ZoneVecEnv(env_id, B)
    env.seed(1000)
    obs = env.reset()
    torch.cuda.synchronize()
    origin, zxy = env.origin.cpu().numpy(), env.zone_xy.cpu().numpy()
    bits = bits_of(env)
    assert np.all(env.seeds.cpu().numpy() == 1001 + np.arange(B)) and np.all(env.episode.cpu().numpy() == 1)
    mism = 0
    for i in list(range(0, 64)) + list(range(B - 40, B)):
        tw = co.philox_reset(env_id, 1000 + i)
        assert np.array_equal(origin[i, :2], tw['xy0']) and origin[i, 2] == np.float32(tw['rot0']), i
        assert np.array_equal(zxy[:, i, :], tw['zone_xy']), i
        if env_id == 'PointTTSP-v0':
            mism += int(np.sum(tmax_of(env)[i] != tw['zone_max_steps']))
        if env_id == 'ColourMatch-v0':
            col = [(bits[i] >> 16 >> (2 * k)) & 3 for k in range(6)]
            assert col == list(tw['colours']), i
    assert mism == 0
    o = obs['obs'].cpu().numpy()
    assert np.all(o[:, 0] == 1.0) and np.all(o[:, 5:] == 0.0)
    assert np.allclose(o[:, 1:3] * 3, origin[:, :2], atol=1e-6)
    assert np.allclose(o[:, 3], np.cos(origin[:, 2]), atol=1e-6) and np.allclose(o[:, 4], np.sin(origin[:, 2]), atol=1e-6)


def test_fixed_range_seed_mode(crl):
    """FixedSeedsWrapper semantics: every reset re-seeds uniformly in [min_seed, max_seed];
    the same seed always builds the same map."""
    B = 256
    env = crl.ZoneVecEnv('PointTSP-v0', B, seed_mode='fixed_range', min_seed=1, max_seed=5, env_offset=4096)
    env.reset()
    torch.cuda.synchronize()
    seeds = env.seeds.cpu().numpy() - 1                     # Engine.reset left seed + 1 behind
    assert set(seeds) <= {1, 2, 3, 4, 5} and len(set(seeds)) == 5
    zxy, origin = env.zone_xy.cpu().numpy(), env.origin.cpu().numpy()
    for s in range(1, 6):
        idx = np.where(seeds == s)[0]
        tw = co.philox_reset('PointTSP-v0', 0, seed_mode=1, min_seed=s, max_seed=s)
        for i in idx[:5]:
            assert np.array_equal(zxy[:, i, :], tw['zone_xy']) and np.array_equal(origin[i, :2], tw['xy0'])
    # the chooser is keyed by the GLOBAL env index and the episode number
    tw = co.philox_reset('PointTSP-v0', 0, seed_mode=1, min_seed=1, max_seed=5, global_env=4096 + 17, episode=0)
    assert tw['seed_after'] - 1 == seeds[17]


@pytest.mark.parametrize('env_id', TASKS)
def test_auto_reset_semantics(crl, env_id):
    """penv.py:9-10: a finished env restarts inside step(); the returned obs is the new
    episode's first observation, reward/done/goal_met are the finished step's."""
    B = 2048
    env = crl.ZoneVecEnv(env_id, B)
    env.seed(50000)
    env.reset()
    # make episodes end soon: put every env a few steps before the step limit
    bits = env.aux[:, 3].view(torch.int32)
    start = torch.randint(1960, 1999, (B,), device='cuda', dtype=torch.int32)
    bits.copy_((bits & ~0xffff) | start)
    n_done = 0
    seen_done = torch.zeros(B, dtype=torch.bool, device='cuda')
    for t in range(45):
        seeds_before, ep_before = env.seeds.clone(), env.episode.clone()
        obs, reward, done, info = env.step_random(action_seed=9)
        d = done.clone()
        n_done += int(d.sum())
        seen_done |= d
        if d.any():
            idx = torch.where(d)[0]
            o = obs['obs'][idx].cpu().numpy()
            assert np.all(o[:, 0] == 1.0) and np.all(o[:, 5:] == 0.0)             # fresh episode
            assert torch.all(env.steps[idx] == 0)
            assert torch.all(env.seeds[idx] == seeds_before[idx] + 1)               # Engine: _seed += 1
            assert torch.all(env.episode[idx] == ep_before[idx] + 1)
            i = int(idx[0])
            tw = co.philox_reset(env_id, int(seeds_before[i]))
            assert np.array_equal(env.zone_xy[:, i, :].cpu().numpy(), tw['zone_xy'])
            assert np.array_equal(obs['zone_obs'][i, :, 0:2].cpu().numpy(),
                                  (tw['zone_xy'] * np.float32(1.0 / 3.0)).astype(np.float32))
        nd = torch.where(~d)[0]
        assert torch.all(env.seeds[nd] == seeds_before[nd])                       # untouched envs
    assert bool(seen_done.all())
    c = env.counters()
    assert c['episodes'] == n_done and c['length_sum'] >= 2000 * n_done * 0.3
    # step_no_reset leaves finished envs alone
    env2 = crl.ZoneVecEnv(env_id, 64)
    env2.reset()
    b2 = env2.aux[:, 3].view(torch.int32)
    b2.copy_((b2 & ~0xffff) | 1999)
    z_before = env2.zone_xy.clone()
    obs, reward, done, info = env2.step_no_reset(torch.zeros(64, 2, device='cuda'))
    assert bool(done.all()) and torch.equal(env2.zone_xy, z_before) and torch.all(env2.steps == 2000)
    assert torch.all(obs['obs'][:, 0] == 0.0)


@pytest.mark.parametrize('env_id', TASKS)
def test_ragged_batch_equals_prefix_of_full_batch(crl, env_id):
    """B not a multiple of 32 (and of 4: the bulk copy falls back to plain stores)."""
    full = crl.ZoneVecEnv(env_id, 128)
    full.seed(7); full.reset()
    acts = torch.rand(40, 128, 2, device='cuda') * 2 - 1
    for B in (1, 33, 99, 100):
        env = crl.ZoneVecEnv(env_id, B)
        env.seed(7); env.reset()
        ref = crl.ZoneVecEnv(env_id, 128)
        ref.seed(7); ref.reset()
        for t in range(40):
            env.step(acts[t, :B].contiguous())
            ref.step(acts[t])
        a, b = snapshot(env), snapshot(ref)
        for k in a:
            if k == 'zone_xy' or k == 'zone_tmax':
                assert torch.equal(a[k], b[k][:, :B]), (B, k)
            else:
                assert torch.equal(a[k], b[k][:B]), (B, k)


def test_sharding_independence(crl):
    """Two shards with env_offset 0 / 1024 == one batch of 2048: Philox counters use the
    global env index, so results do not depend on the GPU count."""
    env_id = 'PointTTSP-v0'
    whole = crl.ZoneVecEnv(env_id, 2048, seed_mode='fixed_range', min_seed=1, max_seed=100)
    parts = [crl.ZoneVecEnv(env_id, 1024, seed_mode='fixed_range', min_seed=1, max_seed=100, env_offset=o)
             for o in (0, 1024)]
    for e in [whole] + parts:
        e.reset()
    for t in range(60):
        whole.step_random(action_seed=4)
        for e in parts:
            e._step_index = whole._step_index - 1
            e.step_random(action_seed=4)
    for k in ('pose', 'aux', 'obs', 'zone_obs', 'result', 'seeds'):
        assert torch.equal(getattr(whole, k), torch.cat([getattr(e, k) for e in parts])), k
    assert torch.equal(whole.zone_xy, torch.cat([e.zone_xy for e in parts], dim=1))


def test_step_host_equals_device_step(crl):
    env_a = crl.ZoneVecEnv('ColourMatch-v0', 300); env_a.seed(3); env_a.reset()
    env_b = crl.ZoneVecEnv('ColourMatch-v0', 300); env_b.seed(3); env_b.reset()
    rs = np.random.RandomState(0)
    for t in range(25):
        a = rs.uniform(-1, 1, (300, 2)).astype(np.float32)
        obs_h, rew_h, done_h, info_h = env_a.step_host(a)
        obs_d, rew_d, done_d, info_d = env_b.step(torch.from_numpy(a).cuda())
        assert np.array_equal(obs_h['obs'], obs_d['obs'].cpu().numpy())
        assert np.array_equal(obs_h['zone_obs'], obs_d['zone_obs'].cpu().numpy())
        assert np.array_equal(rew_h, rew_d.cpu().numpy()) and np.array_equal(done_h, done_d.cpu().numpy())


def test_step_host_no_reset_wait_equals_device_step_no_reset(crl):
    """step_host(auto_reset=False, wait=True) -- its own prepared call object -- against step_no_reset of a WaitWrapper
    env on the device: parked envs (zero observation, reward 0, done) included; then an auto-reset host step."""
    B = 256
    env_a = crl.ZoneVecEnv('PointTSP-v0', B, wait=True); env_a.seed(5); env_a.cfg.num_steps = 12; env_a.reset()
    env_b = crl.ZoneVecEnv('PointTSP-v0', B, wait=True); env_b.seed(5); env_b.cfg.num_steps = 12; env_b.reset()
    rs = np.random.RandomState(1)
    for t in range(30):
        a = rs.uniform(-1, 1, (B, 2)).astype(np.float32)
        last = t % 15 == 14                               # hier_base.py:180-183: skill_len - 1 step_no_reset, then step
        obs_h, rew_h, done_h, _ = env_a.step_host(a, auto_reset=last, wait=True)
        obs_d, rew_d, done_d, _ = (env_b.step if last else env_b.step_no_reset)(torch.from_numpy(a).cuda())
        assert np.array_equal(obs_h['obs'], obs_d['obs'].cpu().numpy()), t
        assert np.array_equal(obs_h['zone_obs'], obs_d['zone_obs'].cpu().numpy()), t
        assert np.array_equal(rew_h, rew_d.cpu().numpy()) and np.array_equal(done_h, done_d.cpu().numpy()), t
        if t == 13:
            assert done_h.all() and not obs_h['obs'].any()     # everyone parked after the 12-step episodes
    assert len(env_a._host_calls) == 2
    env_a.close()
    assert not env_a._host_calls


@pytest.mark.parametrize('actions', ['numpy', 'host_actions', 'pinned_actions'])
@pytest.mark.parametrize('env_id', TASKS + ['PointTTSP-v3', 'ColourMatch-v3'])     # -v3: the EXT kernels (shaped_reward too)
def test_step_host_delta_is_byte_identical_to_full_copy(crl, env_id, actions):
    """The host-direct step (crl_host_call_step: one kernel; the step writes obs / result / changed rows into the pinned
    host buffers itself) moves only the zone_obs rows and result records that changed; what the caller sees in its
    host buffers must be byte for byte what crl_step_host (full copy) delivers -- across zone events, cooldown ticks,
    timeouts and auto-resets (episodes cut short to force many).  The actions come from an ordinary numpy array (copied
    into the env's pinned buffer), from that buffer filled in place (host_actions()) or from a rotation of
    pinned_actions() arrays that the kernel reads where they lie."""
    B = 1000
    envs = []
    for _ in range(2):
        e = crl.ZoneVecEnv(env_id, B); e.seed(11); e.cfg.num_steps = 40; e.reset(); envs.append(e)
    full, delta = envs
    pinned = delta.pinned_actions(4)
    rs = np.random.RandomState(5)
    moved = []
    for t in range(130):
        a = rs.uniform(-1, 1, (B, 2)).astype(np.float32)
        if t == 70:                                   # device-side work in between invalidates the mirror
            for e in envs:
                e.step(torch.from_numpy(a).cuda())
            continue
        if t == 20:                                   # put 200 robots on zone 3: events through the delta path
            for e in envs:
                e.pose[:200, :2] = e.zone_xy[3, :200, :]
        of, rf, df, inf_ = full.step_host(a, delta=False)
        ad = {'numpy': a, 'host_actions': delta.host_actions(), 'pinned_actions': pinned[t % 4]}[actions]
        if ad is not a:
            ad[:] = a
        od, rd, dd, ind = delta.step_host(ad, delta=True)
        rows = delta.delta_rows if delta.delta_rows >= 0 else delta.host_rows_moved(reset=True)   # -1: counted on the device
        if t == 20:
            assert rows >= 200 and (env_id.startswith('ColourMatch') or int((ind['event'] != 0).sum()) >= 200)
        assert np.array_equal(of['zone_obs'].view(np.uint32), od['zone_obs'].view(np.uint32)), t
        assert np.array_equal(of['obs'].view(np.uint32), od['obs'].view(np.uint32)), t
        assert np.array_equal(rf.view(np.uint32), rd.view(np.uint32)) and np.array_equal(df, dd), t
        assert np.array_equal(inf_['event'], ind['event']) and np.array_equal(inf_['goal_met'], ind['goal_met'])
        if 'shaped_reward' in ind:
            assert np.array_equal(inf_['shaped_reward'], ind['shaped_reward']) and np.array_equal(inf_['need_next_goal'], ind['need_next_goal'])
        assert np.array_equal(od['zone_obs'], delta.zone_obs.cpu().numpy()), t
        moved.append(rows)
    assert moved[0] == B and moved[70] == B           # first call and the call after device-side work: full copy
    # result records cross only when they differ from what the host holds: far fewer than one per env and step
    # (equality with the full copy was checked at every step above)
    assert 0 < delta.host_results_moved() < 128 * B // 3
    # between the step-limit resets only a few rows move (TimedTSP: its 40-step episodes also end on timeouts; its
    # time-left column is a plane of its own in the plane-major mirror and is not counted as a row)
    assert max(moved[1:39]) < (B // 2 if env_id.startswith('PointTTSP') else B // 4)
    if not env_id.startswith('PointTTSP'):                  # (TimedTSP's episodes are desynchronised by their timeouts long before)
        assert B in moved[39:42] or max(moved[38:42]) >= B // 2   # the step-limit reset rewrites every row


@pytest.mark.parametrize('env_id,B', [('PointTSP-v0', 65536), ('PointTTSP-v0', 262144), ('ColourMatch-v0', 262144)])
def test_full_size_properties(crl, env_id, B):
    """BASELINE.json configs 2-4 at full size: invariants that hold at any size."""
    env = crl.ZoneVecEnv(env_id, B)
    env.seed(123)
    env.reset()
    N, Z = env.spec.num_zones, env.spec.zone_dim
    n_done, ret_sum = 0, 0.0
    ep_ret = torch.zeros(B, device='cuda')
    hamming0 = None
    if env_id == 'ColourMatch-v0':
        col = (torch.from_numpy(bits_of(env)).cuda() >> 16).unsqueeze(1) >> (2 * torch.arange(N, device='cuda')) & 3
        nb, ng, nr = [(col == c).sum(1) for c in range(3)]
        hamming0 = torch.minimum(torch.minimum(2 * ng + nr, 2 * nr + nb), 2 * nb + ng)
    # shorten episodes so that auto-resets happen within the test
    bits = env.aux[:, 3].view(torch.int32)
    bits.copy_((bits & ~0xffff) | torch.randint(1700, 1990, (B,), device='cuda', dtype=torch.int32))
    for t in range(320):
        obs, reward, done, info = env.step_random(action_seed=77)
        ep_ret += reward
        n_done += int(done.sum())
        ret_sum += float(ep_ret[done].double().sum())
        ep_ret[done] = 0
    torch.cuda.synchronize()
    assert env.check_state() == [0] * 8                     # crl_check_state: no invariant violated anywhere
    c = env.counters()
    assert c['episodes'] == n_done and n_done >= B
    assert abs(c['return_sum'] - ret_sum) <= 1e-3 * max(1.0, abs(ret_sum))
    bits_np = bits_of(env)
    steps, hi = bits_np & 0xffff, bits_np >> 16
    o, z = env.obs.cpu().numpy(), env.zone_obs.cpu().numpy()
    assert np.array_equal(o[:, 0], (1.0 - steps / 2000.0).astype(np.float32))
    assert np.allclose(np.hypot(o[:, 3], o[:, 4]), 1.0, atol=1e-6)
    zxy = env.zone_xy.cpu().numpy().transpose(1, 0, 2)                               # (B, N, 2)
    assert np.allclose(z[:, :, 0:2], zxy / 3.0, atol=1e-6) and np.all(z[:, :, 5] == 0.25)
    pose, aux = env.pose.cpu().numpy(), env.aux.cpu().numpy()
    assert np.all(np.abs(pose[:, 2]) <= np.pi + 1e-5) and np.all(np.isfinite(pose)) and np.all(np.isfinite(aux[:, :3]))
    assert np.all(np.hypot(pose[:, 3], aux[:, 0]) <= 1.5 + 1e-3)                      # terminal speed
    # layouts valid: keepouts and extents
    pts = np.concatenate([env.origin.cpu().numpy()[:, None, :2], zxy], 1).astype(np.float64)[:4096]
    keep = np.array([0.4] + [0.55] * N)
    assert np.all(np.abs(pts) <= (3.0 - keep)[None, :, None] + 1e-5)
    d = np.linalg.norm(pts[:, :, None] - pts[:, None], axis=3)
    iu = np.triu_indices(N + 1, 1)
    assert np.all(d[:, iu[0], iu[1]] >= (keep[:, None] + keep[None])[iu] - 1e-5)
    if env_id == 'ColourMatch-v0':
        colz = (hi[:, None] >> (2 * np.arange(N))) & 3
        assert np.all(colz < 3)
        rgb = np.stack([colz == 2, colz == 1, colz == 0], 2).astype(np.float32)
        assert np.array_equal(z[:, :, 2:5], rgb)
        cd = cooldown_of(env)
        assert cd.max() <= 150 and np.array_equal(z[:, :, 6], cd.astype(np.float32) / np.float32(150))
    else:
        vis = ((hi[:, None] >> np.arange(N)) & 1).astype(bool)
        assert np.array_equal(z[:, :, 2], vis.astype(np.float32)) and np.array_equal(z[:, :, 4], (~vis).astype(np.float32))
        assert np.all(z[:, :, 3] == 1.0)
        # dense TSP reward: the running return of an unfinished episode is its visit count
        assert np.array_equal(aux[:, 2], vis.sum(1).astype(np.float32))
        if env_id == 'PointTTSP-v0':
            tm = tmax_of(env)
            assert np.all((steps[:, None] < tm) | vis)                               # else it would have ended
            want = np.where(vis, np.float32(1.0), ((tm - steps[:, None]) / 2000.0).astype(np.float32))
            assert np.array_equal(z[:, :, 6], want)


@pytest.mark.parametrize('env_id,B', [('PointTSP-v0', 65536), ('PointTTSP-v0', 262144), ('ColourMatch-v0', 262144)])
def test_full_size_sampled_envs_against_the_oracle(crl, env_id, B):
    """BASELINE.json configs 2-4 at FULL size, checked against the oracle directly: 256 envs spread
    over the batch (first and last warp, CTA boundaries, random ones) are stepped by the fp64 oracle
    beside the kernel from identical positions -- events, visited / colour / cooldown state,
    timeouts, done, goal_met and integer rewards bit-exact, rewards 1e-6, observations as in
    test_gpu_parity -- while the whole batch steps in the same launches."""
    from oracle import zone_env as ze
    from tests.test_gpu_parity import REWARD_ATOL, check_obs
    task = ze.TASK_OF_ENV_ID[env_id]
    env = crl.ZoneVecEnv(env_id, B)
    env.seed(4242)
    env.reset()
    N = env.spec.num_zones
    rs = np.random.RandomState(11)
    idx = np.unique(np.concatenate([np.arange(0, 40), np.arange(B - 40, B), np.arange(63, 4096, 64)[:48],
                                    rs.randint(0, B, 160)]))[:256]
    it = torch.from_numpy(idx).cuda()
    # make things happen in the sampled envs: some close to the step limit, some sitting on a zone
    bits = env.aux[:, 3].view(torch.int32)
    near_end = it[::5]
    bits[near_end] = (bits[near_end] & ~0xffff) | torch.randint(1960, 1999, (len(near_end),), device='cuda', dtype=torch.int32)
    refs = []
    zone32 = env.zone_xy[:, it, :].cpu().numpy().astype(np.float64)           # (N, n, 2)
    b0 = bits_of(env)
    tm = tmax_of(env) if task == ze.TTSP else None
    for j, i in enumerate(idx):
        r = ze.ZoneTaskEnv(task)
        lay = {'xy0': np.zeros(2), 'rot0': 0.0, 'zone_xy': zone32[:, j, :]}
        if task == ze.TTSP:
            lay['zone_max_steps'] = tm[i]
        if task == ze.CM:
            lay['colours'] = np.array([(b0[i] >> 16 >> (2 * k)) & 3 for k in range(N)])
        r.reset(layout=lay)
        r.steps = int(b0[i] & 0xffff)
        refs.append(r)
    alive = np.ones(len(idx), dtype=bool)
    n_events = n_done = 0
    for t in range(48):
        if t % 6 == 0:                                                       # teleport a third of them onto a zone
            sel = it[(t // 6) % 3::3]
            z = torch.randint(0, N, (len(sel),), device='cuda')
            env.pose[sel, :2] = env.zone_xy[z, sel, :] + 0.05
        a = torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda()
        pose, aux = env.pose[it].cpu().numpy().astype(np.float64), env.aux[it].cpu().numpy().astype(np.float64)
        obs, reward, done, info = env.step_no_reset(a)
        res = env.result[it].cpu().numpy()
        og, zg = obs['obs'][it].cpu().numpy(), obs['zone_obs'][it].cpu().numpy()
        b1 = bits_of(env)[idx]
        cd = cooldown_of(env)[idx] if task == ze.CM else None
        a_np = a[it].cpu().numpy()
        for j, r in enumerate(refs):
            if not alive[j]:
                continue                                                     # the reference asserts on a finished env
            r.set_state([pose[j, 0], pose[j, 1], pose[j, 2]], [pose[j, 3], aux[j, 0], aux[j, 1]])
            o_ref, r_ref, d_ref, i_ref = r.step(a_np[j])
            where = (env_id, t, int(idx[j]))
            assert bool(res[j, 4]) == d_ref and bool(res[j, 5]) == bool(i_ref.get('goal_met', False)), where
            assert int(res[j, 6:7].view(np.int8)[0]) == r.event, where
            assert abs(float(res[j, :4].view(np.float32)[0]) - r_ref) <= REWARD_ATOL, where
            assert int(b1[j] & 0xffff) == r.steps, where
            if task == ze.CM:
                assert [(int(b1[j]) >> 16 >> (2 * k)) & 3 for k in range(N)] == list(r.colours), where
                assert list(cd[j]) == list(r.cooldown), where
            else:
                assert [bool((int(b1[j]) >> 16 >> k) & 1) for k in range(N)] == list(r.visited), where
            check_obs(task, og[j], zg[j], o_ref['obs'], o_ref['zone_obs'], where)
            n_events += r.event != 0
            if d_ref:
                alive[j] = False
                n_done += 1
    assert n_events >= 20 and n_done >= 20, (n_events, n_done)
    assert env.check_state()[:2] == [0, 0]


@pytest.mark.parametrize('env_id', ['PointTTSP-v0', 'ColourMatch-v0'])
def test_device_sampler_is_distribution_equivalent_to_reference_sampler(crl, env_id):
    """The Philox reset on the device vs Engine.sample_layout / beta / choice on numpy's
    legacy stream (the oracle's C twin): two-sample Kolmogorov-Smirnov / chi-square tests
    on the statistics a layout is made of.  Different streams, same distribution."""
    from scipy import stats
    n = 6000
    env = crl.ZoneVecEnv(env_id, n)
    env.seed(424242)
    env.reset()
    torch.cuda.synchronize()
    N = env.spec.num_zones
    g_xy0 = env.origin[:, :2].cpu().numpy().astype(np.float64)
    g_rot = env.origin[:, 2].cpu().numpy().astype(np.float64)
    g_z = env.zone_xy.cpu().numpy().transpose(1, 0, 2).astype(np.float64)
    r_xy0, r_rot, r_z, r_tm, r_col = [], [], [], [], []
    c = co.CEnv(env_id)
    for s in range(n):
        c.seed(7000000 + s)
        c.reset()
        lay = c.layout()
        r_xy0.append(lay['xy0']); r_rot.append(lay['rot0']); r_z.append(lay['zone_xy'])
        r_tm.append(lay.get('zone_max_steps', np.zeros(N))); r_col.append(lay.get('colours', np.zeros(N)))
    r_xy0, r_rot, r_z = np.array(r_xy0), np.array(r_rot), np.array(r_z)

    def ks(a, b, what):
        p = stats.ks_2samp(np.ravel(a), np.ravel(b)).pvalue
        assert p > 1e-4, (what, p)

    ks(g_xy0[:, 0], r_xy0[:, 0], 'robot x'); ks(g_xy0[:, 1], r_xy0[:, 1], 'robot y'); ks(g_rot, r_rot, 'robot rot')
    for k in (0, N // 2, N - 1):                 # early, middle and last-placed zone differ in distribution
        ks(g_z[:, k, 0], r_z[:, k, 0], f'zone {k} x'); ks(g_z[:, k, 1], r_z[:, k, 1], f'zone {k} y')
        ks(np.linalg.norm(g_z[:, k] - g_xy0, axis=1), np.linalg.norm(r_z[:, k] - r_xy0, axis=1), f'zone {k} - robot')

    def nearest(z):
        d = np.linalg.norm(z[:, :, None] - z[:, None], axis=3) + np.eye(z.shape[1]) * 1e9
        return d.min(2)
    ks(nearest(g_z), nearest(r_z), 'nearest-neighbour distance')
    ks(np.abs(g_z).max(2), np.abs(r_z).max(2), 'distance to the arena edge')
    if env_id == 'PointTTSP-v0':
        ks(tmax_of(env), np.array(r_tm), 'zone_max_steps ~ int(Beta(3,1.5)*2000)')
    else:
        bits = bits_of(env) >> 16
        g_col = (bits[:, None] >> (2 * np.arange(N))) & 3
        obs_counts = np.array([np.bincount(g_col.ravel(), minlength=3), np.bincount(np.array(r_col).astype(int).ravel(), minlength=3)])
        assert stats.chi2_contingency(obs_counts)[1] > 1e-4


@pytest.mark.parametrize('env_id', TASKS)
def test_prefetched_resets_equal_inline_resets(crl, env_id):
    """A reset served from a parked (prefetched) layout and a reset sampled inline give
    bit-identical state: the layout is a pure function of the seed.  Also checks that the
    parked path is the one taken when slots are full, and that re-seeding invalidates it."""
    B = 1000
    a = crl.ZoneVecEnv(env_id, B, prefetch_every=4)
    b = crl.ZoneVecEnv(env_id, B, prefetch_every=0)
    for e in (a, b):
        e.seed(31337); e.reset()
    torch.cuda.synchronize()
    # a full reset() parks the layouts of the next two resets and consumes the first; `a` then tops
    # its slots up again, `b` (never prefetching) is stripped of its parked layout: all inline
    # (slot flags: 0 empty, 16 + r = ready, filled by sampler round r)
    assert bool((a.next_ready >= 16).all()) and bool((b.next_ready[0] == 0).all()) and bool((b.next_ready[1] >= 16).all())
    b.next_ready.zero_()
    gen = torch.Generator(device='cuda'); gen.manual_seed(0)
    for rnd in range(3):
        for e in (a, b):                      # everyone finishes within the next 30 steps
            bits = e.aux[:, 3].view(torch.int32)
            bits.copy_((bits & ~0xffff) | (e.spec.num_steps - 1 - (torch.arange(B, device='cuda', dtype=torch.int32) % 30)))
        for t in range(40):
            act = torch.rand(B, 2, device='cuda', generator=gen) * 2 - 1
            a.step(act); b.step(act)
            torch.cuda.synchronize()          # let the side-stream prefetch land before the next wave
    sa, sb = snapshot(a), snapshot(b)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    ca, cb = a.counters(), b.counters()
    assert cb['resets_prefetched'] == B and cb['resets_inline'] == cb['episodes']   # a full reset() samples through the slots
    assert ca['resets_prefetched'] >= 3 * B and ca['resets_prefetched'] + ca['resets_inline'] == ca['episodes'] + B
    # re-seeding drops the parked layouts: the next reset must not use them
    a.seed(99)
    assert bool((a.next_ready == 0).all())
    a.prefetch_every = 0
    a.reset()
    tw = co.philox_reset(env_id, 99 + 5)
    assert np.array_equal(a.zone_xy[:, 5, :].cpu().numpy(), tw['zone_xy'])


@pytest.mark.parametrize('env_id', TASKS)
def test_chained_steps_equal_plain_steps(crl, env_id):
    """CRL_STEP_CHAINED (a step waits for its own previous step warp by warp instead of for the
    whole preceding grid) must not change a single bit: two envs from the same seeds, one stepped
    with plain launches, one with chained launches -- eagerly, interleaved with a second chained
    env on the same stream, and replayed from a CUDA graph -- end in identical state and output."""
    B = 40000                                    # ragged; several waves of warps
    plain = crl.ZoneVecEnv(env_id, B, prefetch_every=0)
    chain = crl.ZoneVecEnv(env_id, B, prefetch_every=0)
    other = crl.ZoneVecEnv(env_id, 3000, prefetch_every=0, env_offset=B)
    for e in (plain, chain, other):
        e.seed(777); e.reset()
    for e in (plain, chain):                     # make episodes end (and auto-reset) during the run
        bits = e.aux[:, 3].view(torch.int32)
        bits.copy_((bits & ~0xffff) | (e.spec.num_steps - 1 - (torch.arange(B, device='cuda', dtype=torch.int32) % 50)))
    n_eager, n_graph = 25, 30
    for t in range(n_eager + n_graph):
        plain.step_random(action_seed=5)
    for t in range(n_eager):
        chain.step_random(action_seed=5, chained=True)
        other.step_random(action_seed=6, chained=True)
    torch.cuda.synchronize()
    # graph part: explicit (fixed) actions, because a captured step_index is frozen and in-kernel
    # actions would repeat; every replay is then a well-defined step
    g = torch.cuda.CUDAGraph()
    act = torch.rand(B, 2, device='cuda') * 2 - 1
    act_o = torch.rand(3000, 2, device='cuda') * 2 - 1
    plain2 = crl.ZoneVecEnv(env_id, B, prefetch_every=0)
    chain2 = crl.ZoneVecEnv(env_id, B, prefetch_every=0)
    for e in (plain2, chain2):
        e.seed(778); e.reset()
        bits = e.aux[:, 3].view(torch.int32)
        bits.copy_((bits & ~0xffff) | (e.spec.num_steps - 1 - (torch.arange(B, device='cuda', dtype=torch.int32) % 50)))
    for t in range(2 * n_graph + 2):
        plain2.step(act)
    chain2._step(act, 1, chained=True); other._step(act_o, 1, chained=True)      # eager first: chain established
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        chain2._step(act, 1, chained=True); other._step(act_o, 1, chained=True)
        chain2._step(act, 1, chained=True); other._step(act_o, 1, chained=True)
    chain2._step(act, 1, chained=True)
    for t in range(n_graph):
        g.replay()
    torch.cuda.synchronize()
    # the eager chained run only covered n_eager steps: finish it plainly, then compare
    for t in range(n_graph):
        chain.step_random(action_seed=5)
    torch.cuda.synchronize()
    for x, y in ((plain, chain), (plain2, chain2)):
        sx, sy = snapshot(x), snapshot(y)
        for k in sx:
            assert torch.equal(sx[k], sy[k]), k
        assert y.counters()['chain_wait_timeouts'] == 0
    assert chain.counters()['episodes'] > B // 2     # resets did happen under chaining
    st = chain2.stamp.cpu().numpy()
    assert np.all(st[0] == st[1]) and np.all(st[0] == 2 * n_graph + 2)


@pytest.mark.parametrize('env_id', ['PointTTSP-v0', 'ColourMatch-v3'])
def test_state_dict_resumes_bit_for_bit(crl, env_id):
    """A run restored from state_dict() continues exactly as the original did, through auto-resets
    (layouts are pure functions of the seeds, so the parked ones need not be saved)."""
    B = 512
    env = crl.ZoneVecEnv(env_id, B)
    env.seed(31)
    env.cfg.num_steps = 25
    env.reset()
    rs = np.random.RandomState(8)
    acts = [torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda() for _ in range(90)]
    goals = torch.zeros(B, dtype=torch.int32, device='cuda')
    def run(e, lo, hi):
        out = []
        for t in range(lo, hi):
            if e.spec.goals:
                e.set_goal(torch.where(e.needs_goal(), goals + t % 6, goals - 1))
            o, r, d, info = e.step(acts[t])
            out.append((o['obs'].clone(), o['zone_obs'].clone(), e.result.clone(), e.shaped_reward.clone()))
        return out
    run(env, 0, 40)
    snap = env.state_dict()
    first = run(env, 40, 90)
    other = crl.ZoneVecEnv(env_id, B)                    # a fresh object, as after a restart
    other.load_state_dict(snap)
    second = run(other, 40, 90)
    for t, (a, b) in enumerate(zip(first, second)):
        assert all(torch.equal(x, y) for x, y in zip(a, b)), t
    assert other.counters()['episodes'] == env.counters()['episodes'] > B
    assert torch.equal(other.seeds, env.seeds) and torch.equal(other.zone_xy, env.zone_xy)


def test_check_state_detects_corruption(crl):
    """crl_check_state counts, per kind, what a stray write would break."""
    env = crl.ZoneVecEnv('PointTTSP-v3', 256)
    env.reset()
    assert env.check_state() == [0] * 8
    env.pose[3, 0] = float('nan')
    env.pose[4, 2] = 7.0
    env.aux[5, 3] = torch.tensor(2001, dtype=torch.int32).view(torch.float32)
    env.zone_xy[2, 6, 0] = 2.9
    env.aux[7, 3] = torch.tensor(1 << 31, dtype=torch.int64).to(torch.int32).view(torch.float32)
    env.next_ready[1, 8] = 9
    env.goal[9] = 15
    env.zone_tmax[0, 10] = 2001
    # (1 << 31 of the state word is the episode parity, no longer a visited bit: a wrong parity counts with
    # the slot flags, index 5; every one of a 15-zone env's 15 visited bits is legal)
    assert env.check_state() == [1, 1, 1, 1, 0, 2, 1, 1]
    easy = crl.ZoneVecEnv('PointTSP-v1', 64)
    easy.reset()
    easy.aux[7, 3] = (easy.aux[7, 3].view(torch.int32) | (1 << 26)).view(torch.float32)   # "zone 10" of a 5-zone env
    assert easy.check_state() == [0, 0, 0, 0, 1, 0, 0, 0]
    cm = crl.ZoneVecEnv('ColourMatch-v0', 64)
    cm.reset()
    assert cm.check_state() == [0] * 8
    cm.cooldown[1, 0] = 151
    cm.aux[2, 3] = torch.tensor(3 << 16, dtype=torch.int32).view(torch.float32)   # colour code 3 does not exist
    assert cm.check_state()[4] == 2


@pytest.mark.parametrize('env_id', TASKS)
def test_layout_bank_reproduces_the_reference_maps(crl, env_id):
    """A fixed task set exported from the reference side (here: the oracle's numpy-legacy
    Engine.reset for seeds 1..12, as make_train_env(num_training_tasks=12) would build them) is
    installed as a layout bank; every reset -- the first one and every in-step auto-reset -- must
    land on exactly the map of the seed it ran with, timeouts / colours included."""
    from oracle import zone_env as ze
    task = ze.TASK_OF_ENV_ID[env_id]
    K, B = 12, 700
    bank = {'xy0': [], 'rot0': [], 'zone_xy': [], 'zone_max_steps': [], 'colours': []}
    for s in range(1, K + 1):
        e = ze.ZoneTaskEnv(task)
        e.seed(s)
        e.reset()
        bank['xy0'].append(e.xy0); bank['rot0'].append(e.rot0); bank['zone_xy'].append(e.zone_xy)
        bank['zone_max_steps'].append(e.zone_max_steps if task == ze.TTSP else np.zeros(e.N, int))
        bank['colours'].append(e.colours if task == ze.CM else np.zeros(e.N, int))
    bank = {k: np.array(v) for k, v in bank.items()}
    env = crl.ZoneVecEnv(env_id, B, seed_mode='fixed_range', min_seed=1, max_seed=K, layout_bank=bank)
    env.cfg.num_steps = 7
    seen = set()
    env.reset()
    for t in range(40):
        if t:
            env.step_random(action_seed=4)
        torch.cuda.synchronize()
        seeds = env.seeds.cpu().numpy() - 1                  # Engine.reset left seed + 1 behind
        k = seeds - 1
        seen |= set(int(x) for x in k)
        assert k.min() >= 0 and k.max() < K
        assert np.array_equal(env.zone_xy.cpu().numpy().transpose(1, 0, 2), bank['zone_xy'][k].astype(np.float32)), t
        o = env.origin.cpu().numpy()
        assert np.array_equal(o[:, :2], bank['xy0'][k].astype(np.float32)) and np.array_equal(o[:, 2], bank['rot0'][k].astype(np.float32))
        if task == ze.TTSP:
            assert np.array_equal(tmax_of(env), bank['zone_max_steps'][k]), t
        if task == ze.CM and t % 7 == 0:                     # right after a reset the colours are the bank's
            col = (bits_of(env)[:, None] >> 16 >> (2 * np.arange(6))) & 3
            assert np.array_equal(col, bank['colours'][k]), t
    assert seen == set(range(K))
    c = env.counters()
    assert c['resets_inline'] == 0 and c['resets_prefetched'] == B * (1 + 40 // 7)
    env.cfg.num_steps = 2000                                 # the bank's timeouts belong to 2000-step episodes
    assert env.check_state() == [0] * 8
    with pytest.raises(ValueError):
        crl.ZoneVecEnv(env_id, 8, seed_mode='fixed_range', min_seed=1, max_seed=K + 1, layout_bank=bank)
