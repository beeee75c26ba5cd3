"""CRL_STEP_ZONE_OBS_DELTA: a step that writes only the zone_obs rows that change.  ZoneVecEnv passes the flag
whenever its bound zone_obs tensor holds the rows of the current state; what a caller sees must be byte for byte
what a step that writes every row returns."""
import numpy as np
import pytest

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

TASKS = ['PointTSP-v0', 'PointTTSP-v0', 'ColourMatch-v0']


@pytest.fixture(scope='module')
def crl():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    import combinatorial_rl_tasks_b200 as m
    return m


def make_pair(crl, env_id, B, num_steps=None):
    """Two envs with the same seeds: `env` steps through ZoneVecEnv (with the flag once its zone_obs is current),
    `twin` through crl_step without it (full_step)."""
    pair = []
    for _ in range(2):
        e = crl.ZoneVecEnv(env_id, B, prefetch_every=0)
        e.seed(17)
        if num_steps is not None:
            e.cfg.num_steps = num_steps                  # short episodes: timeouts and auto-resets every few steps
        e.reset()
        pair.append(e)
    return pair


def full_step(twin, actions, flags, action_seed=0):
    from combinatorial_rl_tasks_b200 import _lib
    aptr = None if actions is None else actions.data_ptr()
    _lib.check(twin.lib.crl_step(twin.cfg, twin.state, aptr, twin.out, flags, action_seed, 0, twin._stream()))


def same_bytes(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def assert_same_outputs(env, twin, where):
    assert same_bytes(env.zone_obs, twin.zone_obs), where
    assert same_bytes(env.obs, twin.obs), where
    assert torch.equal(env.result, twin.result), where


def put_robots_on_zones(envs, n, zone):
    for e in envs:
        e.pose[:n, :2] = e.zone_xy[zone, :n, :]


@pytest.mark.parametrize('auto_reset', [True, False])
@pytest.mark.parametrize('B', [65536, 1000])
@pytest.mark.parametrize('env_id', TASKS)
def test_delta_step_is_byte_identical_to_full_step(crl, env_id, B, auto_reset):
    """Across zone events (robots put on zones), ColourMatch cooldowns, timeouts and auto-resets, at a full-size and
    a ragged batch (B = 1000: the last warp holds 8 envs)."""
    from combinatorial_rl_tasks_b200 import _lib
    env, twin = make_pair(crl, env_id, B, num_steps=40)
    g = torch.Generator(device='cuda').manual_seed(3)
    step = env.step if auto_reset else env.step_no_reset
    flags = _lib.STEP_AUTO_RESET if auto_reset else 0
    events = 0
    for t in range(90):
        if t in (5, 47):
            put_robots_on_zones((env, twin), B // 5, 3 if t == 5 else 4)
        a = torch.rand(B, 2, device='cuda', generator=g) * 2 - 1
        step(a)
        full_step(twin, a, flags)
        assert_same_outputs(env, twin, t)
        events += int((env.event != 0).sum().item())
    assert env._zone_obs_ok
    assert events >= B // 20
    if auto_reset:
        assert env.counters()['episodes'] >= B                 # every env went through at least one auto-reset


@pytest.mark.parametrize('env_id', TASKS)
def test_delta_step_in_a_replayed_cuda_graph(crl, env_id):
    """As bench.py runs it: in-kernel actions on the device step counter, auto-reset on, the step captured in a CUDA
    graph (with the flag: zone_obs is current after the reset) and replayed."""
    from combinatorial_rl_tasks_b200 import _lib
    B = 65536
    env, twin = make_pair(crl, env_id, B, num_steps=60)
    flags = _lib.STEP_AUTO_RESET | _lib.STEP_ACTION_COUNTER
    env.step_random(action_seed=1234, replayable=True)
    full_step(twin, None, flags, 1234)
    torch.cuda.synchronize()
    assert_same_outputs(env, twin, 'eager')
    graphs = []
    for fn in (lambda: env.step_random(action_seed=1234, replayable=True),
               lambda: full_step(twin, None, flags, 1234)):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        graphs.append(g)
    for t in range(150):
        if t == 20:
            put_robots_on_zones((env, twin), B // 5, 2)
        for g in graphs:
            g.replay()
        torch.cuda.synchronize()
        assert_same_outputs(env, twin, t)
    assert env.counters()['episodes'] >= B


def test_unchanged_rows_are_not_written(crl):
    """PointTSP: rows of envs that cannot change in the next step -- far from every zone (the event is tested at
    the position the step starts from) and far from the step limit -- are left alone: NaNs written there survive."""
    B = 4096
    env = crl.ZoneVecEnv('PointTSP-v0', B, prefetch_every=0)
    env.seed(5)
    env.reset()
    g = torch.Generator(device='cuda').manual_seed(1)
    for _ in range(3):
        env.step(torch.rand(B, 2, device='cuda', generator=g) * 2 - 1)
    d = torch.linalg.vector_norm(env.zone_xy - env.pose[None, :, :2], dim=2).min(dim=0).values   # (B,)
    quiet = (d > 0.6) & (env.steps < env.cfg.num_steps - 10)
    assert int(quiet.sum().item()) > B // 4
    env.zone_obs[quiet] = float('nan')
    env.step(torch.rand(B, 2, device='cuda', generator=g) * 2 - 1)
    assert bool(torch.isnan(env.zone_obs[quiet]).all().item())


def _poison(env):
    env.zone_obs.fill_(float('nan'))


@pytest.mark.parametrize('transition', ['bind_outputs', 'write_zone_obs', 'load_state_dict', 'masked_reset'])
def test_each_not_current_transition_forces_a_full_write(crl, transition):
    """After anything that can leave stale rows in the bound zone_obs tensor, the next step writes every row."""
    B = 1000
    env, twin = make_pair(crl, 'PointTSP-v0', B)
    g = torch.Generator(device='cuda').manual_seed(2)
    acts = lambda: torch.rand(B, 2, device='cuda', generator=g) * 2 - 1
    from combinatorial_rl_tasks_b200 import _lib

    def both(a):
        env.step(a)
        full_step(twin, a, _lib.STEP_AUTO_RESET)

    for _ in range(3):
        both(acts())
    assert env._zone_obs_ok
    if transition == 'bind_outputs':
        N, Z = env.spec.num_zones, env.spec.zone_dim
        env.bind_outputs(torch.zeros(B, 8, device='cuda'), torch.full((B, N, Z), float('nan'), device='cuda'),
                         torch.zeros(B, 8, dtype=torch.uint8, device='cuda'))
    elif transition == 'write_zone_obs':
        env.write_zone_obs = False
        a = acts()
        env.step(a)                                            # builds no zone_obs rows at all
        full_step(twin, a, _lib.STEP_AUTO_RESET)
        env.write_zone_obs = True
        _poison(env)
    elif transition == 'load_state_dict':
        sd = env.state_dict()
        both(acts())
        env.load_state_dict(sd)
        twin.load_state_dict(sd)
        _poison(env)
    else:
        mask = np.zeros(B, dtype=np.uint8)
        mask[::7] = 1
        env.reset(mask=mask)
        twin.reset(mask=mask)
        _poison(env)
    assert not env._zone_obs_ok
    both(acts())
    assert not bool(torch.isnan(env.zone_obs).any().item())
    assert_same_outputs(env, twin, transition)
    assert env._zone_obs_ok
