"""bench.py's timed region and its --dump-outputs: exactly --steps steps are taken, and the same arguments dump the
same outputs, within the size limit."""
import argparse
import os

import numpy as np
import pytest

torch = pytest.importorskip('torch')
import bench  # noqa: E402


class _Outputs:
    """The output surface dump_outputs reads from a ZoneVecEnv, on host tensors."""

    def __init__(self, B, N=15, Z=6):
        g = torch.Generator().manual_seed(0)
        self.num_envs = B
        self.obs, self.zone_obs = torch.randn(B, 8, generator=g), torch.randn(B, N, Z, generator=g)
        result = torch.randint(0, 256, (B, 8), dtype=torch.uint8, generator=g)
        result[:, :4] = torch.randn(B, generator=g).view(torch.uint8).reshape(B, 4)
        self.reward, self.done = result.view(torch.float32)[:, 0], result[:, 4].view(torch.bool)
        self.goal_met, self.event, self.cost = result[:, 5].view(torch.bool), result[:, 6].view(torch.int8), torch.zeros(B)

    def _obs_dict(self):
        return {'zone_obs': self.zone_obs, 'obs': self.obs}

    def _info(self):
        return {'goal_met': self.goal_met, 'cost': self.cost, 'event': self.event}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_writes_every_output_as_float32(tmp_path):
    env = _Outputs(300)
    bench.dump_outputs(env, str(tmp_path))
    got = _load(tmp_path)
    assert sorted(got) == ['done', 'info_cost', 'info_event', 'info_goal_met', 'obs', 'reward', 'zone_obs']
    assert all(a.dtype == np.float32 for a in got.values())
    assert np.array_equal(got['zone_obs'], env.zone_obs.numpy()) and np.array_equal(got['reward'], env.reward.numpy())
    assert np.array_equal(got['info_event'], env.event.numpy().astype(np.float32))
    assert np.array_equal(got['done'], env.done.numpy().astype(np.float32))


def test_dump_outputs_samples_the_same_envs_under_the_size_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, 'DUMP_BYTES', 256 * 1024)
    env = _Outputs(5000)
    for d in ('a', 'b'):
        bench.dump_outputs(env, str(tmp_path / d))
    a, b = _load(tmp_path / 'a'), _load(tmp_path / 'b')
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in os.listdir(tmp_path / 'a')) <= bench.DUMP_BYTES
    keep = a['env_index'].astype(np.int64)
    assert a['env_index'].dtype == np.float64 and 100 < len(keep) < 5000 and np.all(np.diff(keep) > 0)
    assert np.array_equal(a['obs'], env.obs.numpy()[keep]) and np.array_equal(a['zone_obs'], env.zone_obs.numpy()[keep])
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)


@pytest.mark.gpu
def test_bench_times_exactly_the_requested_steps_and_dumps_the_same_outputs(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    import combinatorial_rl_tasks_b200 as crl
    from combinatorial_rl_tasks_b200 import _lib
    dev = torch.device('cuda:0')
    K, W = 37, 5

    def run(d):
        args = argparse.Namespace(bank=0, prefetch_every=32, prefetch_warps=0, cfg=[], no_auto_reset=False,
                                  env='PointTSP-v0', min_replicas=0)
        ring = bench.Ring(crl, _lib, args, 'PointTSP-v0', 65536, dev, 0)
        m = bench.measure(ring, K, W, 1, None)
        bench.dump_outputs(ring.last_env, str(d))
        # the ring's constructor steps each replica once; episodes last 2000 steps, so the median env of a replica
        # counts the steps that replica took
        taken = sum(int(e.steps.cpu().median()) for e in ring.envs)
        return m, taken, ring.R

    m, taken, R = run(tmp_path / 'a')
    assert m['timed_steps'] == K and taken == R + W + K, (m, taken, R)
    assert 0 < m['ms_per_step_best'] <= m['ms_per_step_worst'] and m['timed_region_s'] > 0
    run(tmp_path / 'b')
    a, b = _load(tmp_path / 'a'), _load(tmp_path / 'b')
    assert sorted(a) == ['done', 'info_cost', 'info_event', 'info_goal_met', 'obs', 'reward', 'zone_obs']
    assert a['zone_obs'].shape == (65536, 15, 6) and np.all(np.isfinite(a['obs']))
    assert all(np.array_equal(a[k], b[k]) for k in a), [k for k in a if not np.array_equal(a[k], b[k])]
