"""ZoneVecEnv: the reference's vector-env surface on one B200.

Stands where ``ParallelEnv([make_train_env(...) for _ in range(B)])`` stands in the
reference (main/src/torch_ac/torch_utils/penv.py:23-69 over main/envs/make_env.py:3-51):
``reset() / step(actions) / step_no_reset(actions) / seed(...)``, attributes ``envs``,
``observation_space``, ``action_space``.  Differences, all by design:

* one object holds all B envs; every per-env Python list becomes a device tensor:
  ``obs['obs']`` (B,8) f32, ``obs['zone_obs']`` (B,N,Z) f32 (the layout
  main/src/utils/format.py:27-28 builds), ``reward`` (B,) f32, ``done`` (B,) bool,
  ``info`` = dict of tensors {'goal_met' (B,) bool, 'cost' zeros, 'event' (B,) int8};
* the returned tensors are persistent buffers owned by the env and overwritten by the
  next call (clone what must outlive a step).  They are READ-ONLY for the caller: a step
  rewrites only the ``zone_obs`` rows that change, so an in-place edit would survive it;
* calls are asynchronous on the current CUDA stream.

All arithmetic happens in libcrl_b200.so (include/crl_b200.h); torch only owns the
memory.  There is no CPU path.
"""
import contextlib
import ctypes

import numpy as np
import torch

from . import _lib
from .config import ENV_SPECS
from .spaces import Box, Dict


_NO_GUARD = contextlib.nullcontext()


class _EnvView:
    """What ``penv.envs[i]`` must answer for the reference's callers."""

    def __init__(self, vec, index):
        self._vec, self.index = vec, index
        self.observation_space = vec.observation_space
        self.action_space = vec.action_space

    @property
    def unwrapped(self):
        return self

    @property
    def num_cities(self):
        return self._vec.spec.num_zones

    # zone-goals scripts/train_skill_planner.py:134-135 and penv.py:23 probe these on envs[0]
    @property
    def goal_dim(self):
        return 2

    @property
    def goal_zone(self):
        g = int(self._vec.goal[self.index].item())
        return None if g < 0 else g

    def noop_obs(self):
        """WaitWrapper.noop_obs (wrappers.py:46-50)."""
        N, Z = self._vec.spec.num_zones, self._vec.spec.zone_dim
        return {'zone_obs': np.zeros((N, Z)), 'obs': np.zeros(8)}


_raw_stream = getattr(torch._C, '_cuda_getCurrentRawStream', None) or \
    (lambda index: torch.cuda.current_stream(index).cuda_stream)


# CrlConfig fields that may differ between the two sides of crl_copy_envs: the batch's size, place and seed range
_COPY_FREE_FIELDS = ('num_envs', 'env_offset', 'seed_mode', 'min_seed', 'max_seed')


def _task_config(cfg):
    return tuple(getattr(cfg, f) for f, _ in cfg._fields_ if f not in _COPY_FREE_FIELDS)


def _dev_index(device):
    return device.index if device.index is not None else torch.cuda.current_device()


def _copy_out(side, zone_obs):
    """The CrlOut of one side of a copy; ``zone_obs=False``: the rows are not copied (absent on the other side)."""
    return _lib.CrlOut(obs=side.obs.data_ptr(), zone_obs=side.zone_obs.data_ptr() if zone_obs else None,
                       result=side.result.data_ptr(), shaped_reward=side.shaped_reward.data_ptr())


class EnvSnapshot:
    """The complete state of n envs of a ZoneVecEnv, gathered on the env's device by crl_copy_envs
    (``ZoneVecEnv.snapshot``); ``ZoneVecEnv.copy_envs_from(snapshot, ...)`` restores it onto any envs of any
    ZoneVecEnv with the same env id and config.  Holds the per-env state planes (sized by crl_plane_bytes for n envs,
    no next-layout planes, no counters) and the output rows of the n envs -- the ZoneVecEnv attribute names, env i of
    the snapshot being ``env_ids[i]`` of the source -- and no reference to the source env."""

    _PLANES = (('pose', 0, torch.float32, (4,)), ('aux', 1, torch.float32, (4,)), ('zone_xy', 2, torch.float32, None),
               ('zone_tmax', 3, torch.int32, None), ('cooldown', 4, torch.int32, (2,)), ('seeds', 5, torch.int64, ()),
               ('episode', 6, torch.int32, ()), ('origin', 7, torch.float32, (4,)), ('obs', 14, torch.float32, (8,)),
               ('zone_obs', 15, torch.float32, None), ('result', 16, torch.uint8, (8,)), ('goal', 20, torch.int32, ()),
               ('shaped_reward', 21, torch.float32, ()))

    def __init__(self, env, n):
        self.env_id, self.spec, self.num_envs, self.device = env.env_id, env.spec, int(n), env.device
        self.cfg = _lib.CrlConfig.from_buffer_copy(env.cfg)
        self.cfg.num_envs = self.num_envs
        self.zone_obs_ok = False                  # the zone_obs rows are those of the state (set by the gather)
        sizes = (ctypes.c_int64 * _lib.NUM_PLANES)()
        _lib.check(env.lib.crl_plane_bytes(self.cfg, sizes, _lib.NUM_PLANES))
        N, Z = self.spec.num_zones, self.spec.zone_dim
        shapes = {'zone_xy': (N, n, 2), 'zone_tmax': ((N + 1) // 2, n), 'zone_obs': (n, N, Z)}
        for name, i, dtype, tail in self._PLANES:
            t = None
            if sizes[i]:
                t = torch.zeros(sizes[i], dtype=torch.uint8, device=self.device).view(dtype)
                t = t.view(shapes[name] if tail is None else (n,) + tail)
            setattr(self, name, t)
        ptr = lambda t: None if t is None else t.data_ptr()
        self.state = _lib.CrlState(pose=ptr(self.pose), aux=ptr(self.aux), zone_xy=ptr(self.zone_xy),
                                   zone_tmax=ptr(self.zone_tmax), cooldown=ptr(self.cooldown), seed=ptr(self.seeds),
                                   episode=ptr(self.episode), origin=ptr(self.origin), goal=ptr(self.goal))

    def nbytes(self):
        """Device bytes the snapshot holds."""
        return sum(t.numel() * t.element_size() for t in (getattr(self, k) for k, *_ in self._PLANES) if t is not None)


class ZoneVecEnv:
    def __init__(self, env_id, num_envs, device='cuda:0', seed_mode='increment', min_seed=1, max_seed=100,
                 env_offset=0, auto_reset=True, prefetch_every=32, wait=False, prefetch_warps=0, layout_bank=None):
        if not torch.cuda.is_available():
            raise RuntimeError('ZoneVecEnv needs a CUDA device (sm_100a); there is no CPU fallback')
        self.lib = _lib.load()
        self.env_id = env_id
        self.spec = spec = ENV_SPECS[env_id]
        self.num_envs = B = int(num_envs)
        self.device = torch.device(device)
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.auto_reset = auto_reset
        # top up the parked next layouts every `prefetch_every` steps at most (0: never, resets then
        # sample inline); the interval stretches up to 16x while the sampler finds nothing to do
        self.prefetch_every = prefetch_every
        self._pf_interval, self._pf_due = max(prefetch_every, 1), max(prefetch_every, 1)
        self.prefetch_warps = prefetch_warps      # background sampler warps per SM (0: library default)
        # WaitWrapper semantics (make_train_env(hier=True), wrappers.py:29-54): under
        # step_no_reset an env whose episode ended is parked until it is reset
        self.wait = bool(wait)
        self._mode_flags = (_lib.STEP_GOALS if spec.goals else 0)
        self._write_zone_obs = True
        N, Z = spec.num_zones, spec.zone_dim
        self.cfg = _lib.CrlConfig(
            task=spec.task, num_envs=B, num_zones=N, num_steps=spec.num_steps, frameskip=spec.frameskip,
            max_cooldown=spec.max_cooldown,
            seed_mode=_lib.SEED_FIXED_RANGE if seed_mode == 'fixed_range' else _lib.SEED_INCREMENT,
            env_offset=env_offset, min_seed=min_seed, max_seed=max_seed, zone_size=spec.zone_size,
            time_saved_reward=spec.time_saved_reward, beta_a=spec.beta_a, beta_b=spec.beta_b,
            robot_keepout=spec.robot_keepout, zone_keepout=spec.zone_keepout, extent=spec.extent,
            initial_visited=spec.initial_visited, walled=1 if spec.walled else 0)
        dev = self.device
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=dev)
        # state planes (layout documented in include/crl_b200.h)
        self.pose = z(B, 4)
        self.aux = z(B, 4)
        self.zone_xy = z(N, B, 2)
        self.zone_tmax = z((N + 1) // 2, B, dtype=torch.int32) if spec.task == _lib.TASK_TTSP else None
        self.cooldown = z(B, 2, dtype=torch.int32) if spec.task == _lib.TASK_CM else None
        self.seeds = z(B, dtype=torch.int64)
        self.episode = z(B, dtype=torch.int32)
        self.origin = z(B, 4)
        self.counters_dev = z(8, dtype=torch.float64)
        # next-layout slots, filled in the background by crl_prefetch_layouts
        # (two slots per env: reset number n takes slot n & 1)
        self.next_zone_xy = z(2, N, B, 2)
        if spec.task == _lib.TASK_TTSP:
            self.next_task = z(2, (N + 1) // 2, B, dtype=torch.int32)
        elif spec.task == _lib.TASK_CM:
            self.next_task = z(2, B, dtype=torch.int32)
        else:
            self.next_task = None
        self.next_origin = z(2, B, 4)
        self.next_seed = z(2, B, dtype=torch.int64)
        self.next_ready = z(2, B, dtype=torch.int32)
        self._prefetch_work = z(1 + 2 * B, 4, dtype=torch.int32)
        # sampler rounds: numbered 1, 2, ...; a round's parked layouts become usable by the steps once it
        # has been PUBLISHED on the stepping stream (crl_prefetch_publish), which tick() does two
        # rounds later -- the stepping stream then waits for an event that fired long ago
        self._prefetch_epoch = z(4, dtype=torch.int32)
        self._round = 0
        self._round_done = {}                     # round -> event recorded behind it on its stream
        self._published = 0
        self._pf_found = torch.zeros(1, dtype=torch.int32).pin_memory()   # empty slots the last round found
        self._side = torch.cuda.Stream(device=dev)
        # per-warp completion stamps of crl_step (CRL_STEP_CHAINED)
        self.stamp = z(3, (B + 31) // 32, dtype=torch.int32)
        self._chain_ok = False                    # True: the last kernel enqueued for this state was a ticketed step
        # zone_obs rows and result records the host-direct step_host calls moved (CRL_STEP_TRACK_ROWS, cumulative)
        self._row_list = z(4, dtype=torch.int32)
        self._mirror_ok = False                   # True: the host zone_obs buffer equals the device one
        # True: the bound zone_obs tensor holds the rows of the current state, so a step may write only the rows that
        # change (CRL_STEP_ZONE_OBS_DELTA).  Set by a full reset and by every step that writes zone_obs
        self._zone_obs_ok = False
        self.delta_rows = 0                       # rows the last step_host moved (B = all)
        # outputs
        self._cost = z(B)
        # goal-conditioned variants (PointTSP-v3 ...): goal_zone per env (-1 = None), shaped reward
        self.goal = torch.full((B,), -1, dtype=torch.int32, device=dev)
        self._goal_xy = z(B, 2)
        self._needs_goal = z(B, dtype=torch.uint8)
        self._available = z(B, N, dtype=torch.uint8)
        ptr = lambda t: t.data_ptr() if t is not None else None
        self.state = _lib.CrlState(pose=ptr(self.pose), aux=ptr(self.aux), zone_xy=ptr(self.zone_xy),
                                   zone_tmax=ptr(self.zone_tmax), cooldown=ptr(self.cooldown),
                                   seed=ptr(self.seeds), episode=ptr(self.episode), origin=ptr(self.origin),
                                   counters=ptr(self.counters_dev), next_zone_xy=ptr(self.next_zone_xy),
                                   next_task=ptr(self.next_task), next_origin=ptr(self.next_origin),
                                   next_seed=ptr(self.next_seed), next_ready=ptr(self.next_ready),
                                   stamp=ptr(self.stamp), prefetch_work=ptr(self._prefetch_work),
                                   row_list=ptr(self._row_list), goal=ptr(self.goal),
                                   prefetch_epoch=ptr(self._prefetch_epoch))
        fixed = spec.fixed_layout()               # hard instances: fixed robot / city placements
        if fixed is not None:
            self._fixed = torch.from_numpy(fixed).to(dev).contiguous()
            self.state.fixed_layout = self._fixed.data_ptr()
        if layout_bank is not None:
            self._install_layout_bank(layout_bank, seed_mode, min_seed, max_seed)
        self.bind_outputs(z(B, 8), z(B, N, Z), z(B, 8, dtype=torch.uint8), z(B))
        self._actions_dev = z(B, 2)
        # copy_envs_from: pairs skipped on the device for an id out of range (device ids; cumulative), and the number of
        # copies made INTO this env (Rollout(store='frames') refuses to go on across one)
        self.copy_rejects = z(1, dtype=torch.int32)
        self.copy_count = 0
        self._host = None
        self._host_calls = {}                     # (auto_reset, wait) -> CrlHostCall*, see step_host
        self._host_call_step = self.lib.crl_host_call_step
        self._pinned = {}                         # id(numpy array) -> (pinned tensor, pointer, array): pinned_actions()
        self._step_index = 0
        self.gpu_launches = 0
        # spaces: wrappers.py:144-153 (Box(-inf, inf)), Engine action space Box(-1, 1, (2,))
        self.observation_space = Dict({'zone_obs': Box(-np.inf, np.inf, (N, Z)),
                                       'obs': Box(-np.inf, np.inf, (8,))})
        self.action_space = Box(-1.0, 1.0, (2,))
        self.envs = [_EnvView(self, i) for i in range(min(B, 1))]
        self.seed(torch.arange(B, dtype=torch.int64) + env_offset)

    # -- plumbing ------------------------------------------------------------------
    def _install_layout_bank(self, bank, seed_mode, min_seed, max_seed):
        """The maps of a fixed task set (CrlState.bank_*): ``bank`` = dict with xy0 (K,2), rot0 (K,),
        zone_xy (K,N,2) and, per task, zone_max_steps (K,N) / colours (K,N), entry k being the map
        of seed ``min_seed + k`` -- e.g. what the reference's own ``env.seed(s); env.reset()`` builds
        for each of make_train_env's ``num_training_tasks`` seeds.  Every reset then copies the
        entry of its seed: the device runs on exactly those maps and needs no sampler."""
        N, spec = self.spec.num_zones, self.spec
        xy0 = np.asarray(bank['xy0'], dtype=np.float64).reshape(-1, 2)
        K = xy0.shape[0]
        if K != max_seed - min_seed + 1:
            raise ValueError('a layout bank needs one entry per seed in [min_seed, max_seed]')
        origin = np.zeros((K, 4), dtype=np.float32)
        origin[:, :2], origin[:, 2] = xy0, np.asarray(bank['rot0'], dtype=np.float64).reshape(K)
        zxy = np.asarray(bank['zone_xy'], dtype=np.float64).reshape(K, N, 2).astype(np.float32)
        task = None
        if spec.task == _lib.TASK_TTSP:
            tm = np.clip(np.asarray(bank['zone_max_steps']).reshape(K, N), 0, 65535).astype(np.uint32)
            tm = np.concatenate([tm, np.zeros((K, (-N) % 2), dtype=np.uint32)], axis=1)
            task = (tm[:, 0::2] | (tm[:, 1::2] << 16)).astype(np.uint32).view(np.int32)
        elif spec.task == _lib.TASK_CM:
            col = np.asarray(bank['colours']).reshape(K, N).astype(np.uint32)
            task = (col << (2 * np.arange(N, dtype=np.uint32))).sum(axis=1).astype(np.uint32).view(np.int32).reshape(K, 1)
        dev = self.device
        self._bank = (torch.from_numpy(zxy).to(dev).contiguous(), torch.from_numpy(origin).to(dev).contiguous(),
                      None if task is None else torch.from_numpy(np.ascontiguousarray(task)).to(dev))
        self.state.bank_zone_xy = self._bank[0].data_ptr()
        self.state.bank_origin = self._bank[1].data_ptr()
        self.state.bank_task = None if self._bank[2] is None else self._bank[2].data_ptr()
        if seed_mode == 'fixed_range':
            self.prefetch_every = 0               # every seed is in the bank: nothing to sample

    def prepare_outputs(self, obs, zone_obs, result, shaped_reward=None):
        """Validate a set of caller-owned output tensors once and return a binding that
        ``bind_outputs(binding=...)`` installs with a few attribute stores (rollout.py prepares
        one per slot).  ``zone_obs=None``: for steps that write no zone_obs (``write_zone_obs = False``); a reset or a
        step that would write it then fails."""
        B, N, Z = self.num_envs, self.spec.num_zones, self.spec.zone_dim
        assert obs.shape == (B, 8) and result.shape == (B, 8)
        assert obs.dtype == torch.float32 and result.dtype == torch.uint8
        assert obs.is_contiguous() and result.is_contiguous()
        if zone_obs is not None:
            assert zone_obs.shape == (B, N, Z) and zone_obs.dtype == torch.float32 and zone_obs.is_contiguous()
        if shaped_reward is None:
            shaped_reward = getattr(self, 'shaped_reward', None)
            if shaped_reward is None:
                shaped_reward = torch.zeros(B, dtype=torch.float32, device=self.device)
        out = _lib.CrlOut(obs=obs.data_ptr(), zone_obs=None if zone_obs is None else zone_obs.data_ptr(),
                          result=result.data_ptr(),
                          shaped_reward=shaped_reward.data_ptr())
        return (obs, zone_obs, result, shaped_reward, result.view(torch.float32)[:, 0], result[:, 4].view(torch.bool),
                result[:, 5].view(torch.bool), result[:, 6].view(torch.int8), result[:, 7].view(torch.bool), out)

    def bind_outputs(self, obs=None, zone_obs=None, result=None, shaped_reward=None, binding=None):
        """Point the env's outputs at caller-owned device tensors: the next reset / step writes
        obs (B,8) f32, zone_obs (B,N,Z) f32, result (B,8) u8 and shaped_reward (B,) f32 there, in
        place.  A rollout buffer hands in slot t+1 before step t, so storing a frame costs no copy
        (rollout.py).  The tensors must be contiguous; obs / zone_obs 16-byte aligned."""
        if binding is None:
            binding = self.prepare_outputs(obs, zone_obs, result, shaped_reward)
        (self.obs, self.zone_obs, self.result, self.shaped_reward, self.reward, self.done, self.goal_met, self.event,
         self.need_next_goal, self.out) = binding
        self._mirror_ok = False
        self._zone_obs_ok = False
        self._chain_ok = False

    @property
    def write_zone_obs(self):
        """False: step() / step_no_reset() / step_random() neither build nor write ``zone_obs`` (CRL_STEP_NO_ZONE_OBS)
        -- for rollouts whose only consumer is ``ZoneEncoder.forward_from_state(env)``, which derives the zone rows
        from the state planes.  ``env.zone_obs`` then keeps what the last reset / full step wrote.  step_host always
        writes it."""
        return self._write_zone_obs

    @write_zone_obs.setter
    def write_zone_obs(self, on):
        self._write_zone_obs = bool(on)
        self._mirror_ok = False
        self._zone_obs_ok = False

    def _guard(self):
        """Make this env's device current for the call; free when it already is (the usual case)."""
        return _NO_GUARD if torch.cuda.current_device() == self._dev_index else torch.cuda.device(self.device)

    def _stream(self):
        # the raw handle of torch's current stream on this device (a C call: torch.cuda.current_stream() builds a Stream
        # object, ~2 us of every host-facing call)
        return ctypes.c_void_p(_raw_stream(self._dev_index))

    def _obs_dict(self):
        return {'zone_obs': self.zone_obs, 'obs': self.obs}

    def _info(self):
        info = {'goal_met': self.goal_met, 'cost': self._cost, 'event': self.event}
        if self.spec.goals:
            info['shaped_reward'] = self.shaped_reward
            info['need_next_goal'] = self.need_next_goal
        return info

    def _as_dev(self, x, dtype):
        return torch.as_tensor(x, dtype=dtype, device=self.device).contiguous()

    # -- reference surface ---------------------------------------------------------
    def seed(self, seeds):
        """Engine.seed for every env: an int (env i gets seed + i) or a (B,) tensor."""
        if isinstance(seeds, int):
            seeds = torch.arange(self.num_envs, dtype=torch.int64) + seeds
        # a sampler round still running on the side stream writes slot flags: it must be over before they are zeroed
        torch.cuda.current_stream(self.device).wait_stream(self._side)
        self.seeds.copy_(self._as_dev(seeds, torch.int64))
        self.episode.zero_()
        self.aux[:, 3] = (self.aux[:, 3].view(torch.int32) & 0x7fffffff).view(torch.float32)   # slot parity follows `episode`
        self.next_ready.zero_()          # parked layouts were drawn for the old seeds
        self._pf_interval = self._pf_due = max(self.prefetch_every, 1)
        self._chain_ok = False
        self._mirror_ok = False
        self._zone_obs_ok = False

    def prefetch(self, stream=None, warps_per_sm=0):
        """One sampler round (crl_prefetch_layouts): fill the empty next-layout slots.

        ``stream=None``: in the background, on the side stream, ordered behind the work already queued on
        the stepping stream but never blocking it.  Before launching round r the stepping stream
        publishes round r - 2 (it waits for that round's event, which fired long ago: rounds are at least
        ``prefetch_every`` steps apart), so a round's layouts reach the steps one to two intervals after
        it was launched and the step's reset path needs no acquire / release.  An env that finishes before
        its slot is usable samples inline with the identical result.
        ``stream=<the stepping stream>``: in line (reset, load_state_dict); published at once."""
        cur = torch.cuda.current_stream(self.device)
        background = stream is None
        if torch.cuda.is_current_stream_capturing():
            return
        with self._guard():
            if background:
                stream = self._side
                self._publish(self._round - 1, cur)
                stream.wait_stream(cur)
            else:
                # rounds share one work list: not before a background round still running is over
                stream.wait_stream(self._side)
            self._round += 1
            _lib.check(self.lib.crl_prefetch_layouts(self.cfg, self.state, warps_per_sm or self.prefetch_warps,
                                                     self._round, ctypes.c_void_p(stream.cuda_stream)))
            with torch.cuda.stream(stream):               # how much there was to do, read by tick() later
                self._pf_found.copy_(self._prefetch_work[0, :1], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
            self._round_done[self._round] = ev
            if not background:
                self._publish(self._round, cur)
        self.gpu_launches += 2 if self.spec.task == _lib.TASK_TSP else 3

    def _publish(self, rnd, cur):
        """Make rounds <= rnd usable by the steps enqueued on ``cur`` from here on."""
        if rnd <= self._published:
            return
        for r in [r for r in self._round_done if r <= rnd]:
            cur.wait_event(self._round_done.pop(r))
        _lib.check(self.lib.crl_prefetch_publish(self.state, rnd, ctypes.c_void_p(cur.cuda_stream)))
        self._published = rnd
        self.gpu_launches += 1

    def tick(self, steps=1):
        """Cadence of the background sampler, called once per step (step() does; a caller that
        replays captured steps calls it itself).  A round is launched when `prefetch_every` steps
        have passed -- stretched up to 16x while the previous rounds found no empty slot (PointTSP
        under random actions resets once in 2000 steps), back to the base interval as soon as one
        finds work.  The count read here may be one round old; an env whose slot is empty when it
        needs it samples inline, so the cadence never affects results."""
        if not self.prefetch_every:
            return False
        self._pf_due -= steps
        if self._pf_due > 0:
            return False
        found = int(self._pf_found[0])
        self._pf_interval = min(2 * self._pf_interval, 16 * self.prefetch_every) if found == 0 else self.prefetch_every
        self._pf_due = self._pf_interval
        self.prefetch()
        return True

    def reset(self, layout=None, mask=None, env_ids=None):
        """Engine.reset of all envs (or those in ``mask``).  ``layout`` switches to the
        host-supplied-layout mode: dict with xy0 (n,2), rot0 (n,), zone_xy (n,N,2) and
        zone_max_steps (n,N) / colours (n,N) per task, for envs ``env_ids`` (default 0..n)."""
        with self._guard():
            if layout is None:
                m = None if mask is None else self._as_dev(mask, torch.uint8)
                if not torch.cuda.is_current_stream_capturing():
                    self._publish(self._round, torch.cuda.current_stream(self.device))   # everything parked so far
                if mask is None and self.state.bank_zone_xy is None and not torch.cuda.is_current_stream_capturing():
                    # a full reset: sample every layout with the one-lane-per-env sampler first
                    # (all SMs, nothing else is running), then crl_reset only copies
                    self.prefetch(torch.cuda.current_stream(self.device), warps_per_sm=16)
                _lib.check(self.lib.crl_reset(self.cfg, self.state, self.out,
                                              None if m is None else m.data_ptr(), self._stream()))
            else:
                xy0 = self._as_dev(layout['xy0'], torch.float64).reshape(-1, 2)
                n = xy0.shape[0]
                rot0 = self._as_dev(layout['rot0'], torch.float64).reshape(n)
                zxy = self._as_dev(layout['zone_xy'], torch.float64).reshape(n, self.spec.num_zones, 2)
                tm = self._as_dev(layout['zone_max_steps'], torch.int32) if 'zone_max_steps' in layout else None
                col = self._as_dev(layout['colours'], torch.int32) if 'colours' in layout else None
                ids = None if env_ids is None else self._as_dev(env_ids, torch.int32)
                lay = _lib.CrlLayoutIn(xy0=xy0.data_ptr(), rot0=rot0.data_ptr(), zone_xy=zxy.data_ptr(),
                                       zone_max_steps=None if tm is None else tm.data_ptr(),
                                       colours=None if col is None else col.data_ptr())
                _lib.check(self.lib.crl_reset_from_layout(self.cfg, self.state, self.out, lay,
                                                          None if ids is None else ids.data_ptr(), n,
                                                          self._stream()))
            self.gpu_launches += 1
            self._chain_ok = False
            self._mirror_ok = False
            # a reset of every env writes every row; after a masked reset or host-supplied layouts the next step
            # writes them all
            self._zone_obs_ok = layout is None and mask is None
            if self.prefetch_every and not torch.cuda.is_current_stream_capturing():
                # the reset above must be visible to the prefetcher: same-stream launch
                self.prefetch(torch.cuda.current_stream(self.device))
        return self._obs_dict()

    def _step(self, actions, flags, action_seed=0, chained=False):
        """``chained=True``: the caller asserts that the kernel enqueued just before this call on the
        current stream is a step (of this env or another ZoneVecEnv) that did not write ``actions``
        (CRL_STEP_CHAINED: back-to-back rollout steps overlap across the launch boundary)."""
        if chained:
            flags |= _lib.STEP_CHAINED if self._chain_ok else _lib.STEP_CHAIN_START
        if not flags & _lib.STEP_PHYSICS_ONLY:
            flags |= self._mode_flags
        if not self._write_zone_obs:
            flags |= _lib.STEP_NO_ZONE_OBS
        elif self._zone_obs_ok and not flags & (_lib.STEP_GOALS | _lib.STEP_WAIT) and not self.spec.walled:
            # only the rows that change are written (the goal-conditioned, WaitWrapper and walled kernels write all)
            flags |= _lib.STEP_ZONE_OBS_DELTA
        with self._guard():
            if actions is None:
                aptr = None
            else:
                if not (isinstance(actions, torch.Tensor) and actions.is_cuda and actions.dtype == torch.float32
                        and actions.is_contiguous()):
                    actions = self._as_dev(actions, torch.float32)
                assert actions.shape == (self.num_envs, 2)
                aptr = actions.data_ptr()
            # replayable draws count their steps on the device; the host index then stays out of it
            si = 0 if flags & _lib.STEP_ACTION_COUNTER else self._step_index
            _lib.check(self.lib.crl_step(self.cfg, self.state, aptr, self.out, flags, action_seed, si, self._stream()))
        self._step_index += 1
        self.gpu_launches += 1
        self._chain_ok = bool(chained)
        self._mirror_ok = False
        self._zone_obs_ok = self._write_zone_obs
        if self.prefetch_every and not torch.cuda.is_current_stream_capturing():
            self.tick()
        return self._obs_dict(), self.reward, self.done, self._info()

    def step(self, actions):
        """ParallelEnv.step (penv.py:52-59): finished envs restart inside the call; their
        returned observation is the new episode's first one, reward/done/info the old one's.
        The returned tensors are the env's own buffers and READ-ONLY for the caller: once ``zone_obs``
        holds the current rows, a step rewrites only the rows that change, so an in-place edit would stay."""
        # with wait=True a parked env (finished under step_no_reset) is WaitWrapper's no-op followed by
        # the worker's reset: (first obs of the new episode, 0, True, {}) -- wrappers.py:36-44, penv.py:7-10
        return self._step(actions, (_lib.STEP_AUTO_RESET if self.auto_reset else 0) | (_lib.STEP_WAIT if self.wait else 0))

    def step_no_reset(self, actions):
        """ParallelEnv.step_no_reset (penv.py:61-66).  With ``wait=True`` (the reference wraps each
        env in WaitWrapper for the hierarchical collectors) an env that finished earlier is a
        no-op: zero observation, reward 0, done True, until reset().  The returned tensors are
        read-only for the caller, as with step()."""
        return self._step(actions, _lib.STEP_WAIT if self.wait else 0)

    # -- goal RPCs of the goal-conditioned variants (zone-goals penv.py:75-99), batched ------
    def _need_goals(self):
        if not self.spec.goals:
            raise RuntimeError(f'{self.env_id} is not a goal-conditioned variant (use PointTSP-v3, ...)')

    def set_goal(self, goals):
        """env.set_goal for the whole batch (TSP_next_city_env.py:77-80): ``goals`` (B,) int,
        negative = leave that env alone.  Invalid requests (visited zone, index out of range: the
        reference's assertion) leave the goal unset and are counted in counters()['goals_rejected']."""
        self._need_goals()
        g = self._as_dev(goals, torch.int32).reshape(self.num_envs)
        with self._guard():
            _lib.check(self.lib.crl_set_goal(self.cfg, self.state, g.data_ptr(), self._stream()))
        self._chain_ok = False

    def set_goal_at(self, env_idx, goal):
        """ParallelEnv.set_goal(env_idx, goal) (zone-goals penv.py:75-80): one env."""
        g = torch.full((self.num_envs,), -1, dtype=torch.int32, device=self.device)
        g[int(env_idx)] = int(goal)
        self.set_goal(g)

    def _goal_query(self, xy=False, needs=False, available=False):
        self._need_goals()
        with self._guard():
            _lib.check(self.lib.crl_goal_query(self.cfg, self.state,
                                               self._goal_xy.data_ptr() if xy else None,
                                               self._needs_goal.data_ptr() if needs else None,
                                               self._available.data_ptr() if available else None,
                                               self._stream()))
        self._chain_ok = False

    def get_goal(self, env_idx=None):
        """(B,2) goal coordinates / 3 (zeros where no goal is set); one env if env_idx is given."""
        self._goal_query(xy=True)
        return self._goal_xy if env_idx is None else self._goal_xy[env_idx]

    def needs_goal(self):
        """(B,) bool: goal_zone is None (penv.py:88-93)."""
        self._goal_query(needs=True)
        return self._needs_goal.view(torch.bool)

    def available_goals(self, env_idx=None):
        """(B,N) bool mask of eligible goal zones (penv.py:94-99)."""
        self._goal_query(available=True)
        a = self._available.view(torch.bool)
        return a if env_idx is None else a[env_idx]

    def step_random(self, action_seed=1, auto_reset=True, chained=False, replayable=False):
        """A step with U(-1,1)^2 actions drawn in-kernel (Philox): action_space.sample().
        ``chained=True`` for back-to-back rollout steps with nothing else enqueued in between.
        ``replayable=True`` (CRL_STEP_ACTION_COUNTER): the draw's step index advances on the device, so a
        CUDA graph that captured this call draws fresh iid actions at every replay.  The returned tensors
        are read-only for the caller, as with step().  A captured step keeps the zone_obs mode it was
        captured with: captured while ``zone_obs`` held the current rows, every replay writes only the rows
        that change, so the graph must not be replayed after anything that leaves stale rows there
        (bind_outputs, a step with ``write_zone_obs = False``, load_state_dict, a masked reset)."""
        flags = (_lib.STEP_AUTO_RESET if auto_reset else 0) | (_lib.STEP_ACTION_COUNTER if replayable else 0)
        return self._step(None, flags, action_seed, chained=chained)

    def step_host(self, actions, auto_reset=True, delta=True, wait=False):
        """The reference-facing call with HOST buffers: numpy actions in, numpy obs /
        reward / done out (pinned staging; host<->device copies inside the call).  The returned
        arrays are persistent host buffers overwritten by the next call, as the device ones are --
        READ-ONLY for the caller: on the delta path a zone_obs row or a result record is rewritten only
        when it changes, so an in-place edit (``reward *= scale``) would stay there; copy first.

        ``delta=True``: once the host buffers mirror the device ones (after the first call), a call is ONE kernel and a
        stream synchronisation -- the step kernel reads the actions from, and writes obs / result / shaped_reward and the
        changed zone_obs rows to, the pinned host buffers itself, through a prepared call object (``crl_host_call_step``:
        three arguments per frame, buffers and flags resolved once).  A result record (reward, done, goal_met, event,
        need_next_goal: all zeros except on an event) crosses only when it differs from the one the host array already
        holds.  The arrays returned are byte-identical to a full copy.  The DEVICE tensor ``env.obs`` is then not updated
        by the call (``env.zone_obs`` and ``env.result`` are).  TimedTSP's time-left column moves every step: its host
        mirror is plane-major (``zone_obs`` is then a (B, N, Z) strided view of a [Z][B][N] buffer) and that column
        crosses as one contiguous plane.  ``env.delta_rows`` = rows the call moved (B = all; -1 = counted on the device
        only, see ``host_rows_moved()`` / ``host_results_moved()``)."""
        h = self._host or self._host_buffers()
        if delta and self._mirror_ok:
            # the prepared call (crl_host_call_*): buffers and flags resolved once, three arguments per frame
            call = self._host_calls.get((auto_reset, wait))
            if call is None:
                call = self._host_call(auto_reset, wait)
            pin = self._pinned.get(id(actions))
            if pin is not None:                       # one of pinned_actions(): read where it lies
                aptr = pin[1]
            else:
                aptr = h['actions_ptr']
                if actions is not h['np']['actions']:
                    np.copyto(h['np']['actions'], np.asarray(actions, dtype=np.float32).reshape(self.num_envs, 2))
            if torch.cuda.current_device() == self._dev_index:
                rc = self._host_call_step(call, aptr, _raw_stream(self._dev_index))
            else:
                with torch.cuda.device(self.device):
                    rc = self._host_call_step(call, aptr, _raw_stream(self._dev_index))
            if rc:
                _lib.check(rc)
            self.delta_rows = -1
            self._step_index += 1
            self.gpu_launches += 1
            self._chain_ok = False
            self._zone_obs_ok = True              # the kernel writes all of the device zone_obs as well
            if self.prefetch_every:
                self.tick()
            return h['ret']
        hn = h['np']
        aptr = h['actions_ptr']
        if actions is not hn['actions']:
            pin = self._pinned.get(id(actions))
            if pin is not None:                       # one of pinned_actions(): read where it lies
                aptr = pin[1]
            else:
                np.copyto(hn['actions'], np.asarray(actions, dtype=np.float32).reshape(self.num_envs, 2))
        flags = (_lib.STEP_AUTO_RESET if auto_reset else 0) | self._mode_flags
        if wait:
            flags |= _lib.STEP_WAIT
        with self._guard():
            if self.spec.task == _lib.TASK_TTSP:
                # full copy into the plane-major mirror: step on the device, then everything crosses (the device
                # transposes zone_obs to [Z][B][N] first)
                src = h['actions'] if aptr == h['actions_ptr'] else self._pinned[id(actions)][0]
                self._actions_dev.copy_(src, non_blocking=True)
                _lib.check(self.lib.crl_step(self.cfg, self.state, self._actions_dev.data_ptr(), self.out, flags, 0,
                                             self._step_index, self._stream()))
                h['zone_obs'].copy_(self.zone_obs.permute(2, 0, 1), non_blocking=True)
                h['obs'].copy_(self.obs, non_blocking=True)
                h['result'].copy_(self.result, non_blocking=True)
                if self.spec.goals:
                    h['shaped'].copy_(self.shaped_reward, non_blocking=True)
                torch.cuda.current_stream(self.device).synchronize()
            else:
                _lib.check(self.lib.crl_step_host(self.cfg, self.state, aptr,
                                                  self._actions_dev.data_ptr(), self.out, h['out'],
                                                  flags, self._stream()))
        self.delta_rows = self.num_envs
        self._step_index += 1
        self.gpu_launches += 1
        self._chain_ok = False                    # memcpys follow the step kernel on the stream
        self._mirror_ok = True
        self._zone_obs_ok = True                  # every path above writes all of the device zone_obs
        if self.prefetch_every:
            self.tick()                           # the background sampler's cadence, as in _step
        return h['ret']

    def _host_call(self, auto_reset, wait):
        """crl_host_call_create for one (auto_reset, wait) combination of step_host; kept until close()."""
        h = self._host
        flags = (_lib.STEP_AUTO_RESET if auto_reset else 0) | (_lib.STEP_WAIT if wait else 0) | self._mode_flags
        if self.spec.task == _lib.TASK_TTSP:
            flags |= _lib.STEP_HOST_PLANES            # plane-major host mirror, see _host_buffers
        call = ctypes.c_void_p()
        with self._guard():
            _lib.check(self.lib.crl_host_call_create(self.cfg, self.state, self.out, h['out'], flags, ctypes.byref(call)))
        self._host_calls[(auto_reset, wait)] = call
        return call

    def close(self):
        """Free the prepared host calls (the tensors go with the object)."""
        calls, self._host_calls = self._host_calls, {}
        for call in calls.values():
            self.lib.crl_host_call_destroy(call)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def host_rows_moved(self, reset=False):
        """zone_obs rows the host-direct step_host calls have written to the host mirror since the count was last
        reset (the kernel counts them in CrlState.row_list[0])."""
        n = int(self._row_list[0].item())
        if reset:
            self._row_list[:1].zero_()
        return n

    def host_results_moved(self, reset=False):
        """Result records the host-direct step_host calls have written to the host array since the count was last reset
        (CrlState.row_list[1]); the others were equal to what the host already held."""
        n = int(self._row_list[1].item())
        if reset:
            self._row_list[1:2].zero_()
        return n

    def _host_buffers(self):
        if self._host is None:
            B, N, Z = self.num_envs, self.spec.num_zones, self.spec.zone_dim
            pin = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype).pin_memory()
            # TimedTSP: the host mirror of zone_obs is PLANE-major, [Z][B][N], handed out as a (B, N, Z) strided view:
            # the time-left column, which moves every step, is then one contiguous plane (CRL_STEP_HOST_PLANES)
            zshape = (Z, B, N) if self.spec.task == _lib.TASK_TTSP else (B, N, Z)
            h = {'actions': pin(B, 2, dtype=torch.float32), 'obs': pin(B, 8, dtype=torch.float32),
                 'zone_obs': pin(*zshape, dtype=torch.float32), 'result': pin(B, 8, dtype=torch.uint8),
                 'shaped': pin(B, dtype=torch.float32)}
            h['out'] = _lib.CrlOut(obs=h['obs'].data_ptr(), zone_obs=h['zone_obs'].data_ptr(),
                                   result=h['result'].data_ptr(), shaped_reward=h['shaped'].data_ptr())
            h['np'] = {k: h[k].numpy() for k in ('actions', 'obs', 'zone_obs', 'result', 'shaped')}
            if self.spec.task == _lib.TASK_TTSP:
                h['np']['zone_obs'] = h['np']['zone_obs'].transpose(1, 2, 0)
            h['actions_ptr'] = h['actions'].data_ptr()
            # what every step_host call returns: views of the persistent host buffers, built once
            res = h['np']['result']
            info = {'goal_met': res[:, 5].view(np.bool_), 'event': res[:, 6].view(np.int8)}
            if self.spec.goals:
                info['shaped_reward'] = h['np']['shaped']
                info['need_next_goal'] = res[:, 7].view(np.bool_)
            h['ret'] = ({'zone_obs': h['np']['zone_obs'], 'obs': h['np']['obs']}, res.view(np.float32)[:, 0],
                        res[:, 4].view(np.bool_), info)
            self._host = h
        return self._host

    def pinned_actions(self, n=1):
        """``n`` page-locked (B,2) float32 numpy arrays for the caller to fill with actions: step_host reads an
        array of this pool where it lies (no staging copy).  Any other array is first copied into the env's own
        pinned buffer."""
        out = []
        for _ in range(n):
            t = torch.zeros(self.num_envs, 2, dtype=torch.float32).pin_memory()
            a = t.numpy()
            self._pinned[id(a)] = (t, t.data_ptr(), a)
            out.append(a)
        return out

    def host_actions(self):
        """The pinned (B,2) float32 action buffer step_host stages from; filling it in place and
        passing it to step_host skips one host copy."""
        return self._host_buffers()['np']['actions']

    # -- extras ----------------------------------------------------------------------
    @property
    def steps(self):
        return self.aux[:, 3].view(torch.int32) & 0xffff

    def counters(self, allow_chain_timeouts=False):
        """Episode statistics accumulated in-kernel since construction.  Raises if a chained step ever
        gave up its wait (see CRL_STEP_CHAINED), unless ``allow_chain_timeouts``."""
        out = (ctypes.c_double * 8)()
        with self._guard():
            _lib.check(self.lib.crl_counters_read(self.state, out, self._stream()))
        if out[7] != 0 and not allow_chain_timeouts:
            # a chained step (CRL_STEP_CHAINED) gave up waiting for its own previous step and went on:
            # the state may be corrupt.  Never seen; never to be ignored.
            raise RuntimeError(f'{int(out[7])} chained step(s) stopped waiting for their predecessor '
                               '(counters[7]); the env state is not trustworthy')
        return {'return_sum': out[0], 'episodes': out[1], 'successes': out[2], 'length_sum': out[3],
                'resets_prefetched': out[4], 'resets_inline': out[5], 'goals_rejected': out[6],
                'chain_wait_timeouts': out[7]}

    def check_state(self):
        """Invariant check of the state planes (crl_check_state); returns the eight violation counts
        as a list of ints -- all zero on a healthy env.  Synchronises."""
        v = torch.zeros(8, dtype=torch.int64, device=self.device)
        with self._guard():
            _lib.check(self.lib.crl_check_state(self.cfg, self.state, v.data_ptr(), self._stream()))
        bad = [int(x) for x in v.cpu()]
        if float(self.counters_dev[7].item()) != 0:
            raise RuntimeError('a chained step stopped waiting for its predecessor (counters[7]); the env state is '
                               'not trustworthy')
        return bad

    _STATE_KEYS = ('pose', 'aux', 'zone_xy', 'zone_tmax', 'cooldown', 'seeds', 'episode', 'origin', 'counters_dev',
                   'goal', 'obs', 'zone_obs', 'result', 'shaped_reward')

    def state_dict(self):
        """Everything needed to continue a run bit for bit (the reference has no equivalent: its
        envs live in worker processes and die with them): clones of the state and output planes.
        Parked next layouts are not saved -- they are pure functions of the seeds and are redrawn."""
        torch.cuda.current_stream(self.device).synchronize()
        d = {k: getattr(self, k).clone() for k in self._STATE_KEYS if getattr(self, k) is not None}
        d['step_index'] = self._step_index
        d['action_count'] = self.stamp[2].clone()     # CRL_STEP_ACTION_COUNTER steps taken, per 32 envs
        d['env_id'], d['num_envs'], d['num_steps'] = self.env_id, self.num_envs, int(self.cfg.num_steps)
        return d

    def load_state_dict(self, d):
        assert d['env_id'] == self.env_id and d['num_envs'] == self.num_envs
        torch.cuda.current_stream(self.device).wait_stream(self._side)      # no sampler round in flight while slots are dropped
        for k in self._STATE_KEYS:
            if getattr(self, k) is not None:
                getattr(self, k).copy_(d[k])
        self.cfg.num_steps = d['num_steps']
        self._step_index = d['step_index']
        self.next_ready.zero_()                   # parked layouts belong to the run that was interrupted
        self.stamp[:2].zero_()
        if 'action_count' in d:
            self.stamp[2].copy_(d['action_count'])
        self._chain_ok = False
        self._mirror_ok = False
        self._zone_obs_ok = False
        if self.prefetch_every and self.state.bank_zone_xy is None:
            self.prefetch(torch.cuda.current_stream(self.device))

    # -- env copies (crl_copy_envs) ----------------------------------------------------
    def snapshot(self, env_ids=None):
        """The state and output rows of envs ``env_ids`` (default: all), gathered into an ``EnvSnapshot`` on this env's
        device.  ``env_ids``: a host sequence (checked here) or a CUDA int tensor (an id out of range is skipped on the
        device and counted in ``copy_rejects``; its snapshot env stays zero).  Asynchronous on the current stream."""
        n, sid, _ = self._copy_ids(self, env_ids, None, check_dst=False)
        if not n:
            raise ValueError('snapshot: no envs')
        return self._snapshot(n, sid)

    def _snapshot(self, n, sid, rejected=True):
        snap = EnvSnapshot(self, n)
        both = self.zone_obs is not None
        with self._guard():
            _lib.check(self.lib.crl_copy_envs(snap.cfg, snap.state, _copy_out(snap, both), None,
                                              self.cfg, self.state, _copy_out(self, both),
                                              None if sid is None else sid.data_ptr(), n,
                                              self.copy_rejects.data_ptr() if rejected else None, self._stream()))
        snap.zone_obs_ok = both and self._zone_obs_ok
        self._chain_ok = False                    # the kernel before this env's next step is not a step
        self.gpu_launches += 1
        return snap

    def copy_envs_from(self, src, src_ids=None, dst_ids=None):
        """Make envs ``dst_ids`` of this env exact copies of envs ``src_ids`` of ``src``: state and output rows, bit
        for bit (crl_copy_envs).  ``src`` is an ``EnvSnapshot`` (restore: ids index the snapshot) or a ``ZoneVecEnv``
        (branching; ``src`` may be this env, any permutation of its envs is then copied correctly through a temporary
        snapshot).  ``None`` ids stand for 0..n-1; ``n`` is the length of the ids given, else ``src.num_envs``.

        Ids are host sequences, checked here (range, distinct dst ids, equal lengths: ``ValueError``), or CUDA int
        tensors, passed on unsynchronised: a pair with an id out of range is skipped on the device and counted in
        ``copy_rejects``.  ``src`` must have this env's id, device and config (``num_steps`` included) but may differ in
        size, offset and seed range (``ValueError`` otherwise).  The copies then take the same actions to the same
        outputs and states as their sources -- through auto-resets too with ``seed_mode='increment'`` or a layout bank;
        with ``seed_mode='fixed_range'`` until the episode ends, since the next seed is drawn from the dst's global
        index, as in-kernel random actions are.  Episode counters are not copied.  Asynchronous on the current stream."""
        if not isinstance(src, (ZoneVecEnv, EnvSnapshot)):
            raise TypeError(f'copy_envs_from: src must be a ZoneVecEnv or an EnvSnapshot, not {type(src).__name__}')
        if src.env_id != self.env_id:
            raise ValueError(f'copy_envs_from: src is {src.env_id}, this env is {self.env_id}')
        if _dev_index(src.device) != self._dev_index:
            raise ValueError(f'copy_envs_from: src lives on {src.device}, this env on {self.device}')
        if _task_config(src.cfg) != _task_config(self.cfg):
            raise ValueError('copy_envs_from: src has another config (num_steps, ...) than this env')
        n, sid, did = self._copy_ids(src, src_ids, dst_ids)
        if not n:
            return
        # a sampler round still running on the side stream writes slot flags the copy clears
        if not torch.cuda.is_current_stream_capturing():
            torch.cuda.current_stream(self.device).wait_stream(self._side)
        if src is self:
            # through a snapshot of the src envs: the id sets of one crl_copy_envs on one state must be disjoint
            if sid is not None and did is not None:
                # a src id rejected by the gather leaves a zero env in the snapshot: not to be copied on
                did = torch.where((sid >= 0) & (sid < self.num_envs), did, torch.full_like(did, -1))
            elif sid is not None:
                ar = torch.arange(n, dtype=torch.int32, device=self.device)
                did = torch.where((sid >= 0) & (sid < self.num_envs), ar, torch.full_like(ar, -1))
            src, sid = self._snapshot(n, sid, rejected=False), None
        both = src.zone_obs is not None and self.zone_obs is not None
        src_zone_ok = src.zone_obs_ok if isinstance(src, EnvSnapshot) else src._zone_obs_ok
        with self._guard():
            _lib.check(self.lib.crl_copy_envs(self.cfg, self.state, _copy_out(self, both),
                                              None if did is None else did.data_ptr(),
                                              src.cfg, src.state, _copy_out(src, both),
                                              None if sid is None else sid.data_ptr(), n,
                                              self.copy_rejects.data_ptr(), self._stream()))
        self.gpu_launches += 1
        self.copy_count += 1
        self._mirror_ok = False
        self._chain_ok = False
        # the untouched rows keep what they held; the copied ones are current only if the source's were
        self._zone_obs_ok = self._zone_obs_ok and both and src_zone_ok
        if isinstance(src, ZoneVecEnv):
            src._chain_ok = False

    def _copy_ids(self, src, src_ids, dst_ids, check_dst=True):
        """(n, src ids, dst ids) of a copy from ``src`` into this env: each id list None (= 0..n-1) or a device int32
        tensor.  Host ids are checked here; device ids only for their device and length."""
        def prep(ids, bound, what, distinct):
            if ids is None:
                return None, None
            if isinstance(ids, torch.Tensor) and ids.is_cuda:
                if ids.is_floating_point() or ids.is_complex() or ids.dtype == torch.bool:
                    raise ValueError(f'{what} ids must be integers, not {ids.dtype}')
                if _dev_index(ids.device) != self._dev_index:
                    raise ValueError(f'{what} ids live on {ids.device}, the envs on {self.device}')
                ids = ids.reshape(-1)
                if ids.dtype != torch.int32:     # an id beyond int32 stays out of range instead of wrapping into it
                    ids = ids.clamp(-1, 2 ** 31 - 1).to(torch.int32)
                return ids.numel(), ids.contiguous()
            a = np.asarray(ids.cpu() if isinstance(ids, torch.Tensor) else ids)
            if a.dtype.kind not in 'iu' and a.size:
                raise ValueError(f'{what} ids must be integers, not {a.dtype}')
            a = a.astype(np.int64).reshape(-1)
            if a.size and (a.min() < 0 or a.max() >= bound):
                raise ValueError(f'{what} ids must lie in [0, {bound})')
            if distinct and np.unique(a).size != a.size:
                raise ValueError(f'{what} ids must be distinct')
            return a.size, a.astype(np.int32)
        ns, sid = prep(src_ids, src.num_envs, 'src', False)
        nd, did = prep(dst_ids, self.num_envs, 'dst', check_dst)
        if ns is not None and nd is not None and ns != nd:
            raise ValueError(f'copy_envs_from: {ns} src ids but {nd} dst ids')
        n = ns if ns is not None else nd if nd is not None else src.num_envs
        if sid is None and n > src.num_envs:
            raise ValueError(f'copy_envs_from: {n} envs from a src of {src.num_envs}')
        if check_dst and did is None and n > self.num_envs:
            raise ValueError(f'copy_envs_from: {n} envs into an env of {self.num_envs}')
        if not n:
            return 0, None, None
        up = lambda a: torch.from_numpy(a).to(self.device) if isinstance(a, np.ndarray) else a   # checked host ids
        return n, up(sid), up(did)

    def set_qpos_qvel(self, qpos, qvel, env_ids=None):
        """Overwrite sim.data.qpos / qvel (fp64, reference coordinates) of some envs."""
        qp, qv = self._as_dev(qpos, torch.float64).reshape(-1, 3), self._as_dev(qvel, torch.float64).reshape(-1, 3)
        ids = None if env_ids is None else self._as_dev(env_ids, torch.int32)
        with self._guard():
            _lib.check(self.lib.crl_set_qpos_qvel(self.cfg, self.state, qp.data_ptr(), qv.data_ptr(),
                                                  None if ids is None else ids.data_ptr(), qp.shape[0],
                                                  self._stream()))
        self._chain_ok = False
        self._mirror_ok = False
        self._zone_obs_ok = False

    def get_qpos_qvel(self, env_ids=None):
        n = self.num_envs if env_ids is None else len(env_ids)
        qp = torch.empty(n, 3, dtype=torch.float64, device=self.device)
        qv = torch.empty_like(qp)
        ids = None if env_ids is None else self._as_dev(env_ids, torch.int32)
        with self._guard():
            _lib.check(self.lib.crl_get_qpos_qvel(self.cfg, self.state, qp.data_ptr(), qv.data_ptr(),
                                                  None if ids is None else ids.data_ptr(), n, self._stream()))
        self._chain_ok = False
        return qp, qv

    def physics_substeps(self, actions, n):
        """Debug/parity: integrate n MuJoCo substeps with no task logic."""
        old = self.cfg.frameskip
        self.cfg.frameskip = n
        try:
            return self._step(actions, _lib.STEP_PHYSICS_ONLY)
        finally:
            self.cfg.frameskip = old


def make_vec_env(env_id, num_envs, **kw):
    return ZoneVecEnv(env_id, num_envs, **kw)
