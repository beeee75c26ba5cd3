"""On-device rollout storage and GAE: what BaseAlgo.collect_experiences keeps per update
(main/src/torch_ac/algos/base.py:86-108 buffers, :110-249 loop), without leaving the GPU.

The reference stores each frame by copying Python lists into torch tensors
(base.py:145-166) after pickling them through a pipe.  Here a rollout owns T + 1 output slots
and, before step t, points the env's outputs at slot t + 1 (ZoneVecEnv.bind_outputs): the step
kernel writes obs, zone_obs and the result record straight into the rollout, so storing a frame
is free.  Advantages are computed by crl_gae from those records (bit-identical to
base.py:195-205).

    ro = Rollout(env, num_frames_per_proc=128)
    obs = ro.begin()                              # reset, or carry over from the previous rollout
    for t in range(ro.T):
        dist, value = acmodel(obs)                # obs: {'obs': (B,8), 'zone_obs': (B,N,Z)} views of slot t
        action = dist.sample()
        obs, reward, done, info = ro.step(t, action, value, dist.log_prob(action))
    exps = ro.finish(next_value=acmodel(obs)[1])  # advantages, returns, flattened P x T like base.py:225-231

Layout note: tensors are kept T-major, (T, B, ...), as the reference's own buffers are;
``finish`` returns both the (T, B) tensors and, on request, the reference's P x T flattening
(env-major), which is a transposing copy -- flat (non-recurrent) PPO samples frames at random and
does not need it.

``store='frames'``: zone_obs is not stored at all.  A zone row is a pure function of the zone layout (fixed for an
episode), the state word aux.w and the ColourMatch cooldown bytes, so each frame keeps one 16-byte record per env
(include/crl_b200.h: CrlFrame) and each episode its layout once, in a table of ``layout_capacity`` entries.  The steps
run with ``env.write_zone_obs = False``; a small kernel behind each step writes the records (crl_frame_capture).  The
observation is then ``{'obs': (B,8), 'zone_frames': ZoneFrames}``: ``ZoneEncoder`` / ``FusedZoneEnvModel`` build the
rows inside their kernels, forward and backward; a torch policy calls ``.zone_obs()``.
"""
import ctypes

import torch

from . import _lib


class ZoneFrames:
    """Stored frames of a ``Rollout(store='frames')``: CrlFrame records (int32 ``(..., 4)``, any leading shape) plus
    the rollout's layout table and the env's config.  Indexing and ``reshape`` / ``transpose`` act on the records only
    (``flat(x)[idx]`` of a minibatch gather works as for a tensor); ``zone_obs()`` materialises the rows, bit for bit
    the ``zone_obs`` the step would have written.  Valid until the rollout's next ``begin()``, which refills the table."""

    def __init__(self, records, layout_xy, layout_tmax, cfg, lib=None):
        self.records, self.layout_xy, self.layout_tmax, self.cfg = records, layout_xy, layout_tmax, cfg
        self.lib = lib or _lib.load()

    def _with(self, records):
        return ZoneFrames(records, self.layout_xy, self.layout_tmax, self.cfg, self.lib)

    @property
    def shape(self):
        return self.records.shape[:-1]

    @property
    def device(self):
        return self.records.device

    @property
    def num_zones(self):
        return int(self.cfg.num_zones)

    @property
    def zone_dim(self):
        return 6 if self.cfg.task == _lib.TASK_TSP else 7

    def __len__(self):
        return self.records.shape[0]

    def __getitem__(self, idx):
        return self._with(self.records[idx])

    def reshape(self, *shape):
        shape = tuple(shape[0]) if len(shape) == 1 and isinstance(shape[0], (tuple, list, torch.Size)) else shape
        return self._with(self.records.reshape(*shape, 4))

    def transpose(self, d0, d1):
        n = self.records.dim() - 1
        return self._with(self.records.transpose(d0 % n, d1 % n))

    def flat_records(self):
        """(M, 4) contiguous records: what the library entries take."""
        return self.records.reshape(-1, 4).contiguous()

    def ptrs(self):
        """(layout_xy, layout_tmax) device pointers of the table."""
        return self.layout_xy.data_ptr(), None if self.layout_tmax is None else self.layout_tmax.data_ptr()

    def zone_obs(self, out=None):
        """The rows, ``shape + (N, Z)`` float32 (crl_frames_zone_obs)."""
        rec = self.flat_records()
        M, N, Z = rec.shape[0], self.num_zones, self.zone_dim
        if out is None:
            out = torch.empty(tuple(self.shape) + (N, Z), dtype=torch.float32, device=self.device)
        assert out.shape == tuple(self.shape) + (N, Z) and out.dtype == torch.float32 and out.is_contiguous()
        if M == 0:
            return out
        xy, tm = self.ptrs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_frames_zone_obs(self.cfg, M, rec.data_ptr(), xy, tm, out.data_ptr(),
                                                    ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return out


class Rollout:
    """``store='zone_obs'`` (default): every slot keeps the step's zone_obs rows.  ``store='frames'``: one CrlFrame
    record per env and slot plus a layout table of ``layout_capacity`` entries (default B (1 + ceil(T / 32)): enough
    unless episodes average fewer than about 32 steps); see the module docstring.  ``finish()`` raises if the table was
    too small."""

    def __init__(self, env, num_frames_per_proc, discount=0.99, gae_lambda=0.95, store='zone_obs', layout_capacity=None):
        self.env, self.T = env, int(num_frames_per_proc)
        self.discount, self.gae_lambda = float(discount), float(gae_lambda)
        B, N, Z, T, dev = env.num_envs, env.spec.num_zones, env.spec.zone_dim, self.T, env.device
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=dev)
        if store not in ('zone_obs', 'frames'):
            raise ValueError(f"store must be 'zone_obs' or 'frames', not {store!r}")
        self.store = store
        if store == 'frames':
            self._init_frames(layout_capacity)
            return
        # slot t = what the policy sees before step t; slot t + 1 = what step t returned
        self.obs = z(T + 1, B, 8)
        self.zone_obs = z(T + 1, B, N, Z)
        self.result = z(T + 1, B, 8, dtype=torch.uint8)
        self.shaped = z(T + 1, B) if env.spec.goals else None
        self.actions = z(T, B, 2)
        self.values = z(T, B)
        self.log_probs = z(T, B, 2)
        self.advantages = z(T, B)
        self.returns = z(T, B)
        self.rewards = self.result.view(torch.float32)[1:, :, 0]         # (T, B) view: reward of step t
        self.dones = self.result[1:, :, 4].view(torch.bool)              # (T, B) view
        self._started = False
        assert B % 4 == 0, 'slots of zone_obs must start 16-byte aligned: num_envs must be a multiple of 4'
        # one validated output binding per slot, installed with a few attribute stores per step
        self._bindings = [env.prepare_outputs(self.obs[t], self.zone_obs[t], self.result[t],
                                              None if self.shaped is None else self.shaped[t]) for t in range(T + 1)]
        self._obs_views = [{'zone_obs': self.zone_obs[t], 'obs': self.obs[t]} for t in range(T + 1)]
        self._action_views = [self.actions[t] for t in range(T)]

    def _init_frames(self, layout_capacity):
        env, T = self.env, self.T
        B, N, dev = env.num_envs, env.spec.num_zones, env.device
        if env.wait:
            raise ValueError("Rollout(store='frames'): a WaitWrapper env (wait=True) reports all-zero rows for parked "
                             "envs, which are not a function of the stored record; use store='zone_obs'")
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=dev)
        self.obs = z(T + 1, B, 8)
        self.zone_obs = None
        self.result = z(T + 1, B, 8, dtype=torch.uint8)
        self.shaped = z(T + 1, B) if env.spec.goals else None
        self.actions = z(T, B, 2)
        self.values = z(T, B)
        self.log_probs = z(T, B, 2)
        self.advantages = z(T, B)
        self.returns = z(T, B)
        self.rewards = self.result.view(torch.float32)[1:, :, 0]
        self.dones = self.result[1:, :, 4].view(torch.bool)
        self._started = False
        self.layout_capacity = int(layout_capacity) if layout_capacity is not None else B * (1 + -(-T // 32))
        if not 1 <= self.layout_capacity < 2 ** 32 - 1:
            raise ValueError('layout_capacity must be in [1, 2^32 - 2]')
        self.frames = z(T + 1, B, 4, dtype=torch.int32)                 # CrlFrame[T + 1][B]
        self.layout_xy = z(self.layout_capacity, N, 2)
        self.layout_tmax = z(self.layout_capacity, (N + 1) // 2, dtype=torch.int32) if env.spec.task == _lib.TASK_TTSP else None
        self._fill = z(2, dtype=torch.int32)                            # entries handed out, entries requested
        self._fill_host = torch.zeros(2, dtype=torch.int32).pin_memory()
        self._reset_zone_obs = None                                     # the reset writes zone_obs: a scratch slot
        self._bindings = [env.prepare_outputs(self.obs[t], None, self.result[t], None if self.shaped is None else self.shaped[t])
                          for t in range(T + 1)]
        self._frame_views = [ZoneFrames(self.frames[t], self.layout_xy, self.layout_tmax, env.cfg, env.lib)
                             for t in range(T + 1)]
        self._obs_views = [{'obs': self.obs[t], 'zone_frames': self._frame_views[t]} for t in range(T + 1)]
        self._action_views = [self.actions[t] for t in range(T)]
        # the capture's per-slot pointers, resolved once: a Rollout.step pays one more library call, nothing else
        tmax = None if self.layout_tmax is None else self.layout_tmax.data_ptr()
        self._capture_args = [(self.result[t].data_ptr(), self.frames[t].data_ptr()) for t in range(T + 1)]
        self._table_args = (self.layout_xy.data_ptr(), tmax, self.layout_capacity, self._fill.data_ptr())
        self._capture_fn = env.lib.crl_frame_capture

    def _capture(self, t, initial):
        env = self.env
        result, frames = self._capture_args[t]
        rc = self._capture_fn(env.cfg, env.state, None if initial else result, 1 if initial else 0, frames,
                              *self._table_args, env._stream())
        if rc:
            _lib.check(rc)
        env.gpu_launches += 1

    def storage_bytes(self):
        """Device bytes of the rollout's buffers, by name (computed from the shapes)."""
        names = ('obs', 'zone_obs', 'frames', 'layout_xy', 'layout_tmax', 'result', 'shaped', 'actions', 'values',
                 'log_probs', 'advantages', 'returns')
        return {k: getattr(self, k).numel() * getattr(self, k).element_size() for k in names
                if getattr(self, k, None) is not None}

    def _bind(self, t):
        self.env.bind_outputs(binding=self._bindings[t])

    def obs_at(self, t):
        return self._obs_views[t]

    def begin(self, reset=None):
        """Start a rollout: the first one (or ``reset=True``) resets every env into slot 0; later
        ones carry slot T of the previous rollout over to slot 0 (base.py keeps self.obs and
        self.mask across calls the same way)."""
        if reset is None:
            reset = not self._started
        if self.store == 'frames':
            return self._begin_frames(reset)
        if reset:
            self._bind(0)
            self.env.reset()
            self.result[0].zero_()                        # mask = 1: no env has just finished
        else:
            self.obs[0].copy_(self.obs[self.T])
            self.zone_obs[0].copy_(self.zone_obs[self.T])
            self.result[0].copy_(self.result[self.T])
        self._started = True
        return self.obs_at(0)

    def _begin_frames(self, reset):
        env = self.env
        if reset:
            if self._reset_zone_obs is None:                  # crl_reset writes the first rows: somewhere to put them
                self._reset_zone_obs = torch.zeros(env.num_envs, env.spec.num_zones, env.spec.zone_dim,
                                                   dtype=torch.float32, device=env.device)
            env.bind_outputs(self.obs[0], self._reset_zone_obs, self.result[0],
                             None if self.shaped is None else self.shaped[0])
            env.reset()
            self.result[0].zero_()
        else:
            self.obs[0].copy_(self.obs[self.T])
            self.result[0].copy_(self.result[self.T])
        env.write_zone_obs = False
        self._fill.zero_()                                    # the table restarts with every rollout
        with env._guard():
            self._capture(0, initial=True)
        self._started = True
        return self.obs_at(0)

    def step(self, t, actions, values=None, log_probs=None):
        """ParallelEnv.step for frame t (auto-reset on), outputs written into slot t + 1."""
        a = self._action_views[t]
        if actions.data_ptr() != a.data_ptr():            # a policy may also write into ro.actions[t] directly
            a.copy_(actions)
        if values is not None:
            self.values[t].copy_(values)
        if log_probs is not None:
            self.log_probs[t].copy_(log_probs)
        self._bind(t + 1)
        env = self.env
        if self.store == 'frames':
            if env._write_zone_obs:
                env.write_zone_obs = False
            _, reward, done, info = env.step(a)
            with env._guard():                              # free when the env's device is current
                self._capture(t + 1, initial=False)
            return self._obs_views[t + 1], reward, done, info
        _, reward, done, info = env.step(a)
        return self._obs_views[t + 1], reward, done, info

    def masks(self):
        """(T, B) float: masks[t] = 1 - done of the step before frame t (base.py:151-152)."""
        return 1.0 - self.result[:self.T, :, 4].float()

    def finish(self, next_value, flatten=False):
        """base.py:182-205: advantages and returns of the rollout just collected.  Rewards are the
        shaped rewards for the goal-conditioned variants (base.py:155-159)."""
        env, T, B = self.env, self.T, self.env.num_envs
        if self.store == 'frames':
            self._fill_host.copy_(self._fill, non_blocking=True)
            torch.cuda.current_stream(env.device).synchronize()
            requested = int(self._fill_host[1]) & 0xffffffff
            if requested > self.layout_capacity:
                raise RuntimeError(f'Rollout: the layout table holds {self.layout_capacity} entries but this rollout '
                                   f'needed {requested} (frames of the episodes that did not fit build NaN rows); '
                                   f'pass layout_capacity >= {requested}')
        nv = next_value.to(device=env.device, dtype=torch.float32).reshape(B).contiguous()
        with torch.cuda.device(env.device):
            _lib.check(env.lib.crl_gae(self.result.data_ptr(),
                                       None if self.shaped is None else self.shaped.data_ptr(),
                                       self.values.data_ptr(), nv.data_ptr(), ctypes.c_double(self.discount),
                                       ctypes.c_double(self.gae_lambda), T, B, self.advantages.data_ptr(),
                                       self.returns.data_ptr(), env._stream()))
        env.gpu_launches += 1
        out = {'advantage': self.advantages, 'returnn': self.returns, 'value': self.values, 'action': self.actions,
               'log_prob': self.log_probs, 'reward': self.rewards if self.shaped is None else self.shaped[1:],
               'obs': {'obs': self.obs[:T], 'zone_obs': self.zone_obs[:T]} if self.store == 'zone_obs' else
                      {'obs': self.obs[:T], 'zone_frames': self._frames_view(slice(0, T))}}
        if flatten:                                      # T x P -> P x T -> P * T, base.py:225-231
            pt = lambda x: x.transpose(0, 1).reshape((-1,) + tuple(x.shape[2:]))
            out = {k: ({kk: pt(vv) for kk, vv in v.items()} if isinstance(v, dict) else pt(v)) for k, v in out.items()}
        return out

    def _frames_view(self, idx):
        return ZoneFrames(self.frames[idx], self.layout_xy, self.layout_tmax, self.env.cfg, self.env.lib)
