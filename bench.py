#!/usr/bin/env python
"""bench.py -- env-steps/sec of the fused env.step() hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--env PointTSP-v0] [--envs 65536] [--dump-outputs DIR]

One "step" = one crl_step() launch over one batch of `--envs` envs (10 MuJoCo substeps + task logic +
full observation write per env, auto-reset on, iid U(-1,1)^2 actions drawn IN the kernel per (env, step):
SURVEY 8d).  Default workload = BASELINE.json configs[1]: PointTSP, 65,536 batched envs, 1 x B200.

Timing.  After W warm-up steps the bench times exactly K (= --steps) steps, back to back (CUDA events on the
launching stream, a barrier + synchronize on both sides).  The K steps are queued behind a device-side spin,
so the window holds device work only, not the host's launch of the first step.  `ms_per_step` = window / K
(the fastest and slowest graph replay inside the window are reported beside it).  A 65,536-env batch is
39 MB of state + observation and would sit in the 126 MB L2, so the steps cycle a RING of independent
replicas of the batch (each its own state, layouts and counters; together > 2 x L2): every launch finds its
inputs in HBM.  `value` = steps x envs / device time, max over ranks.  `e2e` = the same metric through
ZoneVecEnv.step_host(): HOST numpy actions in, HOST obs / reward / done out, copies inside every call.  The
same line also carries BASELINE.json configs[2] and [3] (`configs`), and under --gpus N > 1 configs[4] (all
three tasks at 1,048,576 envs per GPU).

Outputs.  Seeds and the in-kernel action draws are fixed, so the same arguments step the same envs with the
same actions in every run.  `--dump-outputs DIR` writes what the timed path's last step returned to its caller
(see dump_outputs()), so that two builds of the project can be compared output for output.

`--impl reference` times the reference's CPU path: mujoco-py / Safety Gym cannot be installed here, so that
is the oracle's port of it (oracle/), in three topologies -- see cpu_baselines().
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

L2_BYTES = 126 * 1024 * 1024
METRIC = 'env_steps_per_sec'
UNIT = 'env-steps/s'
CANON_BYTES = {'PointTSP-v0': 614, 'PointTTSP-v0': 734, 'ColourMatch-v0': 374}   # SURVEY 8d, unpacked layout


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get('hbm_gbs', 6650.0), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md, 6.65 TB/s)'


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc, self.first = index, [], None, 0

    def mark(self):
        """Samples taken before this call (warm-up) are dropped."""
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        self.t.join(timeout=2)
        self.rows = self.rows[max(0, self.first - 1):]
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for k, n in enumerate(names) if any(len(r) > 2 + k and r[2 + k] == 'Active' for r in self.rows)]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx[0] if mx else None,
                'reasons': reasons, 'samples': len(sm)}


# ---- CPU side: the reference's path on the host cores (oracle/ is test infrastructure; this is the one place
# ---- bench.py executes it, as the reported baseline -- never as the thing measured above) -------------------
def cpu_threads_port(env_id, seconds, threads=None):
    """The oracle's fp64 C port, free-running: one env per thread, no IPC (the STRONGEST CPU number)."""
    from oracle import c_oracle
    threads = threads or os.cpu_count() or 1
    rate, steps, wall = c_oracle.timed_rollout(env_id, threads=threads, seconds=seconds)
    return {'value': rate, 'unit': UNIT, 'cores': threads, 'kind': 'port',
            'sample': f'{steps} env-steps of {env_id} (fp64 C port of the reference path incl. numpy-legacy '
                      f'layout resets, random actions, {threads} threads x 1 env each, no IPC, {wall:.1f} s)'}


def cpu_variants(env_id, budget):
    """The reference's own topologies (oracle/penv_baseline.py): evaluate.py's single-process protocol on seeds
    1000000.. (BASELINE.json configs[0]) and ParallelEnv's process-per-env Pipe protocol with os.cpu_count()
    envs, each with the Python restatement of the task code and with the C twin behind the same pipes."""
    from oracle import penv_baseline as pb
    v = {}
    for name, fn in (('eval_single_process_c', lambda: pb.eval_protocol(env_id, impl='c', max_seconds=budget)),
                     ('eval_single_process_python', lambda: pb.eval_protocol(env_id, impl='python', max_seconds=budget)),
                     ('pipe_process_per_env_c', lambda: pb.pipe_vector_env(env_id, seconds=budget, impl='c')),
                     ('pipe_process_per_env_python', lambda: pb.pipe_vector_env(env_id, seconds=budget, impl='python'))):
        try:
            r = fn()
            v[name] = {'value': r['value'], 'unit': UNIT, 'cores': r.get('processes', 1), 'sample': r['sample']}
        except Exception as ex:                                       # a baseline never takes the bench down
            v[name] = {'error': repr(ex)}
    note = ('reference topologies: evaluate.py:47-72 (configs[0]) and penv.py:4-59 (process per env, Pipe, pickle); '
            '"python" = oracle/zone_env.py, the numpy restatement of the reference\'s Python task code; "c" = the C twin '
            'behind the same protocol')
    return v, note


def cpu_baselines(env_id, seconds):
    """cpu_baseline of the JSON line.  `value` = the C port on all host threads (what the reference's
    ALGORITHM costs on these cores: far above what its Python / mujoco-py / pipe implementation reaches, so
    every ratio against it is conservative); `variants` = cpu_variants()."""
    cb = cpu_threads_port(env_id, seconds)
    cb['variants'], cb['variants_note'] = cpu_variants(env_id, max(2.0, seconds / 3.0))
    return cb


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    per_step = 4.0
    cpu_threads_port(args.env, 1.0)                                   # warm-up
    k = max(1, min(args.steps, 5))
    vals = [cpu_threads_port(args.env, per_step) for _ in range(k)]
    v = sorted(x['value'] for x in vals)[len(vals) // 2]
    cb = dict(vals[-1], value=v)
    cb['variants'], cb['variants_note'] = cpu_variants(args.env, 3.0)
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': k,
        'warmup': 1, 'ms_per_step': per_step * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': f'{args.env} random-action rollouts on host cores; each step = {per_step:.0f} s sample',
                   'what': 'C PORT of the reference path (oracle/crl_oracle.c) on all host threads, one env per thread, '
                           'no IPC: mujoco-py / Safety Gym are not installable here. It is much FASTER than the '
                           'reference\'s own Python + pipes implementation (see cpu_baseline.variants), i.e. a '
                           'conservative baseline'},
        'cpu_baseline': cb,
        'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


# ---- GPU side -----------------------------------------------------------------------------------------
class Ring:
    """R independent replicas of one batch (> 2 x L2 together), stepped round-robin with in-kernel iid
    actions, as CUDA graphs of whole ring cycles."""

    def __init__(self, crl, _lib, args, env_id, B, dev, rank, chained=None, streams=1):
        import ctypes
        import torch
        self.torch, self.env_id, self.B, self.dev = torch, env_id, B, dev
        probe = crl.ZoneVecEnv(env_id, 32, device=dev, prefetch_every=0)
        rd, wr = ctypes.c_int64(), ctypes.c_int64()
        probe.lib.crl_step_bytes(probe.cfg, ctypes.byref(rd), ctypes.byref(wr))
        # the in-kernel action draw reads no action plane: 8 B less than crl_step_bytes' figure (SURVEY 8d)
        self.step_bytes = rd.value + wr.value - 8
        self.task = probe.spec.task
        del probe
        self.R = R = max(2, getattr(args, 'min_replicas', 0), -(-2 * L2_BYTES // (B * self.step_bytes)))
        # the replicas are independent batches: by default each is stepped on its own stream (up to 8), so that
        # the tail of one replica's launch overlaps another's body; on ONE stream back-to-back steps of small
        # batches chain warp by warp instead (CRL_STEP_CHAINED)
        self.S = S = max(1, min(streams if streams > 0 else 8, R))
        self.chained = (B <= 131072 and S == 1) if chained is None else bool(chained)
        bank_kw = self._bank(crl, args, dev) if args.bank else {}
        self.envs = []
        for r in range(R):
            e = crl.ZoneVecEnv(env_id, B, device=dev, env_offset=(rank * R + r) * B,
                               prefetch_every=args.prefetch_every, prefetch_warps=args.prefetch_warps, **bank_kw)
            for kv in args.cfg:                                        # diagnostic overrides, e.g. --cfg beta_a=1000
                k, v = kv.split('=')
                setattr(e.cfg, k, type(getattr(e.cfg, k))(float(v)))
            e.seed(1 + (rank * R + r) * B)
            e.reset()
            self.envs.append(e)
        self.auto_reset = not args.no_auto_reset
        self.side = [torch.cuda.Stream(device=dev) for _ in range(S - 1)]
        self.graphs = {}
        self.prefetch_launches = 0
        # a replay must not carry an env past its sampler cadence: tick() runs between replays
        self.max_graph_steps = R * max(args.prefetch_every, 8)
        self._enqueue(R)                                               # eager: smem opt-in, first touch
        torch.cuda.synchronize()

    @staticmethod
    def _bank(crl, args, dev):
        # the training configuration of the reference: a fixed set of K maps (make_train_env), here K maps
        # drawn by the device sampler itself and installed as a layout bank
        import numpy as np
        import torch
        helper = crl.ZoneVecEnv(args.env, args.bank, device=dev)
        helper.seed(1)
        helper.reset()
        torch.cuda.synchronize()
        N = helper.spec.num_zones
        o = helper.origin.cpu().numpy()
        bank = {'xy0': o[:, :2], 'rot0': o[:, 2], 'zone_xy': helper.zone_xy.cpu().numpy().transpose(1, 0, 2)}
        if helper.zone_tmax is not None:
            w = helper.zone_tmax.cpu().numpy().astype(np.int64) & 0xffffffff
            bank['zone_max_steps'] = np.stack([w & 0xffff, w >> 16], 1).reshape(-1, w.shape[1])[:N].T
        if helper.cooldown is not None:
            bits = helper.aux[:, 3].view(torch.int32).cpu().numpy().astype(np.int64) & 0xffffffff
            bank['colours'] = (bits[:, None] >> 16 >> (2 * np.arange(N))) & 3
        return dict(seed_mode='fixed_range', min_seed=1, max_seed=args.bank, layout_bank=bank)

    def _enqueue(self, n):
        """Steps 0..n-1 of the round-robin (step i -> replica i % R, on stream (i % R) % S)."""
        torch = self.torch
        main = torch.cuda.current_stream(self.dev)
        for s in self.side:
            s.wait_stream(main)
        for i in range(n):
            e = self.envs[i % self.R]
            k = (i % self.R) % self.S
            if k == 0:
                e.step_random(action_seed=1234, auto_reset=self.auto_reset, chained=self.chained, replayable=True)
            else:
                with torch.cuda.stream(self.side[k - 1]):
                    e.step_random(action_seed=1234, auto_reset=self.auto_reset, chained=self.chained, replayable=True)
        for s in self.side:
            main.wait_stream(s)

    def _graph(self, n):
        if n not in self.graphs:
            torch = self.torch
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._enqueue(n)
            self.graphs[n] = g
        return self.graphs[n]

    def prepare(self, n_steps):
        """Graphs for a run of n_steps: replays of `per` steps (a whole number of ring cycles) plus one tail."""
        per = min(n_steps, max(self.R, (self.max_graph_steps // self.R) * self.R))
        plan = [per] * (n_steps // per) + ([n_steps % per] if n_steps % per else [])
        for n in set(plan):
            self._graph(n)
        return plan

    def run(self, plan):
        for n in plan:
            self.graphs[n].replay()
            # the envs' own sampler cadence (ZoneVecEnv.tick), outside the graphs, on the side streams
            for r, e in enumerate(self.envs):
                took = n // self.R + (1 if r < n % self.R else 0)
                if took and e.tick(took):
                    self.prefetch_launches += 3 if self.task == 0 else 4
            self.last_env = self.envs[(n - 1) % self.R]                # every graph starts at replica 0

    def counters(self):
        c = self.torch.zeros(8, dtype=self.torch.float64, device=self.dev)
        for e in self.envs:
            c += e.counters_dev
        return c


def measure(ring, K, W, world, dist, spin_cycles=20_000_000):
    """Time exactly K steps after W warm-up steps.  The K steps' graphs are captured first and queued behind a
    spin of `spin_cycles` SM clocks (~10 ms), so the events around them hold device work only, not the host's
    launch of the first graph (slow: a graph's first launch also uploads it).  Returns dict(ms_per_step, ...)."""
    torch = ring.torch
    ring.run(ring.prepare(W))
    plan = ring.prepare(K)
    ring.prefetch_launches = 0
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(plan) + 1)]
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda._sleep(spin_cycles)
    ev[0].record()
    for i, n in enumerate(plan):
        ring.run([n])
        ev[i + 1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    seg = sorted(ev[i].elapsed_time(ev[i + 1]) / n for i, n in enumerate(plan))
    total_ms = ev[0].elapsed_time(ev[-1])
    return {'ms_per_step': total_ms / K, 'ms_per_step_best': seg[0], 'ms_per_step_worst': seg[-1],
            'ms_per_step_mean': total_ms / K, 'timed_steps': K, 'segments': len(plan),
            'timed_region_s': total_ms * 1e-3}


DUMP_BYTES = 64 << 20


def dump_outputs(env, out_dir, seed=0):
    """What the timed path's last step handed its caller (ZoneVecEnv.step_random: obs, zone_obs, reward, done and the
    info arrays) as out_dir/<name>.npy, float32.  When they exceed DUMP_BYTES in all, every array keeps the rows of
    the same fixed, seeded sample of envs, listed in env_index.npy."""
    import numpy as np
    got = dict(env._obs_dict(), reward=env.reward, done=env.done, **{'info_' + k: v for k, v in env._info().items()})
    got = {k: v.float().cpu().numpy() for k, v in got.items()}
    B = env.num_envs
    room = DUMP_BYTES - 4096 * (len(got) + 1)                          # less a generous .npy header per file
    if sum(a.nbytes for a in got.values()) > room:
        row = sum(a.nbytes for a in got.values()) // B
        keep = np.sort(np.random.RandomState(seed).choice(B, room // (row + 8), replace=False))
        got = {k: a[keep] for k, a in got.items()}
        got['env_index'] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in got.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def device_line(ring, m, world, peak):
    """value / roofline of one measured ring."""
    B, sb = ring.B, ring.step_bytes
    ms = m['ms_per_step']
    achieved = sb * B / (ms * 1e-3) / 1e9
    canon = CANON_BYTES.get(ring.env_id)
    return {'value': world * B / (ms * 1e-3), 'ms_per_step': ms, 'achieved_gbs': achieved, 'frac': achieved / peak,
            'best_frac': sb * B / (m['ms_per_step_best'] * 1e-3) / 1e9 / peak,
            'mean_frac': sb * B / (m['ms_per_step_mean'] * 1e-3) / 1e9 / peak,
            'bytes_per_env_step': sb, 'canonical_bytes_per_env_step': canon,
            'frac_canonical': canon * B / (ms * 1e-3) / 1e9 / peak if canon else None}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import combinatorial_rl_tasks_b200 as crl
    from combinatorial_rl_tasks_b200 import _lib

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        # stdout carries the one JSON line and nothing else: while NCCL initialises (it prints its
        # version banner on stdout), file descriptor 1 points at stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=torch.device(f'cuda:{local}'))
            torch.cuda.set_device(local)
            dist.barrier()                                         # creates the communicator now
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    dev = torch.device(f'cuda:{local}')
    torch.cuda.set_device(dev)
    # each rank next to its own GPU: its pinned host buffers (the e2e path moves tens of GB/s per GPU) then live on
    # that GPU's NUMA node instead of wherever torchrun happened to start the process
    from combinatorial_rl_tasks_b200.hostbind import bind_to_gpu_numa_node
    all_cores = os.sched_getaffinity(0)
    numa = {'bound': False, 'why': '--no-numa-bind'} if args.no_numa_bind else bind_to_gpu_numa_node(local)
    peak, peak_src = measured_peaks()
    B, K, W = args.envs, max(1, args.steps), max(3, args.warmup)
    chained = None if args.chained < 0 else bool(args.chained)

    def stats(ring):
        c = ring.counters()
        if world > 1:                                                  # episode statistics: the path's only collective (SURVEY 8e)
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
        c = c.cpu().numpy()
        return {'return_sum': c[0], 'episodes': c[1], 'successes': c[2], 'length_sum': c[3],
                'resets_prefetched': c[4], 'resets_inline': c[5], 'chain_wait_timeouts': c[7],
                'reduction': 'nccl all_reduce(sum)' if world > 1 else 'single rank'}

    def rank_max(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # ---- the headline workload ------------------------------------------------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.5)                                                    # nvidia-smi start-up
    ring = Ring(crl, _lib, args, args.env, B, dev, rank, chained=chained, streams=args.streams)
    sampler.mark()
    m = measure(ring, K, W, world, dist)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(ring.last_env, args.dump_outputs)
    for k in ('ms_per_step', 'ms_per_step_best', 'ms_per_step_mean'):
        m[k] = rank_max(m[k])
    head = device_line(ring, m, world, peak)
    head_R, head_S, head_chained = ring.R, ring.S, ring.chained
    head_stats = stats(ring)
    head_launches = m['timed_steps'] + ring.prefetch_launches

    # ---- e2e: host numpy in, host numpy out, through the public API --------------------------------------
    env = ring.envs[0]
    N, Z = env.spec.num_zones, env.spec.zone_dim
    pageable = [np.random.RandomState(7 + i + 100 * rank).uniform(-1, 1, (B, 2)).astype(np.float32) for i in range(8)]
    pinned = env.pinned_actions(8)                                     # the caller's own page-locked action buffers
    for a, b in zip(pinned, pageable):
        np.copyto(a, b)
    host_actions = pinned

    def timed_host_steps(delta, seconds, host_actions=pinned):
        for i in range(3):
            env.step_host(host_actions[i % 8], delta=delta)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        rows = calls = 0
        per_call = []
        env.host_rows_moved(reset=True)
        env.host_results_moved(reset=True)
        t_start = time.perf_counter()
        while True:
            t0 = time.perf_counter()
            for i in range(25):
                obs, rew, done, info = env.step_host(host_actions[(calls + i) % 8], delta=delta)
                rows += max(env.delta_rows, 0)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            per_call.append((t1 - t0) / 25)
            calls += 25
            if t1 - t_start >= seconds or calls >= args.e2e_max_calls:
                break
        rows += env.host_rows_moved(reset=True)                      # the zero-copy path counts its rows on the device
        timed_host_steps.results_per_step = env.host_results_moved(reset=True) / calls if delta else float(B)
        per_call.sort()
        med = rank_max(per_call[len(per_call) // 2])
        return world * B / med, rows / calls, calls, world * B / rank_max(per_call[0])

    def e2e_of(env_, seconds):
        """step_host end to end for one env batch (page-locked action arrays): env-steps/s, median group of 25 calls."""
        acts = env_.pinned_actions(4)
        rs_ = np.random.RandomState(11 + rank)
        for a_ in acts:
            np.copyto(a_, rs_.uniform(-1, 1, a_.shape).astype(np.float32))
        for i in range(3):
            env_.step_host(acts[i % 4])
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        per, n, t_start = [], 0, time.perf_counter()
        while True:
            t0 = time.perf_counter()
            for i in range(10):
                env_.step_host(acts[(n + i) % 4])
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            per.append((t1 - t0) / 10)
            n += 10
            if t1 - t_start >= seconds or n >= 2000:
                break
        per.sort()
        return world * env_.num_envs / rank_max(per[len(per) // 2])

    full_rate, _, _, _ = timed_host_steps(False, args.e2e_seconds / 3)
    pageable_rate, _, _, _ = timed_host_steps(True, args.e2e_seconds / 3, pageable)
    rate, rows_per_step, e2e_calls, best_rate = timed_host_steps(True, args.e2e_seconds)
    is_delta = rows_per_step < B
    results_per_step = timed_host_steps.results_per_step if is_delta else float(B)

    def copy_engine_floor(seconds=0.2):
        """The copy engine alone moving one call's obs + result (no kernel, no actions) with every rank active: what
        the box's host path allows for these bytes at this N (eight ranks of one VM share it, profiles/r02_notes.md)."""
        hb, s_ = env._host_buffers(), torch.cuda.current_stream(dev)
        def one():
            hb['obs'].copy_(env.obs, non_blocking=True)
            hb['result'].copy_(env.result, non_blocking=True)
            s_.synchronize()
        for _ in range(3):
            one()
        if world > 1:
            dist.barrier()
        per, t_start = [], time.perf_counter()
        while True:
            t0 = time.perf_counter()
            for _ in range(10):
                one()
            t1 = time.perf_counter()
            per.append((t1 - t0) / 10)
            if t1 - t_start >= seconds:
                break
        per.sort()
        return world * B / rank_max(per[len(per) // 2])

    floor_rate = copy_engine_floor()
    e2e = {'value': rate, 'unit': UNIT, 'h2d_bytes_per_step': 8 * B,
           'd2h_bytes_per_step': int(32 * B + 8 * results_per_step + rows_per_step * 4 * N * Z),
           'calls': e2e_calls, 'timing': 'median over groups of 25 calls (host clock, synchronize on both sides)',
           'best_group_value': best_rate,
           'pageable_actions_value': pageable_rate,
           'api': 'ZoneVecEnv.step_host: host numpy actions in (page-locked arrays from env.pinned_actions(), one of 8 per call; '
                  '`pageable_actions_value` = the same with ordinary numpy arrays, staged through a pinned buffer inside the '
                  'call), host numpy obs/zone_obs/reward/done out, transfers + stream sync inside every call'
                  + ('; crl_host_call_step (the prepared form of crl_step_host_delta, zero-copy): ONE kernel per call -- the step kernel reads the actions from, and writes '
                     'obs, and the zone_obs rows and result records that changed (mean %.1f rows and %.1f records of %d per step: a '
                     'record is all zeros except on an event) to, the pinned host buffers itself; host buffers byte-identical to '
                     'a full copy' % (rows_per_step, results_per_step, B) if is_delta
                     else '; crl_step_host: everything copied whole'),
           'host_placement': numa,
           'full_copy_value': full_rate,
           'copy_engine_floor_value': floor_rate,
           'copy_engine_floor_note': 'obs + result of one call moved WHOLE (%d bytes) by the copy engine alone + a stream sync, every '
                                     'rank at once, same max-over-ranks median; no kernel, no action upload: what the host path of '
                                     'this box gives a plain copy of the outputs at this N (the zero-copy call moves fewer bytes: '
                                     'result records cross only when they change, see d2h_bytes_per_step)' % ((32 + 8) * B),
           'full_copy_d2h_bytes_per_step': (32 + 4 * N * Z + 8) * B}
    del ring, env
    torch.cuda.empty_cache()

    # ---- BASELINE.json configs[2], [3] (N = 1) and configs[4] (N > 1): extra keys of the same line ----------
    extra = {}
    if not args.no_extra:
        todo = []
        if world == 1:
            todo += [('configs[2]', 'PointTTSP-v0', 262144), ('configs[3]', 'ColourMatch-v0', 262144)]
        if world > 1 or args.configs4:
            todo += [('configs[4]', e, 1048576) for e in ('PointTSP-v0', 'PointTTSP-v0', 'ColourMatch-v0')]
        for tag, env_id, b in todo:
            if (env_id, b) == (args.env, B):
                continue
            r2 = Ring(crl, _lib, args, env_id, b, dev, rank, chained=chained, streams=args.streams)
            m2 = measure(r2, K, W, world, dist)
            for k in ('ms_per_step', 'ms_per_step_best', 'ms_per_step_mean'):
                m2[k] = rank_max(m2[k])
            d = device_line(r2, m2, world, peak)
            if world == 1:
                d['e2e_value'] = e2e_of(r2.envs[0], 0.4)        # ZoneVecEnv.step_host, host numpy in / out
            d.update({'config': tag, 'env': env_id, 'envs_per_gpu_per_launch': b, 'ring_replicas': r2.R, 'streams': r2.S,
                      'chained_steps': r2.chained, 'timed_steps': m2['timed_steps'], 'timed_region_s': m2['timed_region_s'],
                      'unit': UNIT, 'episode_stats': stats(r2), 'sampler_launches': r2.prefetch_launches})
            extra[f'{env_id}:{b}'] = d
            head_launches += m2['timed_steps'] + r2.prefetch_launches
            del r2
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    traffic = traffic_note = None
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        traffic, traffic_note = tj.get(f'{args.env}:{B}'), tj.get('_note')
    sb = head['bytes_per_env_step']
    out = {
        'metric': METRIC, 'value': head['value'], 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': m['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{args.env}, {B} batched envs per launch, iid U(-1,1)^2 actions drawn in-kernel per (env, step), '
                               f'auto-reset {"off" if args.no_auto_reset else "on"}',
                   'envs_per_gpu_per_launch': B,
                   'l2': f'inputs larger than L2: ring of {head_ring_desc(sb, B)}',
                   'launch': 'CUDA graphs of whole ring cycles, replayed back to back; in-kernel actions advance on a device counter',
                   'ring_replicas': head_R, 'streams': head_S, 'chained_steps': head_chained,
                   'concurrency': 'the ring\'s replicas are independent env batches, each stepped on its own CUDA stream (launches of '
                                  'different replicas overlap; steps of one replica are ordered by its stream)', 'prefetch_every': args.prefetch_every, 'layout_bank': args.bank or None,
                   'timing': f'K={K} steps after W={W} warm-up steps, back to back ({m["timed_region_s"] * 1e3:.2f} ms of device '
                             f'time, CUDA events queued behind a device spin, barrier + synchronize on both sides), '
                             f'{m["segments"]} graph replays; ms_per_step / value = the whole window, max over ranks'},
        'timing': {k: m[k] for k in ('ms_per_step', 'ms_per_step_best', 'ms_per_step_worst', 'ms_per_step_mean', 'timed_steps',
                                     'segments', 'timed_region_s')},
        'roofline': {'bound': 'hbm', 'achieved': head['achieved_gbs'], 'peak': peak, 'unit': 'GB/s', 'frac': head['frac'],
                     'traffic': traffic, 'traffic_note': traffic_note if traffic is not None else None,
                     'algorithmic_bytes_per_launch': sb * B, 'peak_source': peak_src, 'kernel': 'step_kernel',
                     'bytes_per_env_step': sb,
                     'bytes_note': 'crl_step_bytes minus the 8-byte action read (actions are drawn in-kernel)',
                     'canonical_bytes_per_env_step': head['canonical_bytes_per_env_step'],
                     'frac_canonical': head['frac_canonical'], 'frac_best_segment': head['best_frac'],
                     'frac_mean': head['mean_frac'], 'frac_of_nominal_8TBs': head['achieved_gbs'] / 8000.0},
        'clocks': clocks, 'e2e': e2e, 'gpu_launches': head_launches,
        'gpu_launches_detail': {'step_kernel (headline timed region)': m['timed_steps'],
                                'all timed regions incl. extra configs and sampler / publish kernels': head_launches},
        'episode_stats': head_stats,
        'configs': extra,
    }
    if world == 1 and not args.no_extra:
        try:
            out['encoder'] = encoder_leg(crl, torch, dev)
            out['gpu_launches_detail']['encoder leg (zone + head kernels, not in gpu_launches)'] = 'see encoder.timing'
        except Exception as ex:
            out['encoder'] = {'error': repr(ex)}
    if world == 1 and not args.no_cpu_baseline:
        try:
            os.sched_setaffinity(0, all_cores)                        # the CPU baseline gets ALL host cores back
            out['cpu_baseline'] = cpu_baselines(args.env, args.cpu_seconds)
        except Exception as ex:  # the baseline is a reported number, never the product path
            out['cpu_baseline'] = {'error': repr(ex)}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def encoder_leg(crl, torch, dev, envs=65536, hidden=185, seconds=0.3):
    """SURVEY 8f rank 2: the rollout-time ZoneEnvModel.forward (main/src/env_model.py:48-79, h = 185:
    scripts/train_ppo.py:66) on the observations of `envs` PointTSP envs through ZoneEncoder (two tcgen05 kernels of this
    library: zone_net_ + mean-pool fused, then combine_net_([obs, L3(pooled)]) as one folded GEMM).  Device time, CUDA
    events, input replicas larger than 2 x L2 cycled, random-init weights.  Tensor roofline: useful flops of the fused zone
    kernel's two layers against the measured bf16 peak."""
    spec = crl.ENV_SPECS['PointTSP-v0']
    N, Z, h, B = spec.num_zones, spec.zone_dim, hidden, envs
    g = torch.Generator(device=dev).manual_seed(7)
    rn = lambda *sh, scale=1.0: torch.randn(*sh, device=dev, generator=g) * scale
    sd = {'zone_net_.0.weight': rn(h, 8 + Z, scale=0.3), 'zone_net_.0.bias': rn(h, scale=0.1),
          'zone_net_.2.weight': rn(h, h, scale=0.1), 'zone_net_.2.bias': rn(h, scale=0.1),
          'zone_net_.4.weight': rn(h, h, scale=0.1), 'zone_net_.4.bias': rn(h, scale=0.1),
          'combine_net_.weight': rn(h, 8 + h, scale=0.1), 'combine_net_.bias': rn(h, scale=0.1)}
    enc = crl.ZoneEncoder(sd, num_zones=N, device=dev)
    env = crl.ZoneVecEnv('PointTSP-v0', B, device=dev)
    env.seed(3)
    obs = env.reset()
    for _ in range(4):
        obs, *_ = env.step_random(action_seed=9)
    in_bytes = B * (8 + N * Z) * 4
    reps = max(2, -(-2 * L2_BYTES // in_bytes))
    o_r = [obs['obs'].clone() for _ in range(reps)]
    z_r = [obs['zone_obs'].clone() for _ in range(reps)]
    pooled = torch.empty(B, h, device=dev)

    def timed(fn):
        for i in range(5):
            fn(i % reps)
        torch.cuda.synchronize()
        per, n = [], 0
        t_end = time.perf_counter() + seconds
        while time.perf_counter() < t_end or len(per) < 3:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(20):
                fn((n + i) % reps)
            e1.record()
            torch.cuda.synchronize()
            per.append(e0.elapsed_time(e1) / 20 * 1e-3)
            n += 20
        per.sort()
        return per[len(per) // 2]

    t_zone = timed(lambda i: enc.pooled(o_r[i], z_r[i], out=pooled))
    t_fwd = timed(lambda i: enc(o_r[i], z_r[i]))
    t_state = timed(lambda i: enc.forward_from_state(env))
    ok = enc.healthy()
    useful = B * N * 2 * ((8 + Z) * h + h * h)
    pk = 2250.0
    pp = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(pp):
        with open(pp) as f:
            pk = json.load(f).get('bf16_tflops', pk)
    del env
    return {'op': 'ZoneEnvModel.forward (env_model.py:48-79), rollout time, bf16 operands / fp32 accumulation',
            'workload': f'PointTSP-v0 observations of {B} envs, N={N}, Z={Z}, h={h}, random-init weights',
            'healthy': ok, 'forward_us': t_fwd * 1e6, 'zone_kernel_us': t_zone * 1e6,
            'forward_from_state_us': t_state * 1e6, 'envs_per_s': B / t_fwd,
            'launches_per_forward': 2,
            'roofline': {'bound': 'tensor', 'kernel': 'zone_encode_kernel', 'achieved': useful / t_zone / 1e12, 'peak': pk,
                         'unit': 'TFLOP/s', 'frac': useful / t_zone / 1e12 / pk},
            'l2': f'{reps} input replicas ({reps * in_bytes >> 20} MB) cycled; forward_from_state reads one env\'s state planes',
            'timing': 'median group of 20 calls, CUDA events'}


def head_ring_desc(step_bytes, B):
    R = max(2, -(-2 * L2_BYTES // (B * step_bytes)))
    return (f'{R} independent {B}-env replicas ({R * B * step_bytes / 1e6:.0f} MB touched per cycle) > 2x the 126 MB L2, '
            f'so every launch reads HBM')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100000, help='timed steps of the headline workload and of each extra config')
    ap.add_argument('--warmup', type=int, default=200)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--env', default='PointTSP-v0')
    ap.add_argument('--envs', type=int, default=65536)
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step (rank 0\'s envs) to DIR/<name>.npy, <= 64 MB in all')
    ap.add_argument('--e2e-seconds', type=float, default=1.0)
    ap.add_argument('--e2e-max-calls', type=int, default=20000)
    ap.add_argument('--cpu-seconds', type=float, default=9.0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-numa-bind', action='store_true', help='leave the process where the launcher put it')
    ap.add_argument('--no-extra', action='store_true', help='skip the configs[2] / [3] / [4] legs')
    ap.add_argument('--configs4', action='store_true', help='run the 1,048,576-env legs of configs[4] also on one GPU')
    ap.add_argument('--no-auto-reset', action='store_true', help='diagnostic: finished envs keep stepping')
    ap.add_argument('--chained', type=int, default=-1,
                    help='1: back-to-back steps order themselves warp by warp (CRL_STEP_CHAINED); 0: whole-grid '
                         'wait; -1: chained when a launch is at most a wave or two (<= 131072 envs)')
    ap.add_argument('--streams', type=int, default=0,
                    help='the ring\'s replicas are independent batches: step them on this many streams (replica r on stream '
                         'r %% S); 0 = one stream per replica, at most 8')
    ap.add_argument('--min-replicas', type=int, default=0, help='at least this many ring replicas')
    ap.add_argument('--prefetch-every', type=int, default=32,
                    help='top up the next-layout slots every N steps of an env (0: resets sample inline)')
    ap.add_argument('--bank', type=int, default=0,
                    help='fixed task set of K maps (make_train_env): resets copy from a layout bank, no sampler')
    ap.add_argument('--cfg', action='append', default=[], help='diagnostic: override a CrlConfig field, key=value')
    ap.add_argument('--prefetch-warps', type=int, default=0, help='background sampler warps per SM (0: default)')
    args = ap.parse_args()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
