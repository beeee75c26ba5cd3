"""Planning on the simulator: random-shooting MPC on PointTSP with env copies (ZoneVecEnv.copy_envs_from).

    python examples/lookahead.py --env PointTSP-v0 --envs 1024 --branches 64 --horizon 32 --steps 500

Every step, each of the E real envs branches into K planner envs (one crl_copy_envs of E K envs: env e of the real
batch onto planner envs e K .. e K + K - 1).  Each branch takes its own uniform first action, then H - 1 steps of
in-kernel random actions -- keyed by the planner env's global index, so the K branches of an env diverge -- and
sums its rewards up to the end of its episode.  The real env takes the first action of its best branch.  A second
batch with the same seeds takes uniform random actions; the script prints the mean return of both over the run.
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import combinatorial_rl_tasks_b200 as crl  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--env', default='PointTSP-v0')
    ap.add_argument('--envs', type=int, default=1024, help='real envs E')
    ap.add_argument('--branches', type=int, default=64, help='planner branches per real env K')
    ap.add_argument('--horizon', type=int, default=32, help='steps per branch H')
    ap.add_argument('--steps', type=int, default=500, help='real steps')
    ap.add_argument('--seed', type=int, default=1)
    a = ap.parse_args(argv)
    E, K, H, T, dev = a.envs, a.branches, a.horizon, a.steps, torch.device('cuda:0')
    real, rand = crl.ZoneVecEnv(a.env, E, device=dev), crl.ZoneVecEnv(a.env, E, device=dev)
    for env in (real, rand):                      # the same seeds: the same layouts
        env.seed(a.seed)
        env.reset()
    # the planner never auto-resets (a branch's return stops at its episode's end): no background sampler
    plan = crl.ZoneVecEnv(a.env, E * K, device=dev, prefetch_every=0)
    branch_src = torch.arange(E, dtype=torch.int32, device=dev).repeat_interleave(K)
    gen = torch.Generator(device=dev).manual_seed(a.seed)
    rows = torch.arange(E, device=dev)
    mpc_ret, rand_ret = torch.zeros(E, device=dev), torch.zeros(E, device=dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t in range(T):
        plan.copy_envs_from(real, branch_src)
        first = torch.rand(E * K, 2, generator=gen, device=dev) * 2 - 1
        plan.step_no_reset(first)
        ret, alive = plan.reward.clone(), ~plan.done
        for _ in range(H - 1):
            plan.step_random(action_seed=t + 1, auto_reset=False)
            ret += plan.reward * alive
            alive &= ~plan.done
        best = ret.view(E, K).argmax(1)
        real.step(first.view(E, K, 2)[rows, best])
        mpc_ret += real.reward
        rand.step(torch.rand(E, 2, generator=gen, device=dev) * 2 - 1)
        rand_ret += rand.reward
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    res = {'env': a.env, 'envs': E, 'branches': K, 'horizon': H, 'steps': T, 'seconds': round(sec, 3),
           'mpc_return': float(mpc_ret.mean()), 'random_return': float(rand_ret.mean()),
           'planner_env_steps_per_s': E * K * H * T / sec}
    print(f"{a.env}: mean return over {T} steps of {E} envs -- random-shooting MPC (K={K}, H={H}) "
          f"{res['mpc_return']:.3f}, random policy {res['random_return']:.3f} ({sec:.1f} s, "
          f"{res['planner_env_steps_per_s']:.3g} planner env-steps/s)")
    return res


if __name__ == '__main__':
    main()
