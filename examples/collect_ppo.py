"""How the reference's training loop looks on top of this package: the collection half of
BaseAlgo.collect_experiences (main/src/torch_ac/algos/base.py:110-249) with a small policy of the
reference's shape (per-zone MLP, mean over zones: main/src/env_model.py:48-79), everything on the GPU.

    python examples/collect_ppo.py --env PointTSP-v0 --envs 65536 --frames 64 --updates 3 [--fused-encoder | --fused-train]

--fused-encoder: the collection forward runs the embedding on crl.ZoneEncoder (the tcgen05 kernel, bf16 operands);
the update keeps the torch module, whose weights are re-packed after every optimiser step.
--fused-train: the policy embeds through crl.FusedZoneEnvModel in collection AND update: the (B N)-row part of the
embedding runs forward and backward on the tensor cores, the rest is torch autograd.

The env writes each frame straight into the rollout (no per-frame copies), crl_gae computes the
advantages; what is left for torch is the policy itself.
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

import combinatorial_rl_tasks_b200 as crl  # noqa: E402
from combinatorial_rl_tasks_b200.rollout import Rollout  # noqa: E402


class ZonePolicy(nn.Module):
    """ZoneEnvModel (env_model.py:48-79) + Gaussian actor and critic heads."""

    def __init__(self, zone_dim, h=64):
        super().__init__()
        self.zone_net = nn.Sequential(nn.Linear(8 + zone_dim, h), nn.ReLU(), nn.Linear(h, h), nn.ReLU(), nn.Linear(h, h))
        self.combine = nn.Linear(8 + h, h)
        self.actor, self.critic = nn.Linear(h, 2), nn.Linear(h, 1)
        self.log_std = nn.Parameter(torch.zeros(2))

    def forward(self, obs):
        o, z = obs['obs'], obs['zone_obs']
        x = torch.cat([o[:, None, :].expand(-1, z.shape[1], -1), z], dim=-1)
        emb = torch.relu(self.combine(torch.cat([o, self.zone_net(x).mean(dim=1)], dim=-1)))
        return self.heads(emb)

    def heads(self, emb):
        return torch.distributions.Normal(torch.tanh(self.actor(emb)), self.log_std.exp()), self.critic(emb).squeeze(-1)

    def encoder_state_dict(self):
        """The embedding's weights under the reference's parameter names (ZoneEnvModel.state_dict())."""
        sd = {f'zone_net_.{k}': v for k, v in self.zone_net.state_dict().items()}
        sd.update({f'combine_net_.{k}': v for k, v in self.combine.state_dict().items()})
        return sd


class FusedZonePolicy(nn.Module):
    """ZonePolicy with the embedding as crl.FusedZoneEnvModel (the reference's parameter names: env_model.zone_net_.*,
    env_model.combine_net_.*)."""

    def __init__(self, zone_dim, num_zones, h=64):
        super().__init__()
        self.env_model = crl.FusedZoneEnvModel(8, zone_dim, num_zones, h)
        self.actor, self.critic = nn.Linear(h, 2), nn.Linear(h, 1)
        self.log_std = nn.Parameter(torch.zeros(2))

    def forward(self, obs):
        return self.heads(torch.relu(self.env_model(obs)))

    heads = ZonePolicy.heads


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--env', default='PointTSP-v0')
    ap.add_argument('--envs', type=int, default=65536)
    ap.add_argument('--frames', type=int, default=64)
    ap.add_argument('--updates', type=int, default=3)
    ap.add_argument('--fused-encoder', action='store_true')
    ap.add_argument('--fused-train', action='store_true')
    args = ap.parse_args()
    if args.fused_encoder and args.fused_train:
        ap.error('--fused-encoder and --fused-train are alternatives')
    env = crl.ZoneVecEnv(args.env, args.envs, seed_mode='fixed_range', min_seed=1, max_seed=100)   # make_train_env
    if args.fused_train:
        policy = FusedZonePolicy(env.spec.zone_dim, env.spec.num_zones).cuda()
    else:
        policy = ZonePolicy(env.spec.zone_dim).cuda()
    opt = torch.optim.Adam(policy.parameters(), lr=3e-4)
    ro = Rollout(env, args.frames, discount=0.998, gae_lambda=0.95)
    enc = crl.ZoneEncoder(policy.encoder_state_dict(), num_zones=env.spec.num_zones) if args.fused_encoder else None
    act = (lambda o: policy.heads(torch.relu(enc(o)))) if enc else policy
    for it in range(args.updates):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        obs = ro.begin()
        with torch.no_grad():
            for t in range(ro.T):
                dist, value = act(obs)
                action = dist.sample().clamp(-1, 1)
                obs, reward, done, info = ro.step(t, action, value, dist.log_prob(action))
            exps = ro.finish(act(obs)[1])
        torch.cuda.synchronize(); t1 = time.perf_counter()
        # one PPO-style epoch over a random tenth of the frames (the reference's update_parameters, abridged)
        T, B = ro.T, env.num_envs
        idx = torch.randint(0, T * B, (T * B // 10,), device='cuda')
        flat = lambda x: x.reshape((T * B,) + tuple(x.shape[2:]))[idx]
        batch_obs = {k: flat(v) for k, v in exps['obs'].items()}
        dist, value = policy(batch_obs)
        adv = flat(exps['advantage'])
        ratio = (dist.log_prob(flat(exps['action'])) - flat(exps['log_prob'])).sum(-1).exp()
        loss = -torch.min(ratio * adv, ratio.clamp(0.8, 1.2) * adv).mean() + 0.5 * (value - flat(exps['returnn'])).pow(2).mean()
        opt.zero_grad(); loss.backward(); opt.step()
        if enc:
            enc.load_state_dict(policy.encoder_state_dict())
        torch.cuda.synchronize(); t2 = time.perf_counter()
        c = env.counters()
        print(f'update {it}: collected {T * B} frames in {1e3 * (t1 - t0):.1f} ms ({T * B / (t1 - t0):.3e} env-steps/s incl. policy), '
              f'update {1e3 * (t2 - t1):.1f} ms, loss {loss.item():.4f}, episodes so far {int(c["episodes"])}, '
              f'mean return {c["return_sum"] / max(c["episodes"], 1):.3f}')


if __name__ == '__main__':
    main()
