#!/usr/bin/env python
"""Minimal on-device SAC loop over the batched docking env -- the counterpart of the reference's ``train()`` with
``MODEL = SAC`` (gym_dockauv/train.py:64: ``MODEL('MlpPolicy', env).learn(...)``) without a host round trip per step:

    python examples/sac_device_replay.py [--envs 16384] [--slots 16] [--steps 32] [--batch 8192] [--gradient-steps 32]
                                         [--iters 20] [--scenario ObstaclesDocking3d] [--fused]

* collection: ``DeviceReplayBuffer.collect`` -- the step kernels write observation, reward, done flag and terminal
  observation of every step straight into the replay ring; with ``--fused``, ``DeviceReplayBuffer.collect_fused`` --
  the same actor evaluated by the library's tensor-core kernel between the steps of one captured launch chain (bf16
  operands, f32 accumulation);
* minibatches: ``DeviceReplayBuffer.sample`` -- one kernel (``dockauv_replay_sample``) draws the batch and gathers its
  rows, with SB3's ``ReplayBufferSamples`` fields;
* the networks and the update are plain PyTorch with SB3 SAC's defaults: tanh-squashed Gaussian actor, twin Q critics,
  Polyak-averaged target critics (tau = 0.005), entropy coefficient tuned towards a target entropy of -n_u.

Prints, per iteration, the episodes that ended during its collection with their mean return and length (from the env's
statistics vector), the env-steps/s of collection (policy included) and the samples/s of the update (sampling and
gradient steps).
"""
import argparse
import copy
import math
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from gym_dockauv_b200 import envs  # noqa: E402
from gym_dockauv_b200.config import TRAIN_CONFIG  # noqa: E402
from gym_dockauv_b200.policy import FusedSquashedActor  # noqa: E402
from gym_dockauv_b200.replay import DeviceReplayBuffer  # noqa: E402


def mlp(n_in, n_out, hidden=256):
    return nn.Sequential(nn.Linear(n_in, hidden), nn.ReLU(), nn.Linear(hidden, hidden), nn.ReLU(), nn.Linear(hidden, n_out))


class Actor(nn.Module):
    def __init__(self, n_obs, n_act):
        super().__init__()
        self.net = mlp(n_obs, 2 * n_act)

    def forward(self, obs):
        """tanh-squashed Gaussian: (action in [-1, 1], log-probability with the tanh correction)."""
        mu, log_std = self.net(obs).chunk(2, dim=-1)
        std = log_std.clamp(-20, 2).exp()
        u = mu + std * torch.randn_like(mu)
        a = torch.tanh(u)
        logp = (-0.5 * ((u - mu) / std).pow(2) - std.log() - 0.5 * math.log(2 * math.pi)).sum(-1)
        logp = logp - (2 * (math.log(2) - u - F.softplus(-2 * u))).sum(-1)
        return a, logp

    @torch.no_grad()
    def act(self, obs):
        return self(obs)[0]


class Critic(nn.Module):
    def __init__(self, n_obs, n_act):
        super().__init__()
        self.q1, self.q2 = mlp(n_obs + n_act, 1), mlp(n_obs + n_act, 1)

    def forward(self, obs, act):
        x = torch.cat([obs, act], -1)
        return self.q1(x), self.q2(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--slots", type=int, default=16, help="replay slots of the whole batch (2..64)")
    ap.add_argument("--steps", type=int, default=32, help="env steps per iteration")
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--gradient-steps", type=int, default=32)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--scenario", default="ObstaclesDocking3d")
    ap.add_argument("--fused", action="store_true", help="collect with the actor evaluated on the device (collect_fused)")
    args = ap.parse_args()
    env = envs.SCENARIOS[args.scenario](TRAIN_CONFIG, num_envs=args.envs, seed=0)
    buf = DeviceReplayBuffer(env, args.slots, seed=0)
    buf.reset_env()
    dev, n_obs, n_u = env.device, env.n_observations, env.n_actions
    actor, critic = Actor(n_obs, n_u).to(dev), Critic(n_obs, n_u).to(dev)
    critic_target = copy.deepcopy(critic).requires_grad_(False)
    log_alpha = torch.zeros(1, device=dev, requires_grad=True)
    opt_actor = torch.optim.Adam(actor.parameters(), lr=3e-4)
    opt_critic = torch.optim.Adam(critic.parameters(), lr=3e-4)
    opt_alpha = torch.optim.Adam([log_alpha], lr=3e-4)
    gamma, tau, target_entropy = 0.99, 0.005, -float(n_u)
    if args.fused:      # the head's row slices are views of the live parameters: Adam's in-place updates are seen
        net = actor.net
        w, b = net[4].weight, net[4].bias
        fused = FusedSquashedActor([net[0], net[2]], w[:n_u], b[:n_u], w[n_u:], b[n_u:])
    for it in range(args.iters):
        env.clear_stats()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if args.fused:
            buf.collect_fused(fused, args.steps)
        else:
            buf.collect(actor.act, args.steps)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        for _ in range(args.gradient_steps):
            b = buf.sample(args.batch)
            alpha = log_alpha.exp().detach()
            with torch.no_grad():
                a_next, logp_next = actor(b.next_observations)
                q_next = torch.min(*critic_target(b.next_observations, a_next)) - alpha * logp_next.unsqueeze(-1)
                target = b.rewards + (1 - b.dones) * gamma * q_next
            q1, q2 = critic(b.observations, b.actions)
            loss_q = 0.5 * (F.mse_loss(q1, target) + F.mse_loss(q2, target))
            opt_critic.zero_grad(set_to_none=True)
            loss_q.backward()
            opt_critic.step()
            a_pi, logp = actor(b.observations)
            loss_pi = (alpha * logp.unsqueeze(-1) - torch.min(*critic(b.observations, a_pi))).mean()
            opt_actor.zero_grad(set_to_none=True)
            loss_pi.backward()
            opt_actor.step()
            loss_alpha = -(log_alpha * (logp.detach() + target_entropy)).mean()
            opt_alpha.zero_grad(set_to_none=True)
            loss_alpha.backward()
            opt_alpha.step()
            with torch.no_grad():
                for p, pt in zip(critic.parameters(), critic_target.parameters()):
                    pt.lerp_(p, tau)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        st = env.get_stats()
        n_ep = int(st["episodes"])
        means = (f"mean return {st['sum_return'] / n_ep:10.2f}  mean length {st['sum_length'] / n_ep:7.1f}" if n_ep
                 else "mean return        n/a  mean length     n/a")
        print(f"iter {it:3d}  episodes {n_ep:7d}  {means}  collect {args.envs * args.steps / (t1 - t0):.3g} env-steps/s  "
              f"update {args.batch * args.gradient_steps / (t2 - t1):.3g} samples/s  q-loss {loss_q.item():.4g}  "
              f"alpha {float(alpha):.4g}", flush=True)
    env.close()


if __name__ == "__main__":
    main()
