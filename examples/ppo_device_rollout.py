#!/usr/bin/env python
"""Minimal on-device PPO loop over the batched docking env -- the counterpart of the reference's
``train()`` (gym_dockauv/train.py:21-82: ``MODEL('MlpPolicy', env).learn(...)``) without a host round trip per step:

    python examples/ppo_device_rollout.py [--envs 16384] [--steps 64] [--iters 20] [--record-envs K --record-dir DIR]
                                          [--fused]

* rollouts: ``DeviceRolloutBuffer.collect`` -- the step kernels write observation / reward / done of step t straight
  into row t of the buffer; with ``--fused``, ``DeviceRolloutBuffer.collect_fused``: the same networks evaluated by the
  library's policy kernel between the steps of one captured rollout (the graph is captured once and replayed every
  iteration: the update rewrites the parameters in place);
* advantages: ``dockauv_gae`` (one kernel over the stacked rows);
* the policy / value networks and the clipped-surrogate update are plain PyTorch (they are not part of the step path);
* ``--record-envs K``: the episodes of K envs spread over the batch are recorded on the device while the run trains
  (``TrainingRecorder``) and written to ``--record-dir`` as reference-format ``EpisodeDataStorage`` pickles, drained once
  per iteration.

Prints, per iteration, the mean return of the episodes that ended inside the rollout and the env-steps/s of collection.
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

from gym_dockauv_b200 import envs  # noqa: E402
from gym_dockauv_b200.config import TRAIN_CONFIG  # noqa: E402
from gym_dockauv_b200.episode_export import TrainingRecorder  # noqa: E402
from gym_dockauv_b200.policy import FusedActorCritic  # noqa: E402
from gym_dockauv_b200.rollout import DeviceRolloutBuffer  # noqa: E402


class ActorCritic(nn.Module):
    def __init__(self, n_obs, n_act, hidden=64):
        super().__init__()
        self.pi = nn.Sequential(nn.Linear(n_obs, hidden), nn.Tanh(), nn.Linear(hidden, hidden), nn.Tanh(), nn.Linear(hidden, n_act))
        self.v = nn.Sequential(nn.Linear(n_obs, hidden), nn.Tanh(), nn.Linear(hidden, hidden), nn.Tanh(), nn.Linear(hidden, 1))
        self.log_std = nn.Parameter(torch.full((n_act,), -0.5))

    def dist(self, obs):
        return torch.distributions.Normal(self.pi(obs), self.log_std.exp())

    @torch.no_grad()
    def act(self, obs):
        d = self.dist(obs)
        a = d.sample()
        return a, self.v(obs).squeeze(-1), d.log_prob(a).sum(-1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--scenario", default="ObstaclesDocking3d")
    ap.add_argument("--record-envs", type=int, default=0, help="record the episodes of this many envs (at most 1024)")
    ap.add_argument("--record-dir", default="episode_storage")
    ap.add_argument("--fused", action="store_true", help="collect with the policy kernel (DeviceRolloutBuffer.collect_fused)")
    args = ap.parse_args()
    env = envs.SCENARIOS[args.scenario](TRAIN_CONFIG, num_envs=args.envs, seed=0)
    buf = DeviceRolloutBuffer(env, args.steps, gamma=0.99, gae_lambda=0.95)
    buf.reset_env()
    rec = None
    if args.record_envs:
        ids = torch.linspace(0, args.envs - 1, args.record_envs).long().unique().tolist()
        rec = TrainingRecorder(env, ids, args.record_dir, title="ppo", capacity=max(args.steps, 64))
    net = ActorCritic(env.n_observations, env.n_actions).to(env.device)
    opt = torch.optim.Adam(net.parameters(), lr=3e-4)
    fused = FusedActorCritic([net.pi[0], net.pi[2], net.pi[4]], [net.v[0], net.v[2], net.v[4]], net.log_std) \
        if args.fused else None
    for it in range(args.iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if fused is not None:
            buf.compute_returns_and_advantage(buf.collect_fused(fused))
        else:
            last_obs = buf.collect(net.act)
            with torch.no_grad():
                buf.compute_returns_and_advantage(net.v(last_obs).squeeze(-1))
        torch.cuda.synchronize()
        t_collect = time.perf_counter() - t0
        info = buf.episode_infos()
        if rec is not None:
            n_saved = len(rec.drain())
            if n_saved:
                print(f"iter {it:3d}  wrote {n_saved} episode pickles to {args.record_dir}", flush=True)
        for _ in range(4):
            for mb in buf.get(batch_size=1 << 16):
                adv = (mb.advantages - mb.advantages.mean()) / (mb.advantages.std() + 1e-8)
                d = net.dist(mb.observations)
                ratio = (d.log_prob(mb.actions).sum(-1) - mb.old_log_prob).exp()
                loss_pi = -torch.min(ratio * adv, ratio.clamp(0.8, 1.2) * adv).mean()
                loss_v = (net.v(mb.observations).squeeze(-1) - mb.returns).pow(2).mean()
                loss = loss_pi + 0.5 * loss_v - 0.0 * d.entropy().sum(-1).mean()
                opt.zero_grad(set_to_none=True)
                loss.backward()
                nn.utils.clip_grad_norm_(net.parameters(), 0.5)
                opt.step()
        n_ep = info["l"].numel()
        mean_r = float(info["r"].mean()) if n_ep else float("nan")
        mean_l = float(info["l"].float().mean()) if n_ep else float("nan")
        captures = f"  graph captures {env.rollout_policy_captures()} " if fused is not None else ""
        print(f"iter {it:3d}  episodes {n_ep:7d}  mean return {mean_r:10.2f}  mean length {mean_l:7.1f}  "
              f"collect {args.envs * args.steps / t_collect:.3g} env-steps/s (policy included){captures}", flush=True)
    env.close()


if __name__ == "__main__":
    main()
