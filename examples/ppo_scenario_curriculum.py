#!/usr/bin/env python
"""On-device PPO with a scenario-bank curriculum: the PPO loop of ``ppo_device_rollout.py``, with every reset drawn
from a bank of initial conditions whose draw weights follow the policy's failures.

    python examples/ppo_scenario_curriculum.py [--envs 16384] [--steps 64] [--iters 20] [--rows 4096]

* the bank: ``ScenarioBank.from_builtin`` -- ``rows`` draws of the scenario's own start distribution;
* per iteration, on the device: episodes and goal-reached counts per row (``scatter_add`` over ``env.ended_bank_row``
  at ``done``, condition bit 0 = goal reached).  ``ended_bank_row`` holds a row only until the env's next episode ends,
  so the ends of step t - 1 are counted in the policy callback before step t, and those of the last step once
  ``collect`` returns;
* the weights become ``1 - success rate + eps`` (rows never seen keep weight 1) through ``env.set_scenario_weights``,
  which rewrites them in place: the cached step graphs stay valid, the capture count stays flat after iteration 0.

Prints, per iteration, the goal-reached rate of the episodes that ended, the share of rows seen so far and the number of
step-graph captures.
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
from gym_dockauv_b200.rollout import DeviceRolloutBuffer  # noqa: E402
from gym_dockauv_b200.scenario_bank import ScenarioBank  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from ppo_device_rollout import ActorCritic  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rows", type=int, default=4096)
    ap.add_argument("--eps", type=float, default=0.05)
    ap.add_argument("--scenario", default="ObstaclesDocking3d")
    args = ap.parse_args()
    env = envs.SCENARIOS[args.scenario](TRAIN_CONFIG, num_envs=args.envs, seed=0)
    K = args.rows
    bank = ScenarioBank.from_builtin(env, K, seed=1)
    env.set_scenario_bank(bank, weights=torch.ones(K, device=env.device))
    buf = DeviceRolloutBuffer(env, args.steps, gamma=0.99, gae_lambda=0.95)
    buf.reset_env()
    episodes = torch.zeros(K, dtype=torch.float64, device=env.device)
    reached = torch.zeros(K, dtype=torch.float64, device=env.device)

    def count_ends(t):
        """the episodes that ended at step t of the buffer, by the bank row they started from"""
        d = buf.dones[t].bool()
        rows = env.ended_bank_row.long().clamp(min=0)
        episodes.scatter_add_(0, rows, d.double())
        reached.scatter_add_(0, rows, (d & (buf.cond_bits[t] & 1).bool()).double())

    net = ActorCritic(env.n_observations, env.n_actions).to(env.device)
    opt = torch.optim.Adam(net.parameters(), lr=3e-4)
    for it in range(args.iters):
        step = [0]

        def policy(obs):
            t = step[0]
            if t > 0:
                count_ends(t - 1)
            step[0] += 1
            a, v, lp = net.act(obs)
            # the step reads its actions from row t of the buffer: the same pointers at every iteration, so each of
            # the T step graphs is captured once
            return buf.actions[t].copy_(a), v, lp

        ep0, re0 = float(episodes.sum()), float(reached.sum())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        last_obs = buf.collect(policy)
        count_ends(args.steps - 1)
        with torch.no_grad():
            buf.compute_returns_and_advantage(net.v(last_obs).squeeze(-1))
        torch.cuda.synchronize()
        t_collect = time.perf_counter() - t0
        # curriculum: weight a row by how often the policy fails from it (rows not seen yet keep weight 1)
        rate = torch.where(episodes > 0, reached / episodes.clamp(min=1), torch.zeros_like(episodes))
        env.set_scenario_weights(1.0 - rate + args.eps)
        for _ in range(4):
            for mb in buf.get(batch_size=1 << 16):
                adv = (mb.advantages - mb.advantages.mean()) / (mb.advantages.std() + 1e-8)
                d = net.dist(mb.observations)
                ratio = (d.log_prob(mb.actions).sum(-1) - mb.old_log_prob).exp()
                loss_pi = -torch.min(ratio * adv, ratio.clamp(0.8, 1.2) * adv).mean()
                loss_v = (net.v(mb.observations).squeeze(-1) - mb.returns).pow(2).mean()
                loss = loss_pi + 0.5 * loss_v
                opt.zero_grad(set_to_none=True)
                loss.backward()
                nn.utils.clip_grad_norm_(net.parameters(), 0.5)
                opt.step()
        n_ep, n_re = float(episodes.sum()) - ep0, float(reached.sum()) - re0
        goal_rate = n_re / n_ep if n_ep else float("nan")
        seen = float((episodes > 0).double().mean())
        print(f"iter {it:3d}  episodes {int(n_ep):7d}  goal reached {goal_rate:6.3f}  rows seen {seen:6.3f}  "
              f"step-graph captures {env.step_graph_captures()}  collect {args.envs * args.steps / t_collect:.3g} "
              f"env-steps/s (policy included)", flush=True)
    env.close()


if __name__ == "__main__":
    main()
