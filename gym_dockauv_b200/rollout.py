"""Device-resident rollout buffer for the on-policy callers of the env (SURVEY.md 8f-1).

The reference trains with stable-baselines3 ``MODEL('MlpPolicy', env)`` / ``model.learn`` (gym_dockauv/train.py:64-71):
``collect_rollouts`` steps the env ``n_steps`` times, stores (obs, action, reward, episode_start, value, log_prob) per
step in a ``RolloutBuffer``, then ``compute_returns_and_advantage`` (GAE) and minibatch iteration follow.  With 10^5 ..
10^6 envs that loop cannot go through host arrays and python dicts, so this buffer keeps everything in HBM:

* the step kernel writes observation / reward / done of step t straight into row t of the buffer (``env.step_into`` /
  ``env.rollout``) -- no per-step copies;
* GAE runs as one kernel over the stacked rows (``dockauv_gae``);
* ``get(batch_size)`` yields shuffled minibatches as device tensors with the field names of SB3's
  ``RolloutBufferSamples``;
* ``episode_infos()`` returns what ``Monitor`` would have logged (``r``, ``l``) for the episodes that ended inside the
  rollout, from the in-kernel episode counters.

Field semantics follow SB3's ``RolloutBuffer``: ``observations[t]`` is the observation the policy acted on at step t,
``episode_starts[t]`` tells whether that observation is the first of an episode, ``rewards[t]`` the reward of the
action taken at step t.  After an auto-reset the next observation is the env's reset observation (all zeros for this
env family, docking3d.py:269,322).
"""
from collections import namedtuple

import torch

RolloutSamples = namedtuple("RolloutSamples", ["observations", "actions", "old_values", "old_log_prob", "advantages",
                                               "returns"])


class DeviceRolloutBuffer:
    def __init__(self, env, n_steps, gamma=0.99, gae_lambda=0.95):
        self.env, self.n_steps, self.gamma, self.gae_lambda = env, int(n_steps), float(gamma), float(gae_lambda)
        T, N, dev = self.n_steps, env.num_envs, env.device
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=dev)  # noqa: E731
        # obs rows 0..T: row t is the observation before step t, row T the one after the last step (carried over)
        self._obs = z(T + 1, N, env.n_observations)
        self.actions = z(T, N, env.n_actions)
        self.rewards = z(T, N, dtype=env.dtype)
        self.dones = z(T, N, dtype=torch.uint8)          # done flag returned by step t
        self._starts = z(T + 1, N, dtype=torch.uint8)    # row t: observation t starts an episode
        self.values = z(T, N)
        self.log_probs = z(T, N)
        self.advantages = z(T, N)
        self.returns = z(T, N)
        self.last_values = z(N)                          # collect_fused: V(last_obs), the GAE bootstrap
        self.cond_bits = z(T, N, dtype=torch.uint8)
        self.ep_return = z(T, N, dtype=env.dtype)
        self.ep_length = z(T, N, dtype=torch.int32)
        self._starts[0] = 1
        self.full = False

    # ------------------------------------------------------------------ views with SB3's names
    @property
    def observations(self):
        return self._obs[:self.n_steps]

    @property
    def episode_starts(self):
        return self._starts[:self.n_steps]

    @property
    def last_obs(self):
        return self._obs[self.n_steps]

    def reset_env(self, seed=None):
        """env.reset() and its observation into row 0 (all envs start an episode)."""
        self._obs[0].copy_(self.env.reset(seed=seed))
        self._starts[0] = 1
        self.full = False
        return self._obs[0]

    def _carry_over(self):
        if self.full:      # the last observation of the previous rollout is the first of this one
            self._obs[0].copy_(self._obs[self.n_steps])
            self._starts[0].copy_(self._starts[self.n_steps])
        self.ep_length.zero_()

    def _finish(self):
        self._starts[1:].copy_(self.dones)       # observation t + 1 starts an episode when step t ended one
        self.full = True

    # ------------------------------------------------------------------ collection
    def collect(self, policy):
        """Closed-loop rollout: ``policy(obs) -> (actions, values, log_probs)`` (device tensors; actions [N, n_u]
        float32/float64 in the normalised [-1, 1] range, values / log_probs [N]).  Returns the value-bootstrap
        observation (row T)."""
        env = self.env
        self._carry_over()
        for t in range(self.n_steps):
            a, v, lp = policy(self._obs[t])
            self.actions[t].copy_(a)
            self.values[t].copy_(v.reshape(-1))
            self.log_probs[t].copy_(lp.reshape(-1))
            env.step_into(a if a.dtype in (torch.float32, torch.float64) else self.actions[t], self._obs[t + 1],
                          self.rewards[t], self.dones[t], cond_bits=self.cond_bits[t],
                          ep_return_out=self.ep_return[t], ep_len_out=self.ep_length[t])
        self._finish()
        return self.last_obs

    def collect_open_loop(self, actions=None, generator=None, use_graph=True):
        """Rollout with actions known up front (default: i.i.d. U(-1, 1), the benchmark's random-action rollout):
        one ``dockauv_rollout`` call steps the env ``n_steps`` times into the buffer rows."""
        self._carry_over()
        if actions is None:
            self.actions.uniform_(-1.0, 1.0, generator=generator)
        else:
            self.actions.copy_(actions)
        self.env.rollout(self.actions, self._obs[1:], self.rewards, self.dones, cond_bits=self.cond_bits,
                         ep_return_out=self.ep_return, ep_len_out=self.ep_length, use_graph=use_graph)
        self._finish()
        return self.last_obs

    def collect_fused(self, policy, use_graph=True):
        """Closed-loop rollout with the actor-critic evaluated on the device (``env.rollout_policy``): one library call
        fills the rows ``collect`` fills (actions as sampled, before clipping; values; log-probs) and ``last_values``.
        ``policy``: a ``FusedActorCritic``.  Returns ``last_values`` (the value of ``last_obs``)."""
        self._carry_over()
        self.env.rollout_policy(policy, self._obs[0], self._obs[1:], self.rewards, self.dones, self.actions, self.values,
                                self.log_probs, last_values=self.last_values, cond_bits=self.cond_bits,
                                ep_return_out=self.ep_return, ep_len_out=self.ep_length, use_graph=use_graph)
        self._finish()
        return self.last_values

    # ------------------------------------------------------------------ consumption
    def compute_returns_and_advantage(self, last_values):
        """GAE(lambda) on the device; ``last_values``: value estimate of ``last_obs`` ([N])."""
        self.env.gae(self.rewards, self.values, last_values.reshape(-1).to(torch.float32).contiguous(), self.dones,
                     self.gamma, self.gae_lambda, self.advantages, self.returns)

    def get(self, batch_size=None, generator=None):
        """Shuffled minibatches over the T*N transitions (device tensors)."""
        T, N = self.n_steps, self.env.num_envs
        total = T * N
        perm = torch.randperm(total, device=self.env.device, generator=generator)
        flat = RolloutSamples(self.observations.reshape(total, -1), self.actions.reshape(total, -1),
                              self.values.reshape(total), self.log_probs.reshape(total),
                              self.advantages.reshape(total), self.returns.reshape(total))
        batch_size = total if batch_size is None else int(batch_size)
        for b in range(0, total, batch_size):
            idx = perm[b:b + batch_size]
            yield RolloutSamples(*[f[idx] for f in flat])

    def episode_infos(self):
        """Monitor-style summaries of the episodes that ended inside the rollout: dict of device tensors
        ``r`` (return), ``l`` (length), ``cond_bits``, plus (t, env) indices."""
        ended = self.ep_length > 0
        t, i = ended.nonzero(as_tuple=True)
        return {"r": self.ep_return[ended], "l": self.ep_length[ended], "cond_bits": self.cond_bits[ended], "t": t,
                "env": i}
