"""Device-resident replay ring for the off-policy callers of the env (the SAC half of ``MODEL`` at train.py:64).

SB3's off-policy loop (``OffPolicyAlgorithm.collect_rollouts`` / ``_store_transition``, stable-baselines3 1.5.0) stores
one transition per env and step, with ``next_obs = terminal_observation if done else new_obs``, and
``ReplayBuffer.sample`` draws minibatches uniformly over the stored (slot, env) pairs.  At 10^5 .. 10^6 envs neither can
go through host arrays, so this buffer keeps everything in HBM:

* ``collect`` lets the step kernels write observation, reward, done flag and terminal observation of step t straight
  into the ring slots (``env.step_into``); no observation is copied after the kernel;
* ``collect_fused`` does the same with SAC's actor evaluated on the device (``policy.FusedSquashedActor``): the
  actor and step launches of all steps are one library call (``dockauv_replay_collect``), replayed as a CUDA graph;
* ``sample`` is one kernel (``dockauv_replay_sample``) that draws the minibatch and gathers its rows, next observations
  at episode ends included, into float32 tensors with the field names of SB3's ``ReplayBufferSamples``.

Layout: ``S = n_slots`` slots of the whole batch of ``N`` envs.  Slot ``t % S`` holds

* ``obs[t % S]``: the observation the policy acted on at step t (``o_t``);
* ``actions[t % S]``: the action of step t exactly as the step read it, float32 in the normalised [-1, 1] range.  For
  BlueROV2 that is SB3 SAC's ``buffer_action``.  For LAUV the reference declares the physical ``u_bound`` as
  ``action_space`` (docking3d.py:116-125, kept in ``BaseDocking3d.action_space``) while ``step`` expects normalised
  actions; SB3 would rescale its [-1, 1] policy output onto that space before stepping.  Here the policy's output goes
  to the step unchanged;
* ``rewards[t % S]`` (env dtype), ``dones[t % S]`` (uint8): what step t returned;
* ``terminal_obs[t % S]``: the last real observation of the envs whose episode ended at step t (other rows are stale
  and never read).

After T steps since ``reset_env`` the valid transitions are t in [max(0, T - (S - 1)), T - 1]: transition t is
(o_t, a_t, r_t, d_t, next = d_t ? terminal_obs[t % S] : o_{t+1}).  The slot the next step overwrites is never drawn
(SB3's ``optimize_memory_usage`` rule for the newest slot), so a full ring holds (S - 1) * N sampleable transitions,
with exact next observations at episode ends.  The first observation of an episode is the env's all-zero reset
observation (docking3d.py:269,322).

``S`` is limited to 2..64: every ring slot is a different set of output pointers for ``dockauv_step``, which caches one
CUDA graph per pointer set (96 per handle, oldest evicted first).  With more slots than the cache holds every step would
capture its graph anew; 64 leaves room for the caller's other pointer sets.  Capacity scales with N instead: 64 slots of
65,536 envs are 4.2M transitions.

Episode statistics for Monitor-style logging come from the env itself (``env.clear_stats`` / ``env.get_stats``).
"""
import ctypes as C
from collections import namedtuple

import torch

from . import _capi
from .params import F32, F64, DockauvReplayRing, DockauvReplaySample

ReplayBufferSamples = namedtuple("ReplayBufferSamples", ["observations", "actions", "next_observations", "dones",
                                                         "rewards"])

MIN_SLOTS, MAX_SLOTS = 2, 64


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class DeviceReplayBuffer:
    def __init__(self, env, n_slots, seed=0):
        S = int(n_slots)
        if not MIN_SLOTS <= S <= MAX_SLOTS:
            raise ValueError(f"n_slots must be between {MIN_SLOTS} and {MAX_SLOTS}, got {n_slots}: one slot is always being "
                             f"overwritten, and each slot is a pointer set with its own cached step graph (96 per env "
                             f"handle), so more slots would re-capture the step graph on every step; grow num_envs instead")
        self.env, self.n_slots, self.seed = env, S, int(seed) & (2 ** 64 - 1)
        self._lib = _capi.load()
        N, dev = env.num_envs, env.device
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=dev)  # noqa: E731
        self.obs = z(S, N, env.n_observations)
        self.terminal_obs = z(S, N, env.n_observations)
        self.actions = z(S, N, env.n_actions)
        self.rewards = z(S, N, dtype=env.dtype)
        self.dones = z(S, N, dtype=torch.uint8)
        self._ring = DockauvReplayRing(*[_ptr(t) for t in (self.obs, self.terminal_obs, self.actions, self.rewards,
                                                           self.dones)])
        self._precision = F64 if env.dtype == torch.float64 else F32
        self.t = 0          # steps since reset_env
        self.draws = 0      # sample() calls so far: the Philox counter of the next minibatch

    @property
    def n_valid(self):
        """Sampleable transitions per env: min(T, S - 1)."""
        return min(self.t, self.n_slots - 1)

    def size(self):
        """Sampleable transitions in total (SB3's ``ReplayBuffer.size()`` times the env count)."""
        return self.n_valid * self.env.num_envs

    def reset_env(self, seed=None):
        """``env.reset`` and its (all-zero) observation into slot 0; empties the buffer."""
        self.obs[0].copy_(self.env.reset(seed=seed))
        self.t = 0
        return self.obs[0]

    def collect(self, policy, n_steps):
        """``n_steps`` closed-loop steps: ``policy(obs) -> actions`` ([N, n_u] device tensor, normalised [-1, 1]).  The
        actions are copied into their slot and the step reads them from there; the step kernels write observation,
        reward, done and terminal observation into the ring.  Returns the observation the next step acts on."""
        env, S = self.env, self.n_slots
        for _ in range(int(n_steps)):
            s, s1 = self.t % S, (self.t + 1) % S
            self.actions[s].copy_(policy(self.obs[s]))
            env.step_into(self.actions[s], self.obs[s1], self.rewards[s], self.dones[s], terminal_obs=self.terminal_obs[s])
            self.t += 1
        return self.obs[self.t % S]

    def collect_fused(self, actor, n_steps, use_graph=True):
        """``collect`` with a ``FusedSquashedActor`` evaluated on the device before each step: ONE library call on the
        env's current stream for all ``n_steps`` steps.  Step t's actor reads the observation of its slot and writes the
        actions into it (float32, unclipped, unscaled, as ``collect`` stores them), and the step reads them from there.
        With ``use_graph`` the launch sequence is captured once per (actor, start slot, ``n_steps``) and replayed: with
        ``n_steps`` a multiple of ``n_slots`` every call replays the same graph.  Returns the observation the next step
        acts on."""
        env, S, T = self.env, self.n_slots, int(n_steps)
        actor.check_env(env)
        if T <= 0:
            raise ValueError(f"n_steps must be positive, got {n_steps}")
        _capi.check(self._lib.dockauv_replay_collect(env._handle, C.byref(actor.struct), C.byref(self._ring), S,
                                                     self.t % S, T, int(env.auto_reset), int(bool(use_graph)),
                                                     env._stream()))
        self.t += T
        env.t_total_steps += T
        return self.obs[self.t % S]

    def collect_captures(self):
        """How many times ``collect_fused(use_graph=True)`` had to capture its launch sequence (replays do not)."""
        n = C.c_int64()
        _capi.check(self._lib.dockauv_replay_collect_captures(self.env._handle, C.byref(n)))
        return n.value

    def sample(self, batch_size, return_index=False):
        """``batch_size`` transitions drawn uniformly over the valid (transition, env) pairs, as float32 device tensors
        with SB3's field names and shapes: observations / next_observations [B, n_obs], actions [B, n_u], dones and
        rewards [B, 1] (dones = done * (1 - timeouts) with timeouts = 0: the reference never sets TimeLimit.truncated).
        One kernel launch; each call advances the draw counter, so a fixed ``seed`` gives the same minibatch sequence.
        With ``return_index`` also returns the int64 [B] ring index slot * N + env of each row."""
        B, env = int(batch_size), self.env
        if B <= 0:
            raise ValueError(f"batch_size must be positive, got {batch_size}")
        if self.t == 0:
            raise ValueError("the buffer is empty: collect at least one step after reset_env")
        n_obs, n_u = env.n_observations, env.n_actions
        flat = torch.empty(B * (2 * n_obs + n_u + 2), dtype=torch.float32, device=env.device)
        o, nx, a, d, r = flat.split([B * n_obs, B * n_obs, B * n_u, B, B])
        idx = torch.empty(B, dtype=torch.int64, device=env.device) if return_index else None
        out = DockauvReplaySample(*[_ptr(t) for t in (o, a, nx, d, r, idx)])
        n_valid = self.n_valid
        with torch.cuda.device(env.device):
            _capi.check(self._lib.dockauv_replay_sample(
                C.byref(self._ring), self._precision, self.n_slots, env.num_envs, n_obs, n_u, self.t - n_valid, n_valid,
                B, self.seed, self.draws, C.byref(out), C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)))
        self.draws += 1
        samples = ReplayBufferSamples(o.view(B, n_obs), a.view(B, n_u), nx.view(B, n_obs), d.view(B, 1), r.view(B, 1))
        return (samples, idx) if return_index else samples
