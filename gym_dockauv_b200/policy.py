"""The networks the library evaluates on the device between the steps: the actor-critic of
``BaseDocking3d.rollout_policy`` (PPO) and the squashed-Gaussian actor of ``DeviceReplayBuffer.collect_fused`` (SAC).

It is stable-baselines3 1.5.0's default ``MlpPolicy`` as PPO builds it from ``MODEL('MlpPolicy', env)``
(gym_dockauv/train.py:64): separate ``pi`` and ``vf`` MLPs ``n_obs -> H -> H`` with Tanh after each hidden layer,
``action_net`` ``H -> n_u``, ``value_net`` ``H -> 1``, a state-independent ``log_std`` and a diagonal Gaussian.  The
library reads the parameters through their device pointers, so an in-place ``optimizer.step()`` is seen by the next
rollout (also by a replayed CUDA graph); parameters that are re-allocated (``.to()``, ``load_state_dict`` into new
tensors) need a new ``FusedActorCritic``.

From an SB3 ``ActorCriticPolicy`` ``p``::

    FusedActorCritic([p.mlp_extractor.policy_net[0], p.mlp_extractor.policy_net[2], p.action_net],
                     [p.mlp_extractor.value_net[0], p.mlp_extractor.value_net[2], p.value_net], p.log_std)
"""
import ctypes as C

import torch

from .params import (POLICY_MAX_SMEM, SAC_ACTOR_HIDDEN, DockauvPolicy, DockauvSquashedActor, policy_smem_bytes,
                     sac_actor_smem_bytes)


class FusedActorCritic:
    """``pi_layers`` / ``vf_layers``: three ``nn.Linear`` each (``n_obs -> H``, ``H -> H``, ``H -> n_u`` / ``H -> 1``),
    ``log_std``: ``[n_u]``; all float32, contiguous, on one CUDA device.  ``deterministic=True`` takes the mean action
    (SB3's ``predict(deterministic=True)``).  Keeps references to the tensors it hands to the library."""

    def __init__(self, pi_layers, vf_layers, log_std, deterministic=False):
        pi, vf = list(pi_layers), list(vf_layers)
        if len(pi) != 3 or len(vf) != 3:
            raise ValueError("pi_layers and vf_layers take three nn.Linear each")
        n_obs, H, n_u = pi[0].in_features, pi[0].out_features, pi[2].out_features
        if H % 32 != 0 or not 32 <= H <= 128:
            raise ValueError(f"the hidden width must be a multiple of 32 in 32..128, got {H}")
        for layers, n_out, name in ((pi, n_u, "pi"), (vf, 1, "vf")):
            for k, (n_in, n_o) in enumerate(((n_obs, H), (H, H), (H, n_out))):
                lin = layers[k]
                if tuple(lin.weight.shape) != (n_o, n_in) or lin.bias is None or tuple(lin.bias.shape) != (n_o,):
                    raise ValueError(f"{name} layer {k} must be nn.Linear({n_in}, {n_o}) with a bias")
        if tuple(log_std.shape) != (n_u,):
            raise ValueError(f"log_std must have shape ({n_u},), got {tuple(log_std.shape)}")
        smem = policy_smem_bytes(n_obs, H, n_u)
        if smem > POLICY_MAX_SMEM:
            raise ValueError(f"the weights need {smem} bytes of shared memory (n_obs {n_obs}, hidden {H}, n_u {n_u}); one "
                             f"CTA holds at most {POLICY_MAX_SMEM}")
        self._tensors = [lin.weight for lin in pi] + [lin.bias for lin in pi] + [lin.weight for lin in vf] + \
            [lin.bias for lin in vf] + [log_std]
        device = log_std.device
        for t in self._tensors:
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError("policy parameters must be contiguous float32 tensors")
            if t.device.type != "cuda" or t.device != device:
                raise ValueError("policy parameters must all live on the same CUDA device")
        self.n_obs, self.hidden, self.n_actions, self.device = n_obs, H, n_u, device
        self.deterministic = bool(deterministic)
        p = [C.c_void_p(t.data_ptr()) for t in self._tensors]
        self.struct = DockauvPolicy((C.c_void_p * 3)(*p[0:3]), (C.c_void_p * 3)(*p[3:6]), (C.c_void_p * 3)(*p[6:9]),
                                    (C.c_void_p * 3)(*p[9:12]), p[12], H, int(self.deterministic))

    def check_env(self, env):
        """Refuses an env whose observation / action sizes or device differ from the policy's."""
        if (self.n_obs, self.n_actions) != (env.n_observations, env.n_actions):
            raise ValueError(f"policy is {self.n_obs} -> {self.n_actions}, env has {env.n_observations} observations and "
                             f"{env.n_actions} actions")
        if self.device != env.device:
            raise ValueError(f"policy lives on {self.device}, env on {env.device}")


class FusedSquashedActor:
    """stable-baselines3 1.5.0's SAC ``Actor`` for ``DeviceReplayBuffer.collect_fused``: ``latent_pi`` (two
    ``nn.Linear``, ``n_obs -> H -> H``, ReLU after each), ``mu`` and ``log_std`` (``H -> n_u``, log_std clamped to
    [-20, 2]); the action is ``tanh(mu + exp(log_std) eps)``, or ``tanh(mu)`` with ``deterministic=True`` (SB3's
    ``predict(deterministic=True)``).  H is 64, 128 or 256 (SB3's SAC default is 256).  The parameters are float32,
    contiguous, on one CUDA device; the library reads them through their device pointers (bf16 operands on the tensor
    cores, f32 accumulation, include/dockauv.h), so an in-place ``optimizer.step()`` is seen by the next collection, also
    by a replayed CUDA graph.  Keeps references to the tensors it hands to the library.

    From an SB3 SAC policy ``p``::

        a = p.actor
        FusedSquashedActor([a.latent_pi[0], a.latent_pi[2]], a.mu.weight, a.mu.bias, a.log_std.weight, a.log_std.bias)

    From one ``Linear(H, 2 n_u)`` head whose output is split into (mu, log_std), as in examples/sac_device_replay.py
    (the row slices are contiguous views of the live parameter, so in-place updates are seen)::

        net = actor.net      # Linear(n_obs, H), ReLU, Linear(H, H), ReLU, Linear(H, 2 n_u)
        w, b = net[4].weight, net[4].bias
        FusedSquashedActor([net[0], net[2]], w[:n_u], b[:n_u], w[n_u:], b[n_u:])
    """

    def __init__(self, latent_pi, mu_weight, mu_bias, log_std_weight, log_std_bias, deterministic=False):
        lat = list(latent_pi)
        if len(lat) != 2:
            raise ValueError("latent_pi takes two nn.Linear (n_obs -> H, H -> H)")
        n_obs, H = lat[0].in_features, lat[0].out_features
        if H not in SAC_ACTOR_HIDDEN:
            raise ValueError(f"the hidden width must be one of {SAC_ACTOR_HIDDEN}, got {H}")
        for k, (n_in, n_o) in enumerate(((n_obs, H), (H, H))):
            lin = lat[k]
            if tuple(lin.weight.shape) != (n_o, n_in) or lin.bias is None or tuple(lin.bias.shape) != (n_o,):
                raise ValueError(f"latent_pi layer {k} must be nn.Linear({n_in}, {n_o}) with a bias")
        n_u = int(mu_weight.shape[0]) if mu_weight.dim() == 2 else -1
        if n_u not in (3, 6, 8):
            raise ValueError(f"mu_weight must be [n_u, {H}] with n_u 3, 6 or 8, got {tuple(mu_weight.shape)}")
        for name, t, shape in (("mu_weight", mu_weight, (n_u, H)), ("mu_bias", mu_bias, (n_u,)),
                               ("log_std_weight", log_std_weight, (n_u, H)), ("log_std_bias", log_std_bias, (n_u,))):
            if tuple(t.shape) != shape:
                raise ValueError(f"{name} must have shape {shape}, got {tuple(t.shape)}")
        smem = sac_actor_smem_bytes(n_obs, H, n_u)
        if smem > POLICY_MAX_SMEM:
            raise ValueError(f"the weights need {smem} bytes of shared memory (n_obs {n_obs}, hidden {H}, n_u {n_u}); one "
                             f"CTA holds at most {POLICY_MAX_SMEM}")
        self._tensors = [lat[0].weight, lat[1].weight, lat[0].bias, lat[1].bias, mu_weight, mu_bias, log_std_weight,
                         log_std_bias]
        device = mu_weight.device
        if any(t.dtype != torch.float32 or not t.is_contiguous() for t in self._tensors):
            raise ValueError("actor parameters must be contiguous float32 tensors")
        if any(t.device.type != "cuda" or t.device != device for t in self._tensors):
            raise ValueError("actor parameters must all live on the same CUDA device")
        self.n_obs, self.hidden, self.n_actions, self.device = n_obs, H, n_u, device
        self.deterministic = bool(deterministic)
        p = [C.c_void_p(t.data_ptr()) for t in self._tensors]
        self.struct = DockauvSquashedActor((C.c_void_p * 2)(*p[0:2]), (C.c_void_p * 2)(*p[2:4]), *p[4:8], H,
                                           int(self.deterministic))

    check_env = FusedActorCritic.check_env
