"""The actor-critic that ``BaseDocking3d.rollout_policy`` evaluates on the device between the steps of a rollout.

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

from .params import POLICY_MAX_SMEM, DockauvPolicy, policy_smem_bytes


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
