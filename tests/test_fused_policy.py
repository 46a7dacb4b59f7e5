"""Closed-loop rollouts on the device (dockauv_rollout_policy): SB3's MlpPolicy evaluated between the steps.

CPU: every refusal that needs no handle comes before the handle is looked at; FusedActorCritic refuses bad layers
before any device is touched; the ctypes structs match the header.  GPU: the closed loop equals the open loop replayed
with its own clipped actions, bit for bit, across layouts, precisions, vehicles, auto-reset, step parts and scenario
banks; the policy's numerics against a float64 evaluation; the noise against a numpy Philox + Box-Muller; graphs;
launch counts; the PPO example."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M32 = np.uint64(0xFFFFFFFF)


# ------------------------------------------------------------------------------------------- the noise, restated
def philox4x32_10(c, k0, k1):
    """Philox4x32-10 over numpy uint64 arrays holding 32-bit words (gym_dockauv_b200/csrc/dockauv_device.cuh)."""
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in c]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & M32, p1 & M32, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & M32, p0 & M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c


def policy_eps(seed, gids, episodes, t_steps, n_u):
    """eps [n, n_u] of the documented counters (include/dockauv.h, dockauv_rollout_policy), in float64."""
    gids = np.asarray(gids, dtype=np.uint64)
    ep = np.asarray(episodes, dtype=np.int64).astype(np.uint64) & M32
    t = np.asarray(t_steps, dtype=np.int64).astype(np.uint64) & np.uint64(0x1FFFFFFF)
    out = []
    for j in range((n_u + 3) // 4):
        w = philox4x32_10([gids & M32, gids >> np.uint64(32), ep, np.uint64(0xC0000000) | (t << np.uint64(1)) | np.uint64(j)],
                          seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
        for m in range(2):
            u = ((w[2 * m] >> np.uint64(8)) + np.uint64(1)).astype(np.float64) * 2.0 ** -24
            v = (w[2 * m + 1] >> np.uint64(8)).astype(np.float64) * 2.0 ** -24
            r = np.sqrt(-2.0 * np.log(u))
            out += [r * np.cos(2 * np.pi * v), r * np.sin(2 * np.pi * v)]
    return np.stack(out[:n_u], axis=1)


# ------------------------------------------------------------------------------------------- CPU
def test_refusals_that_need_no_handle_come_first():
    from gym_dockauv_b200 import _capi
    from gym_dockauv_b200.params import DockauvPolicy, DockauvPolicyOut, DockauvRolloutOut
    lib = _capi.load()
    fake = 0x10000

    def call(h=None, hidden=64, n_steps=8, null=(), pol=True, out=True, pout=True, obs0=fake):
        ptrs = {k: (C.c_void_p * 3)(*[None if f"{k}{i}" in null else fake for i in range(3)])
                for k in ("pi_w", "pi_b", "vf_w", "vf_b")}
        p = DockauvPolicy(ptrs["pi_w"], ptrs["pi_b"], ptrs["vf_w"], ptrs["vf_b"], None if "log_std" in null else fake,
                          hidden, 0)
        o = DockauvRolloutOut(*[None if k in null else fake for k in ("obs", "reward", "done")], *[None] * 5)
        po = DockauvPolicyOut(*[None if k in null else fake for k in ("actions", "values", "log_probs")], None)
        rc = lib.dockauv_rollout_policy(h, C.byref(p) if pol else None, obs0, n_steps, C.byref(o) if out else None,
                                        C.byref(po) if pout else None, 1, 1, None)
        return rc, lib.dockauv_last_error().decode()

    rc, msg = call()
    assert rc == -1 and "null handle" in msg          # every argument passed: only then is the handle looked at
    for kw, word in ((dict(pol=False), "null argument"), (dict(out=False), "null argument"),
                     (dict(pout=False), "null argument"), (dict(obs0=None), "null argument"),
                     (dict(null=("pi_w0",)), "layer 0"), (dict(null=("vf_b2",)), "layer 2"),
                     (dict(null=("pi_b1",)), "layer 1"), (dict(null=("log_std",)), "log_std"),
                     (dict(hidden=0), "hidden"), (dict(hidden=48), "hidden"), (dict(hidden=160), "hidden"),
                     (dict(n_steps=0), "n_steps"), (dict(n_steps=-3), "n_steps"),
                     (dict(null=("obs",)), "obs, reward and done"), (dict(null=("done",)), "obs, reward and done"),
                     (dict(null=("actions",)), "actions, values and log_probs"),
                     (dict(null=("log_probs",)), "actions, values and log_probs")):
        rc, msg = call(**kw)
        assert rc == -1 and word in msg, (kw, msg)
    for hidden in (32, 64, 96, 128):
        assert "null handle" in call(hidden=hidden)[1]
    assert lib.dockauv_rollout_policy_captures(None, None) == -1


def test_structs_match_the_header(tmp_path):
    """Field offsets and sizes of DockauvPolicy / DockauvPolicyOut as the C compiler lays them out."""
    from gym_dockauv_b200.params import DockauvPolicy, DockauvPolicyOut
    fields = {"DockauvPolicy": ["pi_w", "pi_b", "vf_w", "vf_b", "log_std", "hidden", "deterministic"],
              "DockauvPolicyOut": ["actions", "values", "log_probs", "last_values"]}
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "dockauv.h"', 'int main(void) {']
    for s, fs in fields.items():
        src.append(f'printf("{s} %zu\\n", sizeof({s}));')
        src += [f'printf("{s}.{f} %zu\\n", offsetof({s}, {f}));' for f in fs]
    src.append("return 0; }")
    (tmp_path / "layout.c").write_text("\n".join(src))
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(ROOT, "include"), str(tmp_path / "layout.c"), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True)
               .stdout.splitlines())
    for s, cls in (("DockauvPolicy", DockauvPolicy), ("DockauvPolicyOut", DockauvPolicyOut)):
        assert int(got[s]) == C.sizeof(cls), s
        assert [f[0] for f in cls._fields_] == fields[s]
        for f in fields[s]:
            assert int(got[f"{s}.{f}"]) == getattr(cls, f).offset, (s, f)


def _layers(n_obs, H, n_u, dtype=None, device="cpu"):
    import torch.nn as nn
    kw = dict(dtype=dtype, device=device)
    return ([nn.Linear(n_obs, H, **kw), nn.Linear(H, H, **kw), nn.Linear(H, n_u, **kw)],
            [nn.Linear(n_obs, H, **kw), nn.Linear(H, H, **kw), nn.Linear(H, 1, **kw)])


def test_fused_actor_critic_refuses_bad_layers_before_the_device():
    import torch
    from gym_dockauv_b200.params import POLICY_MAX_SMEM, policy_smem_bytes
    from gym_dockauv_b200.policy import FusedActorCritic
    assert policy_smem_bytes(36, 64, 6) == 54096          # the stock obstacle env: 36 observations, 6 actions
    assert policy_smem_bytes(80, 128, 8) <= POLICY_MAX_SMEM < policy_smem_bytes(100, 128, 6)
    for H in (16, 48, 160):
        pi, vf = _layers(36, H, 6)
        with pytest.raises(ValueError, match="hidden"):
            FusedActorCritic(pi, vf, torch.zeros(6))
    pi, vf = _layers(100, 128, 6)
    with pytest.raises(ValueError, match="shared memory"):
        FusedActorCritic(pi, vf, torch.zeros(6))
    pi, vf = _layers(36, 64, 6)
    with pytest.raises(ValueError, match="log_std"):
        FusedActorCritic(pi, vf, torch.zeros(5))
    with pytest.raises(ValueError, match="vf layer 2"):
        FusedActorCritic(pi, vf[:2] + [torch.nn.Linear(64, 2)], torch.zeros(6))
    with pytest.raises(ValueError, match="three"):
        FusedActorCritic(pi[:2], vf, torch.zeros(6))
    pi64, vf64 = _layers(36, 64, 6, dtype=torch.float64)
    with pytest.raises(ValueError, match="float32"):
        FusedActorCritic(pi64, vf64, torch.zeros(6, dtype=torch.float64))
    with pytest.raises(ValueError, match="CUDA"):
        FusedActorCritic(pi, vf, torch.zeros(6))


# ------------------------------------------------------------------------------------------- GPU helpers
def _cfg(max_timesteps=None, vehicle=None):
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    if max_timesteps is not None:
        cfg["max_timesteps"] = max_timesteps
    if vehicle is not None:
        cfg["vehicle"] = vehicle
    if vehicle == "LAUV":
        cfg["t_step_size"] = 0.02      # the reference's integrator diverges at the stock 0.1 for this vehicle
    return cfg


def _policy(env, H=64, init="torch", seed=0, log_std=-0.5, deterministic=False):
    """(FusedActorCritic, its modules): torch-default or SB3's orthogonal initialisation (gain sqrt(2) for the hidden
    layers, 0.01 for action_net, 1 for value_net, zero biases)."""
    import torch
    import torch.nn as nn
    from gym_dockauv_b200.policy import FusedActorCritic
    torch.manual_seed(seed)
    pi, vf = _layers(env.n_observations, H, env.n_actions, device=env.device)
    if init == "orthogonal":
        for layers in (pi, vf):
            for k, lin in enumerate(layers):
                nn.init.orthogonal_(lin.weight, gain=2 ** 0.5 if k < 2 else (0.01 if layers is pi else 1.0))
                nn.init.zeros_(lin.bias)
    ls = nn.Parameter(torch.full((env.n_actions,), float(log_std), device=env.device))
    return FusedActorCritic(pi, vf, ls, deterministic=deterministic), (pi, vf, ls)


def _eval(mods, obs, dtype):
    import torch
    pi, vf, _ = mods

    def net(layers, x):
        w = [(lin.weight.detach().to(dtype), lin.bias.detach().to(dtype)) for lin in layers]
        x = torch.tanh(torch.nn.functional.linear(x, *w[0]))
        x = torch.tanh(torch.nn.functional.linear(x, *w[1]))
        return torch.nn.functional.linear(x, *w[2])
    x = obs.to(dtype)
    return net(pi, x), net(vf, x)[..., 0]


class _Rollout:
    """Output tensors of one closed-loop rollout of T steps."""

    def __init__(self, env, T):
        import torch
        N, dev = env.num_envs, env.device
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=dev)  # noqa: E731
        self.obs0 = z(N, env.n_observations)
        self.obs = z(T, N, env.n_observations)
        self.reward = z(T, N, dtype=env.dtype)
        self.done = z(T, N, dtype=torch.uint8)
        self.cond_bits = z(T, N, dtype=torch.uint8)
        self.ep_return = z(T, N, dtype=env.dtype)
        self.ep_len = z(T, N, dtype=torch.int32)
        self.actions = z(T, N, env.n_actions)
        self.values = z(T, N)
        self.log_probs = z(T, N)
        self.last_values = z(N)

    def run(self, env, policy, use_graph=True):
        self.ep_return.zero_()         # only the entries of episodes that end are written: zeros elsewhere compare equal
        env.rollout_policy(policy, self.obs0, self.obs, self.reward, self.done, self.actions, self.values, self.log_probs,
                           last_values=self.last_values, cond_bits=self.cond_bits, ep_return_out=self.ep_return,
                           ep_len_out=self.ep_len, use_graph=use_graph)
        return self

    def fields(self):
        return dict(obs=self.obs, reward=self.reward, done=self.done, cond_bits=self.cond_bits, ep_return=self.ep_return,
                    ep_len=self.ep_len, actions=self.actions, values=self.values, log_probs=self.log_probs,
                    last_values=self.last_values)

    def clone(self):
        return {k: v.clone() for k, v in self.fields().items()}


def _state(env):
    return [t.clone() for t in (env.state, env.u_prev, env.goal, env.current, env.capsules, env.spheres, env.ep_return,
                                env.t_steps, env.episode)]


def _pre_step_counters(episode0, t0, done):
    """(episode, t_steps) of every env before each step of a rollout with auto-reset, from the done flags."""
    import torch
    ep, t = episode0.clone().long(), t0.clone().long()
    eps, ts = [], []
    for d in done.bool():
        eps.append(ep.clone())
        ts.append(t.clone())
        ep = torch.where(d, ep + 1, ep)
        t = torch.where(d, torch.zeros_like(t), t + 1)
    return torch.stack(eps), torch.stack(ts)


# ------------------------------------------------------------------------------------------- GPU: closed = open loop
CASES = {
    "pipeline_f64": dict(num_envs=4096, n_synthetic_spheres=3),
    "pipeline_parts_f32": dict(num_envs=1 << 17, n_synthetic_spheres=3, precision="f32"),
    "warp_rays_f32": dict(num_envs=3000, n_synthetic_spheres=3, layout="warp_rays", precision="f32"),
    "thread_per_env_f64": dict(num_envs=3000, n_synthetic_spheres=3, layout="thread_per_env"),
    "lauv_f64": dict(num_envs=4096, n_synthetic_spheres=3, vehicle="LAUV"),
    "lauv_parts_f32": dict(num_envs=1 << 17, precision="f32", vehicle="LAUV"),
    "bank_f64": dict(num_envs=4096, n_synthetic_spheres=3, bank=True),
    "bank_parts_f32": dict(num_envs=1 << 17, n_synthetic_spheres=3, precision="f32", bank=True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_closed_loop_equals_open_loop_replay(case):
    """After rollout_policy, a twin handle replaying clamp(actions, u_lo, u_hi) as float32 actions with rollout()
    reproduces every output and the final state exactly (max_timesteps 10: every env ends an episode inside)."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.scenario_bank import ScenarioBank
    kw = dict(CASES[case])
    vehicle, bank = kw.pop("vehicle", None), kw.pop("bank", False)
    T, seed = 24, 11
    cfg = _cfg(max_timesteps=10, vehicle=vehicle)
    a, b = envs.ObstaclesDocking3d(cfg, seed=seed, **kw), envs.ObstaclesDocking3d(cfg, seed=seed, **kw)
    if bank:
        rows = ScenarioBank.from_builtin(a, 257, seed=5)
        a.set_scenario_bank(rows)
        b.set_scenario_bank(ScenarioBank.from_builtin(b, 257, seed=5))
    policy, _ = _policy(a, log_std=0.3)          # wide enough that clipping matters
    ra = _Rollout(a, T)
    for env in (a, b):
        env.reset(seed=seed)
    ra.run(a, policy)
    lo = torch.as_tensor(a.action_space.low, device=a.device)
    hi = torch.as_tensor(a.action_space.high, device=a.device)
    clipped = torch.clamp(ra.actions, lo, hi).float()
    assert not torch.equal(clipped, ra.actions)
    rb = _Rollout(b, T)
    b.rollout(clipped, rb.obs, rb.reward, rb.done, cond_bits=rb.cond_bits, ep_return_out=rb.ep_return,
              ep_len_out=rb.ep_len)
    torch.cuda.synchronize()
    assert int(ra.done.sum()) >= a.num_envs         # every env ended at least one episode inside the rollout
    for k in ("obs", "reward", "done", "cond_bits", "ep_return", "ep_len"):
        assert torch.equal(getattr(ra, k), getattr(rb, k)), k
    for x, y in zip(_state(a), _state(b)):
        assert torch.equal(x, y)
    if bank:
        assert torch.equal(a.bank_row, b.bank_row)
    a.close(); b.close()


# ------------------------------------------------------------------------------------------- GPU: numerics
@pytest.mark.gpu
@pytest.mark.parametrize("init", ["torch", "orthogonal"])
@pytest.mark.parametrize("H", [64, 128])
def test_policy_numerics_against_float64(H, init):
    """Means (deterministic actions, and a - sigma eps of a stochastic run), values, log-probs and last_values on the
    rollout's own observation rows against a float64 torch evaluation of the same weights: within 1e-5 (log-probs
    1e-4) and no worse than 4x the float32 torch module's own error; eps against the numpy restatement within 1e-5."""
    import torch
    from gym_dockauv_b200 import envs
    T, N, seed = 12, 8192, 3
    env = envs.ObstaclesDocking3d(_cfg(max_timesteps=6), num_envs=N, seed=seed, n_synthetic_spheres=3)
    sigma_log = torch.tensor([-0.7, -0.2, 0.1, -1.0, 0.0, -0.4], device=env.device)
    for deterministic in (True, False):
        policy, mods = _policy(env, H=H, init=init, seed=7, deterministic=deterministic)
        with torch.no_grad():
            mods[2].copy_(sigma_log)
        r = _Rollout(env, T)
        env.reset(seed=seed)
        ep0, t0 = env.episode.clone(), env.t_steps.clone()
        r.obs0.copy_(env.obs)
        r.run(env, policy)
        torch.cuda.synchronize()
        obs_in = torch.cat([r.obs0[None], r.obs[:-1]])
        mu64, v64 = _eval(mods, obs_in, torch.float64)
        mu32, v32 = _eval(mods, obs_in, torch.float32)
        _, lv64 = _eval(mods, r.obs[-1], torch.float64)
        _, lv32 = _eval(mods, r.obs[-1], torch.float32)
        ls = mods[2].detach().double()
        if deterministic:
            eps = torch.zeros_like(mu64)
        else:
            pe, pt = _pre_step_counters(ep0, t0, r.done)
            gids = np.tile(np.arange(N), T)
            eps = torch.as_tensor(policy_eps(seed, gids, pe.cpu().numpy().ravel(), pt.cpu().numpy().ravel(), 6),
                                  device=env.device).reshape(T, N, 6)
            eps_kernel = (r.actions.double() - mu64) / ls.exp()
            assert float((eps_kernel - eps).abs().max()) < 1e-5
        # a stochastic sample holds the mean only to the rounding of a itself (|a| up to ~8): 1e-5 there, and the
        # comparison with the f32 module's own error on the deterministic means
        mu_kernel = r.actions.double() - ls.exp() * eps
        for got, ref, f32, own_bound in ((mu_kernel, mu64, mu32, deterministic), (r.values, v64, v32, True),
                                         (r.last_values, lv64, lv32, True)):
            err = float((got.double() - ref).abs().max())
            own = float((f32.double() - ref).abs().max())
            assert err < 1e-5, (err, own)
            assert not own_bound or err <= 4 * max(own, 1e-7), (err, own)
        lp_ref = (-0.5 * eps * eps - ls - 0.5 * np.log(2 * np.pi)).sum(-1)
        assert float((r.log_probs.double() - lp_ref).abs().max()) < 1e-4
    env.close()


# ------------------------------------------------------------------------------------------- GPU: noise
@pytest.mark.gpu
def test_noise_is_reproducible_and_independent_of_sharding():
    """Two runs from reset(seed=s) are bit-equal, another seed differs, and a 2M-env handle equals two M-env handles
    with env_id0 = 0 and M (the 2M handle is stepped in two parts)."""
    import torch
    from gym_dockauv_b200 import envs
    M, T = 1 << 16, 16
    cfg = _cfg(max_timesteps=7)
    big = envs.ObstaclesDocking3d(cfg, num_envs=2 * M, seed=4, n_synthetic_spheres=3)
    policy, mods = _policy(big)
    r = _Rollout(big, T)
    runs = []
    for s in (4, 4, 5):
        big.reset(seed=s)
        r.run(big, policy)
        runs.append(r.clone())
    for k in runs[0]:
        assert torch.equal(runs[0][k], runs[1][k]), k
    assert not torch.equal(runs[0]["actions"], runs[2]["actions"])
    for part, id0 in ((0, 0), (1, M)):
        small = envs.ObstaclesDocking3d(cfg, num_envs=M, seed=4, env_id0=id0, n_synthetic_spheres=3)
        p, _ = _policy(small)
        rs = _Rollout(small, T)
        small.reset(seed=4)
        rs.run(small, p)
        torch.cuda.synchronize()
        for k, v in rs.fields().items():
            ref = runs[0][k]
            ref = ref[part * M:(part + 1) * M] if ref.dim() == 1 else ref[:, part * M:(part + 1) * M]
            assert torch.equal(v, ref), (k, part)
        small.close()
    big.close()


# ------------------------------------------------------------------------------------------- GPU: graphs and launches
@pytest.mark.gpu
def test_graph_replays_read_weights_updated_in_place():
    """Same tensors: no re-capture; after an in-place optimizer.step() the replay equals a use_graph=False call with the
    new weights bit for bit; a deterministic evaluation policy alternating with the training one re-captures nothing
    after its first call; graph, no graph and taps set give equal outputs, and the tap ring advances by T."""
    import torch
    from gym_dockauv_b200 import envs
    T, seed = 20, 9
    env = envs.ObstaclesDocking3d(_cfg(max_timesteps=8), num_envs=4096, seed=seed, n_synthetic_spheres=3)
    policy, mods = _policy(env)
    evaluation = type(policy)(mods[0], mods[1], mods[2], deterministic=True)
    r = _Rollout(env, T)

    def run(p, use_graph=True):
        env.reset(seed=seed)
        r.run(env, p, use_graph=use_graph)
        torch.cuda.synchronize()
        return r.clone()
    first = run(policy)
    assert env.rollout_policy_captures() == 1
    again = run(policy)
    assert env.rollout_policy_captures() == 1
    for k in first:
        assert torch.equal(first[k], again[k]), k
    params = [p for lin in mods[0] + mods[1] for p in lin.parameters()] + [mods[2]]
    opt = torch.optim.SGD(params, lr=0.05)
    x = torch.randn(64, env.n_observations, device=env.device)
    loss = _eval(mods, x, torch.float32)[0].pow(2).sum() + _eval(mods, x, torch.float32)[1].pow(2).sum() + mods[2].sum()
    loss.backward()
    opt.step()
    replay = run(policy)
    assert env.rollout_policy_captures() == 1
    plain = run(policy, use_graph=False)
    assert not torch.equal(replay["actions"], first["actions"])
    for k in replay:
        assert torch.equal(replay[k], plain[k]), k
    for _ in range(2):
        ev = run(evaluation)
        tr = run(policy)
    assert env.rollout_policy_captures() == 2
    assert torch.equal(tr["actions"], plain["actions"])
    assert not torch.equal(ev["actions"], tr["actions"])
    ring = env.set_taps([0, 17, 4095], capacity=64)
    tapped = run(policy)
    assert int(ring["count"][0]) == T
    tapped_plain = run(policy, use_graph=False)
    assert int(ring["count"][0]) == 2 * T
    for k in tapped:
        assert torch.equal(tapped[k], plain[k]) and torch.equal(tapped_plain[k], plain[k]), k
    # the ring holds the tapped envs' observations of the last rollout's steps, in order (before any auto-reset: rows
    # of steps that ended an episode hold the last real observation, obs the zero reset observation)
    slots = torch.arange(T, 2 * T) % 64
    live = plain["done"][:, 17] == 0
    assert torch.equal(ring["obs"][slots][:, 1][live], plain["obs"][:, 17][live])
    assert torch.equal(ring["done"][slots][:, 1], plain["done"][:, 17])
    env.clear_taps()
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("N,ranges", [(4096, 1), (1 << 17, 2)])
def test_launch_count(N, ranges):
    """dockauv_launch_count grows by ranges x (T x (1 + step launches) + 1) per rollout (graph or not)."""
    import torch
    from gym_dockauv_b200 import envs
    T = 6
    env = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=1, n_synthetic_spheres=3)
    env.reset(seed=1)
    r = _Rollout(env, T)
    n0 = env.launch_count()
    env.rollout(torch.zeros(T, N, env.n_actions, device=env.device), r.obs, r.reward, r.done, use_graph=False)
    step_launches = (env.launch_count() - n0) // (ranges * T)
    assert env.launch_count() - n0 == ranges * T * step_launches
    policy, _ = _policy(env)
    for use_graph in (False, True, True):
        n0 = env.launch_count()
        r.run(env, policy, use_graph=use_graph)
        assert env.launch_count() - n0 == ranges * (T * (1 + step_launches) + 1), use_graph
    torch.cuda.synchronize()
    env.close()


@pytest.mark.gpu
def test_refusals_with_a_handle_touch_nothing():
    """Weights too large for shared memory and misaligned observation rows are refused before any launch."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG
    from gym_dockauv_b200.params import DockauvPolicy, DockauvPolicyOut, DockauvRolloutOut
    cfg = dict(BASE_CONFIG)
    deg = np.pi / 180
    cfg["radar"] = dict(freq=1, alpha=75 * deg, beta=75 * deg, ray_per_deg=5 * deg, max_dist=10, blocksize_reduce=1)
    T, N = 4, 256
    env = envs.ObstaclesDocking3d(cfg, num_envs=N, seed=1)
    assert env.n_observations == 16 + 256
    env.reset(seed=1)
    buf = torch.zeros(1 << 20, device=env.device)
    p = [C.c_void_p(buf.data_ptr())] * 3
    pol = DockauvPolicy((C.c_void_p * 3)(*p), (C.c_void_p * 3)(*p), (C.c_void_p * 3)(*p), (C.c_void_p * 3)(*p),
                        p[0], 32, 0)
    obs = torch.full((T * N * 272 + 4,), 7.0, device=env.device)
    rew = torch.zeros(T, N, dtype=torch.float64, device=env.device)
    done = torch.zeros(T, N, dtype=torch.uint8, device=env.device)
    out = DockauvRolloutOut(obs.data_ptr(), rew.data_ptr(), done.data_ptr(), *[None] * 5)
    pout = DockauvPolicyOut(buf.data_ptr(), buf.data_ptr(), buf.data_ptr(), None)
    lib = env._lib
    n0 = env.launch_count()
    for hidden in (96, 128):       # n_obs 272: 2 x 272 x 96 floats of layer 0 alone exceed 227 KB
        pol.hidden = hidden
        assert lib.dockauv_rollout_policy(env._handle, C.byref(pol), C.c_void_p(buf.data_ptr()), T, C.byref(out),
                                          C.byref(pout), 1, 0, None) == -1
        assert b"shared memory" in lib.dockauv_last_error()
    torch.cuda.synchronize()
    assert env.launch_count() == n0 and bool((obs == 7.0).all())
    env.close()
    env = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=1, n_synthetic_spheres=3)       # n_obs 36
    env.reset(seed=1)
    n0 = env.launch_count()
    out.obs = obs.data_ptr() + 4        # rows are written with 128-bit stores
    pol.hidden = 64
    assert env._lib.dockauv_rollout_policy(env._handle, C.byref(pol), C.c_void_p(buf.data_ptr()), T, C.byref(out),
                                           C.byref(pout), 1, 0, None) == -1
    assert b"16-byte aligned" in env._lib.dockauv_last_error()
    torch.cuda.synchronize()
    assert env.launch_count() == n0 and bool((obs == 7.0).all())
    env.close()


# ------------------------------------------------------------------------------------------- GPU: the PPO example
@pytest.mark.gpu
def test_ppo_example_fused_captures_once():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "ppo_device_rollout.py"), "--fused", "--iters", "3",
                        "--envs", "4096", "--steps", "16"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("iter")]
    assert len(lines) == 3
    assert all("graph captures 1 " in ln for ln in lines), r.stdout
