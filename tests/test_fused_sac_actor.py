"""Off-policy collection on the device (dockauv_replay_collect): SAC's actor on the tensor cores fills the replay ring.

CPU: every refusal that needs no handle comes before the handle is looked at; the ctypes struct matches the header;
FusedSquashedActor refuses bad layers before any device is touched; the shared-memory size agrees between C and
Python.  GPU: the ring equals an open-loop replay of its own actions through step_into, bit for bit, across layouts,
precisions, vehicles, step parts, scenario banks and start slots; the actor's numerics against a float64 evaluation
with the documented bf16 roundings; determinism and sharding; graphs; launch counts; taps; the SAC example."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.test_fused_policy import _cfg, _pre_step_counters, policy_eps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------- CPU
def _actor_struct(hidden=256, null=(), det=0, ptr=0x10000):
    from gym_dockauv_b200.params import DockauvSquashedActor
    f = lambda k: None if k in null else ptr  # noqa: E731
    return DockauvSquashedActor((C.c_void_p * 2)(f("w0"), f("w1")), (C.c_void_p * 2)(f("b0"), f("b1")), f("mu_w"),
                                f("mu_b"), f("log_std_w"), f("log_std_b"), hidden, det)


def test_refusals_that_need_no_handle_come_first():
    from gym_dockauv_b200 import _capi
    from gym_dockauv_b200.params import DockauvReplayRing
    lib = _capi.load()
    fake = 0x10000

    def call(hidden=256, null=(), actor=True, ring=True, n_slots=16, start_slot=3, n_steps=32):
        a = _actor_struct(hidden, null)
        r = DockauvReplayRing(*[None if k in null else fake for k in ("obs", "terminal_obs", "actions", "reward", "done")])
        rc = lib.dockauv_replay_collect(None, C.byref(a) if actor else None, C.byref(r) if ring else None, n_slots,
                                        start_slot, n_steps, 1, 1, None)
        return rc, lib.dockauv_last_error().decode()

    rc, msg = call()
    assert rc == -1 and "null handle" in msg          # every argument passed: only then is the handle looked at
    for kw, word in ((dict(actor=False), "null argument"), (dict(ring=False), "null argument"),
                     (dict(null=("w0",)), "layer 0"), (dict(null=("b1",)), "layer 1"), (dict(null=("mu_w",)), "mu"),
                     (dict(null=("mu_b",)), "mu"), (dict(null=("log_std_w",)), "log_std"),
                     (dict(null=("log_std_b",)), "log_std"),
                     *[(dict(null=(k,)), "ring buffer") for k in ("obs", "terminal_obs", "actions", "reward", "done")],
                     (dict(hidden=32), "hidden"), (dict(hidden=96), "hidden"), (dict(hidden=512), "hidden"),
                     (dict(n_steps=0), "n_steps"), (dict(n_steps=-4), "n_steps"),
                     (dict(n_slots=1, start_slot=0), "n_slots"), (dict(n_slots=65), "n_slots"),
                     (dict(start_slot=16), "start_slot"), (dict(start_slot=-1), "start_slot")):
        rc, msg = call(**kw)
        assert rc == -1 and word in msg, (kw, msg)
    for hidden in (64, 128, 256):
        assert "null handle" in call(hidden=hidden)[1]
    assert "null handle" in call(n_slots=64, start_slot=63)[1] and "null handle" in call(n_slots=2, start_slot=0)[1]
    assert lib.dockauv_replay_collect_captures(None, None) == -1


def test_struct_matches_the_header(tmp_path):
    """Field offsets and size of DockauvSquashedActor as the C compiler lays them out."""
    from gym_dockauv_b200.params import DockauvSquashedActor
    fields = ["w", "b", "mu_w", "mu_b", "log_std_w", "log_std_b", "hidden", "deterministic"]
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "dockauv.h"', 'int main(void) {',
           'printf("size %zu\\n", sizeof(DockauvSquashedActor));']
    src += [f'printf("{f} %zu\\n", offsetof(DockauvSquashedActor, {f}));' for f in fields]
    src.append("return 0; }")
    (tmp_path / "layout.c").write_text("\n".join(src))
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(ROOT, "include"), str(tmp_path / "layout.c"), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True)
               .stdout.splitlines())
    assert int(got["size"]) == C.sizeof(DockauvSquashedActor)
    assert [f[0] for f in DockauvSquashedActor._fields_] == fields
    for f in fields:
        assert int(got[f]) == getattr(DockauvSquashedActor, f).offset, f


SMEM_SHAPES = [(36, 256, 6), (36, 64, 3), (41, 128, 8), (144, 256, 6), (145, 256, 6), (272, 64, 6)]


def test_smem_size_agrees_between_c_and_python(tmp_path):
    """sac_actor_smem_bytes of dockauv_sac_actor.cuh, compiled by nvcc for the host, against params.py; and the
    refusal boundary: H 256, n_u 6 fits up to 144 observations."""
    from gym_dockauv_b200.build import _nvcc
    from gym_dockauv_b200.params import POLICY_MAX_SMEM, sac_actor_smem_bytes
    src = ['#include <cstdio>', '#include "dockauv_sac_actor.cuh"', 'int main() {']
    src += [f'printf("%zu\\n", dockauv::sac_actor_smem_bytes({a}, {b}, {c}));' for a, b, c in SMEM_SHAPES]
    src += ['printf("%zu\\n", dockauv::kPolicyMaxSmem);', "return 0; }"]
    (tmp_path / "smem.cu").write_text("\n".join(src))
    exe = tmp_path / "smem"
    subprocess.run([_nvcc(), "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I",
                    os.path.join(ROOT, "gym_dockauv_b200", "csrc"), str(tmp_path / "smem.cu"), "-o", str(exe)],
                   check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got[:-1] == [sac_actor_smem_bytes(*s) for s in SMEM_SHAPES]
    assert got[-1] == POLICY_MAX_SMEM
    assert sac_actor_smem_bytes(36, 256, 6) == 182592
    assert sac_actor_smem_bytes(144, 256, 6) <= POLICY_MAX_SMEM < sac_actor_smem_bytes(145, 256, 6)


def _latent(n_obs, H, dtype=None, device="cpu"):
    import torch.nn as nn
    return [nn.Linear(n_obs, H, dtype=dtype, device=device), nn.Linear(H, H, dtype=dtype, device=device)]


def test_fused_squashed_actor_refuses_bad_layers_before_the_device():
    import torch
    from gym_dockauv_b200.policy import FusedSquashedActor

    def heads(H, n_u, dtype=torch.float32):
        return torch.zeros(n_u, H, dtype=dtype), torch.zeros(n_u, dtype=dtype), torch.zeros(n_u, H, dtype=dtype), \
            torch.zeros(n_u, dtype=dtype)
    for H in (32, 96, 512):
        with pytest.raises(ValueError, match="hidden"):
            FusedSquashedActor(_latent(36, H), *heads(H, 6))
    with pytest.raises(ValueError, match="two"):
        FusedSquashedActor(_latent(36, 256)[:1], *heads(256, 6))
    with pytest.raises(ValueError, match="latent_pi layer 1"):
        FusedSquashedActor([_latent(36, 256)[0], torch.nn.Linear(256, 128)], *heads(256, 6))
    with pytest.raises(ValueError, match="mu_weight"):
        FusedSquashedActor(_latent(36, 256), *heads(256, 5))
    mw, mb, lw, lb = heads(256, 6)
    with pytest.raises(ValueError, match="mu_weight"):
        FusedSquashedActor(_latent(36, 256), mw[:, :128], mb, lw, lb)
    with pytest.raises(ValueError, match="log_std_bias"):
        FusedSquashedActor(_latent(36, 256), mw, mb, lw, lb[:5])
    with pytest.raises(ValueError, match="shared memory"):
        FusedSquashedActor(_latent(145, 256), *heads(256, 6))
    with pytest.raises(ValueError, match="float32"):
        FusedSquashedActor(_latent(36, 256, dtype=torch.float64), *heads(256, 6, torch.float64))
    w = torch.zeros(256, 12)
    with pytest.raises(ValueError, match="contiguous"):
        FusedSquashedActor(_latent(36, 256), w.t()[:6], mb, lw, lb)
    with pytest.raises(ValueError, match="CUDA"):            # n_obs 144 fits; CPU tensors are refused next
        FusedSquashedActor(_latent(144, 256), *heads(256, 6))
    # the example's single Linear(H, 2 n_u) head: its row slices are contiguous views
    head = torch.nn.Linear(256, 12)
    with pytest.raises(ValueError, match="CUDA"):
        FusedSquashedActor(_latent(36, 256), head.weight[:6], head.bias[:6], head.weight[6:], head.bias[6:])


# ------------------------------------------------------------------------------------------- GPU helpers
def _env(n_envs=4096, seed=11, max_timesteps=10, vehicle=None, bank=False, **kw):
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.scenario_bank import ScenarioBank
    env = envs.ObstaclesDocking3d(_cfg(max_timesteps=max_timesteps, vehicle=vehicle), num_envs=n_envs, seed=seed, **kw)
    if bank:
        env.set_scenario_bank(ScenarioBank.from_builtin(env, 257, seed=5))
    return env


def _actor(env, H=256, seed=0, log_std_bias=-0.5, deterministic=False):
    """(FusedSquashedActor, modules): torch-default initialisation, log_std bias shifted so the noise matters."""
    import torch
    import torch.nn as nn
    from gym_dockauv_b200.policy import FusedSquashedActor
    torch.manual_seed(seed)
    lat = _latent(env.n_observations, H, device=env.device)
    mu, log_std = nn.Linear(H, env.n_actions, device=env.device), nn.Linear(H, env.n_actions, device=env.device)
    with torch.no_grad():
        log_std.bias.add_(log_std_bias)
    mods = (lat, mu, log_std)
    return FusedSquashedActor(lat, mu.weight, mu.bias, log_std.weight, log_std.bias, deterministic=deterministic), mods


def _ring(buf):
    import torch
    torch.cuda.synchronize()
    return dict(obs=buf.obs.clone(), actions=buf.actions.clone(), rewards=buf.rewards.clone(), dones=buf.dones.clone(),
                terminal_obs=buf.terminal_obs.clone())


def _same_ring(x, y):
    import torch
    for k in ("obs", "actions", "rewards", "dones"):
        assert torch.equal(x[k], y[k]), k
    done = x["dones"].bool()
    assert torch.equal(x["terminal_obs"][done], y["terminal_obs"][done])


# ------------------------------------------------------------------------------------------- GPU: ring = open loop
CASES = {
    "pipeline_f64": dict(n_envs=4096, n_synthetic_spheres=3),
    "pipeline_parts_f32": dict(n_envs=1 << 17, n_synthetic_spheres=3, precision="f32"),
    "warp_rays_f32": dict(n_envs=3000, n_synthetic_spheres=3, layout="warp_rays", precision="f32"),
    "thread_per_env_f64": dict(n_envs=3000, n_synthetic_spheres=3, layout="thread_per_env"),
    "direct_f64": dict(n_envs=4096, n_synthetic_spheres=3, control_mode="direct"),
    "lauv_f64": dict(n_envs=4096, vehicle="LAUV"),
    "lauv_parts_f32": dict(n_envs=1 << 17, precision="f32", vehicle="LAUV"),
    "bank_f64": dict(n_envs=4096, n_synthetic_spheres=3, bank=True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_ring_equals_open_loop_replay(case):
    """collect_fused in calls of 16, 11 and 16 steps on a 16-slot ring (the ring wraps, the third call starts at slot 11,
    max_timesteps 10 forces auto-resets); after each call a twin env with the same seed steps the ring's own actions
    through step_into (DeviceReplayBuffer.collect) into a second ring, which must be identical."""
    import torch
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    S, seed = 16, 11
    a, b = _env(**CASES[case]), _env(**CASES[case])
    assert a.n_actions == {"direct_f64": 8, "lauv_f64": 3, "lauv_parts_f32": 3}.get(case, 6)
    actor, _ = _actor(a)
    ba, bb = DeviceReplayBuffer(a, S), DeviceReplayBuffer(b, S)
    ba.reset_env(seed=seed)
    bb.reset_env(seed=seed)
    n_done = 0
    for T in (16, 11, 16):
        start = ba.t % S
        nxt = ba.collect_fused(actor, T)
        bb.collect(lambda obs: ba.actions[bb.t % S], T)
        assert ba.t == bb.t and a.t_total_steps == b.t_total_steps == ba.t
        assert nxt.data_ptr() == ba.obs[ba.t % S].data_ptr()
        x, y = _ring(ba), _ring(bb)
        _same_ring(x, y)
        slots = [(start + t) % S for t in range(T)]
        n_done += int(x["dones"][slots].sum())
        assert bool(torch.isfinite(x["actions"]).all()) and float(x["actions"].abs().max()) <= 1.0
    assert n_done >= a.num_envs             # every env ended at least one episode
    if CASES[case].get("bank"):
        assert torch.equal(a.bank_row, b.bank_row)
    a.close(); b.close()


# ------------------------------------------------------------------------------------------- GPU: numerics
def _bf16(x):
    import torch
    return x.float().to(torch.bfloat16).double()


def _reference(mods, obs, eps, deterministic):
    """float64 evaluation with the kernel's bf16 roundings: (a, bound).  Each layer's f32 accumulation may differ from
    the exact sum by at most K 2^-22 of the sum of |terms| (generous for the tensor cores' f32 adds); a hidden
    activation then lies between the bf16 roundings of ReLU(p - e) and ReLU(p + e), and that spread goes into the next
    layer's e through |W|.  The epilogue adds f32 rounding (expf, fmaf, tanhf) and the 1e-5 of eps's f32 Box-Muller."""
    import torch
    lat, mu, log_std = mods
    gam = lambda K: K * 2.0 ** -22  # noqa: E731
    h, d = _bf16(obs), torch.zeros_like(obs, dtype=torch.float64)
    for lin in lat:
        w, bias = _bf16(lin.weight.detach()), lin.bias.detach().double()
        p = bias + h @ w.t()
        e = d @ w.abs().t() + gam(w.shape[1] + 1) * (bias.abs() + (h.abs() + d) @ w.abs().t())
        h = _bf16(torch.relu(p))
        lo, hi = _bf16(torch.relu(p - e)), _bf16(torch.relu(p + e))
        d = torch.maximum(hi - h, h - lo)
    outs = []
    for lin in (mu, log_std):
        w, bias = _bf16(lin.weight.detach()), lin.bias.detach().double()
        p = bias + h @ w.t()
        outs.append((p, d @ w.abs().t() + gam(w.shape[1] + 1) * (bias.abs() + (h.abs() + d) @ w.abs().t())))
    (m, em), (ls, els) = outs
    if deterministic:
        u, du = m, em
    else:
        std = ls.clamp(-20, 2).exp()
        u = m + std * eps
        du = em + std * (els.exp() - 1 + 2.0 ** -21) * eps.abs() + std * els.exp() * 1e-5 + 2.0 ** -22 * u.abs()
    return torch.tanh(u), du + 2.0 ** -21


def _f32_torch(mods, obs, eps, deterministic):
    import torch
    lat, mu, log_std = mods
    with torch.no_grad():
        x = torch.relu(lat[1](torch.relu(lat[0](obs))))
        m, ls = mu(x), log_std(x).clamp(-20, 2)
        return torch.tanh(m if deterministic else m + ls.exp() * eps.float())


@pytest.mark.gpu
@pytest.mark.parametrize("H", [64, 256])
def test_actor_numerics_against_float64(H):
    """Deterministic and stochastic actions on the ring's own observations against the float64 evaluation with the
    documented bf16 roundings, within the bound derived from them; the gap to a plain f32 PyTorch evaluation is printed
    (the cost of bf16), not asserted."""
    import torch
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    T, N, seed = 8, 8192, 3
    env = _env(n_envs=N, seed=seed, max_timesteps=6, n_synthetic_spheres=3)
    buf = DeviceReplayBuffer(env, T + 1)
    for deterministic in (True, False):
        actor, mods = _actor(env, H=H, seed=7, deterministic=deterministic)
        buf.reset_env(seed=seed)
        ep0, t0 = env.episode.clone(), env.t_steps.clone()
        buf.collect_fused(actor, T)
        torch.cuda.synchronize()
        obs, got = buf.obs[:T], buf.actions[:T].double()
        if deterministic:
            eps = torch.zeros(T, N, env.n_actions, dtype=torch.float64, device=env.device)
        else:
            pe, pt = _pre_step_counters(ep0, t0, buf.dones[:T])
            eps = torch.as_tensor(policy_eps(seed, np.tile(np.arange(N), T), pe.cpu().numpy().ravel(),
                                             pt.cpu().numpy().ravel(), env.n_actions),
                                  device=env.device).reshape(T, N, env.n_actions)
        ref, bound = _reference(mods, obs, eps, deterministic)
        err = (got - ref).abs()
        f32_gap = float((got - _f32_torch(mods, obs, eps, deterministic).double()).abs().max())
        print(f"H {H} deterministic {deterministic}: max |a - ref| {float(err.max()):.3g} (bound max "
              f"{float(bound.max()):.3g}, median {float(bound.median()):.3g}); max |a - f32 torch| {f32_gap:.3g}")
        assert bool((err <= bound).all()), float((err - bound).max())
        assert float(bound.median()) < 1e-2           # the bound stays well below the bf16 spacing of |a| ~ 1
        assert int(buf.dones[:T].sum()) > 0
    env.close()


# ------------------------------------------------------------------------------------------- GPU: determinism
@pytest.mark.gpu
def test_reset_reproduces_and_sharding_does_not_matter():
    """reset(seed) + collect_fused reproduces the ring bit for bit; a 2M-env handle (stepped in two parts) writes the
    same actions as two M-env handles with env_id0 = 0 and M."""
    import torch
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    M, S, T = 1 << 16, 8, 12
    big = _env(n_envs=2 * M, seed=4, max_timesteps=7, n_synthetic_spheres=3)
    actor, _ = _actor(big)
    buf = DeviceReplayBuffer(big, S)
    runs = []
    for s in (4, 4):
        buf.reset_env(seed=s)
        buf.collect_fused(actor, T)
        runs.append(_ring(buf))
    _same_ring(runs[0], runs[1])
    for part, id0 in ((0, 0), (1, M)):
        small = _env(n_envs=M, seed=4, max_timesteps=7, env_id0=id0, n_synthetic_spheres=3)
        act, _ = _actor(small)
        sb = DeviceReplayBuffer(small, S)
        sb.reset_env(seed=4)
        sb.collect_fused(act, T)
        torch.cuda.synchronize()
        half = {k: v[:, part * M:(part + 1) * M] for k, v in runs[0].items()}
        assert torch.equal(sb.actions, half["actions"]), part
        _same_ring(_ring(sb), half)
        small.close()
    big.close()


# ------------------------------------------------------------------------------------------- GPU: graphs, launches, taps
@pytest.mark.gpu
def test_graphs():
    """T = S replays one graph; after an in-place optimizer step the replay equals a use_graph=False call; a new start
    slot or a deterministic actor captures anew, within the cache of four; the step graphs are not touched."""
    import torch
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    S, seed = 8, 9
    env = _env(n_envs=4096, seed=seed, max_timesteps=8, n_synthetic_spheres=3)
    actor, mods = _actor(env)
    buf = DeviceReplayBuffer(env, S)
    sg0 = env.step_graph_captures()
    buf.reset_env(seed=seed)
    for _ in range(3):
        buf.collect_fused(actor, S)
    assert buf.collect_captures() == 1

    def run(a, use_graph=True):
        buf.reset_env(seed=seed)
        buf.collect_fused(a, S, use_graph=use_graph)
        return _ring(buf)
    first = run(actor)
    lat, mu, log_std = mods
    params = [p for m in (*lat, mu, log_std) for p in m.parameters()]
    opt = torch.optim.SGD(params, lr=0.05)
    x = torch.randn(64, env.n_observations, device=env.device)
    h = torch.relu(lat[1](torch.relu(lat[0](x))))
    (mu(h).pow(2).sum() + log_std(h).sum()).backward()
    opt.step()
    replay = run(actor)
    assert buf.collect_captures() == 1
    plain = run(actor, use_graph=False)
    assert not torch.equal(replay["actions"], first["actions"])
    _same_ring(replay, plain)
    buf.reset_env(seed=seed)
    buf.collect_fused(actor, 3)                # (s0 0, T 3): new
    buf.collect_fused(actor, S)                # (s0 3, T S): new
    assert buf.collect_captures() == 3
    evaluation = type(actor)(lat, mu.weight, mu.bias, log_std.weight, log_std.bias, deterministic=True)
    for _ in range(2):
        ev = run(evaluation)
        tr = run(actor)
    assert buf.collect_captures() == 4
    _same_ring(tr, plain)
    assert not torch.equal(ev["actions"], tr["actions"])
    assert env.step_graph_captures() == sg0
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("N,ranges", [(4096, 1), (1 << 17, 2)])
def test_launch_count(N, ranges):
    """The fused collection of T steps launches exactly T actor kernels per env range more than the open-loop rollout."""
    import torch
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    T = 6
    env = _env(n_envs=N, seed=1, max_timesteps=400, n_synthetic_spheres=3)
    env.reset(seed=1)
    obs = torch.zeros(T, N, env.n_observations, device=env.device)
    rew = torch.zeros(T, N, dtype=env.dtype, device=env.device)
    done = torch.zeros(T, N, dtype=torch.uint8, device=env.device)
    n0 = env.launch_count()
    env.rollout(torch.zeros(T, N, env.n_actions, device=env.device), obs, rew, done, use_graph=False)
    open_loop = env.launch_count() - n0
    actor, _ = _actor(env)
    buf = DeviceReplayBuffer(env, 8)
    buf.reset_env(seed=1)
    for use_graph in (False, True, True):
        n0 = env.launch_count()
        buf.collect_fused(actor, T, use_graph=use_graph)
        assert env.launch_count() - n0 == open_loop + ranges * T, use_graph
    torch.cuda.synchronize()
    env.close()


@pytest.mark.gpu
def test_taps_leave_the_ring_unchanged():
    """With 64 taps set the ring is identical to the untapped run, and the tap ring advances by T."""
    import torch
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    S, T, seed = 16, 20, 5
    env = _env(n_envs=4096, seed=seed, max_timesteps=8, n_synthetic_spheres=3)
    actor, _ = _actor(env)
    buf = DeviceReplayBuffer(env, S)
    buf.reset_env(seed=seed)
    buf.collect_fused(actor, T)
    plain = _ring(buf)
    taps = env.set_taps(list(range(0, 4096, 64)), capacity=64)
    for use_graph in (True, False):
        buf.reset_env(seed=seed)
        buf.collect_fused(actor, T, use_graph=use_graph)
        _same_ring(_ring(buf), plain)
    assert int(taps["count"][0]) == 2 * T
    env.clear_taps()
    torch.cuda.synchronize()
    env.close()


@pytest.mark.gpu
def test_refusals_with_a_handle_touch_nothing():
    """Weights too large for shared memory (n_obs 272) and misaligned ring rows are refused before any launch."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG
    from gym_dockauv_b200.params import DockauvReplayRing
    cfg = dict(BASE_CONFIG)
    deg = np.pi / 180
    cfg["radar"] = dict(freq=1, alpha=75 * deg, beta=75 * deg, ray_per_deg=5 * deg, max_dist=10, blocksize_reduce=1)
    env = envs.ObstaclesDocking3d(cfg, num_envs=256, seed=1)
    assert env.n_observations == 272
    env.reset(seed=1)
    buf = torch.full((1 << 20,), 7.0, device=env.device)
    p = buf.data_ptr()
    ring = DockauvReplayRing(p, p, p, p, p)
    n0 = env.launch_count()
    for hidden in (256,):                   # 2 x 256 x 280 bf16 of layer 0 and 2 x 256 x 264 of layer 1 exceed 227 KB
        a = _actor_struct(hidden, ptr=p)
        assert env._lib.dockauv_replay_collect(env._handle, C.byref(a), C.byref(ring), 4, 0, 4, 1, 0, None) == -1
        assert b"shared memory" in env._lib.dockauv_last_error()
    torch.cuda.synchronize()
    assert env.launch_count() == n0 and bool((buf == 7.0).all())
    env.close()
    env = _env(n_envs=256, seed=1)          # n_obs 36
    env.reset(seed=1)
    n0 = env.launch_count()
    ring.terminal_obs = p + 4               # rows are written with 128-bit stores
    a = _actor_struct(256, ptr=p)
    assert env._lib.dockauv_replay_collect(env._handle, C.byref(a), C.byref(ring), 4, 0, 4, 1, 0, None) == -1
    assert b"16-byte aligned" in env._lib.dockauv_last_error()
    torch.cuda.synchronize()
    assert env.launch_count() == n0 and bool((buf == 7.0).all())
    env.close()


# ------------------------------------------------------------------------------------------- GPU: the SAC example
@pytest.mark.gpu
def test_sac_example_fused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "sac_device_replay.py"), "--fused", "--envs",
                        "2048", "--iters", "2"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("iter")]
    assert len(lines) == 2, r.stdout
    for ln in lines:
        assert "nan" not in ln.lower() and "inf" not in ln.lower(), ln
        assert "env-steps/s" in ln and "q-loss" in ln, ln
