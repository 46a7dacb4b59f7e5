"""The two networks evaluated inside the rollouts, fed caller-chosen observations, against float64 at every
instantiation: policy_kernel<H, NU> (dockauv_policy.cuh, PPO's actor-critic in f32) and sac_actor_kernel<H, NU>
(dockauv_sac_actor.cuh, SAC's actor on bf16 tensor cores).

Each case is one handle and one T = 1 call per weight variant and mode: the kernel acts on exactly the rows the test wrote (obs0 of
rollout_policy, the ring slot of collect_fused).  The cases cover every (H, n_u) the host code dispatches, and every H
with an observation width that is not a multiple of 16 (SAC's zero-padded layer-0 columns), one that is not a multiple
of 4 (SAC's scalar W0 staging and the k < n_obs guard inside a 16-column chunk) and the largest the shared memory
takes.  Rows are uniform, all-zero (the reset observation), one-hot per column (a misplaced W0 column shows in the one
row that reads it) and scaled to +-8; weights are torch's default or scaled to O(3) pre-activations (tanh saturates,
ReLU and tanh switch units off).  Batches of 1, 5, 17 and 4099 envs and one of 2^17 + 5 stepped in two parts end in
partial tiles; one case per kernel puts the noise counters in their high words.

CPU: the case table against the radar geometry, the shared-memory sizes and the instantiations of dockauv_capi.cu;
the references and bounds on CPU tensors.  GPU: actions, values, last values and log-probs within the derived bounds;
SAC rows independent of their position; the networks independent of the env's precision."""
import os
import re

import numpy as np
import pytest

from tests.test_fused_policy import _Rollout, _cfg, _eval, _layers, policy_eps
from tests.test_fused_sac_actor import _latent, _reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U32 = 2.0 ** -24            # unit roundoff of float32
TANHF = 2 * 2.0 ** -23      # tanhf: at most 2 ulp of its result (CUDA C++ Programming Guide, single-precision functions)
EXPF = 2 * 2.0 ** -23       # expf: at most 2 ulp
EPS_F32 = 1e-5              # the f32 Box-Muller noise against policy_eps (asserted below)

# n_obs: (alpha, beta, ray_per_deg in degrees, blocksize_reduce); n_obs = 16 + the pooled ray count
RADARS = {20: (10, 10, 10, 1), 25: (70, 70, 10, 3), 32: (70, 70, 10, 2), 36: (60, 80, 10, 2), 79: (60, 80, 5, 2),
          92: (30, 180, 10, 1), 144: (70, 150, 10, 1), 272: (150, 150, 10, 1)}
BIG = (1 << 17) + 5         # stepped in two 4096-aligned parts; the second ends in a partial tile of 5 envs

# name: H, n_u (3 LAUV, 6 BlueROV2, 8 BlueROV2 direct), n_obs; N (4099), unaligned (every parameter a view at a storage
# offset of one float), counters (noise counters in their high words), precision (f64).  Every case runs both weight
# variants (WEIGHTS) in both modes.
PPO_CASES = {
    "h32_lauv_25": dict(H=32, n_u=3, n_obs=25),
    "h32_rov_272": dict(H=32, n_u=6, n_obs=272),
    "h32_direct_36_counters": dict(H=32, n_u=8, n_obs=36, N=17, counters=True),
    "h64_lauv_272": dict(H=64, n_u=3, n_obs=272),
    "h64_rov_36": dict(H=64, n_u=6, n_obs=36),
    "h64_direct_79": dict(H=64, n_u=8, n_obs=79),
    "h64_rov_36_unaligned": dict(H=64, n_u=6, n_obs=36, unaligned=True),
    "h64_rov_36_big_f32": dict(H=64, n_u=6, n_obs=36, N=BIG, precision="f32"),
    "h96_lauv_144": dict(H=96, n_u=3, n_obs=144),
    "h96_rov_20": dict(H=96, n_u=6, n_obs=20, N=5),
    "h96_direct_25": dict(H=96, n_u=8, n_obs=25),
    "h128_lauv_79": dict(H=128, n_u=3, n_obs=79),
    "h128_rov_32": dict(H=128, n_u=6, n_obs=32, N=1),
    "h128_direct_92": dict(H=128, n_u=8, n_obs=92),
}
SAC_CASES = {
    "h64_lauv_272": dict(H=64, n_u=3, n_obs=272),
    "h64_rov_25": dict(H=64, n_u=6, n_obs=25),
    "h64_direct_36_counters": dict(H=64, n_u=8, n_obs=36, N=17, counters=True),
    "h64_rov_79_unaligned": dict(H=64, n_u=6, n_obs=79, unaligned=True),
    "h128_lauv_20": dict(H=128, n_u=3, n_obs=20, N=5),
    "h128_rov_79": dict(H=128, n_u=6, n_obs=79),
    "h128_direct_272": dict(H=128, n_u=8, n_obs=272),
    "h128_direct_25_unaligned": dict(H=128, n_u=8, n_obs=25, unaligned=True),
    "h256_lauv_36": dict(H=256, n_u=3, n_obs=36),
    "h256_lauv_79_unaligned": dict(H=256, n_u=3, n_obs=79, unaligned=True),
    "h256_rov_144": dict(H=256, n_u=6, n_obs=144),
    "h256_rov_36_big_f32": dict(H=256, n_u=6, n_obs=36, N=BIG, precision="f32"),
    "h256_direct_25": dict(H=256, n_u=8, n_obs=25, N=1),
}
WEIGHTS = ("torch", "scaled")
COUNTER_SEED, COUNTER_ID0 = 0x9E3779B97F4A7C15, (1 << 32) - 8     # both seed halves set; ids 8.. cross 2^32


def _radar(n_obs):
    alpha, beta, step, block = RADARS[n_obs]
    deg = np.pi / 180
    return dict(freq=1, alpha=alpha * deg, beta=beta * deg, ray_per_deg=step * deg, max_dist=10, blocksize_reduce=block)


def _case_cfg(c):
    cfg = _cfg(vehicle="LAUV" if c["n_u"] == 3 else None)
    cfg["radar"] = _radar(c["n_obs"])
    return cfg, ("direct" if c["n_u"] == 8 else "joystick")


# ------------------------------------------------------------------------------------------- inputs
def _rows(N, n_obs, device="cpu", seed=0):
    """N observation rows: uniform in [-1, 1], then one all-zero row, four rows scaled to +-8 (three uniform in [-8, 8],
    one of signs), one one-hot row per column, uniform after that; a batch shorter than that takes the first N."""
    import torch
    g = torch.Generator().manual_seed(seed)
    uni = lambda n: 2 * torch.rand(n, n_obs, generator=g, dtype=torch.float64) - 1  # noqa: E731
    rows = torch.cat([uni(4), torch.zeros(1, n_obs, dtype=torch.float64), 8 * uni(3), 8 * torch.sign(uni(1)),
                      torch.eye(n_obs, dtype=torch.float64)])
    rows = torch.cat([rows, uni(max(N - rows.shape[0], 0))])[:N]
    return rows.float().to(device)


def _calibration_rows(n_obs, device):
    import torch
    g = torch.Generator().manual_seed(1234)
    return (2 * torch.rand(256, n_obs, generator=g) - 1).to(device)


def _scale_hidden(layers, act, x):
    """Scales the weight and bias of each layer so that its pre-activations on the rows x have an RMS of 3."""
    import torch
    with torch.no_grad():
        h = x.double()
        for lin in layers:
            p = torch.nn.functional.linear(h, lin.weight.double(), lin.bias.double())
            s = 3.0 / float(p.pow(2).mean().sqrt())
            lin.weight.mul_(s)
            lin.bias.mul_(s)
            h = act(p * s)


def _unaligned(t):
    """A contiguous copy of t at a storage offset of one float: 4 bytes past a 16-byte boundary."""
    import torch
    flat = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    flat[1:].copy_(t.reshape(-1))
    v = flat[1:].view(t.shape)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4
    return v


def _ppo_mods(c, w, device, seed=7):
    """(pi, vf, log_std) of a case: torch-default layers, optionally scaled; log_std spread over [-5, 1.5]."""
    import torch
    import torch.nn as nn
    torch.manual_seed(seed)
    pi, vf = _layers(c["n_obs"], c["H"], c["n_u"], device=device)
    if w == "scaled":
        x = _calibration_rows(c["n_obs"], device)
        _scale_hidden(pi[:2], torch.tanh, x)
        _scale_hidden(vf[:2], torch.tanh, x)
    log_std = nn.Parameter(torch.linspace(-5, 1.5, c["n_u"], device=device))
    if c.get("unaligned"):
        for p in [q for lin in pi + vf for q in (lin.weight, lin.bias)] + [log_std]:
            p.data = _unaligned(p.data)
    return pi, vf, log_std


def _sac_latent64(lat, x):
    import torch
    h = x.double()
    for lin in lat:
        h = torch.relu(_linear64(h, lin))
    return h


def _sac_mods(c, w, device, seed=7):
    """(latent_pi, mu, log_std) of a case: torch-default layers, optionally scaled; the log_std head set so that its
    pre-clamp values on uniform rows spread +-2.5 around centres from -26 to 4, across both clamp bounds."""
    import torch
    import torch.nn as nn
    torch.manual_seed(seed)
    H, n_u = c["H"], c["n_u"]
    lat = _latent(c["n_obs"], H, device=device)
    mu, log_std = nn.Linear(H, n_u, device=device), nn.Linear(H, n_u, device=device)
    x = _calibration_rows(c["n_obs"], device)
    with torch.no_grad():
        if w == "scaled":      # ReLU is positively homogeneous: mu's head takes the latent's scale back out
            rms = lambda: float(_linear64(_sac_latent64(lat, x), mu).pow(2).mean().sqrt())  # noqa: E731
            mu0 = rms()
            _scale_hidden(lat, torch.relu, x)
            mu.weight.mul_(mu0 / rms())
        z = _sac_latent64(lat, x) @ log_std.weight.double().t()
        s = 2.5 / z.std(0)
        log_std.weight.mul_(s[:, None].float())
        log_std.bias.copy_(torch.linspace(-26, 4, n_u, dtype=torch.float64, device=device) - (z * s).mean(0))
    if c.get("unaligned"):
        for p in [q for lin in (*lat, mu, log_std) for q in (lin.weight, lin.bias)]:
            p.data = _unaligned(p.data)
    return lat, mu, log_std


def _linear64(h, lin):
    import torch
    return torch.nn.functional.linear(h, lin.weight.detach().double(), lin.bias.detach().double())


def _sac_log_std_pre_clamp(mods, obs):
    lat, _, log_std = mods
    return _linear64(_sac_latent64(lat, obs), log_std)


def _assert_clamp_sides_hit(ls):
    """Some (env, action) pair below -20, some between the bounds, some above 2, each by a margin of 0.5."""
    assert bool((ls < -20.5).any()) and bool(((ls > -19.5) & (ls < 1.5)).any()) and bool((ls > 2.5).any()), \
        (float(ls.min()), float(ls.max()))


# ------------------------------------------------------------------------------------------- PPO bound
def _ppo_bound(mods, obs):
    """Elementwise bounds on |policy_kernel - _eval(float64)| of the means and values.  A layer of K inputs is an f32
    fma chain from the bias: at most (K + 1) 2^-24 (|b| + |W| |h|) from the exact sum; the error d of its input adds
    |W| d.  tanh is increasing, so a pre-activation within e of p gives tanh within max(tanh(p + e) - tanh(p),
    tanh(p) - tanh(p - e)) <= e of tanh(p) (a saturated unit passes almost none of e on); tanhf adds 2 ulp of its
    result."""
    import torch
    pi, vf, _ = mods

    def net(layers):
        h = obs.double()
        d = torch.zeros_like(h)
        for k, lin in enumerate(layers):
            w, b = lin.weight.detach().double(), lin.bias.detach().double()
            p = b + h @ w.t()
            e = d @ w.abs().t() + (w.shape[1] + 1) * U32 * (b.abs() + (h.abs() + d) @ w.abs().t())
            if k == 2:
                return e
            h = torch.tanh(p)
            d = torch.maximum(torch.tanh(p + e) - h, h - torch.tanh(p - e))
            d = d + TANHF * (h.abs() + d)
    return net(pi), net(vf)[..., 0]


def _stochastic_bound(bmu, std, eps, a):
    """a = fmaf(expf(log_std), eps_f32, mu_f32), one rounding: the mean's bound, std |eps_f32 - eps|, the expf error on
    |eps_f32| and the rounding of a."""
    return bmu + std * (EPS_F32 + EXPF * (eps.abs() + EPS_F32)) + 2.0 ** -23 * a.abs()


# ------------------------------------------------------------------------------------------- CPU
def _dispatched(src, fn_h, fn_hu):
    """(H, n_u) pairs a launch switch instantiates: `case H: err = fn_h<H>` x `case n: return fn_hu<H, n>`."""
    hs = re.findall(rf"case (\d+): err = {fn_h}<(\d+)>", src)
    nus = re.findall(rf"case (\d+): return {fn_hu}<H, (\d+)>", src)
    assert hs and nus and all(a == b for a, b in hs + nus), (hs, nus)
    return {(int(h), int(n)) for h, _ in hs for n, _ in nus}


def test_case_tables_match_the_code():
    """Each radar gives its n_obs and each vehicle its n_u; each case fits the shared memory, and each H reaches the
    largest table width that fits, one not a multiple of 16 and one not a multiple of 4 (with 4099 envs, so that every
    column gets its one-hot row); the (H, n_u) pairs are those dockauv_capi.cu instantiates; the batch sizes, unaligned
    parameters and noise counters are all there."""
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    from gym_dockauv_b200.params import POLICY_MAX_SMEM, pack_params, policy_smem_bytes, sac_actor_smem_bytes
    for n_obs in RADARS:
        for n_u in (3, 6, 8):
            cfg, mode = _case_cfg(dict(n_obs=n_obs, n_u=n_u))
            _, meta = pack_params(cfg, "ObstaclesDocking3d", control_mode=mode)
            assert (meta["n_obs"], meta["n_u"]) == (n_obs, n_u)
    for n_obs, radar in ((32, RADAR_64), (36, BASE_CONFIG["radar"])):
        assert all(np.isclose(_radar(n_obs)[k], radar[k]) for k in ("alpha", "beta", "ray_per_deg", "blocksize_reduce"))
    assert policy_smem_bytes(92, 128, 8) == 232016 and sac_actor_smem_bytes(144, 256, 6) == 231744
    with open(os.path.join(ROOT, "gym_dockauv_b200", "csrc", "dockauv_capi.cu")) as f:
        src = f.read()
    for cases, smem, fn_h, fn_hu in ((PPO_CASES, policy_smem_bytes, "launch_policy_h", "launch_policy_hu"),
                                     (SAC_CASES, sac_actor_smem_bytes, "launch_sac_actor_h", "launch_sac_actor_hu")):
        assert {(c["H"], c["n_u"]) for c in cases.values()} == _dispatched(src, fn_h, fn_hu)
        for c in cases.values():
            assert smem(c["n_obs"], c["H"], c["n_u"]) <= POLICY_MAX_SMEM, c
        for H in {c["H"] for c in cases.values()}:
            mine = [c for c in cases.values() if c["H"] == H]
            assert max(c["n_obs"] for c in mine) == max(n for n in RADARS if smem(n, H, 8) <= POLICY_MAX_SMEM), H
            assert any(c["n_obs"] % 16 and c.get("N", 4099) >= 4099 for c in mine), H
            assert any(c["n_obs"] % 4 and c.get("N", 4099) >= 4099 for c in mine), H
        assert {c.get("N", 4099) for c in cases.values()} == {1, 5, 17, 4099, BIG}
        assert any(c.get("counters") and c.get("N") == 17 for c in cases.values())
    assert {c["H"] for c in SAC_CASES.values() if c.get("unaligned")} == {64, 128, 256}
    assert any(c.get("unaligned") for c in PPO_CASES.values())


def test_references_and_bounds_on_the_cpu():
    """At the smallest width, both weight variants: the PPO bound holds for torch's own float32 evaluation (another f32
    implementation of the same sums) and its median stays small; the scaled weights saturate tanh; the SAC reference
    and its bound run in both modes with the noise of the counter case, and the bound's median stays small; the
    log_std head reaches every side of both clamp bounds; the unaligned views hold the same values."""
    import torch
    N, n_obs = 4099, 20
    obs = _rows(N, n_obs)
    assert bool((obs[4] == 0).all()) and float(obs[5:9].abs().max()) > 4
    assert torch.equal(obs[9:9 + n_obs], torch.eye(n_obs)) and torch.equal(_rows(17, n_obs), obs[:17])
    gids = np.arange(N, dtype=np.uint64) + np.uint64(COUNTER_ID0)
    ep = (0x80000000 + np.arange(N)) & 0xFFFFFFFF
    eps = torch.as_tensor(policy_eps(COUNTER_SEED, gids, ep, (1 << 29) | np.arange(N), 8))
    c = dict(H=32, n_u=8, n_obs=n_obs)
    for w in WEIGHTS:
        mods = _ppo_mods(c, w, "cpu")
        mu64, v64 = _eval(mods, obs, torch.float64)
        mu32, v32 = _eval(mods, obs, torch.float32)
        bmu, bv = _ppo_bound(mods, obs)
        assert bool(((mu32.double() - mu64).abs() <= bmu).all()) and bool(((v32.double() - v64).abs() <= bv).all())
        assert float(bmu.median()) < 1e-3 and float(bv.median()) < 1e-3
        saturated = float((_linear64(obs[9 + n_obs:].double(), mods[0][0]).abs() > 3).double().mean())
        assert (saturated > 0.1) == (w == "scaled"), saturated          # on the uniform rows
        ua = _ppo_mods(dict(c, unaligned=True), w, "cpu")
        assert all(torch.equal(x.weight, y.weight) and x.weight.data_ptr() % 16 == 4 for x, y in zip(ua[0], mods[0]))
        mods = _sac_mods(dict(c, H=64), w, "cpu")
        _assert_clamp_sides_hit(_sac_log_std_pre_clamp(mods, obs))
        for deterministic in (True, False):
            ref, bound = _reference(mods, obs, torch.zeros_like(eps) if deterministic else eps, deterministic)
            assert bool(torch.isfinite(ref).all()) and float(ref.abs().max()) <= 1
            assert float(bound.median()) < 1e-2, float(bound.median())


# ------------------------------------------------------------------------------------------- GPU helpers
def _case_env(c, precision=None):
    """(handle of the case, its seed), reset."""
    from gym_dockauv_b200 import envs
    cfg, mode = _case_cfg(c)
    seed, id0 = (COUNTER_SEED, COUNTER_ID0) if c.get("counters") else (3, 0)
    env = envs.ObstaclesDocking3d(cfg, num_envs=c.get("N", 4099), seed=seed, env_id0=id0, control_mode=mode,
                                  precision=precision or c.get("precision", "f64"), n_synthetic_spheres=3)
    assert (env.n_observations, env.n_actions) == (c["n_obs"], c["n_u"])
    env.reset(seed=seed)
    return env, seed


def _counters(env, c):
    """For the counter case, episodes >= 2^31 as uint32 and t_steps with bit 29 set, written in place; then the
    (episode, t_steps) the next call reads."""
    import torch
    if c.get("counters"):
        k = torch.arange(env.num_envs, dtype=torch.int64, device=env.device)
        ep = (0x80000000 + 0x01000193 * k) % (1 << 32)
        env.episode.copy_(torch.where(ep >= 1 << 31, ep - (1 << 32), ep).to(torch.int32))
        env.t_steps.copy_(((1 << 29) | (37 * k) % 1000).to(torch.int32))
        assert bool((env.episode < 0).all())
    return env.episode.clone(), env.t_steps.clone()


def _noise(env, seed, c, ep, t):
    import torch
    gids = np.arange(env.num_envs, dtype=np.uint64) + np.uint64(COUNTER_ID0 if c.get("counters") else 0)
    return torch.as_tensor(policy_eps(seed, gids, ep.cpu().numpy(), t.cpu().numpy(), env.n_actions), device=env.device)


def _ppo_call(env, c, policy, obs):
    import torch
    r = _Rollout(env, 1)
    r.obs0.copy_(obs)
    ep, t = _counters(env, c)
    r.run(env, policy, use_graph=False)
    torch.cuda.synchronize()
    return r, ep, t


def _sac_call(buf, c, actor, obs):
    import torch
    s = buf.t % buf.n_slots
    buf.obs[s].copy_(obs)
    ep, t = _counters(buf.env, c)
    buf.collect_fused(actor, 1, use_graph=False)
    torch.cuda.synchronize()
    return buf.actions[s].clone(), ep, t


def _report(case, what, err, bound):
    print(f"{case} {what}: max err {float(err.max()):.3g}, max bound {float(bound.max()):.3g}, "
          f"max err/bound {float((err / bound.clamp_min(1e-30)).max()):.3g}")


# ------------------------------------------------------------------------------------------- GPU: PPO
@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(PPO_CASES))
def test_policy_kernel_against_float64(case):
    """Both weight variants, deterministic and stochastic: means (the deterministic actions), stochastic actions,
    values and last_values within _ppo_bound of _eval in float64, the bound's median small; the kernel's eps,
    recovered from the two runs, within 1e-5 of policy_eps (beyond the recovery's own rounding); log-probs within
    1e-4."""
    import torch
    from gym_dockauv_b200.policy import FusedActorCritic
    c = PPO_CASES[case]
    env, seed = _case_env(c)
    obs = _rows(env.num_envs, c["n_obs"], env.device)
    for w in WEIGHTS:
        mods = _ppo_mods(c, w, env.device)
        ls = mods[2].detach().double()
        std = ls.exp()
        mu64, v64 = _eval(mods, obs, torch.float64)
        bmu, bv = _ppo_bound(mods, obs)
        assert float(bmu.median()) < 1e-2 and float(bv.median()) < 1e-2
        for deterministic in (True, False):
            r, ep, t = _ppo_call(env, c, FusedActorCritic(*mods, deterministic=deterministic), obs)
            a, v, lp = r.actions[0].double(), r.values[0].double(), r.log_probs[0].double()
            if deterministic:
                eps, ref, bound = torch.zeros_like(mu64), mu64, bmu
                mean, values = a, r.values[0].clone()
            else:
                eps = _noise(env, seed, c, ep, t)
                ref = mu64 + std * eps
                bound = _stochastic_bound(bmu, std, eps, a)
                eps_kernel = (a - mean) / std        # a - mu_f32 is exact in float64
                slack = EXPF * (eps.abs() + EPS_F32) + 2.0 ** -23 * a.abs() / std
                assert float(((eps_kernel - eps).abs() - slack).max()) < EPS_F32
                assert torch.equal(r.values[0], values)
            err = (a - ref).abs()
            _report(case, f"{w} deterministic {deterministic} actions", err, bound)
            assert bool((err <= bound).all()), float((err - bound).max())
            verr = (v - v64).abs()
            assert bool((verr <= bv).all()), float((verr - bv).max())
            lp_ref = (-0.5 * eps * eps - ls - 0.5 * np.log(2 * np.pi)).sum(-1)
            assert float((lp - lp_ref).abs().max()) < 1e-4
            _, lv64 = _eval(mods, r.obs[0], torch.float64)
            _, blv = _ppo_bound(mods, r.obs[0])
            lverr = (r.last_values.double() - lv64).abs()
            assert bool((lverr <= blv).all()), float((lverr - blv).max())
        _report(case, f"{w} values", verr, bv)
        _report(case, f"{w} last values", lverr, blv)
    env.close()


# ------------------------------------------------------------------------------------------- GPU: SAC
@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(SAC_CASES))
def test_sac_actor_kernel_against_float64(case):
    """Both weight variants, deterministic and stochastic: actions within the bound of _reference (float64 with the
    kernel's bf16 roundings), the bound's median small; with 4099 envs or more the log_std head crosses both clamp
    bounds."""
    import torch
    from gym_dockauv_b200.policy import FusedSquashedActor
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    c = SAC_CASES[case]
    env, seed = _case_env(c)
    buf = DeviceReplayBuffer(env, 2)
    obs = _rows(env.num_envs, c["n_obs"], env.device)
    for w in WEIGHTS:
        mods = _sac_mods(c, w, env.device)
        lat, mu, log_std = mods
        if env.num_envs >= 4099:
            _assert_clamp_sides_hit(_sac_log_std_pre_clamp(mods, obs))
        for deterministic in (True, False):
            actor = FusedSquashedActor(lat, mu.weight, mu.bias, log_std.weight, log_std.bias,
                                       deterministic=deterministic)
            a, ep, t = _sac_call(buf, c, actor, obs)
            eps = torch.zeros(env.num_envs, env.n_actions, dtype=torch.float64, device=env.device) if deterministic \
                else _noise(env, seed, c, ep, t)
            ref, bound = _reference(mods, obs, eps, deterministic)
            err = (a.double() - ref).abs()
            _report(case, f"{w} deterministic {deterministic}", err, bound)
            assert bool((err <= bound).all()), float((err - bound).max())
            assert float(bound.median()) < 1e-2          # the bound stays well below the bf16 spacing of |a| ~ 1
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("H", [64, 128, 256])
def test_sac_rows_do_not_depend_on_their_position(H):
    """The deterministic actor on 4099 rows (a partial last tile) and on a random permutation of them: the actions
    permute bit for bit; 4099 copies of one row give that row's action in every env, bit for bit."""
    import torch
    from gym_dockauv_b200.policy import FusedSquashedActor
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    c = dict(H=H, n_u=6, n_obs=25)
    env, _ = _case_env(c)
    buf = DeviceReplayBuffer(env, 2)
    lat, mu, log_std = _sac_mods(c, "torch", env.device)
    actor = FusedSquashedActor(lat, mu.weight, mu.bias, log_std.weight, log_std.bias, deterministic=True)
    obs = _rows(env.num_envs, c["n_obs"], env.device)
    perm = torch.randperm(env.num_envs, generator=torch.Generator().manual_seed(5)).to(env.device)
    a, _, _ = _sac_call(buf, c, actor, obs)
    b, _, _ = _sac_call(buf, c, actor, obs[perm])
    assert torch.equal(b, a[perm])
    for row in (6, 4098):                            # a +-8 row; the last row of the partial tile
        same, _, _ = _sac_call(buf, c, actor, obs[row].expand_as(obs).contiguous())
        assert torch.equal(same, a[row].expand_as(same))
    env.close()


@pytest.mark.gpu
def test_networks_do_not_depend_on_the_env_precision():
    """The same observations and weights on an f64 and an f32 handle (same seed and counters): bit-equal stochastic
    actions of both kernels, and bit-equal PPO values and log-probs."""
    import torch
    from gym_dockauv_b200.policy import FusedActorCritic, FusedSquashedActor
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    c = dict(H=64, n_u=6, n_obs=36)
    out = []
    for precision in ("f64", "f32"):
        env, seed = _case_env(c, precision)
        obs = _rows(env.num_envs, c["n_obs"], env.device)
        r, _, _ = _ppo_call(env, c, FusedActorCritic(*_ppo_mods(c, "scaled", env.device)), obs)
        buf = DeviceReplayBuffer(env, 2)
        buf.reset_env(seed=seed)                     # the counters the PPO call left differ between precisions
        lat, mu, log_std = _sac_mods(dict(c, H=256), "scaled", env.device)
        a, _, _ = _sac_call(buf, c, FusedSquashedActor(lat, mu.weight, mu.bias, log_std.weight, log_std.bias), obs)
        out.append((r.actions.clone(), r.values.clone(), r.log_probs.clone(), a))
        env.close()
    for x, y in zip(*out):
        assert torch.equal(x, y)
