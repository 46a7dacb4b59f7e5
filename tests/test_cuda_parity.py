"""Parity of the CUDA step path (through the C ABI, via gym_dockauv_b200.envs) against

* the golden traces recorded from the unmodified reference (tests/golden/*.npz) -- every episode of a trace is
  one env of the batch, initial conditions injected with set_state(), actions replayed step by step; and
* the CPU oracle (oracle/) on seeded random rollouts, including the in-kernel auto-reset.

Bars (BASELINE.json north_star): done / collision / condition bits and termination step bit-exact; FP64 state,
pre-cast observation, ray distances and reward within 1e-9 relative (floor 1.0) over the whole rollout; float32
observations at most one float32 ulp apart.  FP32 variant: stated looser bounds in test_fp32_variant.
"""
import ctypes as C

import numpy as np
import pytest

from tests.golden_utils import case_names, load_case, rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-9
BLOWUP = 1e3


def _env_for_case(g, layout, precision="f64", debug=True):
    import torch  # noqa: F401
    from gym_dockauv_b200 import envs
    meta = g["meta"]
    mu, sigma = g["current_mu_sigma"][0]
    has_cur = bool(np.any(g["current"][:, 0] != 0) or sigma > 0)
    E = len(g["ep_len"])
    cls = envs.SCENARIOS[meta["env_id"]]
    env = cls(meta["config"], num_envs=E, precision=precision, layout=layout, n_capsules=int(g["n_capsules"].max()),
              n_spheres=int(g["n_spheres"].max()), cur_mu=float(mu), cur_sigma=float(sigma), force_current=has_cur,
              auto_reset=False, debug_outputs=debug)
    assert env.n_rays == meta["n_rays"] and env.n_observations == meta["n_obs"] and env.n_actions == meta["n_u"]
    env.set_state(state=g["init_state"], goal=g["goal"], heading_goal=g["heading_goal"], current=g["current"],
                  capsules=g["capsules"] if env.n_capsules else None, spheres=g["spheres"] if env.n_spheres else None,
                  u_prev=np.zeros((E, env.n_actions)), t_steps=np.zeros(E), ep_return=np.zeros(E))
    return env


@pytest.mark.parametrize("layout", ["thread_per_env", "warp_rays", "pipeline"])
@pytest.mark.parametrize("name", case_names())
def test_cuda_matches_reference_trace(name, layout):
    import torch
    g = load_case(name)
    meta = g["meta"]
    # the multi-launch layouts are built without debug outputs (a debug call is served by the fused kernel), so they
    # are compared through everything the step returns: observations, rewards, flags, state, counters
    dbg = layout in ("thread_per_env", "warp_rays")
    env = _env_for_case(g, layout, debug=dbg)
    E, T = g["action"].shape[:2]
    f32 = meta["action_dtype"] == "f32"
    unstable = meta["vehicle"] == "LAUV" and meta["config"]["t_step_size"] > 0.05
    alive = np.ones(E, dtype=bool)           # still inside the recorded episode and not blown up
    worst = dict(state=0.0, u=0.0, ray=0.0, reward=0.0, rarr=0.0, nav=0.0, edot=0.0, nu_c=0.0, ret=0.0, delta_d=0.0)
    obs_mismatch, compared = 0, 0
    for t in range(T):
        alive &= t < g["ep_len"]
        if unstable:
            alive &= ~(np.abs(g["state"][:, t]).max(axis=1) > BLOWUP)
        if not alive.any():
            break
        a = torch.as_tensor(g["action"][:, t].astype(np.float32 if f32 else np.float64), device=env.device)
        noise = torch.as_tensor(g["noise_w"][:, t], device=env.device) if env._params.cur_sigma > 0 else None
        obs, reward, done, info = env.step(a, noise=noise)
        m = alive
        n = int(m.sum())
        compared += n
        st = env.state.t().cpu().numpy()
        # ---- discrete outputs: bit-exact
        bits = info["cond_bits"].cpu().numpy()
        cond = np.stack([(bits >> k) & 1 for k in range(5)], axis=1).astype(np.uint8)
        assert np.array_equal(cond[m], g["conditions"][m, t]), (name, t)
        assert np.array_equal(done.cpu().numpy()[m], g["done"][m, t]), (name, t)
        assert np.array_equal(cond[m, 4], g["collision"][m, t]), (name, t)
        assert np.array_equal(env.t_steps.cpu().numpy()[m], g["t_steps"][m, t]), (name, t)
        # ---- continuous outputs
        worst["state"] = max(worst["state"], rel_err(st[m], g["state"][m, t]))
        worst["u"] = max(worst["u"], rel_err(env.u_prev.t().cpu().numpy()[m, :meta["n_u"]], g["u"][m, t]))
        worst["reward"] = max(worst["reward"], rel_err(reward.cpu().numpy()[m], g["reward"][m, t]))
        worst["delta_d"] = max(worst["delta_d"], rel_err(info["delta_d"].cpu().numpy()[m], g["delta_d"][m, t]))   # info["delta_d"]
        if dbg:
            worst["ray"] = max(worst["ray"], rel_err(env.debug["ray_dist"].t().cpu().numpy()[m], g["ray_dist"][m, t]))
            worst["rarr"] = max(worst["rarr"], rel_err(env.debug["reward_arr"].t().cpu().numpy()[m], g["reward_arr"][m, t]))
            nav = env.debug["nav"].t().cpu().numpy()
            ref_nav = np.stack([g["delta_d"][:, t], g["delta_theta"][:, t], g["delta_psi"][:, t]], axis=1)
            worst["nav"] = max(worst["nav"], rel_err(nav[m], ref_nav[m]))
            worst["edot"] = max(worst["edot"], rel_err(env.debug["euler_dot"].t().cpu().numpy()[m], g["state_dot"][m, t, 3:6]))
            worst["nu_c"] = max(worst["nu_c"], rel_err(env.debug["nu_c"].t().cpu().numpy()[m], g["nu_c"][m, t, :3]))
        worst["ret"] = max(worst["ret"], rel_err(env.ep_return.cpu().numpy()[m], g["cum_reward"][m, t]))
        ob = obs.cpu().numpy()[m]
        ref_ob = g["obs"][m, t]
        same = (ob == ref_ob) | (np.isnan(ob) & np.isnan(ref_ob))
        obs_mismatch += int((~same).sum())
        assert rel_err(ob, ref_ob) < 2e-7, (name, t)
        # pre-cast observation vs the reference's float32-rounded value: half a float32 ulp of slack
        assert not dbg or rel_err(env.debug["obs_f64"].t().cpu().numpy()[m], ref_ob.astype(np.float64)) < 6.1e-8, (name, t)
    assert compared >= (150 if unstable else int(g["ep_len"].sum()))
    for k, v in worst.items():
        assert v < TOL, (name, layout, k, v, worst)
    assert obs_mismatch <= max(2, compared * meta["n_obs"] // 2000), (obs_mismatch, compared)
    env.close()


def _oracle_rollout(config, scenario, n, steps, seed, n_synth, dtype, layout, precision="f64", lauv=False):
    """Random-action rollout with auto-reset on both sides; returns per-step comparison stats."""
    import torch
    from gym_dockauv_b200 import envs
    from oracle import oracle as orc
    env = envs.SCENARIOS[scenario](config, num_envs=n, seed=seed, n_synthetic_spheres=n_synth, layout=layout,
                                   precision=precision, env_id0=1000)
    env.reset()
    bo = orc.BatchOracle(config, scenario, n, seed=seed, n_extra_spheres=n_synth, env_id0=1000)
    # reset parity: same Philox stream, same distributions
    st0 = env.state.t().cpu().numpy()
    ref0 = bo.field("state")
    assert rel_err(st0, ref0) < (1e-12 if precision == "f64" else 1e-6)
    assert rel_err(env.goal.t().cpu().numpy(), bo.field("goal")) < (1e-12 if precision == "f64" else 1e-6)
    rng = np.random.default_rng(seed)
    out = dict(done_mismatch=0, worst_reward=0.0, worst_state=0.0, episodes=0, obs_worst=0.0)
    n_u = env.n_actions
    for t in range(steps):
        a = rng.uniform(-1, 1, (n, n_u)).astype(dtype)
        obs, reward, done, info = env.step(torch.as_tensor(a, device=env.device))
        robs, rrew, rdone, fin = bo.step(a)
        out["episodes"] += int(fin)
        d = done.cpu().numpy()
        out["done_mismatch"] += int((d != rdone).sum())
        out["worst_reward"] = max(out["worst_reward"], rel_err(reward.cpu().numpy(), rrew))
        out["worst_state"] = max(out["worst_state"], rel_err(env.state.t().cpu().numpy(), bo.field("state")))
        out["obs_worst"] = max(out["obs_worst"], rel_err(obs.cpu().numpy(), robs))
    out["stats"] = env.get_stats()
    env.close()
    return out


@pytest.mark.parametrize("layout", ["warp_rays", "pipeline"])
@pytest.mark.parametrize("radar,n_synth", [
    (dict(alpha=60, beta=80, ray_per_deg=5, blocksize_reduce=2), 3),     # 13 x 17 = 221 rays (8 per lane), 63 pooled cells
    (dict(alpha=70, beta=70, ray_per_deg=10, blocksize_reduce=3), 8),    # 3 x 3 pooling blocks; 13 obstacles (16-slot path)
    (dict(alpha=60, beta=80, ray_per_deg=10, blocksize_reduce=1), 0),    # no pooling: 63 cells, n_obs = 79
])
def test_radar_extremes_vs_oracle(layout, radar, n_synth):
    """Edge sizes of the radar path: close to DOCKAUV_MAX_RAYS rays, pooled grids wider than a warp, block sizes other
    than 2 (generic pooling), more than 8 obstacles per env."""
    from gym_dockauv_b200.config import BASE_CONFIG
    deg = np.pi / 180
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(freq=1, alpha=radar["alpha"] * deg, beta=radar["beta"] * deg, ray_per_deg=radar["ray_per_deg"] * deg,
                        max_dist=10, blocksize_reduce=radar["blocksize_reduce"])
    r = _oracle_rollout(cfg, "ObstaclesDocking3d", 192, 120, seed=9, n_synth=n_synth, dtype=np.float64, layout=layout)
    assert r["done_mismatch"] == 0
    assert r["worst_state"] < TOL and r["worst_reward"] < TOL and r["obs_worst"] < 2e-7, r


@pytest.mark.parametrize("layout", ["thread_per_env", "warp_rays", "pipeline"])
def test_random_rollout_with_autoreset_vs_oracle(layout):
    """256 envs x 300 steps of the BASELINE C4 workload (64 rays, 5 capsules + 3 spheres), auto-reset on."""
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    r = _oracle_rollout(cfg, "ObstaclesDocking3d", 256, 300, seed=5, n_synth=3, dtype=np.float32, layout=layout)
    assert r["done_mismatch"] == 0
    assert r["episodes"] > 100
    assert r["worst_state"] < TOL and r["worst_reward"] < TOL and r["obs_worst"] < 2e-7, r
    assert r["stats"]["episodes"] == r["episodes"]
    assert r["stats"]["env_steps"] == 256 * 300


def test_thousand_step_rollout_vs_oracle():
    """north_star: 1e-9 relative over a 1000-step rollout (SimpleDocking3d = BASELINE config C2, 512 envs)."""
    from gym_dockauv_b200.config import BASE_CONFIG
    r = _oracle_rollout(dict(BASE_CONFIG), "SimpleDocking3d", 512, 1000, seed=11, n_synth=0, dtype=np.float64,
                        layout="auto")
    assert r["done_mismatch"] == 0
    assert r["worst_state"] < TOL and r["worst_reward"] < TOL and r["obs_worst"] < 2e-7, r


def test_lauv_current_rollout_vs_oracle():
    """BASELINE config C3 at the stable step size: CapsuleCurrentDocking3d, LAUV, h = 0.02."""
    from gym_dockauv_b200.config import BASE_CONFIG
    cfg = dict(BASE_CONFIG)
    cfg["vehicle"] = "LAUV"
    cfg["t_step_size"] = 0.02
    r = _oracle_rollout(cfg, "CapsuleCurrentDocking3d", 256, 400, seed=3, n_synth=0, dtype=np.float64, layout="auto")
    assert r["done_mismatch"] == 0
    assert r["worst_state"] < TOL and r["worst_reward"] < TOL, r


def test_fp32_variant():
    """FP32 kernels (precision="f32"): the stated looser bound.  2048 envs of the C4 workload, 60 steps from identical
    initial conditions against the FP64 oracle, comparing every env until its first episode end on either side:
    state within 2e-5, reward within 5e-5, observation within 5e-4 (relative, floor 1.0; measured 3.6e-6 / 1.7e-5 /
    3e-4, profiles/tools/fp32_check.py), done flags may differ for at most 0.1 % of the envs (threshold crossings)."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    from oracle import oracle as orc
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    n = 2048
    env = envs.ObstaclesDocking3d(cfg, num_envs=n, seed=9, n_synthetic_spheres=3, precision="f32")
    env.reset()
    bo = orc.BatchOracle(cfg, "ObstaclesDocking3d", n, seed=9, n_extra_spheres=3)
    assert env.state.dtype == torch.float32 and env.reward.dtype == torch.float32
    rng = np.random.default_rng(9)
    alive = np.ones(n, bool)
    mismatches, worst = 0, dict(state=0.0, reward=0.0, obs=0.0)
    for t in range(60):
        a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
        obs, rew, done, _ = env.step(torch.as_tensor(a, device=env.device))
        robs, rrew, rdone, _ = bo.step(a)
        d, rd = done.cpu().numpy().astype(bool), rdone.astype(bool)
        mismatches += int(((d != rd) & alive).sum())
        m = alive & ~d & ~rd
        # the FP32 bound is stated with a floor of 1.0 (absolute below 1): float32 carries 7 digits of O(10) positions
        worst["state"] = max(worst["state"], rel_err(env.state.t().cpu().numpy().astype(np.float64)[m], bo.field("state")[m], floor=1.0))
        worst["reward"] = max(worst["reward"], rel_err(rew.cpu().numpy().astype(np.float64)[alive], rrew[alive], floor=1.0))
        worst["obs"] = max(worst["obs"], rel_err(obs.cpu().numpy()[m], robs[m], floor=1.0))
        alive &= ~(d | rd)
    assert alive.sum() > n // 3
    assert worst["state"] < 2e-5 and worst["reward"] < 5e-5 and worst["obs"] < 5e-4, worst
    assert mismatches <= n // 1000, mismatches
    env.close()


def test_bluerov2_direct_mode_vs_reference():
    """control_mode="direct" (n_u = 8, dense 6 x 8 thrust map): 60 AUVSim steps recorded from the reference with a
    constant current; the CUDA env is driven with an injected constant current of the same body-frame value by
    freezing the attitude dependence: compared on state and command with the current switched off instead."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG
    from oracle import oracle as orc
    import ctypes as C
    uv = np.load(__import__("os").path.join(__import__("tests.golden_utils", fromlist=["GOLDEN_DIR"]).GOLDEN_DIR,
                                            "unit_vectors.npz"))
    # reference trace has a constant body-frame current, which the env API cannot express (the env rotates a NED
    # current); so: oracle (pinned to that trace by tests/test_oracle_golden.py) vs CUDA on a no-current rollout
    cfg = dict(BASE_CONFIG)
    P = orc.make_params(cfg, vehicle_key="BlueROV2_direct")
    L = orc.lib()
    L.orc_auv_step.argtypes = [C.POINTER(orc.OrcParams), C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p,
                               C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    env = envs.SimpleDocking3d(cfg, num_envs=4, control_mode="direct", auto_reset=False)
    assert env.n_actions == 8
    st0 = np.zeros((4, 12))
    st0[:, 3:6] = [0.1, -0.05, 0.7]
    st0[:, 0] = [1.0, 2.0, 3.0, 4.0]
    env.set_state(state=st0, goal=np.zeros((4, 3)), heading_goal=np.zeros(4), current=np.zeros((4, 5)),
                  u_prev=np.zeros((4, 8)), t_steps=np.zeros(4), ep_return=np.zeros(4))
    ref_state = st0.copy()
    ref_u = np.zeros((4, 8))
    sd = np.zeros(12)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))  # noqa: E731
    for t, a in enumerate(uv["direct_actions"][:40]):
        acts = np.tile(a, (4, 1)) * np.array([[1.0], [0.5], [-0.7], [0.2]])
        env.step(torch.as_tensor(acts, device=env.device))
        for e in range(4):
            s_e, u_e, a_e = ref_state[e].copy(), ref_u[e].copy(), np.ascontiguousarray(acts[e])
            L.orc_auv_step(C.byref(P), dp(s_e), dp(u_e), a_e.ctypes.data_as(C.c_void_p), 0, dp(np.zeros(6)), dp(sd))
            ref_state[e], ref_u[e] = s_e, u_e
        assert rel_err(env.state.t().cpu().numpy(), ref_state) < TOL, t
        assert rel_err(env.u_prev.t().cpu().numpy(), ref_u) < TOL, t
    env.close()


def test_step_host_matches_device_step():
    """The host-buffer entry point (dockauv_step_host) gives the same results as the device-pointer one."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG
    n = 40000   # > one pipeline chunk, not a multiple of the CTA size
    e1 = envs.ObstaclesDocking3d(dict(BASE_CONFIG), num_envs=n, seed=2)
    e2 = envs.ObstaclesDocking3d(dict(BASE_CONFIG), num_envs=n, seed=2)
    e1.reset()
    e2.reset()
    rng = np.random.default_rng(0)
    for _ in range(5):
        a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
        o1, r1, d1, _ = e1.step(torch.as_tensor(a, device=e1.device))
        o2, r2, d2, _ = e2.step_host(a)
        assert np.array_equal(o1.cpu().numpy(), o2)
        assert np.array_equal(r1.cpu().numpy(), r2)
        assert np.array_equal(d1.cpu().numpy().astype(bool), d2)
    e1.close()
    e2.close()


def test_device_without_index_and_misaligned_rows():
    """device="cuda" means the current device (handle, tensors and the device checks agree); observation rows that do not
    start at a 16-byte boundary are refused instead of faulting in a 128-bit store."""
    import torch
    from gym_dockauv_b200 import _capi, envs
    from gym_dockauv_b200.config import BASE_CONFIG
    env = envs.ObstaclesDocking3d(dict(BASE_CONFIG), num_envs=300, device="cuda")
    assert env.device == torch.device("cuda", torch.cuda.current_device())
    env.reset()
    a = torch.zeros(300, 6, device="cuda")
    obs, reward, done, info = env.step(a)
    assert torch.isfinite(obs).all() and info["delta_d"].shape == (300,) and (info["delta_d"] > 0).all()
    d = env.info_dict(0)
    assert d["delta_d"] == float(info["delta_d"][0]) and abs(d["simulation_time"] - 0.1) < 1e-15
    # a view whose storage offset is one float: misaligned rows
    big = torch.zeros(300 * env.n_observations + 4, dtype=torch.float32, device="cuda")
    bad = big[1:1 + 300 * env.n_observations].view(300, env.n_observations)
    with pytest.raises(ValueError):
        env.step_into(a, bad, env.reward, env.done)
    out = envs.DockauvStepOut(*[C.c_void_p(t.data_ptr()) for t in (bad, env.reward, env.done)], None, None, None, None, None)
    rc = env._lib.dockauv_step(env._handle, C.c_void_p(a.data_ptr()), 1, None, C.byref(out), None, 1, None)
    assert rc == -1 and b"16-byte" in env._lib.dockauv_last_error()
    env.close()


def test_rollout_graph_is_replayed_not_recaptured():
    """dockauv_rollout(use_graph): the same pointers replay the captured launch sequence; other pointers re-capture."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG
    n, T = 4096, 6
    env = envs.ObstaclesDocking3d(dict(BASE_CONFIG), num_envs=n, seed=3)
    ref = envs.ObstaclesDocking3d(dict(BASE_CONFIG), num_envs=n, seed=3)
    env.reset()
    ref.reset()
    gen = torch.Generator(device="cuda").manual_seed(1)
    acts = torch.rand(T, n, 6, device="cuda", generator=gen) * 2 - 1
    obs = torch.zeros(T, n, env.n_observations, device="cuda")
    rew = torch.zeros(T, n, dtype=torch.float64, device="cuda")
    done = torch.zeros(T, n, dtype=torch.uint8, device="cuda")
    dd = torch.zeros(T, n, dtype=torch.float64, device="cuda")
    for rep in range(4):
        env.rollout(acts, obs, rew, done, delta_d_out=dd)
        for t in range(T):
            o, r, d, info = ref.step(acts[t])
            assert torch.equal(o, obs[t]) and torch.equal(r, rew[t]) and torch.equal(d, done[t])
            assert torch.equal(info["delta_d"], dd[t])
        assert env.rollout_captures() == 1, rep
    obs2 = torch.zeros_like(obs)
    env.rollout(acts, obs2, rew, done)
    assert env.rollout_captures() == 2
    env.close()
    ref.close()


def test_layouts_agree_bitwise_on_flags_large_batch():
    """65,536 envs, 40 steps: all kernel layouts give identical done flags / observations and rewards within 1e-12."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG
    n = 65536
    es = [envs.ObstaclesCurrentDocking3d(dict(BASE_CONFIG), num_envs=n, seed=4, layout=l)
          for l in ("thread_per_env", "warp_rays", "pipeline")]
    for e in es:
        e.reset()
    gen = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(40):
        a = torch.rand(n, 6, device="cuda", generator=gen) * 2 - 1
        outs = [e.step(a) for e in es]
        for o in outs[1:]:
            assert torch.equal(outs[0][2], o[2])
            assert rel_err(outs[0][1].cpu().numpy(), o[1].cpu().numpy()) < 1e-12
            assert torch.equal(outs[0][0], o[0])
    for e in es[1:]:
        assert rel_err(es[0].state.cpu().numpy(), e.state.cpu().numpy()) < 1e-12
        assert torch.equal(es[0].t_steps, e.t_steps) and torch.equal(es[0].episode, e.episode)
    for e in es:
        e.close()


def test_step_in_parts_equals_one_launch_group():
    """A batch that is stepped in two parts on two streams (>= 131,072 envs, odd size) gives the same bits as the same
    envs stepped as one launch group (split_chunk_envs = N disables the parts; so does any other non-zero value, 4096
    included)."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    n = (1 << 19) + 4097
    es = [envs.ObstaclesDocking3d(cfg, num_envs=n, seed=21, n_synthetic_spheres=3, split_chunk_envs=c) for c in (0, n, 4096)]
    for e in es:
        e.reset()
    gen = torch.Generator(device="cuda").manual_seed(2)
    for _ in range(12):
        a = torch.rand(n, 6, device="cuda", generator=gen) * 2 - 1
        (o0, r0, d0, _), (o1, r1, d1, _), (o2, r2, d2, _) = [e.step(a) for e in es]
        assert torch.equal(o0, o1) and torch.equal(r0, r1) and torch.equal(d0, d1)
        assert torch.equal(o0, o2) and torch.equal(r0, r2) and torch.equal(d0, d2)
    assert torch.equal(es[0].state, es[1].state) and torch.equal(es[0].episode, es[1].episode)
    assert torch.equal(es[0].state, es[2].state) and torch.equal(es[0].episode, es[2].episode)
    s0, s1, s2 = es[0].get_stats(), es[1].get_stats(), es[2].get_stats()
    assert s0["env_steps"] == s1["env_steps"] == s2["env_steps"] == 12 * n and s0["episodes"] == s1["episodes"] == s2["episodes"]
    assert es[0].launch_count() - es[1].launch_count() == 12 * 3      # 6 launches per step against 3 (dynamics + cull, rays, episode end)
    assert es[2].launch_count() == es[1].launch_count()
    for e in es:
        e.close()


def test_scale_invariants_full_size():
    """BASELINE-size batch (1,048,576 envs, C4 workload): size-independent properties instead of the oracle --
    observation bounds, zero rows exactly where done, statistics add up, determinism across two identical runs."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    n = 1 << 20
    sums = []
    for rep in range(2):
        env = envs.ObstaclesDocking3d(cfg, num_envs=n, seed=123, n_synthetic_spheres=3)
        env.reset()
        gen = torch.Generator(device="cuda").manual_seed(7)
        total_done = 0
        for t in range(12):
            a = torch.rand(n, 6, device="cuda", generator=gen) * 2 - 1
            obs, reward, done, info = env.step(a)
            assert torch.isfinite(obs).all() and torch.isfinite(reward).all()
            assert (obs <= 1).all() and (obs >= -1).all() and (obs[:, 0] >= 0).all() and (obs[:, 16:] >= 0).all()
            dn = done.bool()
            total_done += int(dn.sum())
            assert not obs[dn].any()                       # finished envs hand back the zero reset observation
            assert (env.t_steps[dn] == 0).all() and (env.t_steps[~dn] > 0).all()
        st = env.get_stats()
        assert st["episodes"] == total_done and st["env_steps"] == 12 * n
        assert st["done_goal_reached"] + st["done_out_pos"] + st["done_out_att"] + st["done_max_t"] + st["done_collision"] >= total_done
        sums.append((float(env.state.double().sum()), float(reward.double().sum()), total_done))
        env.close()
    assert sums[0] == sums[1]


def test_results_do_not_depend_on_sharding():
    """Contiguous shards keyed by the global env id (SURVEY.md 8e): one batch of 4096 envs and two shards of 2048 with
    env_id0 = 0 / 2048 produce bit-identical states, observations, rewards and flags, including auto-resets."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG
    from gym_dockauv_b200.stats import shard_env_range
    n = 4096
    whole = envs.ObstaclesCurrentDocking3d(dict(BASE_CONFIG), num_envs=n, seed=21)
    shards = []
    for r in range(2):
        b, e = shard_env_range(n, r, 2)
        shards.append(envs.ObstaclesCurrentDocking3d(dict(BASE_CONFIG), num_envs=e - b, seed=21, env_id0=b))
    whole.reset()
    for sh in shards:
        sh.reset()
    gen = torch.Generator(device="cuda").manual_seed(3)
    for t in range(150):
        a = torch.rand(n, 6, device="cuda", generator=gen) * 2 - 1
        ow, rw, dw, _ = whole.step(a)
        outs = [sh.step(a[k * 2048:(k + 1) * 2048].contiguous()) for k, sh in enumerate(shards)]
        assert torch.equal(ow, torch.cat([o[0] for o in outs]))
        assert torch.equal(rw, torch.cat([o[1] for o in outs]))
        assert torch.equal(dw, torch.cat([o[2] for o in outs]))
    assert torch.equal(whole.state, torch.cat([sh.state for sh in shards], dim=1))
    sw = whole.get_stats()
    ss = [sh.get_stats() for sh in shards]
    assert sw["episodes"] == ss[0]["episodes"] + ss[1]["episodes"] > 0
    for e in [whole] + shards:
        e.close()


@pytest.mark.parametrize("scenario,vehicle,n,h", [("SimpleDocking3d", "BlueROV2", 65536, 0.1),          # BASELINE C2
                                                  ("CapsuleCurrentDocking3d", "LAUV", 262144, 0.1),    # BASELINE C3
                                                  ("CapsuleCurrentDocking3d", "LAUV", 262144, 0.02)])
def test_baseline_config_sizes(scenario, vehicle, n, h):
    """BASELINE.json configs C2 / C3 at their full sizes: size-independent properties (bounded finite observations
    for finite states, zero rows and reset counters exactly where done, statistics that add up, determinism).
    LAUV at the stock h = 0.1 blows up like the reference does; there only the bookkeeping invariants are checked."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG
    cfg = dict(BASE_CONFIG, vehicle=vehicle, t_step_size=h)
    n_u = 3 if vehicle == "LAUV" else 6
    stable = not (vehicle == "LAUV" and h > 0.05)
    sums = []
    for rep in range(2):
        env = envs.SCENARIOS[scenario](cfg, num_envs=n, seed=77)
        env.reset()
        gen = torch.Generator(device="cuda").manual_seed(5)
        total_done = 0
        for t in range(30):
            a = torch.rand(n, n_u, device="cuda", generator=gen) * 2 - 1
            obs, reward, done, info = env.step(a)
            dn = done.bool()
            total_done += int(dn.sum())
            assert not obs[dn].any()
            assert (env.t_steps[dn] == 0).all() and (env.t_steps[~dn] > 0).all()
            if stable:
                assert torch.isfinite(obs).all() and torch.isfinite(reward).all()
                assert (obs <= 1).all() and (obs >= -1).all() and (obs[:, 0] >= 0).all() and (obs[:, 16:] >= 0).all()
        st = env.get_stats()
        assert st["episodes"] == total_done and st["env_steps"] == 30 * n
        sums.append((total_done, float(torch.nan_to_num(env.state.double()).sum()), st["sum_length"]))
        env.close()
    assert sums[0] == sums[1]
