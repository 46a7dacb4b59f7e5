"""GPU tests of the episode taps (dockauv_set_taps) and the TrainingRecorder built on them: taps leave every env, output
and statistic of the real step as it is, their records agree with the real step and with the debug-output step, the
recorder reproduces the reference's own EpisodeDataStorage pickles from a graph-replayed auto-reset rollout, and the
ring wraps, spans drains and reports lost episodes as documented."""
import os
import pickle

import numpy as np
import pytest

from tests.golden_utils import rel_err

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "episode_storage_obstacles.npz")
PERSISTENT = ("state", "u_prev", "goal", "heading_goal", "current", "capsules", "spheres", "ep_return", "t_steps", "episode")


def _cfg(max_timesteps=None):
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    if max_timesteps is not None:
        cfg["max_timesteps"] = max_timesteps
    return cfg


def _tap_ids(N, K=64):
    """ids 0 and N - 1 and ids spread over both halves of the batch"""
    rest = np.random.default_rng(5).choice(np.arange(1, N - 1), K - 2, replace=False)
    return [0, N - 1] + sorted(int(i) for i in rest)


def _env(N, layout="auto", **kw):
    import torch
    from gym_dockauv_b200 import envs
    e = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=7, n_synthetic_spheres=3, layout=layout, **kw)
    e.reset()
    # episodes end inside the run (max_t) and through the auto-reset
    e.t_steps += torch.randint(990, 1001, (N,), device=e.device, dtype=torch.int32,
                               generator=torch.Generator(device=e.device).manual_seed(3))
    return e


def _drive(env, mode, actions):
    """Steps env through `mode`; returns the stacked outputs."""
    import torch
    T, N = actions.shape[0], env.num_envs
    z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=env.device)  # noqa: E731
    out = dict(obs=z(T, N, env.n_observations), reward=z(T, N, dtype=env.dtype), done=z(T, N, dtype=torch.uint8),
               cond_bits=z(T, N, dtype=torch.uint8), terminal_obs=z(T, N, env.n_observations),
               ep_return_out=z(T, N, dtype=env.dtype), ep_len_out=z(T, N, dtype=torch.int32),
               delta_d_out=z(T, N, dtype=env.dtype))
    if mode.startswith("rollout"):
        env.rollout(actions, out["obs"], out["reward"], out["done"], cond_bits=out["cond_bits"],
                    terminal_obs=out["terminal_obs"], ep_return_out=out["ep_return_out"], ep_len_out=out["ep_len_out"],
                    delta_d_out=out["delta_d_out"], use_graph=mode == "rollout_graph")
    else:
        env.enable_step_graph(mode == "step_graph")
        for t in range(T):
            env.step_into(actions[t], out["obs"][t], out["reward"][t], out["done"][t], cond_bits=out["cond_bits"][t],
                          terminal_obs=out["terminal_obs"][t], ep_return_out=out["ep_return_out"][t],
                          ep_len_out=out["ep_len_out"][t], delta_d_out=out["delta_d_out"][t])
    return out


@pytest.mark.parametrize("layout", ["pipeline", "warp_rays"])
@pytest.mark.parametrize("mode", ["step_graph", "step", "rollout_graph", "rollout"])
@pytest.mark.parametrize("N", [1000, 1 << 18])      # odd CTA tail; two parts on two streams (pipeline)
def test_taps_do_not_perturb(N, mode, layout):
    import torch
    T = 12
    a = torch.rand(T, N, 6, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0)) * 2 - 1
    plain, tapped = _env(N, layout), _env(N, layout)
    ring = tapped.set_taps(_tap_ids(N), 16)
    o0 = _drive(plain, mode, a)
    o1 = _drive(tapped, mode, a)
    torch.cuda.synchronize()
    assert int(ring["count"].item()) == T
    for k in o0:
        assert torch.equal(o0[k], o1[k]), k
    for k in PERSISTENT:
        assert torch.equal(getattr(plain, k), getattr(tapped, k)), k
    assert int(o0["done"].sum()) > 0
    s0, s1 = plain.get_stats(), tapped.get_stats()
    for k in s0:
        if k.startswith("sum_") and k != "sum_length":     # accumulated by atomics in no fixed order
            assert rel_err(s1[k], s0[k]) < 1e-10, k
        else:
            assert s0[k] == s1[k], k
    plain.close(); tapped.close()


@pytest.mark.parametrize("precision,noise", [("f64", "philox"), ("f64", "caller"), ("f32", "philox")])
def test_records_match_the_real_step(precision, noise):
    import torch
    N, T, S = 1000, 40, 16
    env = _env(N, precision=precision, cur_sigma=0.05, env_id0=123457)
    ids = _tap_ids(N)
    sel = torch.as_tensor(ids, device=env.device)
    ring = env.set_taps(ids, S)
    gen = torch.Generator(device="cuda").manual_seed(2)
    worst_state, n_done, state_bits_equal, reward_bits_equal = 0.0, 0, True, True
    for t in range(T):
        pre = {k: getattr(env, k).clone() for k in ("state", "current", "t_steps", "episode", "ep_return", "goal")}
        a = torch.rand(N, 6, device="cuda", generator=gen) * 2 - 1
        w = torch.randn(N, device="cuda", dtype=env.dtype, generator=gen) * 0.05 if noise == "caller" else None
        obs, reward, done, info = env.step(a, noise=w)
        torch.cuda.synchronize()
        s = t % S
        assert int(ring["count"].item()) == t + 1
        # pre-step inputs: copies of what the real step read (after the auto-reset of the previous step)
        assert torch.equal(ring["pre_state"][s], pre["state"][:, sel])
        assert torch.equal(ring["pre_current"][s], pre["current"][:, sel])
        assert torch.equal(ring["pre_scene"][s, 0:3], pre["goal"][:, sel])
        assert torch.equal(ring["pre_t_steps"][s], pre["t_steps"][sel])
        assert torch.equal(ring["pre_episode"][s], pre["episode"][sel])
        assert torch.equal(ring["pre_ep_return"][s], pre["ep_return"][sel])
        d = done[sel].bool()
        n_done += int(d.sum())
        assert torch.equal(ring["done"][s], done[sel])
        assert torch.equal(ring["cond_bits"][s], info["cond_bits"][sel])
        real_obs = torch.where(d[:, None], info["terminal_observation"][sel], obs[sel])
        assert torch.equal(ring["obs"][s], real_obs), t
        assert rel_err(ring["reward"][s].cpu().numpy(), reward[sel].cpu().numpy()) < 1e-12, t
        reward_bits_equal &= bool(torch.equal(ring["reward"][s], reward[sel]))
        live = ~d      # the real state of a finished env is already the reset one
        got, ref = ring["state"][s][:, live], env.state[:, sel][:, live]
        state_bits_equal &= bool(torch.equal(got, ref))
        worst_state = max(worst_state, rel_err(got.cpu().numpy(), ref.cpu().numpy()))
    assert n_done > 0
    assert worst_state < 1e-12, worst_state
    print(f"{precision} {noise}: post-step state max rel err {worst_state:.2e}, bit-equal: {state_bits_equal}; "
          f"reward bit-equal: {reward_bits_equal}")
    env.close()


@pytest.mark.parametrize("layout", ["pipeline", "warp_rays"])
def test_records_match_the_debug_step(layout):
    import torch
    from gym_dockauv_b200 import envs
    N, T, S = 1000, 60, 64
    tapped = _env(N, layout)
    dbg = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=7, n_synthetic_spheres=3, auto_reset=False, debug_outputs=True)
    dbg.reset()
    dbg.t_steps.copy_(tapped.t_steps)
    ids = _tap_ids(N)
    sel = torch.as_tensor(ids, device="cuda")
    ring = tapped.set_taps(ids, S)
    gen = torch.Generator(device="cuda").manual_seed(4)
    alive = torch.ones(len(ids), dtype=torch.bool, device="cuda")     # tap still in its first episode
    worst = 0.0
    for t in range(T):
        a = torch.rand(N, 6, device="cuda", generator=gen) * 2 - 1
        tapped.step(a)
        _, _, done, _ = dbg.step(a)
        torch.cuda.synchronize()
        if not bool(alive.any()):
            break
        for k in ("state_dot", "nu_c", "ray_dist", "reward_arr"):
            got, ref = ring[k][t][:, alive], dbg.debug[k][:, sel][:, alive]
            if layout == "warp_rays":
                assert torch.equal(got, ref), (k, t)
            worst = max(worst, rel_err(got.cpu().numpy(), ref.cpu().numpy()))
        alive &= ~done[sel].bool()
    assert not bool(alive.all())
    assert worst < 1e-10, worst
    print(f"{layout}: max rel diff to the debug step {worst:.2e}")
    tapped.close(); dbg.close()


def test_training_recorder_matches_reference_pickles(tmp_path):
    """The two reference episodes of episode_storage_obstacles.npz replayed into env 2 of a 4,096-env auto-reset
    pipeline batch through rollout(use_graph=True); same assertions as test_episode_export_matches_reference_pickles."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG
    from gym_dockauv_b200.episode_export import TrainingRecorder
    g = np.load(GOLD)
    N, i = 4096, 2
    for e in g["episodes"]:
        env = envs.ObstaclesDocking3d(BASE_CONFIG, num_envs=N, seed=1, env_id0=1000)
        env.reset()
        env.set_state(state=g[f"init_state_{e}"][None], goal=g[f"goal_{e}"][None], heading_goal=[g[f"heading_goal_{e}"]],
                      capsules=g[f"capsules_{e}"][None], u_prev=np.zeros((1, 6)), t_steps=[0], ep_return=[0.0],
                      env_ids=[i])
        rec = TrainingRecorder(env, [i, 7], str(tmp_path / f"ep{e}"), title="t", capacity=2048)
        acts = g[f"action_{e}"]
        a = torch.zeros(len(acts), N, 6, dtype=torch.float64, device=env.device)
        a[:, i] = torch.as_tensor(acts, device=env.device)
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=env.device)  # noqa: E731
        T = len(acts)
        done = z(T, N, dtype=torch.uint8)
        env.rollout(a, z(T, N, env.n_observations), z(T, N, dtype=torch.float64), done, use_graph=True)
        assert bool(done[-1, i]) and not bool(done[:-1, i].any())
        saved = [s for s in rec.drain() if s[0] == 1000 + i]
        (gid, k, path), = saved
        assert os.path.basename(path).endswith(f"__t__ENV_{1000 + i}__EPISODE_{k}_DATA_STORAGE.pkl")
        st = pickle.load(open(path, "rb"))
        assert sorted(st.keys()) == list(g["keys"]) and sorted(st["vehicle"].keys()) == list(g["vehicle_keys"])
        assert list(st["meta_data_reward"]) == list(g[f"meta_data_reward_{e}"])
        assert len(st["shapes"]) == int(g[f"n_shapes_{e}"])
        for key in ("states", "states_dot", "u"):
            ref = g[f"{key}_{e}"]
            assert st["vehicle"][key].shape == ref.shape, key
            assert rel_err(st["vehicle"][key], ref) < 1e-9, key
        for key in ("radar", "nu_c", "rewards", "cum_rewards"):
            ref = g[f"{key}_{e}"]
            assert st[key].shape == ref.shape, key
            assert rel_err(st[key], ref) < 1e-9, key
        assert np.max(np.abs(st["observation"] - g[f"observation_{e}"])) < 2e-7
        # the episode after the auto-reset starts from the real post-reset state
        post = env.state[:, i].cpu().numpy().copy()
        env.step(torch.zeros(N, 6, dtype=torch.float64, device=env.device))
        rec.drain()
        assert np.array_equal(rec._rows[0]["states"][0], post) and len(rec._rows[0]["states"]) == 2
        rec.close()
        env.close()


def test_ring_wraps_at_capacity():
    import torch
    N, S = 1000, 8
    env = _env(N)
    ids = _tap_ids(N, 5)
    sel = torch.as_tensor(ids, device="cuda")
    ring = env.set_taps(ids, S)
    snaps = []
    gen = torch.Generator(device="cuda").manual_seed(9)
    for t in range(S + 1):
        snaps.append(env.state[:, sel].clone())
        env.step(torch.rand(N, 6, device="cuda", generator=gen) * 2 - 1)
        if t == S - 1:
            torch.cuda.synchronize()
            assert int(ring["count"].item()) == S
            for j in range(S):
                assert torch.equal(ring["pre_state"][j], snaps[j]), j
    torch.cuda.synchronize()
    assert int(ring["count"].item()) == S + 1
    assert torch.equal(ring["pre_state"][0], snaps[S]) and torch.equal(ring["pre_state"][1], snaps[1])
    env.close()


def _short_episode_run(tmp_path, name, capacity, drain_every, T=70):
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.episode_export import TrainingRecorder
    N = 1000
    env = envs.ObstaclesDocking3d(_cfg(max_timesteps=12), num_envs=N, seed=3, n_synthetic_spheres=3)
    env.reset()
    rec = TrainingRecorder(env, [0, 17, 999], str(tmp_path / name), title=name, capacity=capacity, save=False)
    gen = torch.Generator(device="cuda").manual_seed(6)
    for t in range(T):
        env.step(torch.rand(N, 6, device="cuda", generator=gen) * 2 - 1)
        if (t + 1) % drain_every == 0:
            rec.drain()
    rec.drain()
    env.close()
    return rec


def test_episodes_span_drains_and_lost_records_are_dropped(tmp_path):
    ref = _short_episode_run(tmp_path, "ref", 128, 1000)          # one drain at the end, nothing lost
    often = _short_episode_run(tmp_path, "often", 8, 5)           # many drains, episodes across them
    lossy = _short_episode_run(tmp_path, "lossy", 30, 1000)       # one drain after 70 steps: 40 records lost
    assert ref.lost_episodes == 0 and often.lost_episodes == 0 and lossy.lost_episodes > 0
    by_key = {(g, k): st for g, k, st in ref.saved}
    assert len(by_key) >= 9          # every tap ended several episodes of at most 13 steps
    assert [(g, k) for g, k, _ in often.saved] == [(g, k) for g, k, _ in ref.saved]
    assert 0 < len(lossy.saved) < len(ref.saved)
    for rec in (often, lossy):
        for g, k, st in rec.saved:
            r = by_key[(g, k)]
            for key in ("states", "states_dot", "u"):
                assert np.array_equal(st["vehicle"][key], r["vehicle"][key]), (g, k, key)
            for key in ("radar", "nu_c", "rewards", "cum_rewards", "observation"):
                assert np.array_equal(st[key], r[key]), (g, k, key)


def test_invalid_taps_and_step_host_are_refused():
    import torch
    from gym_dockauv_b200 import _capi, envs
    env = envs.SimpleDocking3d(_cfg(), num_envs=2000, seed=1)
    env.reset()
    for ids in ([0, 2000], [-1], [3, 5, 3], list(range(1025))):
        with pytest.raises((_capi.DockauvError, ValueError)):
            env.set_taps(ids, 4)
    # the library's own checks, beneath the python wrapper
    import ctypes as C
    from gym_dockauv_b200.params import DockauvTapBuffers
    ring = env.set_taps([1, 2], 4)
    bufs = DockauvTapBuffers(*[C.c_void_p(ring["pre_state"].data_ptr())] * 17)
    ids = (C.c_int64 * 1025)(*range(1025))
    assert env._lib.dockauv_set_taps(env._handle, ids, 1025, 4, C.byref(bufs)) == -1
    assert env._lib.dockauv_set_taps(env._handle, ids, 2, 0, C.byref(bufs)) == -1
    assert env._lib.dockauv_set_taps(env._handle, ids, 2, 4, None) == -1
    dup = (C.c_int64 * 2)(4, 4)
    assert env._lib.dockauv_set_taps(env._handle, dup, 2, 4, C.byref(bufs)) == -1
    assert b"twice" in env._lib.dockauv_last_error()
    with pytest.raises(_capi.DockauvError, match="taps"):
        env.step_host(np.zeros((2000, 6), np.float32))
    env.clear_taps()
    env.step_host(np.zeros((2000, 6), np.float32))
    env.close()


@pytest.mark.parametrize("N", [65536, 1 << 18])
def test_clear_taps_restores_the_launch_sequence(N):
    """Taps add the gather, the shadow's step in the handle's layout (three pipeline launches for this scenario), the
    debug shadow step and the commit; after clear_taps the handle launches exactly what a handle that never had taps
    launches, through freshly captured step graphs."""
    import torch
    from gym_dockauv_b200 import envs
    es = [envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=2, n_synthetic_spheres=3) for _ in range(2)]
    for e in es:
        e.reset()
    a = torch.zeros(N, 6, device="cuda")

    def per_step(e, n=3):
        n0 = e.launch_count()
        for _ in range(n):
            e.step(a)
        return (e.launch_count() - n0) / n

    base = per_step(es[0])
    es[1].set_taps([0, 5, N - 1], 32)
    assert per_step(es[1]) == base + 3 + 3
    es[1].clear_taps()
    assert per_step(es[1]) == base == per_step(es[0])
    torch.cuda.synchronize()
    assert torch.equal(es[0].state, es[1].state)
    for e in es:
        e.close()
