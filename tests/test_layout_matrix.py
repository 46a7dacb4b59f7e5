"""Every scenario family through every kernel layout on a batch that is not a multiple of any CTA size, with episodes
forced to end inside the run (max_t) so that auto-resets, terminal observations and statistics are exercised: all
layouts must agree with the independently written thread-per-env kernel (flags / observations identical, rewards and
state within 1e-12), and the host-buffer entry point must agree with the device one."""
import numpy as np
import pytest

from tests.golden_utils import rel_err

pytestmark = pytest.mark.gpu

# (8 capsule + 8 sphere slots = 24 float records per env, the most a handle can have: 96 KB of them in shared memory per
# CTA of the dynamics launch)
CASES = [("ObstaclesDocking3d", dict(n_synthetic_spheres=3)), ("ObstaclesCurrentDocking3d", dict(n_synthetic_spheres=8)),
         ("ObstaclesDocking3d", dict(n_synthetic_spheres=8, n_capsules=8)),
         ("ObstaclesNoCapDocking3d", {}), ("CapsuleCurrentDocking3d", {}), ("SimpleCurrentDocking3d", {}),
         ("SimpleDocking3d", {})]


@pytest.mark.parametrize("name,kw", CASES)
def test_all_layouts_agree_on_odd_batch(name, kw):
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    N = 1000
    layouts = ("thread_per_env", "warp_rays", "pipeline")
    es = [envs.SCENARIOS[name](cfg, num_envs=N, seed=11, layout=l, **kw) for l in layouts]
    for e in es:
        e.reset()
        e.t_steps += torch.randint(985, 1001, (N,), device=e.device, dtype=torch.int32,
                                   generator=torch.Generator(device=e.device).manual_seed(3))
    gen = torch.Generator(device="cuda").manual_seed(0)
    n_done = 0
    # a pipeline step: dynamics + cull + finish, rays + finish (with obstacles), episode end
    step_launches = 3 if es[2].n_capsules + es[2].n_spheres > 0 else 2
    for t in range(24):
        a = torch.rand(N, es[0].n_actions, device="cuda", generator=gen) * 2 - 1
        n0 = es[2].launch_count()
        outs = [e.step(a) for e in es]
        assert es[2].launch_count() - n0 == step_launches, (name, t)
        o0, r0, d0, i0 = outs[0]
        n_done += int(d0.sum())
        for (o, r, d, info), l in zip(outs[1:], layouts[1:]):
            assert torch.equal(d0, d), (name, l, t)
            assert torch.equal(i0["cond_bits"], info["cond_bits"]), (name, l, t)
            assert torch.equal(o0, o), (name, l, t)
            assert rel_err(r.cpu().numpy(), r0.cpu().numpy()) < 1e-12, (name, l, t)
            dm = d0.bool()
            assert torch.equal(i0["terminal_observation"][dm], info["terminal_observation"][dm]), (name, l, t)
            assert torch.equal(i0["episode_length"][dm], info["episode_length"][dm]), (name, l, t)
    assert n_done >= N          # every env ran into max_t at least once
    s0 = es[0].get_stats()
    for e, l in zip(es[1:], layouts[1:]):
        assert rel_err(e.state.cpu().numpy(), es[0].state.cpu().numpy()) < 1e-12, (name, l)
        assert torch.equal(e.t_steps, es[0].t_steps) and torch.equal(e.episode, es[0].episode), (name, l)
        if es[0].n_capsules:
            assert torch.equal(e.capsules, es[0].capsules), (name, l)      # re-initialised obstacles: same bits
        s = e.get_stats()
        for k in ("episodes", "sum_length", "done_max_t", "done_collision", "done_out_att", "env_steps"):
            assert s[k] == s0[k], (name, l, k)
        assert rel_err(s["sum_return"], s0["sum_return"]) < 1e-10
    # host-buffer entry point on the default layout vs the device one
    a = np.random.default_rng(1).uniform(-1, 1, (N, es[0].n_actions)).astype(np.float32)
    oh, rh, dh, _ = es[2].step_host(a)
    od, rd, dd, _ = es[1].step(torch.as_tensor(a, device="cuda"))
    assert np.array_equal(dh, dd.cpu().numpy().astype(bool)) and np.array_equal(oh, od.cpu().numpy())
    assert rel_err(rh, rd.cpu().numpy()) < 1e-12
    for e in es:
        e.close()


def test_exact_cull_matches_float_cull():
    """Handles whose coordinates are too large for float obstacle records (max_dist_from_goal + max_dist > 2 km) cull in
    double, in the same three launches per step: same flags / observations / rewards as the thread-per-env kernel."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    cfg["max_dist_from_goal"] = 2500.0
    N = 777
    es = [envs.ObstaclesDocking3d(cfg, num_envs=N, seed=5, n_synthetic_spheres=3, layout=l) for l in ("thread_per_env", "pipeline")]
    for e in es:
        e.reset()
    gen = torch.Generator(device="cuda").manual_seed(4)
    for t in range(40):
        a = torch.rand(N, 6, device="cuda", generator=gen) * 2 - 1
        n0 = es[1].launch_count()
        (o0, r0, d0, i0), (o1, r1, d1, i1) = [e.step(a) for e in es]
        assert es[1].launch_count() - n0 == 3, t
        assert torch.equal(d0, d1) and torch.equal(i0["cond_bits"], i1["cond_bits"]) and torch.equal(o0, o1), t
        assert rel_err(r1.cpu().numpy(), r0.cpu().numpy()) < 1e-12, t
    assert rel_err(es[1].state.cpu().numpy(), es[0].state.cpu().numpy()) < 1e-12
    for e in es:
        e.close()


@pytest.mark.parametrize("kw", [dict(n_synthetic_spheres=3), dict(n_synthetic_spheres=8, n_capsules=8),
                                dict(scenario="SimpleDocking3d")])
def test_list_counts_match_the_step_outputs(kw):
    """dockauv_last_list_counts after a step: the ended count is the number of done flags, the listed count the number of
    envs with a pooled ray cell below 1 or more (listed = something in view, a superset of real hits; none without
    obstacles), with few and with the most float records per env and without obstacles.  A count is the difference of a
    running counter and its value when the step began; the counters start all ones, so every run crosses the 2^32 wrap.
    After a rollout the counts are those of its last step: without a graph, at the capture and at a replay.
    2^18 envs are stepped in two parts, except in steps with timing enabled (the whole batch as one range, on the first
    part's counter block): those alternate with the others, and every step's outputs equal a never-timed twin's."""
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    kw = dict(kw)
    make = envs.SCENARIOS[kw.pop("scenario", "ObstaclesDocking3d")]
    N = 40000                      # one launch group; also stepped in two parts below
    T = 4

    def check(n, obs, done, where):
        n_listed, n_ended = env.last_list_counts()
        assert n_ended == int(done.sum()), where
        if env.n_capsules + env.n_spheres == 0:
            assert n_listed == 0, (where, n_listed)
        # observation rows of finished envs are zeroed; among the others a cell below 1 needs an obstacle in view
        hit = int(((obs[:, 16:] < 1.0).any(1) & ~done.bool()).sum())
        assert hit <= n_listed <= n, (where, hit, n_listed)

    def bits(x):
        return x.view(torch.uint8)

    for n in (N, 1 << 18):
        mixed = n == 1 << 18
        env = make(cfg, num_envs=n, seed=2, **kw)
        twin = make(cfg, num_envs=n, seed=2, **kw) if mixed else None
        for e in (env, twin) if mixed else (env,):
            e.reset()
            e.t_steps += 990        # episodes end inside the run
        gen = torch.Generator(device="cuda").manual_seed(1)
        for t in range(14):
            a = torch.rand(n, env.n_actions, device="cuda", generator=gen) * 2 - 1
            if mixed:
                env.enable_timing(t % 2 == 1)
            obs, rew, done, info = env.step(a)
            check(n, obs, done, (n, t))
            if mixed:
                obs2, rew2, done2, info2 = twin.step(a)
                assert torch.equal(bits(obs), bits(obs2)) and torch.equal(done, done2), (n, t)
                assert torch.equal(info["cond_bits"], info2["cond_bits"]) and torch.equal(bits(rew), bits(rew2)), (n, t)
        assert env.get_stats()["episodes"] > 0
        if mixed:
            env.enable_timing(False)
            twin.close()
        acts = torch.empty(T, n, env.n_actions, device="cuda")
        obs = torch.zeros(T, n, env.n_observations, device="cuda")
        rew = torch.zeros(T, n, dtype=env.dtype, device="cuda")
        done = torch.zeros(T, n, dtype=torch.uint8, device="cuda")
        for use_graph in (False, True, True):
            # step counters in the last T steps of an episode: at every step of the rollout some episodes reach max_t
            env.t_steps.copy_(torch.randint(env.max_timesteps - T + 1, env.max_timesteps + 1, (n,), device="cuda",
                                            dtype=torch.int32, generator=gen))
            acts.uniform_(-1, 1, generator=gen)
            env.rollout(acts, obs, rew, done, use_graph=use_graph)
            assert int(done[T - 1].sum()) > 0
            check(n, obs[T - 1], done[T - 1], (n, "rollout", use_graph))
        assert env.rollout_captures() == 1
        env.close()
