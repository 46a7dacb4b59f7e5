"""Obstacles and goals written straight into the bound tensors, followed by ``refresh_obstacles``: the pipeline layout
reads the obstacles through library-owned copies (float records for the cull, env-major rows for the ray launch), and
this is the one path on which only the refresh brings those copies up to date.

The envs are first reset (so the copies hold other obstacles), then their pose and counters are injected with
``set_state`` without any obstacle or goal, then the obstacles and goals of the cases of ``test_obstacle_edges`` are
written into ``env.capsules`` / ``env.spheres`` / ``env.goal`` directly.  Group "e" places 1 to 16 obstacles in view,
so the ray launch reads the refreshed rows both in its thread-per-env tiles (one or two in view) and in its
warp-per-env loop (three or more).
"""
import numpy as np
import pytest

from tests.test_obstacle_edges import _check_vs_oracle, _make_env, build_cases


def _direct_write_step(env, scenes):
    import torch
    n = len(scenes)
    nc, ns = env.n_capsules, env.n_spheres
    env.reset()
    env.set_state(state=np.stack([s.state for s in scenes]), u_prev=np.stack([s.u0 for s in scenes]),
                  heading_goal=np.array([s.heading for s in scenes]), current=np.zeros((n, 5)),
                  t_steps=np.array([s.t_steps for s in scenes]), ep_return=np.array([s.ep_return for s in scenes]))

    def put(dst, rows):
        dst[:, :n] = torch.as_tensor(np.asarray(rows).reshape(n, -1).T, dtype=dst.dtype, device=env.device)

    put(env.goal, np.stack([s.goal for s in scenes]))
    if nc:
        put(env.capsules, np.stack([s.caps for s in scenes]))
    if ns:
        put(env.spheres, np.stack([s.sph for s in scenes]))
    env.refresh_obstacles()
    a = torch.as_tensor(np.stack([s.action for s in scenes]), device=env.device)
    obs, reward, done, info = env.step(a)
    return dict(obs=obs.cpu().numpy(), reward=reward.cpu().numpy(), done=done.cpu().numpy(),
                cond=info["cond_bits"].cpu().numpy(), state=env.state.t().cpu().numpy(), ray=None)


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["e", "c4"])
def test_direct_write_then_refresh(group):
    """One pipeline step after a direct write + refresh against the oracle (outside the ambiguity window), and with
    every in-view count the ray launch sorts into its two mappings."""
    P, cases, _ = build_cases(group)
    env = _make_env(group, len(cases), "pipeline", auto_reset=False, debug=False)
    res = _direct_write_step(env, [c.scene for c in cases])
    n_listed = env.last_list_counts()[0]
    env.close()
    inside = _check_vs_oracle(P, cases, res, range(len(cases)), "direct write + refresh")
    checked = [c for c in cases if c not in inside]
    assert n_listed > 0
    if group == "e":
        views = {c.n_in_view for c in checked}
        assert views & {1, 2} and any(v >= 3 for v in views), views
