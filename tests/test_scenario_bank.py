"""Scenario banks (dockauv_set_scenario_bank): resets draw caller-supplied initial conditions, uniformly or by weight.

CPU: argument checks of the C call, the ctypes struct against the header, the row packing.  GPU: the rows every reset
takes are the ones a numpy restatement of the Philox draw predicts, bit for bit, in every layout and with the auto-reset;
the oracle follows envs across bank resets; banks from the reference's own generator; sharding; the weighted draw;
graph caching; refusals; clearing; taps."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.golden_utils import rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M32 = np.uint64(0xFFFFFFFF)
BANK_COUNTER = 0x40000000


# ------------------------------------------------------------------------------------------- the draw, restated
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


def predict_rows(seed, gids, episodes, K, cdf=None):
    """Row drawn by the reset of env `gid` whose episode counter is `episode` before the reset."""
    gids = np.asarray(gids, dtype=np.uint64)
    ep = np.broadcast_to(np.asarray(episodes, dtype=np.uint64), gids.shape)
    c = philox4x32_10([gids & M32, gids >> np.uint64(32), ep, np.full(gids.shape, BANK_COUNTER, np.uint64)],
                      seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    if cdf is None:     # high 64 bits of ((c0 << 32) | c1) * K
        A, B = c[0] * np.uint64(K), c[1] * np.uint64(K)
        return ((A + (B >> np.uint64(32))) >> np.uint64(32)).astype(np.int64)
    cdf = np.asarray(cdf, dtype=np.float64)
    x = ((c[0] >> np.uint64(5)).astype(np.float64) * 67108864.0 + (c[1] >> np.uint64(6)).astype(np.float64)) \
        * (1.0 / 9007199254740992.0) * cdf[-1]
    return np.searchsorted(cdf, x, side="right").astype(np.int64)


# ------------------------------------------------------------------------------------------- CPU
def test_bad_arguments_are_refused_with_a_message_that_names_them():
    from gym_dockauv_b200 import _capi
    from gym_dockauv_b200.params import DockauvScenarioBank
    lib = _capi.load()

    def call(h, **kw):
        b = dict(rows=0x10000, cdf=None, row_of_env=None, n_rows=4, row_stride=16)
        b.update(kw)
        rc = lib.dockauv_set_scenario_bank(h, C.byref(DockauvScenarioBank(**b)), None)
        return rc, lib.dockauv_last_error().decode()

    assert lib.dockauv_set_scenario_bank(None, None, None) == -1
    assert "null handle" in lib.dockauv_last_error().decode()
    rc, msg = call(None)
    assert rc == -1 and "null handle" in msg
    for kw, word in ((dict(n_rows=0), "n_rows"), (dict(n_rows=1 << 31), "n_rows"), (dict(rows=0x10008), "16-byte aligned"),
                     (dict(row_stride=14), "row_stride"), (dict(rows=None), "rows is null"),
                     (dict(cdf=0x20004), "cdf")):
        rc, msg = call(None, **kw)
        assert rc == -1 and word in msg, (kw, msg)


def test_bank_struct_matches_header():
    import re
    from gym_dockauv_b200.params import SCENARIO_BANK_FIELDS, DockauvScenarioBank
    text = open(os.path.join(ROOT, "include", "dockauv.h")).read()
    body = re.search(r"typedef struct DockauvScenarioBank \{(.*?)\} DockauvScenarioBank;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [re.findall(r"(\w+)\s*$", decl.strip())[0] for decl in body.split(";") if decl.strip()]
    assert tuple(names) == SCENARIO_BANK_FIELDS
    assert C.sizeof(DockauvScenarioBank) == 40
    assert [f for f, _ in DockauvScenarioBank._fields_] == list(SCENARIO_BANK_FIELDS)
    from gym_dockauv_b200 import _capi
    assert "dockauv_set_scenario_bank" in _capi.SYMBOLS


@pytest.mark.parametrize("scenario", ["ObstaclesDocking3d", "ObstaclesCurrentDocking3d", "SimpleCurrentDocking3d"])
def test_rows_from_reference_dicts_follow_the_documented_column_order(scenario):
    import torch
    from gym_dockauv_b200.config import BASE_CONFIG
    from gym_dockauv_b200.reference_reset import ReferenceResetStream
    from gym_dockauv_b200.scenario_bank import UNUSED_CAPSULE, UNUSED_SPHERE, pack, row_width
    nc, ns = 6, 2          # one capsule slot and the spheres unused
    ds = [ReferenceResetStream(scenario, BASE_CONFIG, seed=3).generate() for _ in range(5)]
    caps = np.zeros((5, nc, 7))
    caps[:] = UNUSED_CAPSULE
    for k, d in enumerate(ds):
        caps[k, :len(d["capsules"])] = d["capsules"]
    rows = pack([d["init_state"][:6] for d in ds], [d["goal"] for d in ds], [d["heading_goal"] for d in ds], nc, ns,
                current=[d["current"] for d in ds], capsules=caps, dtype=torch.float64).numpy()
    W = row_width(nc, ns)
    assert W == 15 + 7 * nc + 4 * ns and rows.shape == (5, W + (-W) % 2)
    for k, d in enumerate(ds):
        r = rows[k]
        assert np.array_equal(r[0:6], d["init_state"][:6])
        assert np.array_equal(r[6:9], d["goal"]) and r[9] == d["heading_goal"]
        assert np.array_equal(r[10:15], d["current"])
        nk = len(d["capsules"])
        assert np.array_equal(r[15:15 + 7 * nk].reshape(nk, 7), d["capsules"])
        assert np.array_equal(r[15 + 7 * nk:15 + 7 * nc].reshape(-1, 7), np.tile(UNUSED_CAPSULE, (nc - nk, 1)))
        assert np.array_equal(r[15 + 7 * nc:W].reshape(ns, 4), np.tile(UNUSED_SPHERE, (ns, 1)))
        assert np.all(r[W:] == 0)
    f32 = pack(np.zeros((3, 6)), np.zeros((3, 3)), np.zeros(3), 5, 3, dtype=torch.float32)
    assert (f32.shape[1] * 4) % 16 == 0 and f32.shape[1] >= row_width(5, 3)


# ------------------------------------------------------------------------------------------- GPU helpers
def _cfg():
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    return cfg


def _random_bank(env, K, seed, current=False):
    """K distinct valid rows: poses 5..20 m from the goal, live obstacles near the goal, some unused slots."""
    from gym_dockauv_b200.scenario_bank import ScenarioBank, UNUSED_CAPSULE, UNUSED_SPHERE
    rng = np.random.default_rng(seed)
    goal = rng.uniform(-3, 3, (K, 3))
    pose = np.concatenate([goal + rng.uniform(-15, 15, (K, 3)), rng.uniform(-0.5, 0.5, (K, 3))], 1)
    heading = rng.uniform(-np.pi, np.pi, K)
    cur = np.zeros((K, 5))
    if current:
        cur[:, 0] = 0.5
        cur[:, 1:3] = rng.uniform(-1.5, 1.5, (K, 2))
        cur[:, 3:5] = rng.uniform(0, 1, (K, 1))
    nc, ns = env.n_capsules, env.n_spheres
    caps = np.zeros((K, nc, 7))
    for k in range(nc):
        c = goal + rng.uniform(-10, 10, (K, 3))
        caps[:, k, 0:3] = c
        caps[:, k, 3:6] = c + rng.uniform(-3, 3, (K, 3))
        caps[:, k, 6] = rng.uniform(0.3, 1.5, K)
    sph = np.zeros((K, ns, 4))
    for s in range(ns):
        sph[:, s, 0:3] = goal + rng.uniform(-10, 10, (K, 3))
        sph[:, s, 3] = rng.uniform(0.3, 1.5, K)
    if nc:
        caps[::3, nc - 1] = UNUSED_CAPSULE
    if ns:
        sph[::4, ns - 1] = UNUSED_SPHERE
    return ScenarioBank(env, pose, goal, heading, current=cur, capsules=caps, spheres=sph)


def _env_rows(env, idx):
    """What a bank row holds, read back from the env's buffers for envs idx: [n, W]"""
    import torch
    nc, ns = env.n_capsules, env.n_spheres
    parts = [env.state[:6, idx], env.goal[:, idx], env.heading_goal[idx][None], env.current[:, idx],
             env.capsules[:7 * nc, idx], env.spheres[:4 * ns, idx]]
    return torch.cat(parts, 0).t()


def _check_rows(env, bank, idx, rows, where=""):
    import torch
    idx = torch.as_tensor(np.asarray(idx, dtype=np.int64), device=env.device)
    rows_t = torch.as_tensor(np.asarray(rows, dtype=np.int64), device=env.device)
    got = _env_rows(env, idx)
    want = bank.rows[rows_t, :bank.width]
    assert torch.equal(got.view(torch.int64 if env.dtype == torch.float64 else torch.int32),
                       want.view(torch.int64 if env.dtype == torch.float64 else torch.int32)), where
    assert torch.all(env.state[6:, idx] == 0) and torch.all(env.u_prev[:, idx] == 0), where
    assert torch.all(env.t_steps[idx] == 0) and torch.all(env.ep_return[idx] == 0), where
    assert torch.equal(env.bank_row[idx], rows_t.to(torch.int32)), where


# ------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("weighted", [False, True])
def test_reset_takes_the_predicted_rows_exactly(precision, weighted):
    import torch
    from gym_dockauv_b200 import envs
    N, K, seed = 1000, 97, 0x1234_5678_9ABC
    env = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=1, precision=precision, n_synthetic_spheres=3)
    bank = _random_bank(env, K, 5)
    w = None
    if weighted:
        w = np.random.default_rng(2).uniform(0, 1, K)
        w[::5] = 0.0
    env.set_scenario_bank(bank, weights=None if w is None else torch.as_tensor(w))
    cdf = None if w is None else np.cumsum(w)
    gids = np.arange(N, dtype=np.uint64)
    prev = np.full(N, -1)
    env.reset(seed=seed)
    for ep in range(3):
        if ep:
            env.reset()
        rows = predict_rows(seed, gids, ep, K, cdf)
        _check_rows(env, bank, np.arange(N), rows, (precision, weighted, ep))
        assert np.array_equal(env.ended_bank_row.cpu().numpy(), prev)
        assert np.all(env.episode.cpu().numpy() == ep + 1)
        assert torch.all(env.obs == 0)
        if w is not None:
            assert not np.any(w[rows] == 0)
        prev = rows
    assert len(np.unique(prev)) > K // 2
    env.close()


LAYOUT_CASES = [("ObstaclesDocking3d", dict(n_synthetic_spheres=3), False),
                ("ObstaclesDocking3d", dict(n_synthetic_spheres=8, n_capsules=8), True),
                ("ObstaclesCurrentDocking3d", dict(n_synthetic_spheres=3), True)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw,weighted", LAYOUT_CASES)
def test_every_layout_resets_from_the_bank_inside_the_step(name, kw, weighted):
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.scenario_bank import ScenarioBank
    N, K, seed = 1000, 300, 11
    layouts = ("thread_per_env", "warp_rays", "pipeline")
    es = [envs.SCENARIOS[name](_cfg(), num_envs=N, seed=seed, layout=l, **kw) for l in layouts]
    bank = ScenarioBank.from_builtin(es[0], K, seed=77)
    w = np.random.default_rng(0).uniform(0, 2, K) if weighted else None
    cdf = None if w is None else np.cumsum(w)
    for e in es:
        e.set_scenario_bank(bank, weights=None if w is None else torch.as_tensor(w))
        e.reset()
        _check_rows(e, bank, np.arange(N), predict_rows(seed, np.arange(N, dtype=np.uint64), 0, K, cdf))
        e.t_steps += torch.randint(985, 1001, (N,), device=e.device, dtype=torch.int32,
                                   generator=torch.Generator(device=e.device).manual_seed(3))
    gen = torch.Generator(device="cuda").manual_seed(0)
    n_done = 0
    for t in range(24):
        a = torch.rand(N, es[0].n_actions, device="cuda", generator=gen) * 2 - 1
        outs = [e.step(a) for e in es]
        o0, r0, d0, i0 = outs[0]
        for (o, r, d, info), l in zip(outs[1:], layouts[1:]):
            assert torch.equal(d0, d) and torch.equal(i0["cond_bits"], info["cond_bits"]), (name, l, t)
            assert torch.equal(o0, o), (name, l, t)
            assert rel_err(r.cpu().numpy(), r0.cpu().numpy()) < 1e-12, (name, l, t)
        ended = np.flatnonzero(d0.cpu().numpy())
        n_done += len(ended)
        if len(ended):
            ep_before = es[0].episode[torch.as_tensor(ended, device="cuda")].cpu().numpy().astype(np.int64) - 1
            rows = predict_rows(seed, ended.astype(np.uint64), ep_before, K, cdf)
            for e, l in zip(es, layouts):
                _check_rows(e, bank, ended, rows, (name, l, t))
        for e, l in zip(es[1:], layouts[1:]):
            assert rel_err(e.state.cpu().numpy(), es[0].state.cpu().numpy()) < 1e-12, (name, l, t)
            assert torch.equal(e.ended_bank_row, es[0].ended_bank_row), (name, l, t)
    assert n_done >= N
    for e in es:
        e.close()


def _follow_oracle(scenario, cfg, N, n_synth, make_bank, steps, n_sample=None, seed=2024, **env_kw):
    """GPU batch with a bank vs the CPU oracle; the predicted row is injected into the oracle env at every reset."""
    import torch
    from gym_dockauv_b200 import envs
    from oracle import oracle as orc
    env = envs.SCENARIOS[scenario](cfg, num_envs=N, seed=seed, n_synthetic_spheres=n_synth, **env_kw)
    bank, w = make_bank(env)
    cdf = None if w is None else np.cumsum(w)
    env.set_scenario_bank(bank, weights=None if w is None else torch.as_tensor(w))
    env.reset()
    if n_sample is None:
        ids = np.arange(N, dtype=np.uint64)
    else:
        ids = np.sort(np.random.default_rng(seed).choice(N, n_sample, replace=False)).astype(np.uint64)
        ids[0], ids[-1] = 0, N - 1
    n = len(ids)
    bo = orc.BatchOracle(cfg, scenario, n, seed=seed, n_extra_spheres=n_synth, env_ids=ids)
    rows_h = bank.rows[:, :bank.width].double().cpu().numpy()
    nc, ns = env.n_capsules, env.n_spheres

    def inject(k_list, rows):
        for k, r in zip(k_list, rows):
            row = rows_h[r]
            st = np.zeros(12)
            st[:6] = row[:6]
            orc.set_env(bo.envs[int(k)], st, row[6:9], row[9], row[15:15 + 7 * nc].reshape(nc, 7),
                        row[15 + 7 * nc:15 + 7 * nc + 4 * ns].reshape(ns, 4), row[10:15])

    inject(range(n), predict_rows(seed, ids, 0, bank.n_rows, cdf))
    idx = torch.as_tensor(ids.astype(np.int64), device=env.device)
    assert rel_err(env.state[:, idx].t().cpu().numpy(), bo.field("state")) == 0
    gen = torch.Generator(device=env.device).manual_seed(seed)
    worst = dict(state=0.0, reward=0.0, obs=0.0)
    n_resets = 0
    for t in range(steps):
        a = torch.rand(N, env.n_actions, device=env.device, generator=gen) * 2 - 1
        obs, reward, done, info = env.step(a)
        robs, rrew, rdone, _ = bo.step(a[idx].cpu().numpy())
        assert np.array_equal(done[idx].cpu().numpy(), rdone), (scenario, t)
        assert np.array_equal(info["cond_bits"][idx].cpu().numpy(), bo.cond_bits), (scenario, t)
        worst["reward"] = max(worst["reward"], rel_err(reward[idx].cpu().numpy(), rrew))
        worst["obs"] = max(worst["obs"], float(np.max(np.abs(obs[idx].cpu().numpy() - robs))))
        ended = np.flatnonzero(rdone)
        if len(ended):
            ep_before = env.episode[idx[torch.as_tensor(ended, device=env.device)]].cpu().numpy().astype(np.int64) - 1
            rows = predict_rows(seed, ids[ended], ep_before, bank.n_rows, cdf)
            assert np.array_equal(env.bank_row[idx].cpu().numpy()[ended], rows)
            inject(ended, rows)
            n_resets += len(ended)
        # after the injection, robs of re-initialised envs is the zero reset observation on both sides
        if t % 8 == 7 or t == steps - 1:
            worst["state"] = max(worst["state"], rel_err(env.state[:, idx].t().cpu().numpy(), bo.field("state")))
    assert n_resets > 0, scenario
    assert worst["state"] < 1e-9 and worst["reward"] < 1e-9 and worst["obs"] < 2e-7, (scenario, worst)
    env.close()
    return n_resets


@pytest.mark.gpu
@pytest.mark.parametrize("N,n_sample", [(384, None), (1 << 20, 4096)])
def test_oracle_follows_envs_across_bank_resets(N, n_sample):
    import torch
    from gym_dockauv_b200.scenario_bank import ScenarioBank
    cfg = _cfg()

    def make(env):
        bank = ScenarioBank.from_builtin(env, 4096, seed=9)
        # shorter episodes: start every row near the goal so some reach it, and end others on max_t
        return bank, np.random.default_rng(1).uniform(0.5, 1.5, 4096)

    cfg["max_timesteps"] = 120
    _follow_oracle("ObstaclesDocking3d", cfg, N, 3, make, 300, n_sample=n_sample)
    assert torch.cuda.is_available()


@pytest.mark.gpu
@pytest.mark.parametrize("scenario", ["CapsuleDocking3d", "ObstaclesDocking3d", "ObstaclesCurrentDocking3d"])
def test_bank_from_the_reference_generator(scenario):
    from gym_dockauv_b200.reference_reset import ReferenceResetStream
    from gym_dockauv_b200.scenario_bank import ScenarioBank
    cfg = _cfg()
    cfg["max_timesteps"] = 80

    def make(env):
        return ScenarioBank.from_generator(env, ReferenceResetStream(scenario, cfg, seed=4).generate, 512), None

    _follow_oracle(scenario, cfg, 256, 0, make, 200)


@pytest.mark.gpu
def test_shards_draw_the_rows_of_one_batch():
    import torch
    from gym_dockauv_b200 import envs
    N, seed = 1000, 21
    whole = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=seed, n_synthetic_spheres=3)
    parts = [envs.ObstaclesDocking3d(_cfg(), num_envs=N // 2, seed=seed, env_id0=b, n_synthetic_spheres=3)
             for b in (0, N // 2)]
    bank = _random_bank(whole, 211, 3)
    w = torch.rand(211, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    for e in [whole] + parts:
        e.set_scenario_bank(bank, weights=w)
    for _ in range(3):
        for e in [whole] + parts:
            e.reset()
        assert torch.equal(whole.bank_row, torch.cat([p.bank_row for p in parts]))
        assert torch.equal(whole.state, torch.cat([p.state for p in parts], 1))
        assert torch.equal(whole.capsules, torch.cat([p.capsules for p in parts], 1))
    for e in [whole] + parts:
        e.close()


@pytest.mark.gpu
def test_weighted_draw_follows_the_weights():
    import torch
    from scipy import stats
    from gym_dockauv_b200 import envs
    N, K, R = 65536, 256, 16
    env = envs.SimpleDocking3d(_cfg(), num_envs=N, seed=8)
    bank = _random_bank(env, K, 1)
    w = np.random.default_rng(5).uniform(0.2, 3.0, K)
    w[np.random.default_rng(6).choice(K, 32, replace=False)] = 0.0
    env.set_scenario_bank(bank, weights=torch.as_tensor(w))
    counts = torch.zeros(K, dtype=torch.int64, device=env.device)
    for _ in range(R):
        env.reset()
        counts += torch.bincount(env.bank_row.long(), minlength=K)
    counts = counts.cpu().numpy()
    assert counts.sum() == N * R
    assert np.all(counts[w == 0] == 0)
    live = w > 0
    expected = N * R * w[live] / w.sum()
    chi2 = float(((counts[live] - expected) ** 2 / expected).sum())
    assert stats.chi2.sf(chi2, live.sum() - 1) > 1e-4, chi2
    env.close()


@pytest.mark.gpu
def test_same_pointer_updates_keep_every_graph():
    import torch
    from gym_dockauv_b200 import envs
    N, K, T, seed = 1000, 64, 4, 13
    env = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=seed, n_synthetic_spheres=3)
    bank = _random_bank(env, K, 2)
    w = np.ones(K)
    env.set_scenario_bank(bank, weights=torch.as_tensor(w))
    env.reset()
    gen = torch.Generator(device="cuda").manual_seed(0)
    acts = torch.empty(T, N, 6, device="cuda")
    obs = torch.zeros(T, N, env.n_observations, device="cuda")
    rew = torch.zeros(T, N, dtype=env.dtype, device="cuda")
    done = torch.zeros(T, N, dtype=torch.uint8, device="cuda")
    act = torch.empty(N, 6, device="cuda")            # one action tensor: one step graph

    def run():
        env.t_steps.fill_(env.max_timesteps)          # every episode ends at the next step
        env.step(act.uniform_(-1, 1, generator=gen))
        acts.uniform_(-1, 1, generator=gen)
        env.rollout(acts, obs, rew, done)

    run()
    sg, rg = env.step_graph_captures(), env.rollout_captures()
    # rewrite rows and weights in place and publish them with same-pointer calls
    g = bank.field("goal")
    bank.field("pose")[:, :3] += 1.0
    g += 0.5
    bank.field("capsules")[:, :, :6] += 0.5
    bank.field("spheres")[:, :, :3] += 0.5
    w = np.zeros(K)
    w[[3, 17, 40]] = [1.0, 2.0, 0.5]
    env.set_scenario_bank(bank)            # same tensor: published in place (also re-publishes the weights below)
    env.set_scenario_weights(torch.as_tensor(w))
    env.t_steps.fill_(env.max_timesteps)
    ep_before = env.episode.cpu().numpy().astype(np.int64)
    env.step(act.uniform_(-1, 1, generator=gen))
    rows = predict_rows(seed, np.arange(N, dtype=np.uint64), ep_before, K, np.cumsum(w))
    assert set(np.unique(rows)) <= {3, 17, 40}
    _check_rows(env, bank, np.arange(N), rows)
    acts.uniform_(-1, 1, generator=gen)
    env.rollout(acts, obs, rew, done)
    assert env.step_graph_captures() == sg and env.rollout_captures() == rg
    # new pointers: captured once more
    env.set_scenario_bank(_random_bank(env, K, 3))
    run()
    assert env.step_graph_captures() == sg + 1 and env.rollout_captures() == rg + 1
    env.close()


@pytest.mark.gpu
def test_bad_banks_are_refused_and_the_previous_bank_stays():
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200._capi import DockauvError
    N, K = 256, 32
    env = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=3, n_synthetic_spheres=3)
    good = _random_bank(env, K, 0)
    env.set_scenario_bank(good)

    def refused(bank, weights, row, word):
        with pytest.raises(DockauvError) as ei:
            env.set_scenario_bank(bank, weights=weights)
        msg = str(ei.value)
        assert f"row {row}" in msg and word in msg, msg
        assert env._bank[0] is good.rows
        env.reset(seed=3)
        _check_rows(env, good, np.arange(N), predict_rows(3, np.arange(N, dtype=np.uint64), 0, K))

    b = _random_bank(env, K, 1)
    b.rows[5, 2] = float("nan")
    refused(b, None, 5, "pose z")
    b = _random_bank(env, K, 1)
    b.field("capsules")[7, 0, 0] = b.field("goal")[7, 0] + 3000.0
    refused(b, None, 7, "capsule 0")
    b = _random_bank(env, K, 1)
    refused(b, torch.as_tensor(np.r_[np.ones(9), -0.5, np.ones(K - 10)]), 9, "cdf")
    refused(b, torch.zeros(K), K - 1, "cdf")
    b.field("current")[3, 0] = 0.5
    refused(b, None, 3, "force_current")
    # the same row on a handle that evaluates the current is accepted
    env2 = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=3, n_synthetic_spheres=3, force_current=True)
    env2.set_scenario_bank(b)
    env2.close()
    # weights refused on the bank that is set: the old weights stay in effect
    env.set_scenario_bank(good, weights=torch.ones(K))
    with pytest.raises(DockauvError):
        env.set_scenario_weights(torch.zeros(K))
    assert float(env._bank[1][-1]) == K
    env.close()


@pytest.mark.gpu
def test_cleared_bank_resets_like_a_handle_that_never_had_one():
    import torch
    from gym_dockauv_b200 import envs
    N = 1000
    a, b = [envs.ObstaclesCurrentDocking3d(_cfg(), num_envs=N, seed=6, n_synthetic_spheres=3) for _ in range(2)]
    a.set_scenario_bank(_random_bank(a, 50, 0, current=True))
    a.reset()
    a.step(torch.zeros(N, 6, device="cuda"))
    a.clear_scenario_bank()
    assert a.bank_row is None
    gen = torch.Generator(device="cuda").manual_seed(1)
    for e in (a, b):
        e.reset(seed=44)
        e.t_steps += 995
    for t in range(12):
        act = torch.rand(N, 6, device="cuda", generator=gen) * 2 - 1
        (o0, r0, d0, _), (o1, r1, d1, _) = a.step(act), b.step(act)
        assert torch.equal(d0, d1) and torch.equal(o0, o1) and torch.equal(r0, r1), t
    for f in ("state", "goal", "heading_goal", "current", "capsules", "spheres", "episode", "t_steps", "u_prev"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    a.close()
    b.close()


@pytest.mark.gpu
def test_taps_record_the_bank_row_after_an_auto_reset():
    import torch
    from gym_dockauv_b200 import envs
    N, K, seed = 1000, 40, 5
    env = envs.ObstaclesDocking3d(_cfg(), num_envs=N, seed=seed, n_synthetic_spheres=3)
    bank = _random_bank(env, K, 4)
    env.set_scenario_bank(bank)
    env.reset()
    ids = [3, 500, 999]
    ring = env.set_taps(ids, capacity=8)
    env.t_steps[ids] = env.max_timesteps             # the tapped envs end at the first step
    env.step(torch.zeros(N, 6, device="cuda"))
    rows = env.bank_row[ids].long()
    env.step(torch.zeros(N, 6, device="cuda"))
    torch.cuda.synchronize()
    assert int(ring["count"]) == 2
    W = bank.width
    scene = torch.cat([bank.rows[rows, 6:10], bank.rows[rows, 15:W]], 1).t()       # goal, heading, capsules, spheres
    assert torch.equal(ring["pre_scene"][1], scene)
    assert torch.equal(ring["pre_state"][1][:6], bank.rows[rows, :6].t())
    assert torch.equal(ring["pre_current"][1], bank.rows[rows, 10:15].t())
    env.close()


@pytest.mark.gpu
def test_curriculum_example_runs():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "ppo_scenario_curriculum.py"), "--envs", "4096",
                        "--steps", "16", "--iters", "2", "--rows", "512"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("iter")]
    assert len(lines) == 2
    caps = [int(l.split("step-graph captures")[1].split()[0]) for l in lines]
    assert caps[0] == caps[1], lines
