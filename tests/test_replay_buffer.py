"""Replay ring and fused minibatch sampler of the off-policy (SAC) caller: argument checks of dockauv_replay_sample and
DeviceReplayBuffer on the CPU; on the GPU, equality with SB3's ``_store_transition`` arrays built from plain steps, the
valid range, uniformity and determinism of the draws, the two-stream large batch, step-graph reuse and the example."""
import ctypes as C
import os
import re
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------- CPU: argument checks
def _sample_args(**over):
    from gym_dockauv_b200.params import DockauvReplayRing, DockauvReplaySample
    fake = 1 << 20                       # 16-byte aligned, never dereferenced: every call below is refused first
    ring = DockauvReplayRing(*([fake] * 5))
    out = DockauvReplaySample(*([fake] * 5 + [None]))
    a = dict(ring=C.byref(ring), reward_precision=0, n_slots=8, n_envs=1024, n_obs=32, n_u=6, t_first=3, n_valid=7,
             batch=256, seed=0, draw=0, out=C.byref(out), stream=None)
    a["_keep"] = (ring, out)
    for k, v in over.items():
        if k.startswith("ring_"):
            setattr(ring, k[5:], v)
        elif k.startswith("out_"):
            setattr(out, k[4:], v)
        else:
            a[k] = v
    return a


def _call(a):
    from gym_dockauv_b200 import _capi
    lib = _capi.load()
    rc = lib.dockauv_replay_sample(a["ring"], a["reward_precision"], a["n_slots"], a["n_envs"], a["n_obs"], a["n_u"],
                                   a["t_first"], a["n_valid"], a["batch"], a["seed"], a["draw"], a["out"], a["stream"])
    return rc, lib.dockauv_last_error().decode()


@pytest.mark.parametrize("over,word", [
    (dict(ring=None), "ring"), (dict(out=None), "out"),
    (dict(ring_obs=None), "ring"), (dict(ring_terminal_obs=None), "ring"), (dict(ring_actions=None), "ring"),
    (dict(ring_reward=None), "ring"), (dict(ring_done=None), "ring"),
    (dict(out_obs=None), "out"), (dict(out_actions=None), "out"), (dict(out_next_obs=None), "out"),
    (dict(out_done=None), "out"), (dict(out_reward=None), "out"),
    (dict(n_slots=1, n_valid=1), "n_slots"), (dict(n_slots=0, n_valid=1), "n_slots"),
    (dict(n_valid=0), "n_valid"), (dict(n_valid=8), "n_valid"), (dict(n_valid=-1), "n_valid"),
    (dict(batch=0), "batch"), (dict(batch=-5), "batch"),
    (dict(reward_precision=2), "reward_precision"), (dict(reward_precision=-1), "reward_precision"),
    (dict(n_obs=0), "n_obs"), (dict(n_obs=16 + 256 + 1), "n_obs"), (dict(n_u=0), "n_u"), (dict(n_u=9), "n_u"),
    (dict(n_envs=0), "n_envs"), (dict(t_first=-1), "t_first"),
    (dict(ring_terminal_obs=(1 << 20) + 4), "aligned"), (dict(out_next_obs=(1 << 20) + 8), "aligned"),
])
def test_replay_sample_refuses_bad_arguments(over, word):
    rc, msg = _call(_sample_args(**over))
    assert rc == -1, over
    assert word in msg, (over, msg)


def test_replay_sample_header_struct_fields():
    """The ctypes mirrors carry the header's fields in the header's order."""
    from gym_dockauv_b200.params import DockauvReplayRing, DockauvReplaySample
    text = open(os.path.join(ROOT, "include", "dockauv.h")).read()
    ring = re.search(r"typedef struct DockauvReplayRing \{(.*?)\} DockauvReplayRing;", text, re.S).group(1)
    assert [f for f, _ in DockauvReplayRing._fields_] == re.findall(r"\*(\w+);", ring)
    smp = re.search(r"typedef struct DockauvReplaySample \{(.*?)\} DockauvReplaySample;", text, re.S).group(1)
    assert [f for f, _ in DockauvReplaySample._fields_] == re.findall(r"\*(\w+)", re.sub(r"/\*.*?\*/", "", smp))


@pytest.mark.parametrize("n_slots", [1, 65, 0])
def test_buffer_refuses_slot_counts_before_allocating(n_slots):
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    stand_in = types.SimpleNamespace()       # no attribute of the env is touched before the check
    with pytest.raises(ValueError, match="n_slots.*graph"):
        DeviceReplayBuffer(stand_in, n_slots)


# ------------------------------------------------------------------------------------------- GPU
def _cfg64():
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    return cfg


def _policy(n_obs, n_u, seed=0):
    """tanh-linear policy written without a matrix product, so two envs fed equal observations get equal actions."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    w = torch.randn(n_obs, n_u, device="cuda", generator=g) * 0.8
    b = torch.randn(n_u, device="cuda", generator=g) * 0.3
    return lambda obs: torch.tanh((obs.unsqueeze(2) * w).sum(1) + b)


def _sb3_arrays(env, policy, T):
    """SB3 _store_transition from plain env.step + clones: obs_t, a_t, r_t (f32), d_t, next_obs_t."""
    obs = env.reset().clone()
    O, A, R, D, NX = [], [], [], [], []
    for _ in range(T):
        a = policy(obs)
        new_obs, r, d, info = env.step(a)
        nx = new_obs.clone()
        m = d.bool()
        nx[m] = info["terminal_observation"][m]
        O.append(obs.cpu().numpy()); A.append(a.cpu().numpy()); R.append(r.cpu().numpy().astype(np.float32))
        D.append(d.cpu().numpy().astype(np.float32)); NX.append(nx.cpu().numpy())
        obs = new_obs.clone()
    return [np.stack(x) for x in (O, A, R, D, NX)]


def _check_rows(buf, smp, idx, ref, T):
    O, A, R, D, NX = ref
    S, N = buf.n_slots, buf.env.num_envs
    idx = idx.cpu().numpy()
    slot, env_i = idx // N, idx % N
    lo = max(0, T - (S - 1))
    t = lo + (slot - lo % S) % S           # the one valid t with t % S == slot
    assert np.all((t >= lo) & (t < T)) and np.all(t % S == slot)
    assert np.array_equal(smp.observations.cpu().numpy(), O[t, env_i])
    assert np.array_equal(smp.actions.cpu().numpy(), A[t, env_i])
    assert np.array_equal(smp.rewards.cpu().numpy()[:, 0], R[t, env_i])
    assert np.array_equal(smp.dones.cpu().numpy()[:, 0], D[t, env_i])
    assert np.array_equal(smp.next_observations.cpu().numpy(), NX[t, env_i])
    return t, env_i


@pytest.mark.gpu
def test_buffer_equals_sb3_store_transition():
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    N, S, T = 4096, 8, 30
    kw = dict(num_envs=N, seed=5, n_synthetic_spheres=3)
    e1 = envs.ObstaclesDocking3d(_cfg64(), **kw)
    pol = _policy(e1.n_observations, e1.n_actions)
    buf = DeviceReplayBuffer(e1, S, seed=11)
    buf.reset_env()
    buf.collect(pol, T)
    e2 = envs.ObstaclesDocking3d(_cfg64(), **kw)
    ref = _sb3_arrays(e2, pol, T)
    O, D = ref[0], ref[3]
    assert D.sum() > 50, "the run must contain auto-resets"
    smp, idx = buf.sample(1 << 18, return_index=True)
    t, env_i = _check_rows(buf, smp, idx, ref, T)
    # sampled rows include episode ends (next = terminal observation) and episode starts
    d_rows = smp.dones.cpu().numpy()[:, 0] == 1
    assert d_rows.sum() > 0
    starts = (t > 0) & (D[np.maximum(t - 1, 0), env_i] == 1)
    assert starts.sum() > 0
    assert np.all(smp.observations.cpu().numpy()[starts] == 0)
    # the first observation of every new episode is the all-zero reset observation
    assert np.all(O[1:][D[:-1] == 1] == 0)
    e1.close(); e2.close()


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 7, 11])        # S = 8: T = 1, S - 1, S + 3
def test_valid_range(T):
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    N, S = 512, 8
    env = envs.ObstaclesDocking3d(_cfg64(), num_envs=N, seed=2, n_synthetic_spheres=3)
    buf = DeviceReplayBuffer(env, S)
    buf.reset_env()
    buf.collect(_policy(env.n_observations, env.n_actions), T)
    assert buf.n_valid == min(T, S - 1) and buf.size() == buf.n_valid * N
    _, idx = buf.sample(1 << 16, return_index=True)
    slot = (idx // N).cpu().numpy()
    assert not np.any(slot == T % S), "drew from the slot the next step overwrites"
    if T < S:
        assert slot.max() < T
    assert len(np.unique(slot)) == min(T, S - 1)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_uniform_and_deterministic(precision):
    import torch
    from scipy.stats import chisquare
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    N, S = 256, 9
    env = envs.ObstaclesDocking3d(_cfg64(), num_envs=N, seed=4, n_synthetic_spheres=3, precision=precision)
    buf = DeviceReplayBuffer(env, S, seed=1234)
    buf.reset_env()
    buf.collect(_policy(env.n_observations, env.n_actions), 12)
    _, idx = buf.sample(1 << 22, return_index=True)
    counts = np.bincount(idx.cpu().numpy(), minlength=S * N).reshape(S, N)
    overwritten = buf.t % S
    assert counts[overwritten].sum() == 0
    bins = np.delete(counts, overwritten, axis=0).ravel()
    assert bins.size == 2048
    assert chisquare(bins).pvalue > 1e-4
    # same (seed, draw): bit-identical outputs; another draw: other rows
    buf.draws = 3
    a, ia = buf.sample(4096, return_index=True)
    buf.draws = 3
    b, ib = buf.sample(4096, return_index=True)
    c, ic = buf.sample(4096, return_index=True)
    assert torch.equal(ia, ib) and all(torch.equal(x, y) for x, y in zip(a, b))
    assert not torch.equal(ia, ic)
    assert buf.draws == 5
    # the reward is the env-dtype ring value rounded to float32 once
    flat_r = buf.rewards.reshape(-1)[ia]
    assert torch.equal(a.rewards[:, 0], flat_r.to(torch.float32))
    env.close()


@pytest.mark.gpu
def test_large_batch_two_streams():
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    N, S, T = 262_144, 4, 6          # stepped in two halves on two streams
    kw = dict(num_envs=N, seed=9, n_synthetic_spheres=3)
    e1 = envs.ObstaclesDocking3d(_cfg64(), **kw)
    pol = _policy(e1.n_observations, e1.n_actions, seed=3)
    buf = DeviceReplayBuffer(e1, S, seed=7)
    buf.reset_env()
    buf.collect(pol, T)
    e2 = envs.ObstaclesDocking3d(_cfg64(), **kw)
    ref = _sb3_arrays(e2, pol, T)
    smp, idx = buf.sample(4096, return_index=True)
    _check_rows(buf, smp, idx, ref, T)
    e1.close(); e2.close()


@pytest.mark.gpu
def test_ring_reuses_step_graphs():
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.replay import DeviceReplayBuffer
    S = 8
    env = envs.ObstaclesDocking3d(_cfg64(), num_envs=2048, seed=1, n_synthetic_spheres=3)
    buf = DeviceReplayBuffer(env, S)
    buf.reset_env()
    pol = _policy(env.n_observations, env.n_actions)
    n0 = env.step_graph_captures()
    buf.collect(pol, S)
    lap = env.step_graph_captures()
    assert lap - n0 <= S
    for _ in range(3):
        buf.collect(pol, 5)
        buf.sample(1024)
    assert env.step_graph_captures() == lap
    env.close()


@pytest.mark.gpu
def test_sac_example_runs():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "sac_device_replay.py"), "--envs", "2048",
                        "--iters", "2"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("iter")]
    assert len(lines) == 2, r.stdout
    for ln in lines:
        nums = [float(x) for x in re.findall(r"[-+]?(?:\d+\.?\d*(?:e[-+]?\d+)?|nan|inf)", ln, re.I)]
        assert nums and all(np.isfinite(nums)), ln
