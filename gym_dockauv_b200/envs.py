"""Batched docking environments: the reference's gym.Env contract (gym_dockauv/envs/docking3d.py:31-402),
vectorised over N independent envs that live in HBM and are stepped by a short sequence of sm_100a kernel launches
(dynamics + cull + finish, rays + finish, episode end; include/dockauv.h).

    env = ObstaclesDocking3d(env_config, num_envs=1 << 20, device="cuda:0")
    obs = env.reset(seed=0)                      # f32 [N, n_obs], all zeros like the reference's reset()
    obs, reward, done, info = env.step(actions)  # actions: [N, n_u] cuda tensor (float32 or float64)

Same scenario class names, same ``env_config`` dict, same observation / reward / done semantics, including the
reference's quirks (zero observation after reset, max-timestep done on step max_timesteps + 1, raw action in
the action penalty, float32 observation cast, hard-coded safety radius).  Finished envs are re-initialised in
the same launch (SB3 VecEnv behaviour): ``obs`` rows of finished envs are the (all-zero) reset observation and
``info["terminal_observation"]`` holds their last real observation.

PyTorch is used for device memory and streams only; all arithmetic of the step path runs in
libdockauv_b200.so (include/dockauv.h).  There is no CPU path.
"""
import ctypes as C

import numpy as np
import torch

from . import _capi
from .config import BASE_CONFIG, REGISTRATION_DICT
from .params import (ACT_F32, ACT_F64, F32, F64, MAX_TAPS, N_STATS, SCENARIO_IDS, STAT_NAMES, TAP_FIELDS, DockauvBuffers,
                     DockauvDebugOut, DockauvPolicyOut, DockauvRolloutOut, DockauvScenarioBank, DockauvStepOut,
                     DockauvTapBuffers, pack_params)

DONE_NAMES = ("Done-Goal_reached", "Done-out_pos", "Done-out_att", "Done-max_t", "Done-collision")


class Box:
    """Minimal stand-in for gym.spaces.Box (gym is not a dependency): low / high / shape / dtype / sample()."""

    def __init__(self, low, high, dtype=np.float32):
        self.low = np.asarray(low, dtype=dtype)
        self.high = np.asarray(high, dtype=dtype)
        self.shape = self.low.shape
        self.dtype = np.dtype(dtype)

    def sample(self):
        return np.random.uniform(self.low, self.high).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))

    def __repr__(self):
        return f"Box({self.low.min()}, {self.high.max()}, {self.shape}, {self.dtype})"


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class BaseDocking3d:
    """N independent docking envs of one scenario on one GPU."""

    scenario = None   # set by the subclasses

    def __init__(self, env_config=BASE_CONFIG, num_envs=1, device="cuda:0", precision="f64", seed=0, env_id0=0,
                 layout="auto", n_spheres=0, n_synthetic_spheres=0, n_capsules=None, vehicle_xml=None,
                 control_mode="joystick", cur_mu=0.005, cur_sigma=0.0, force_current=False, auto_reset=True,
                 debug_outputs=False, split_chunk_envs=0):
        if self.scenario is None:
            raise TypeError("instantiate one of the scenario classes (SimpleDocking3d, ObstaclesDocking3d, ...)")
        self._lib = _capi.load()
        self.config = env_config
        self._init_kwargs = dict(device=device, precision=precision, seed=seed, env_id0=env_id0, layout=layout,
                                 n_spheres=n_spheres, n_synthetic_spheres=n_synthetic_spheres, n_capsules=n_capsules,
                                 vehicle_xml=vehicle_xml, control_mode=control_mode, cur_mu=cur_mu, cur_sigma=cur_sigma,
                                 force_current=force_current, auto_reset=auto_reset, debug_outputs=debug_outputs,
                                 split_chunk_envs=split_chunk_envs)
        self.num_envs = int(num_envs)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _capi.DockauvError("gym_dockauv_b200 runs on CUDA devices only (no CPU fallback)")
        if not torch.cuda.is_available():
            raise _capi.DockauvError("no CUDA device available; gym_dockauv_b200 has no CPU fallback")
        if self.device.index is None:      # "cuda" -> the current device, so that tensors, handle and checks agree
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.precision = precision
        self.dtype = torch.float64 if precision == "f64" else torch.float32
        self.auto_reset = bool(auto_reset)
        self._params, meta = pack_params(
            env_config, self.scenario, precision=precision, seed=seed, env_id0=env_id0, layout=layout,
            n_capsules=n_capsules, n_spheres=n_spheres, n_synthetic_spheres=n_synthetic_spheres,
            vehicle_xml=vehicle_xml, control_mode=control_mode, cur_mu=cur_mu, cur_sigma=cur_sigma,
            force_current=force_current, split_chunk_envs=split_chunk_envs)
        self._meta = meta
        self.n_observations = meta["n_obs"]
        self.n_actions = meta["n_u"]
        self.n_rays = self._params.n_rays
        self.n_capsules = self._params.n_capsules
        self.n_spheres = self._params.n_spheres
        self.max_timesteps = self._params.max_timesteps
        # spaces exactly as the reference declares them (docking3d.py:116-125); note LAUV's action_space is its
        # physical u_bound although step() expects normalised [-1, 1] actions -- reference quirk kept.
        ub = meta["u_bound"]
        self.action_space = Box(ub[:, 0], ub[:, 1], np.float32)
        lo = -np.ones(self.n_observations)
        lo[0] = 0
        lo[16:] = 0
        self.observation_space = Box(lo, np.ones(self.n_observations), np.float32)
        self.meta_data_done = list(DONE_NAMES)

        N, dev, dt = self.num_envs, self.device, self.dtype
        z = lambda *shape, dtype=dt: torch.zeros(*shape, dtype=dtype, device=dev)  # noqa: E731
        # persistent state, SoA [component][env]
        self.state = z(12, N)
        self.u_prev = z(max(self.n_actions, 1), N)
        self.goal = z(3, N)
        self.heading_goal = z(N)
        self.current = z(5, N)
        self.capsules = z(max(self.n_capsules * 7, 1), N)
        self.spheres = z(max(self.n_spheres * 4, 1), N)
        self.ep_return = z(N)
        self.t_steps = z(N, dtype=torch.int32)
        self.episode = z(N, dtype=torch.int32)
        # step outputs
        self.obs = z(N, self.n_observations, dtype=torch.float32)
        self.terminal_obs = z(N, self.n_observations, dtype=torch.float32)
        self.reward = z(N)
        self.done = z(N, dtype=torch.uint8)
        self.cond_bits = z(N, dtype=torch.uint8)
        self.ep_return_out = z(N)
        self.ep_len_out = z(N, dtype=torch.int32)
        self.delta_d = z(N)           # info["delta_d"] of the reference (docking3d.py:400)
        self.debug = None
        if debug_outputs:
            self.debug = dict(ray_dist=z(self.n_rays, N), reward_arr=z(13, N), euler_dot=z(3, N), nu_c=z(3, N),
                              nav=z(3, N), obs_f64=z(self.n_observations, N), state_dot=z(12, N))

        self._handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _capi.check(self._lib.dockauv_create(C.byref(self._params), N, self.device.index, C.byref(self._handle)))
        bufs = DockauvBuffers(*[_ptr(t) for t in (self.state, self.u_prev, self.goal, self.heading_goal,
                                                  self.current, self.capsules, self.spheres, self.ep_return,
                                                  self.t_steps, self.episode)])
        _capi.check(self._lib.dockauv_bind(self._handle, C.byref(bufs)))
        self._out = DockauvStepOut(*[_ptr(t) for t in (self.obs, self.reward, self.done, self.cond_bits,
                                                       self.terminal_obs, self.ep_return_out, self.ep_len_out,
                                                       self.delta_d)])
        self._dbg = None
        if self.debug is not None:
            self._dbg = DockauvDebugOut(*[_ptr(self.debug[k]) for k in ("ray_dist", "reward_arr", "euler_dot", "nu_c",
                                                                       "nav", "obs_f64", "state_dot")])
        self._host = None
        self.taps = None
        self._bank = None
        self.bank_row = None           # scenario bank: row of each env's running episode (-1 = not from the bank)
        self.ended_bank_row = None     # ... and of the episode its most recent reset ended
        self.t_total_steps = 0

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        if getattr(self, "_handle", None) is not None and self._handle.value:
            self._lib.dockauv_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ gym contract
    def reset(self, seed=None, return_info=False, options=None, mask=None):
        """Re-initialise all envs (or those where ``mask`` is non-zero) from the scenario's distributions and
        return the observation -- all zeros, as BaseDocking3d.reset does (docking3d.py:269,322).  ``seed`` restarts
        the counter-based random stream (episode counters back to 0) under a new key."""
        if seed is not None:
            self._params.seed = int(seed) & (2 ** 64 - 1)
            _capi.check(self._lib.dockauv_set_seed(self._handle, self._params.seed))
            self.episode.zero_()
        m = None
        if mask is not None:
            m = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _capi.check(self._lib.dockauv_reset(self._handle, _ptr(m), self._stream()))
        if m is None:
            self.obs.zero_()
        else:
            self.obs[m.bool()] = 0
        if return_info:
            return self.obs, {}
        return self.obs

    def step(self, actions, noise=None):
        """One env.step() for every env.  ``actions``: [N, n_u] CUDA tensor, float32 or float64 (the dtype selects
        the reference's dtype-dependent arithmetic, see include/dockauv.h).  Returns (obs, reward, done, info);
        all tensors are views of buffers that the next step overwrites."""
        adt = self._action_dtype(actions, (self.num_envs, self.n_actions))
        actions = actions.contiguous()
        if noise is not None:
            noise = noise.to(device=self.device, dtype=self.dtype).contiguous()
        _capi.check(self._lib.dockauv_step(self._handle, _ptr(actions), adt, _ptr(noise), C.byref(self._out),
                                           C.byref(self._dbg) if self._dbg is not None else None,
                                           int(self.auto_reset), self._stream()))
        self.t_total_steps += 1
        info = {"cond_bits": self.cond_bits, "terminal_observation": self.terminal_obs,
                "episode_return": self.ep_return_out, "episode_length": self.ep_len_out, "delta_d": self.delta_d}
        return self.obs, self.reward, self.done, info

    def _action_dtype(self, actions, shape):
        if actions.device != self.device:
            raise ValueError(f"actions live on {actions.device}, env on {self.device}; use step_host for host arrays")
        if tuple(actions.shape) != shape:
            raise ValueError(f"actions must have shape {shape}, got {tuple(actions.shape)}")
        if actions.dtype == torch.float32:
            return ACT_F32
        if actions.dtype == torch.float64:
            return ACT_F64
        raise TypeError("actions must be float32 or float64")

    def _check_tensors(self, *checks):
        """Every (tensor, shape, dtype): that shape and dtype, contiguous, on the env's device."""
        for t, shape, dt in checks:
            if tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous() or t.device != self.device:
                raise ValueError(f"tensor must be contiguous {dt} {shape} on {self.device}")

    def _check_rows(self, *rows):
        """Observation rows are written with 128-bit stores when n_obs is a multiple of 4 (include/dockauv.h)."""
        if self.n_observations % 4 == 0:
            for t in rows:
                if t is not None and t.data_ptr() % 16 != 0:
                    raise ValueError("obs / terminal_obs tensors must start at a 16-byte aligned address")

    def step_into(self, actions, obs, reward, done, cond_bits=None, terminal_obs=None, ep_return_out=None,
                  ep_len_out=None, delta_d_out=None):
        """``step`` with caller-chosen output tensors (e.g. row t of a device-resident rollout buffer): the kernel
        writes the observation / reward / done of this step straight into them, nothing is copied afterwards.
        ``obs`` f32 [N, n_obs], ``reward`` env dtype [N], ``done`` uint8 [N]; all contiguous, on the env's device."""
        adt = self._action_dtype(actions, (self.num_envs, self.n_actions))
        self._check_tensors((obs, (self.num_envs, self.n_observations), torch.float32),
                            (reward, (self.num_envs,), self.dtype), (done, (self.num_envs,), torch.uint8))
        self._check_rows(obs, terminal_obs)
        out = DockauvStepOut(*[_ptr(t) for t in (obs, reward, done, cond_bits, terminal_obs, ep_return_out,
                                                 ep_len_out, delta_d_out)])
        actions = actions.contiguous()
        _capi.check(self._lib.dockauv_step(self._handle, _ptr(actions), adt, None, C.byref(out), None,
                                           int(self.auto_reset), self._stream()))
        self.t_total_steps += 1

    def rollout(self, actions, obs, reward, done, cond_bits=None, terminal_obs=None, ep_return_out=None,
                ep_len_out=None, use_graph=True, delta_d_out=None):
        """T steps with actions known up front (``actions`` [T, N, n_u] on the device; random-action rollouts,
        replayed logs) in ONE library call: row t of ``obs`` [T, N, n_obs] / ``reward`` [T, N] / ``done`` [T, N]
        receives the outputs of step t.  With ``use_graph`` the launch sequence is captured into a CUDA graph the
        first time and replayed afterwards (same tensors -> same graph)."""
        T, N = int(actions.shape[0]), self.num_envs
        adt = self._action_dtype(actions, (T, N, self.n_actions))
        self._check_tensors((obs, (T, N, self.n_observations), torch.float32), (reward, (T, N), self.dtype),
                            (done, (T, N), torch.uint8), (actions, (T, N, self.n_actions), actions.dtype))
        out = self._rollout_out(obs, reward, done, cond_bits, terminal_obs, ep_return_out, ep_len_out, delta_d_out)
        _capi.check(self._lib.dockauv_rollout(self._handle, _ptr(actions), adt, T, C.byref(out), int(self.auto_reset),
                                              int(bool(use_graph)), self._stream()))
        self.t_total_steps += T

    def rollout_policy(self, policy, obs0, obs, reward, done, actions, values, log_probs, last_values=None,
                       cond_bits=None, terminal_obs=None, ep_return_out=None, ep_len_out=None, use_graph=True,
                       delta_d_out=None):
        """T steps of a closed loop in ONE library call (dockauv_rollout_policy): ``policy`` (a ``FusedActorCritic``)
        picks each step's actions on the device from ``obs0`` [N, n_obs] for step 0 and row t - 1 of ``obs`` after that.
        Row t of ``actions`` f32 [T, N, n_u] (raw samples, before clipping to ``action_space``), ``values`` and
        ``log_probs`` f32 [T, N] receive the policy's outputs, rows of ``obs`` / ``reward`` / ``done`` (and the optional
        outputs) the step's, as in ``rollout``; ``last_values`` f32 [N] (optional) receives V(row T - 1 of ``obs``).
        With ``use_graph`` the launch sequence is captured once per set of tensors and replayed; parameters updated in
        place are read by the replay."""
        policy.check_env(self)
        T, N = int(obs.shape[0]), self.num_envs
        checks = [(obs0, (N, self.n_observations), torch.float32), (obs, (T, N, self.n_observations), torch.float32),
                  (reward, (T, N), self.dtype), (done, (T, N), torch.uint8),
                  (actions, (T, N, self.n_actions), torch.float32), (values, (T, N), torch.float32),
                  (log_probs, (T, N), torch.float32)]
        if last_values is not None:
            checks.append((last_values, (N,), torch.float32))
        self._check_tensors(*checks)
        out = self._rollout_out(obs, reward, done, cond_bits, terminal_obs, ep_return_out, ep_len_out, delta_d_out)
        pout = DockauvPolicyOut(*[_ptr(t) for t in (actions, values, log_probs, last_values)])
        _capi.check(self._lib.dockauv_rollout_policy(self._handle, C.byref(policy.struct), _ptr(obs0), T, C.byref(out),
                                                     C.byref(pout), int(self.auto_reset), int(bool(use_graph)),
                                                     self._stream()))
        self.t_total_steps += T

    def _rollout_out(self, obs, reward, done, cond_bits, terminal_obs, ep_return_out, ep_len_out, delta_d_out):
        """The stacked outputs of ``rollout`` and ``rollout_policy`` as the library's struct."""
        self._check_rows(obs, terminal_obs)
        return DockauvRolloutOut(*[_ptr(t) for t in (obs, reward, done, cond_bits, terminal_obs, ep_return_out,
                                                     ep_len_out, delta_d_out)])

    def gae(self, rewards, values, last_values, dones, gamma, gae_lambda, advantages, returns):
        """Generalised advantage estimation over a stacked rollout on the device (dockauv_gae): ``rewards`` [T, N]
        in the env dtype or float32, ``values`` f32 [T, N], ``last_values`` f32 [N], ``dones`` uint8 [T, N];
        writes ``advantages`` and ``returns`` (f32 [T, N])."""
        T, N = rewards.shape
        prec = F64 if rewards.dtype == torch.float64 else F32
        if rewards.dtype not in (torch.float64, torch.float32):
            raise TypeError("rewards must be float64 or float32")
        self._check_tensors((values, (T, N), torch.float32), (last_values, (N,), torch.float32),
                            (dones, (T, N), torch.uint8), (advantages, (T, N), torch.float32),
                            (returns, (T, N), torch.float32), (rewards, (T, N), rewards.dtype))
        with torch.cuda.device(self.device):
            _capi.check(self._lib.dockauv_gae(_ptr(rewards), prec, _ptr(values), _ptr(last_values), _ptr(dones), T, N,
                                              float(gamma), float(gae_lambda), _ptr(advantages), _ptr(returns),
                                              self._stream()))

    def step_host(self, actions):
        """The same step for HOST actions (numpy [N, n_u], float32 / float64): actions are copied to the GPU,
        observations, rewards and done flags come back as numpy arrays backed by pinned memory.  This is the call
        a CPU-side training loop (SB3's VecEnv.step) makes; copies are pipelined with the kernel in chunks."""
        a = np.ascontiguousarray(actions)
        if a.shape != (self.num_envs, self.n_actions):
            raise ValueError(f"actions must have shape {(self.num_envs, self.n_actions)}, got {a.shape}")
        if a.dtype == np.float32:
            adt = ACT_F32
        elif a.dtype == np.float64:
            adt = ACT_F64
        else:
            raise TypeError("actions must be float32 or float64")
        if self._host is None:
            N = self.num_envs
            pin = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype).pin_memory()  # noqa: E731
            self._host = dict(obs=pin(N, self.n_observations, dtype=torch.float32), reward=pin(N, dtype=self.dtype),
                              done=pin(N, dtype=torch.uint8), cond=pin(N, dtype=torch.uint8))
        hb = self._host
        cur = torch.cuda.current_stream(self.device)
        if cur.cuda_stream != 0:       # the library orders itself after the legacy default stream only
            cur.synchronize()
        _capi.check(self._lib.dockauv_step_host(self._handle, C.c_void_p(a.ctypes.data), adt,
                                                C.c_void_p(hb["obs"].data_ptr()), C.c_void_p(hb["reward"].data_ptr()),
                                                C.c_void_p(hb["done"].data_ptr()), C.c_void_p(hb["cond"].data_ptr()),
                                                int(self.auto_reset), C.byref(self._out)))
        self.t_total_steps += 1
        return hb["obs"].numpy(), hb["reward"].numpy(), hb["done"].numpy().view(np.bool_), {"cond_bits": hb["cond"].numpy()}

    # ------------------------------------------------------------------ episode taps (dockauv_set_taps)
    def set_taps(self, env_ids, capacity):
        """Record every following ``step`` / ``step_into`` / ``rollout`` of the envs ``env_ids`` (local indices, at most
        1024) into a device ring of ``capacity`` steps, without changing any env's trajectory or output.  Returns the
        ring: a dict of device tensors, ``count`` (int64[1], steps recorded so far; step j sits in slot j % capacity)
        and per slot the pre-step inputs (``pre_state`` [S, 12, K], ``pre_current``, ``pre_scene`` (goal, heading goal,
        capsules, spheres), ``pre_t_steps``, ``pre_episode``, ``pre_ep_return``) and the post-step values before any
        auto-reset (``state``, ``u``, ``state_dot``, ``nu_c``, ``ray_dist``, ``reward_arr`` [S, n, K], ``obs``
        [S, K, n_obs], ``reward``, ``done``, ``cond_bits`` [S, K]).  ``step_host`` refuses to run while taps are set."""
        ids = [int(i) for i in env_ids]
        K, S = len(ids), int(capacity)
        if not 0 < K <= MAX_TAPS:
            raise ValueError(f"between 1 and {MAX_TAPS} env ids, got {K}")
        dev, dt = self.device, self.dtype
        z = lambda *shape, dtype=dt: torch.zeros(*shape, dtype=dtype, device=dev)  # noqa: E731
        n_scene = 4 + 7 * self.n_capsules + 4 * self.n_spheres
        ring = dict(count=z(1, dtype=torch.int64), pre_state=z(S, 12, K), pre_current=z(S, 5, K),
                    pre_scene=z(S, n_scene, K), pre_t_steps=z(S, K, dtype=torch.int32),
                    pre_episode=z(S, K, dtype=torch.int32), pre_ep_return=z(S, K), state=z(S, 12, K),
                    u=z(S, self.n_actions, K), state_dot=z(S, 12, K), nu_c=z(S, 3, K), ray_dist=z(S, self.n_rays, K),
                    reward_arr=z(S, 13, K), obs=z(S, K, self.n_observations, dtype=torch.float32), reward=z(S, K),
                    done=z(S, K, dtype=torch.uint8), cond_bits=z(S, K, dtype=torch.uint8))
        bufs = DockauvTapBuffers(*[_ptr(ring[k]) for k in TAP_FIELDS])
        id_arr = (C.c_int64 * K)(*ids)
        torch.cuda.current_stream(dev).synchronize()      # the ring tensors are zero-filled on the current stream
        _capi.check(self._lib.dockauv_set_taps(self._handle, id_arr, K, S, C.byref(bufs)))
        self.taps = dict(ring, env_ids=ids, capacity=S)
        return self.taps

    def clear_taps(self):
        """Remove the taps: the next steps are launched exactly as without them."""
        _capi.check(self._lib.dockauv_set_taps(self._handle, None, 0, 0, None))
        self.taps = None

    # ------------------------------------------------------------------ scenario bank (dockauv_set_scenario_bank)
    def set_scenario_bank(self, bank, weights=None):
        """Draw every following reset (``reset`` and the in-step auto-reset) from ``bank``: a ``ScenarioBank`` or a
        row table [K, stride] in the env dtype on its device (layout in gym_dockauv_b200/scenario_bank.py).  Rows are
        drawn uniformly, or in proportion to ``weights`` [K] (non-negative).  The library validates the rows on the
        device and refuses the bank (DockauvError naming the row and field) without changing the previous setting.
        Passing the bank that is already set again publishes rows rewritten in place (with ``weights``: new weights,
        as ``set_scenario_weights``); the pointers stay the same, so no step or rollout graph is re-captured.
        ``bank_row`` / ``ended_bank_row`` then hold the row of each env's running episode and of the episode its
        most recent reset ended: at a step whose ``done`` is set, ``ended_bank_row[i]`` is the row of the episode that
        just ended.  The env keeps references to the tensors it hands to the library."""
        rows = getattr(bank, "rows", bank)
        if not torch.is_tensor(rows) or rows.dim() != 2 or rows.dtype != self.dtype or rows.device != self.device \
                or rows.stride(1) != 1:
            raise ValueError(f"bank rows must be a 2-D {self.dtype} tensor on {self.device} with contiguous rows")
        if self._bank is not None and self._bank[0] is rows:
            if weights is None:
                self._set_bank(*self._bank)
            else:
                self.set_scenario_weights(weights)
            return
        cdf = None if weights is None else self._cdf(weights, rows.shape[0])
        row_of_env = torch.full((2, self.num_envs), -1, dtype=torch.int32, device=self.device)
        self._set_bank(rows, cdf, row_of_env)

    def set_scenario_weights(self, weights):
        """New draw weights [K] for the bank that is set.  The running sums are rewritten in place (float64
        ``torch.cumsum``) and re-validated: cached step and rollout graphs stay valid, nothing is re-captured.  On a
        bank set without weights the first call allocates the sums (one re-capture)."""
        if self._bank is None:
            raise RuntimeError("no scenario bank is set")
        rows, cdf, row_of_env = self._bank
        K = rows.shape[0]
        if cdf is None:
            self._set_bank(rows, self._cdf(weights, K), row_of_env)
            return
        old = cdf.clone()
        torch.cumsum(self._weights(weights, K), 0, out=cdf)
        try:
            self._set_bank(rows, cdf, row_of_env)
        except _capi.DockauvError:
            cdf.copy_(old)            # the previous weights stay in effect
            raise

    def clear_scenario_bank(self):
        """Back to the scenario's built-in reset distributions."""
        _capi.check(self._lib.dockauv_set_scenario_bank(self._handle, None, self._stream()))
        self._bank = None
        self.bank_row = self.ended_bank_row = None

    def _weights(self, weights, K):
        w = torch.as_tensor(weights).to(device=self.device, dtype=torch.float64).reshape(-1)
        if w.shape[0] != K:
            raise ValueError(f"{K} weights expected, got {w.shape[0]}")
        return w

    def _cdf(self, weights, K):
        return torch.cumsum(self._weights(weights, K), 0).contiguous()

    def _set_bank(self, rows, cdf, row_of_env):
        b = DockauvScenarioBank(_ptr(rows), _ptr(cdf), _ptr(row_of_env), rows.shape[0], rows.stride(0))
        _capi.check(self._lib.dockauv_set_scenario_bank(self._handle, C.byref(b), self._stream()))
        self._bank = (rows, cdf, row_of_env)
        self.bank_row, self.ended_bank_row = row_of_env[0], row_of_env[1]

    # ------------------------------------------------------------------ exact-state injection (parity tests, resume)
    def set_state(self, state=None, u_prev=None, goal=None, heading_goal=None, current=None, capsules=None,
                  spheres=None, t_steps=None, ep_return=None, env_ids=None):
        """Overwrite per-env state with host values.  Arrays are env-major (``state[n, 12]``, ``capsules[n, K, 7]``
        = (vec_bot, vec_top, radius), ``spheres[n, K, 4]`` = (centre, radius), ``current[n, 5]`` = (V_c, alpha,
        beta, V_min, V_max)); ``env_ids`` selects the envs (default: the first n)."""
        def put(dst, src, rows):
            if src is None:
                return
            src = torch.as_tensor(np.asarray(src), dtype=dst.dtype, device=self.device)
            src = src.reshape(src.shape[0], -1)
            n = src.shape[0]
            idx = torch.arange(n, device=self.device) if env_ids is None else torch.as_tensor(env_ids, device=self.device)
            if rows is None:
                dst[idx] = src[:, 0]
            else:
                if src.shape[1] != rows:
                    raise ValueError(f"expected {rows} values per env, got {src.shape[1]}")
                dst[:rows, idx] = src.t()
        put(self.state, state, 12)
        put(self.u_prev, u_prev, self.n_actions)
        put(self.goal, goal, 3)
        put(self.heading_goal, None if heading_goal is None else np.asarray(heading_goal).reshape(-1, 1), None)
        put(self.current, current, 5)
        if capsules is not None:
            put(self.capsules, np.asarray(capsules).reshape(len(capsules), -1), self.n_capsules * 7)
        if spheres is not None:
            put(self.spheres, np.asarray(spheres).reshape(len(spheres), -1), self.n_spheres * 4)
        put(self.t_steps, None if t_steps is None else np.asarray(t_steps).reshape(-1, 1), None)
        put(self.ep_return, None if ep_return is None else np.asarray(ep_return).reshape(-1, 1), None)
        if goal is not None or capsules is not None or spheres is not None:
            self.refresh_obstacles()

    def refresh_obstacles(self):
        """Call after writing ``self.capsules``, ``self.spheres`` or ``self.goal`` directly: the cull code reads a
        float copy of the obstacles relative to the goal that the library keeps (dockauv_refresh_obstacles);
        ``reset`` and ``set_state`` do it themselves."""
        _capi.check(self._lib.dockauv_refresh_obstacles(self._handle, self._stream()))

    # ------------------------------------------------------------------ statistics (FullDataStorage bookkeeping)
    def stats_tensor(self):
        """The device-side statistics vector (float64[16]) as a tensor view -- the all-reduce send buffer."""
        p = C.c_void_p()
        _capi.check(self._lib.dockauv_fold_stats(self._handle, self._stream()))   # per-CTA replicas -> the public vector
        _capi.check(self._lib.dockauv_stats_ptr(self._handle, C.byref(p)))
        return _DevView(p.value, N_STATS, self.device).tensor()

    def get_stats(self):
        out = (C.c_double * N_STATS)()
        _capi.check(self._lib.dockauv_get_stats(self._handle, out, self._stream()))
        return {k: out[i] for i, k in enumerate(STAT_NAMES)}

    def clear_stats(self):
        _capi.check(self._lib.dockauv_clear_stats(self._handle, self._stream()))

    def enable_timing(self, enabled=True):
        """CUDA-event timing of every following step (dockauv_enable_timing); read with ``last_step_ms``."""
        _capi.check(self._lib.dockauv_enable_timing(self._handle, int(bool(enabled))))

    def last_step_ms(self):
        """(ms of the most recent timed step, [ms of each of its launches]) -- the per-launch list is empty for the
        single-launch layouts; pipeline layout: dynamics + cull + finish, rays + finish (with obstacles), episode end."""
        ms = C.c_float()
        _capi.check(self._lib.dockauv_last_step_ms(self._handle, C.byref(ms)))
        per = (C.c_float * 8)()
        n = C.c_int()
        _capi.check(self._lib.dockauv_last_step_launch_ms(self._handle, per, 8, C.byref(n)))
        return ms.value, [per[k] for k in range(n.value)]

    def launch_count(self):
        n = C.c_int64()
        _capi.check(self._lib.dockauv_launch_count(self._handle, C.byref(n)))
        return n.value

    def enable_step_graph(self, enabled=True):
        """``step`` / ``step_into`` replay a cached CUDA graph of their launch sequence (default); False = plain launches."""
        _capi.check(self._lib.dockauv_enable_step_graph(self._handle, int(bool(enabled))))

    def step_graph_captures(self):
        n = C.c_int64()
        _capi.check(self._lib.dockauv_step_graph_captures(self._handle, C.byref(n)))
        return n.value

    def last_list_counts(self):
        """(envs with an obstacle in view, envs whose episode ended) in the most recent step (pipeline layout)."""
        a, b = C.c_int64(), C.c_int64()
        _capi.check(self._lib.dockauv_last_list_counts(self._handle, C.byref(a), C.byref(b), self._stream()))
        return a.value, b.value

    def rollout_captures(self):
        """How many times ``rollout(use_graph=True)`` had to capture its launch sequence (replays do not)."""
        n = C.c_int64()
        _capi.check(self._lib.dockauv_rollout_captures(self._handle, C.byref(n)))
        return n.value

    def rollout_policy_captures(self):
        """How many times ``rollout_policy(use_graph=True)`` had to capture its launch sequence (replays do not)."""
        n = C.c_int64()
        _capi.check(self._lib.dockauv_rollout_policy_captures(self._handle, C.byref(n)))
        return n.value

    # ------------------------------------------------------------------ conveniences mirroring the reference's info dict
    def info_dict(self, i):
        """The reference's per-step info dict (docking3d.py:388-400) for env i (device -> host read; small N only)."""
        bits = int(self.cond_bits[i].item())
        idx = [k for k in range(5) if bits >> k & 1]
        return {"episode_number": int(self.episode[i].item()), "t_step": int(self.t_steps[i].item()),
                "t_total_steps": self.t_total_steps, "cumulative_reward": float(self.ep_return[i].item()),
                "last_reward": float(self.reward[i].item()), "done": bool(self.done[i].item()),
                "conditions_true": idx, "conditions_true_info": [DONE_NAMES[k] for k in idx],
                "collision": bool(bits >> 4 & 1), "goal_reached": bool(bits & 1),
                "simulation_time": self.t_total_steps * float(self._params.h), "delta_d": float(self.delta_d[i].item())}


class _DevView:
    """Wraps a raw device pointer owned by the library as a torch tensor (no copy) via __cuda_array_interface__."""

    def __init__(self, ptr, n, device):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}
        self._device = device

    def tensor(self):
        return torch.as_tensor(self, device=self._device)


def _scenario(name):
    return type(name, (BaseDocking3d,), {"scenario": name, "__doc__": f"{name} (reference: docking3d.py) -- "
                                         f"batched; see BaseDocking3d."})


SimpleDocking3d = _scenario("SimpleDocking3d")                      # docking3d.py:795-825
SimpleCurrentDocking3d = _scenario("SimpleCurrentDocking3d")        # :828-849
CapsuleDocking3d = _scenario("CapsuleDocking3d")                    # :852-886
CapsuleCurrentDocking3d = _scenario("CapsuleCurrentDocking3d")      # :889-908
ObstaclesDocking3d = _scenario("ObstaclesDocking3d")                # :911-946
ObstaclesNoCapDocking3d = _scenario("ObstaclesNoCapDocking3d")      # :949-965
ObstaclesCurrentDocking3d = _scenario("ObstaclesCurrentDocking3d")  # :968-988

SCENARIOS = {n: globals()[n] for n in SCENARIO_IDS}


def make_gym(gym_env, env_config, **kwargs):
    """Counterpart of gym_dockauv/train.py:248-261: env id string -> (batched) env, KeyError on unknown ids."""
    if gym_env in REGISTRATION_DICT:
        return SCENARIOS[REGISTRATION_DICT[gym_env].split(":")[1]](env_config, **kwargs)
    raise KeyError(f"Not valid gym environment registration string, available options are {REGISTRATION_DICT.keys()}")
