"""Trajectory export in the reference's ``EpisodeDataStorage`` pickle schema (SURVEY.md 8f-3) for selected envs of a
batch, so the reference's post-analysis tooling (``EpisodeDataStorage.load`` and its ``plot_*`` wrappers,
gym_dockauv/utils/datastorage.py:184-420) can read episodes simulated on the GPU.

Row layout, exactly as the reference produces it (datastorage.py:218-288, call sites docking3d.py:252-254, 363-364,
676-684):

* row 0 is written at ``reset()``: initial state, zero ``state_dot`` / ``u``, the reset ``nu_c``, zero rewards and the
  zero observation; its radar end points are those of the radar reset, which the reference performs while the vehicle
  still sits at the origin with zero attitude (docking3d.py:262,285 run before generate_environment, :311);
* one row per ``step()``, appended in the MIDDLE of the step (after the radar / collision update, before
  observe / reward): the post-step ``state``, ``state_dot``, ``u``, radar end points and this step's ``nu_c`` together
  with the rewards / observation of the PREVIOUS step;
* one closing row at the next ``reset()``: the last state again, now with the last step's rewards / observation.

An episode of T steps therefore has T + 2 rows.  The pickle is a dict with the reference's keys.  ``vehicle.object`` and
``shapes`` hold instances of the reference's own classes when ``gym_dockauv`` is importable in the exporting process;
otherwise plain records with the same attribute names (``position``, ``radius``, ``vec_top``, ``vec_bot``).

Two recorders build these rows:

* ``EpisodeRecorder`` drives an env built with ``auto_reset=False, debug_outputs=True`` itself (one small
  device-to-host read per step, finished envs reset from the host): inspection tooling for a handful of envs;
* ``TrainingRecorder`` rides along a training run on any auto-reset env: the library records the chosen envs on the
  device (``BaseDocking3d.set_taps``, include/dockauv.h ``dockauv_set_taps``) and ``drain()`` turns the records into
  pickles, once per rollout or whenever the caller likes.
"""
import datetime
import os
import pickle

import numpy as np
import torch

META_DATA_REWARD = ["Nav_delta_d", "Nav_delta_theta", "Nav_delta_psi", "Att_phi", "Att_theta", "Thetadot",
                    "obstacle_avoid", "action", "Done-Goal_reached", "Done-out_pos", "Done-out_att", "Done-max_t",
                    "Done-collision"]                       # docking3d.py:160-182
N_CONT_REWARDS = 8                                          # docking3d.py:153


class ShapeRecord:
    """Stand-in for gym_dockauv.objects.shape.Sphere / Capsule when the reference package is not importable."""

    def __init__(self, kind, position, radius, vec_top=None):
        self.kind = kind
        self.position = np.asarray(position, dtype=float)
        self.radius = float(radius)
        if vec_top is not None:
            self.vec_top = np.asarray(vec_top, dtype=float)
            self.vec_bot = 2 * self.position - self.vec_top        # shape.py:105-108

    def __repr__(self):
        return f"ShapeRecord({self.kind}, position={self.position}, radius={self.radius})"


class VehicleRecord:
    """Stand-in for the AUVSim instance stored under storage['vehicle']['object']."""

    def __init__(self, name, step_size, u_bound):
        self.name, self.step_size, self.u_bound = name, float(step_size), np.asarray(u_bound)


def _rzyx(phi, theta, psi):
    cphi, sphi, cth, sth, cpsi, spsi = np.cos(phi), np.sin(phi), np.cos(theta), np.sin(theta), np.cos(psi), np.sin(psi)
    return np.array([[cpsi * cth, -spsi * cphi + cpsi * sth * sphi, spsi * sphi + cpsi * cphi * sth],
                     [spsi * cth, cpsi * cphi + sphi * sth * spsi, -cpsi * sphi + sth * spsi * cphi],
                     [-sth, cth * sphi, cth * cphi]])


def meta_data_observation(n_rays_reduced):
    return [["delta_d", "delta_theta", "delta_psi"], ["u", "v", "w"], ["phi", "theta", "psi_sin", "psi_cos"],
            ["p", "q", "r"], ["u_c", "v_c", "w_c"], [f"ray_{i}" for i in range(n_rays_reduced)]]   # docking3d.py:128-135


# ---------------------------------------------------------------------- row assembly shared by both recorders
def nu_c_reset(current, att):
    """nu_c right after reset() (docking3d.py:283): the spawned current (V_c, alpha, beta, ...) at the initial attitude."""
    cur = np.asarray(current, dtype=float)
    vn = cur[0] * np.array([np.cos(cur[1]) * np.cos(cur[2]), np.sin(cur[2]), np.sin(cur[1]) * np.cos(cur[2])])
    return np.concatenate([_rzyx(*att).T.dot(vn), np.zeros(3)])


def end_points(rd_b, state, dist):
    """Radar end points in the NED frame (sensor.py:96-102, 120)."""
    rd_n = rd_b.dot(_rzyx(*state[3:6]).T)
    rd_n /= np.linalg.norm(rd_n, axis=1)[:, None]
    return state[0:3] + rd_n * dist[:, None]


def start_rows(state, current, goal, capsules, spheres, n_actions, n_obs, rd_b, max_dist):
    """Row 0 of an episode, written at reset(); ``state`` / ``current`` are the env's values after the reset,
    ``capsules`` [n, 7] and ``spheres`` [n, 4] its obstacles."""
    state = np.asarray(state, dtype=float)
    return dict(states=[state], states_dot=[np.zeros(12)], u=[np.zeros(n_actions)],
                nu_c=[nu_c_reset(current, state[3:6])],
                radar=[end_points(rd_b, np.zeros(12), np.full(rd_b.shape[0], max_dist))],
                rewards=[np.zeros(13)], cum_rewards=[np.zeros(13)], observation=[np.zeros(n_obs)],
                goal=np.asarray(goal, dtype=float), capsules=np.asarray(capsules, dtype=float).reshape(-1, 7),
                spheres=np.asarray(spheres, dtype=float).reshape(-1, 4))


def append_step(r, rd_b, state, state_dot, u, nu_c, dist, reward_arr, obs):
    """The mid-step row of one step: this step's kinematics with the previous step's rewards / observation; this step's
    rewards and observation are kept for the next row."""
    n_obs = len(r["observation"][0])
    r["states"].append(state); r["states_dot"].append(state_dot); r["u"].append(u)
    r["nu_c"].append(np.concatenate([nu_c, np.zeros(3)]))
    r["radar"].append(end_points(rd_b, state, dist))
    r["rewards"].append(r.get("_last_r", np.zeros(13))); r["cum_rewards"].append(r.get("_cum", np.zeros(13)))
    r["observation"].append(r.get("_last_obs", np.zeros(n_obs)))
    r["_last_r"] = reward_arr
    r["_cum"] = r.get("_cum", np.zeros(13)) + reward_arr
    r["_last_obs"] = np.asarray(obs, dtype=float)


def finish_rows(r, env, title, episode, shape_module=None):
    """Appends the closing row (written by the next reset(), docking3d.py:252-254) and returns the storage dict."""
    for key in ("states", "states_dot", "u", "nu_c", "radar"):
        r[key].append(r[key][-1])
    r["rewards"].append(r["_last_r"]); r["cum_rewards"].append(r["_cum"]); r["observation"].append(r["_last_obs"])
    if shape_module is not None:
        shapes = [shape_module.Capsule(position=(c[0:3] + c[3:6]) / 2, radius=c[6], vec_top=c[3:6]) for c in r["capsules"]]
        shapes += [shape_module.Sphere(position=s[0:3], radius=s[3]) for s in r["spheres"]]
        shapes.append(shape_module.Sphere(r["goal"], 0.15))
    else:
        shapes = [ShapeRecord("capsule", (c[0:3] + c[3:6]) / 2, c[6], vec_top=c[3:6]) for c in r["capsules"]]
        shapes += [ShapeRecord("sphere", s[0:3], s[3]) for s in r["spheres"]]
        shapes.append(ShapeRecord("sphere", r["goal"], 0.15))
    return {
        "vehicle": {"object": VehicleRecord(env.config.get("vehicle", "BlueROV2"), env.config["t_step_size"],
                                            env._meta["u_bound"]),
                    "states": np.array(r["states"]), "states_dot": np.array(r["states_dot"]), "u": np.array(r["u"])},
        "radar": np.array(r["radar"]), "nu_c": np.array(r["nu_c"]), "shapes": shapes, "title": title,
        "episode": episode, "step_size": env.config["t_step_size"],
        "cum_rewards": np.array(r["cum_rewards"]), "rewards": np.array(r["rewards"]),
        "meta_data_reward": list(META_DATA_REWARD), "n_cont_rewards": N_CONT_REWARDS,
        "observation": np.array(r["observation"]),
        "meta_data_observation": meta_data_observation(env.n_observations - 16),
    }


def save_storage(storage, path_folder, title, env_id, episode):
    """Writes ``<utc>__<title>__ENV_<env_id>__EPISODE_<episode>_DATA_STORAGE.pkl`` and returns its path."""
    utc = datetime.datetime.now(datetime.timezone.utc).strftime('%Y_%m_%dT%H_%M_%S')
    if path_folder:
        os.makedirs(path_folder, exist_ok=True)
    name = os.path.join(path_folder, f"{utc}__{title}__ENV_{env_id}__EPISODE_{episode}_DATA_STORAGE.pkl")
    with open(name, "wb") as f:
        pickle.dump(storage, f, pickle.HIGHEST_PROTOCOL)
    return name


def _radar_table(env):
    rd_b = np.ctypeslib.as_array(env._params.rd_b)[:3 * env.n_rays].reshape(env.n_rays, 3).copy()
    return rd_b, float(env._params.radar_max_dist)


class EpisodeRecorder:
    """Wraps a batched env built with ``auto_reset=False, debug_outputs=True`` and records the episodes of the envs
    in ``env_ids``; every finished episode is written to ``path_folder`` as
    ``<utc>__<title>__EPISODE_<k>_DATA_STORAGE.pkl`` and all finished envs are reset (``env.reset(mask=done)``)."""

    def __init__(self, env, env_ids, path_folder, title="", save=True, shape_module=None):
        """``shape_module``: optionally the reference's own ``gym_dockauv.objects.shape`` module, passed in by a caller
        that has the reference installed and wants its ``Capsule`` / ``Sphere`` classes inside the pickles (what
        ``plot_*`` of the reference draws); by default the files hold ``ShapeRecord`` stand-ins with the same
        attributes.  This package never imports the reference on its own."""
        if env.auto_reset or env.debug is None:
            raise ValueError("create the env with auto_reset=False and debug_outputs=True")
        self.shape_module = shape_module
        self.env, self.ids = env, [int(i) for i in env_ids]
        self.path_folder, self.title, self.save = path_folder, title, save
        self._sel = torch.as_tensor(self.ids, device=env.device)
        self.rd_b, self.max_dist = _radar_table(env)
        self.episode_no = {i: 0 for i in self.ids}
        self.rows = {}
        self.saved = []      # (env id, episode number, path or storage dict)

    # ------------------------------------------------------------------ device -> host snapshot of the tracked envs
    def _snapshot(self):
        e, s = self.env, self._sel
        parts = [e.state[:, s], e.u_prev[:e.n_actions, s], e.debug["state_dot"][:, s], e.debug["nu_c"][:, s],
                 e.debug["ray_dist"][:, s], e.debug["reward_arr"][:, s]]
        flat = torch.cat([p.to(torch.float64) for p in parts], dim=0).cpu().numpy()
        obs = e.obs[s].cpu().numpy()
        out, o = [], 0
        for n in (12, e.n_actions, 12, 3, e.n_rays, 13):
            out.append(flat[o:o + n].T)
            o += n
        return (*out, obs)

    def _nu_c_reset(self, k):
        return nu_c_reset(self.env.current[:, self.ids[k]].cpu().numpy(), self.env.state[3:6, self.ids[k]].cpu().numpy())

    def _end_points(self, state, dist):
        return end_points(self.rd_b, state, dist)

    def _start_rows(self, k):
        e, i = self.env, self.ids[k]
        self.episode_no[i] += 1
        self.rows[i] = start_rows(e.state[:, i].cpu().numpy(), e.current[:, i].cpu().numpy(), e.goal[:, i].cpu().numpy(),
                                  e.capsules[:e.n_capsules * 7, i].cpu().numpy(), e.spheres[:e.n_spheres * 4, i].cpu().numpy(),
                                  e.n_actions, e.n_observations, self.rd_b, self.max_dist)

    # ------------------------------------------------------------------ gym-like surface
    def reset(self, seed=None):
        obs = self.env.reset(seed=seed)
        for k in range(len(self.ids)):
            self._start_rows(k)
        return obs

    def step(self, actions):
        e = self.env
        obs, reward, done, info = e.step(actions)
        state, u, sdot, nu_c, dist, rarr, obs_sel = self._snapshot()
        d = done.bool()
        d_sel = d[self._sel].cpu().numpy()
        for k, i in enumerate(self.ids):
            append_step(self.rows[i], self.rd_b, state[k], sdot[k], u[k], nu_c[k], dist[k], rarr[k], obs_sel[k])
            if d_sel[k]:
                self._finish(k)
        if bool(d.any()):
            e.reset(mask=done)
            for k, i in enumerate(self.ids):
                if d_sel[k]:
                    self._start_rows(k)
        return obs, reward, done, info

    def _finish(self, k):
        i = self.ids[k]
        storage = finish_rows(self.rows[i], self.env, self.title, self.episode_no[i], self.shape_module)
        if self.save:
            name = save_storage(storage, self.path_folder, self.title, i, self.episode_no[i])
            self.saved.append((i, self.episode_no[i], name))
        else:
            self.saved.append((i, self.episode_no[i], storage))


class TrainingRecorder:
    """Records the episodes of the envs ``env_ids`` (local indices, at most 1024) of an auto-reset env of any layout
    while it trains: ``env.set_taps`` makes every ``step`` / ``step_into`` / ``rollout`` write a record of these envs
    into a device ring of ``capacity`` steps, and ``drain()`` copies the new records to the host, assembles the
    reference's T + 2 rows per episode and writes
    ``<utc>__<title>__ENV_<global id>__EPISODE_<k>_DATA_STORAGE.pkl`` for every finished episode whose number k (the
    env's episode counter, 1 for its first episode) is a multiple of ``every``.

    * An episode starts at a record whose pre-step step counter is 0 (row 0: the pre-step state, scene and current)
      and ends at a record with ``done``.  Episodes already running when the recorder was created are skipped.
    * An episode cut short by an explicit ``env.reset()`` (a new start before any ``done``) is discarded.
    * Episodes may span drains.  If more than ``capacity`` steps passed since the last drain, the oldest records are
      gone: the episodes that lost records are dropped and counted in ``lost_episodes``; no pickle has a gap.
    """

    def __init__(self, env, env_ids, path_folder, title="", capacity=1024, every=1, shape_module=None, save=True):
        if not env.auto_reset:
            raise ValueError("TrainingRecorder records auto-reset envs; use EpisodeRecorder for auto_reset=False")
        self.env, self.ids = env, [int(i) for i in env_ids]
        self.path_folder, self.title, self.save = path_folder, title, save
        self.every, self.shape_module = max(1, int(every)), shape_module
        self.capacity = int(capacity)
        self.rd_b, self.max_dist = _radar_table(env)
        self.env_id0 = int(env._params.env_id0)
        self.ring = env.set_taps(self.ids, self.capacity)
        self._drained = 0                            # records consumed so far
        self._rows = [None] * len(self.ids)          # rows of the running episode of each tap (None: waiting for a start)
        self._last_episode = [None] * len(self.ids)  # episode number of the last record consumed
        self._gap = [None] * len(self.ids)           # True: records were lost since the last one consumed
        self.lost_episodes = 0
        self.saved = []      # (global env id, episode number, path or storage dict)

    def close(self):
        """Removes the taps (the env steps exactly as it did before the recorder existed)."""
        self.env.clear_taps()

    def drain(self):
        """Consumes the records written since the last call; returns the (global env id, episode, path) entries of the
        pickles written by this call."""
        count = int(self.ring["count"].item())       # ordered after every step issued so far on the current stream
        n = count - self._drained
        if n <= 0:
            return []
        S = self.capacity
        if n > S:                                    # records _drained .. count - S were overwritten
            for k in range(len(self.ids)):
                if self._rows[k] is not None:
                    self.lost_episodes += 1
                self._gap[k] = True
                self._rows[k] = None
            self._drained, n = count - S, S
        a = self._drained % S
        host = {}
        for name in ("pre_state", "pre_current", "pre_scene", "pre_t_steps", "pre_episode", "state", "u", "state_dot",
                     "nu_c", "ray_dist", "reward_arr", "obs", "done"):
            t = self.ring[name]
            part = t[a:a + n] if a + n <= S else torch.cat([t[a:], t[:a + n - S]])
            host[name] = part.cpu().numpy()
        self._drained = count
        before = len(self.saved)
        for j in range(n):
            for k in range(len(self.ids)):
                self._consume(k, host, j)
        return self.saved[before:]

    def _consume(self, k, h, j):
        e = self.env
        ep = int(h["pre_episode"][j, k])
        start = int(h["pre_t_steps"][j, k]) == 0
        if self._gap[k] is not None:                 # first record after lost ones
            last = self._last_episode[k]             # the dropped episode (already counted) or one being skipped
            if last is not None and ep > last + 1:
                self.lost_episodes += ep - last - 1  # episodes that began and ended inside the lost records
            if not start and (last is None or ep != last):
                self.lost_episodes += 1              # the episode running here lost its first records
            self._gap[k] = None
        self._last_episode[k] = ep
        if start:
            nc, ns = e.n_capsules, e.n_spheres
            scene = h["pre_scene"][j, :, k].astype(float)
            self._rows[k] = start_rows(h["pre_state"][j, :, k], h["pre_current"][j, :, k], scene[0:3],
                                       scene[4:4 + 7 * nc], scene[4 + 7 * nc:4 + 7 * nc + 4 * ns], e.n_actions,
                                       e.n_observations, self.rd_b, self.max_dist)
        r = self._rows[k]
        if r is None:
            return
        f = lambda name: h[name][j, :, k].astype(float)  # noqa: E731
        append_step(r, self.rd_b, f("state"), f("state_dot"), f("u"), f("nu_c"), f("ray_dist"), f("reward_arr"),
                    h["obs"][j, k])
        if h["done"][j, k]:
            self._rows[k] = None
            if ep % self.every == 0:
                gid = self.env_id0 + self.ids[k]
                storage = finish_rows(r, e, self.title, ep, self.shape_module)
                if self.save:
                    self.saved.append((gid, ep, save_storage(storage, self.path_folder, self.title, gid, ep)))
                else:
                    self.saved.append((gid, ep, storage))
