"""Scenario banks: tables of initial conditions that every reset draws from (dockauv_set_scenario_bank).

A bank replaces the reference's extension point for new tasks, a subclass overriding ``generate_environment``
(docking3d.py:795-988).  Rows are packed here from per-field tensors and handed to ``env.set_scenario_bank``:

    bank = ScenarioBank.from_generator(env, ReferenceResetStream("ObstaclesDocking3d", cfg, seed=0).generate, 4096)
    env.set_scenario_bank(bank)                  # every reset (auto-reset included) now starts from a bank row
    env.set_scenario_weights(w)                  # weighted draw; cheap to repeat, no graph re-capture

Row layout (include/dockauv.h): pose [0:6], goal [6:9], heading goal [9], current [10:15] (V_c, alpha, beta, V_min,
V_max), then the capsule slots (bot[3], top[3], r) and the sphere slots (centre[3], r).  Rows are padded to a multiple
of 16 bytes.  Slots a generator leaves empty take the library's unused-slot form (radius 0, far from the goal).
"""
import numpy as np
import torch

UNUSED_CAPSULE = (1e6, 1e6, 1e6, 1e6, 1e6, 1e6 + 1.0, 0.0)      # what the built-in reset writes to unused slots
UNUSED_SPHERE = (1e6, 1e6, 1e6, 0.0)
FIELDS = (("pose", 6), ("goal", 3), ("heading_goal", 1), ("current", 5))


def row_width(n_capsules, n_spheres):
    """W = 15 + 7 n_capsules + 4 n_spheres reals."""
    return 15 + 7 * n_capsules + 4 * n_spheres


def pack(pose, goal, heading_goal, n_capsules, n_spheres, current=None, capsules=None, spheres=None,
         dtype=torch.float64, device="cpu"):
    """Per-field arrays of K rows -> the row table [K, stride] (stride = W rounded up to 16 bytes, zero padding).
    ``pose`` [K, 6], ``goal`` [K, 3], ``heading_goal`` [K], ``current`` [K, 5] (default zero), ``capsules``
    [K, kc, 7] with kc <= n_capsules, ``spheres`` [K, ks, 4] with ks <= n_spheres (missing slots: unused form)."""
    t = lambda a: torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a).to(device=device, dtype=dtype)  # noqa: E731
    pose, goal, heading_goal = t(pose), t(goal), t(heading_goal).reshape(-1)
    K = pose.shape[0]
    if pose.shape != (K, 6) or goal.shape != (K, 3) or heading_goal.shape != (K,):
        raise ValueError("pose [K, 6], goal [K, 3] and heading_goal [K] expected")
    W = row_width(n_capsules, n_spheres)
    per = 16 // torch.tensor([], dtype=dtype).element_size()
    stride = -(-W // per) * per
    rows = torch.zeros(K, stride, dtype=dtype, device=device)
    rows[:, 0:6] = pose
    rows[:, 6:9] = goal
    rows[:, 9] = heading_goal
    if current is not None:
        rows[:, 10:15] = t(current).reshape(K, 5)
    caps = rows[:, 15:15 + 7 * n_capsules].view(K, n_capsules, 7)
    sph = rows[:, 15 + 7 * n_capsules:W].view(K, n_spheres, 4)
    caps[:] = torch.tensor(UNUSED_CAPSULE, dtype=dtype, device=device)
    sph[:] = torch.tensor(UNUSED_SPHERE, dtype=dtype, device=device)
    for src, dst, name in ((capsules, caps, "capsules"), (spheres, sph, "spheres")):
        if src is None:
            continue
        src = t(src)
        n = src.shape[1] if src.dim() == 3 else 0
        if src.shape[0] != K or n > dst.shape[1]:
            raise ValueError(f"{name}: {tuple(src.shape)} does not fit {dst.shape[1]} slots of {K} rows")
        if n:
            dst[:, :n] = src
    return rows


class ScenarioBank:
    """K initial conditions packed into the row table of one env (its dtype, device and obstacle slots)."""

    def __init__(self, env, pose, goal, heading_goal, current=None, capsules=None, spheres=None):
        self.n_capsules, self.n_spheres = env.n_capsules, env.n_spheres
        self.rows = pack(pose, goal, heading_goal, self.n_capsules, self.n_spheres, current=current, capsules=capsules,
                         spheres=spheres, dtype=env.dtype, device=env.device)
        self.n_rows = self.rows.shape[0]
        self.width = row_width(self.n_capsules, self.n_spheres)

    def field(self, name):
        """One field of every row as a view: pose, goal, heading_goal, current, capsules [K, nc, 7], spheres."""
        o = 0
        for f, n in FIELDS:
            if f == name:
                return self.rows[:, o] if n == 1 else self.rows[:, o:o + n]
            o += n
        nc, K = self.n_capsules, self.n_rows
        if name == "capsules":
            return self.rows[:, 15:15 + 7 * nc].view(K, nc, 7)
        if name == "spheres":
            return self.rows[:, 15 + 7 * nc:self.width].view(K, self.n_spheres, 4)
        raise KeyError(name)

    @classmethod
    def from_dicts(cls, env, dicts):
        """Rows from dicts in the format of ``ReferenceResetStream.generate()``: ``init_state`` (12; the pose is its
        first six entries, velocities must be zero), ``goal``, ``heading_goal``, ``current`` (5), ``capsules`` [kc, 7],
        optional ``spheres`` [ks, 4]."""
        K = len(dicts)
        nc, ns = env.n_capsules, env.n_spheres
        init = np.stack([np.asarray(d["init_state"], dtype=float) for d in dicts])
        if np.any(init[:, 6:] != 0):
            raise ValueError("bank rows start at rest: init_state[6:12] must be zero")
        caps = np.zeros((K, nc, 7))
        caps[:] = UNUSED_CAPSULE
        sph = np.zeros((K, ns, 4))
        sph[:] = UNUSED_SPHERE
        for k, d in enumerate(dicts):
            for src, dst, name in ((d.get("capsules"), caps, "capsules"), (d.get("spheres"), sph, "spheres")):
                src = np.zeros((0, dst.shape[2])) if src is None else np.asarray(src, dtype=float).reshape(-1, dst.shape[2])
                if src.shape[0] > dst.shape[1]:
                    raise ValueError(f"row {k}: {src.shape[0]} {name}, the env has {dst.shape[1]} slots")
                dst[k, :src.shape[0]] = src
        return cls(env, init[:, :6], np.stack([d["goal"] for d in dicts]), np.array([d["heading_goal"] for d in dicts]),
                   current=np.stack([d["current"] for d in dicts]), capsules=caps, spheres=sph)

    @classmethod
    def from_generator(cls, env, generate, K):
        """K rows from K calls of ``generate()`` (dict format of ``ReferenceResetStream.generate()``)."""
        return cls.from_dicts(env, [generate() for _ in range(int(K))])

    @classmethod
    def from_builtin(cls, env, K, seed):
        """K draws of the env's built-in distributions: ``reset()`` of a scratch env of K envs with the same
        parameters (global ids 0..K-1, key ``seed``), read back on the device."""
        kw = dict(env._init_kwargs, num_envs=int(K), seed=int(seed), env_id0=0, layout="thread_per_env",
                  auto_reset=False, debug_outputs=False)
        scratch = type(env)(env.config, **kw)
        try:
            scratch.reset()
            nc, ns = scratch.n_capsules, scratch.n_spheres
            return cls(env, scratch.state[:6].t(), scratch.goal.t(), scratch.heading_goal, current=scratch.current.t(),
                       capsules=scratch.capsules[:7 * nc].t().reshape(int(K), nc, 7) if nc else None,
                       spheres=scratch.spheres[:4 * ns].t().reshape(int(K), ns, 4) if ns else None)
        finally:
            scratch.close()
