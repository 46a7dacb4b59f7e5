"""Python face of the CPU oracle -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Loads ``oracle/_build/libdockauv_oracle.so`` (compiled from oracle/dockauv_oracle.c by oracle/Makefile) and
prepares its parameter block.  The init-time part of the reference (mass matrices, radar ray table,
obstacle-avoidance weights) is restated here in numpy, each function citing the reference file:line it
follows.  Only tests/, ``__graft_entry__.smoke()`` and bench.py's cpu_baseline / ``--impl reference`` legs
may import this module; the product package (gym_dockauv_b200/) never does.

Vehicle numbers come from tests/golden/vehicles.json, which tests/golden/make_golden.py dumped from the
reference's own vehicle objects (i.e. from its XML files).
"""
import ctypes as C
import json
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "libdockauv_oracle.so")
VEHICLES_JSON = os.path.join(HERE, "..", "tests", "golden", "vehicles.json")

MAX_U, MAX_CAPS, MAX_SPH, MAX_RAYS, N_REWARDS = 8, 8, 8, 1024, 13
c_d, c_i = C.c_double, C.c_int32

SCENARIOS = {"SimpleDocking3d": 0, "SimpleCurrentDocking3d": 1, "CapsuleDocking3d": 2,
             "CapsuleCurrentDocking3d": 3, "ObstaclesDocking3d": 4, "ObstaclesCurrentDocking3d": 5,
             "ObstaclesNoCapDocking3d": 6}


class OrcParams(C.Structure):
    _fields_ = [
        ("vehicle", c_i), ("n_u", c_i), ("m", c_d), ("W", c_d), ("BY", c_d), ("r_G", c_d * 3), ("r_B", c_d * 3),
        ("I_b", c_d * 9), ("M_A", c_d * 36), ("M_inv", c_d * 36), ("D_lin", c_d * 36), ("D_quad", c_d * 36),
        ("L_lift", c_d * 36), ("B_const", c_d * (6 * MAX_U)), ("lauv_B", c_d * 4), ("u_lo", c_d * MAX_U),
        ("u_hi", c_d * MAX_U), ("lp_alpha", c_d), ("h", c_d), ("safety_radius", c_d),
        ("max_timesteps", c_i), ("reward_set", c_i), ("max_dist_from_goal", c_d), ("max_attitude", c_d),
        ("dist_goal_reached_tol", c_d), ("u_max", c_d), ("v_max", c_d), ("w_max", c_d), ("p_max", c_d),
        ("q_max", c_d), ("r_max", c_d), ("w_d", c_d), ("w_delta_psi", c_d), ("w_delta_theta", c_d),
        ("w_phi", c_d), ("w_theta", c_d), ("w_Thetadot", c_d), ("w_oa", c_d), ("w_done", c_d * 5),
        ("action_reward_factors", c_d * MAX_U), ("action_factor_is_scalar", c_i),
        ("cur_mu", c_d), ("cur_sigma", c_d),
        ("n_rays", c_i), ("n_vert", c_i), ("n_horiz", c_i), ("block", c_i), ("n_rays_reduced", c_i),
        ("radar_max_dist", c_d), ("rd_b", c_d * (MAX_RAYS * 3)), ("beta_oa", c_d * MAX_RAYS), ("n_obs", c_i),
    ]


class OrcEnv(C.Structure):
    _fields_ = [
        ("state", c_d * 12), ("u", c_d * MAX_U), ("goal", c_d * 3), ("heading_goal", c_d), ("cur", c_d * 5),
        ("n_caps", c_i), ("n_sph", c_i), ("caps", (c_d * 7) * MAX_CAPS), ("sph", (c_d * 4) * MAX_SPH),
        ("t_steps", c_i), ("episode", c_i), ("cum_reward", c_d),
    ]


class OrcStepOut(C.Structure):
    _fields_ = [
        ("obs", C.c_float * (16 + MAX_RAYS // 4 + 64)), ("reward", c_d), ("reward_arr", c_d * N_REWARDS),
        ("cond", C.c_uint8 * 5), ("collision", C.c_uint8), ("done", C.c_uint8), ("goal_reached", C.c_uint8),
        ("ray_dist", c_d * MAX_RAYS), ("state_dot", c_d * 12), ("nu_c", c_d * 6),
        ("delta_d", c_d), ("delta_theta", c_d), ("delta_psi", c_d), ("delta_heading_goal", c_d),
    ]


def build(force=False):
    """Compile the C restatement (gcc, -O2, no -ffast-math: IEEE semantics are part of the contract)."""
    src = [os.path.join(HERE, "dockauv_oracle.c"), os.path.join(HERE, "dockauv_oracle.h")]
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in src):
        return LIB_PATH
    subprocess.check_call(["make", "-s", "-C", HERE])
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        build()
    L = C.CDLL(LIB_PATH)
    dp = C.POINTER(c_d)
    L.orc_ssa.restype = c_d
    L.orc_ssa.argtypes = [c_d]
    L.orc_Rzyx.restype = None
    L.orc_Rzyx.argtypes = [c_d, c_d, c_d, dp]
    L.orc_ray_capsule.restype = c_d
    L.orc_ray_capsule.argtypes = [dp, dp, dp, dp, c_d]
    L.orc_ray_spheres.restype = c_d
    L.orc_ray_spheres.argtypes = [dp, dp, dp, dp, C.c_int]
    L.orc_dist_line_point.restype = c_d
    L.orc_dist_line_point.argtypes = [dp, dp, dp]
    L.orc_collision_capsule_sphere.restype = C.c_int
    L.orc_collision_capsule_sphere.argtypes = [dp, dp, c_d, dp, c_d]
    L.orc_collision_sphere_spheres.restype = C.c_int
    L.orc_collision_sphere_spheres.argtypes = [dp, c_d, dp, dp, C.c_int]
    L.orc_obstacle_avoidance.restype = c_d
    L.orc_obstacle_avoidance.argtypes = [C.POINTER(OrcParams), dp]
    L.orc_log_precision.restype = c_d
    L.orc_log_precision.argtypes = [c_d, c_d, c_d]
    L.orc_step.restype = None
    L.orc_step.argtypes = [C.POINTER(OrcParams), C.POINTER(OrcEnv), C.c_void_p, C.c_int, c_d, C.POINTER(OrcStepOut)]
    L.orc_reset_env.restype = None
    L.orc_reset_env.argtypes = [C.POINTER(OrcParams), C.POINTER(OrcEnv), C.c_int, C.c_uint64, C.c_uint64]
    L.orc_step_batch.restype = C.c_int64
    L.orc_step_batch.argtypes = [C.POINTER(OrcParams), C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int,
                                 C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    L.orc_step_batch_ids.restype = C.c_int64
    L.orc_step_batch_ids.argtypes = [C.POINTER(OrcParams), C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int,
                                     C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_int]
    assert L.orc_sizeof_params() == C.sizeof(OrcParams), (L.orc_sizeof_params(), C.sizeof(OrcParams))
    assert L.orc_sizeof_env() == C.sizeof(OrcEnv)
    assert L.orc_sizeof_stepout() == C.sizeof(OrcStepOut)
    _lib = L
    return L


def _dp(a):
    return a.ctypes.data_as(C.POINTER(c_d))


def vehicle_table(name):
    with open(VEHICLES_JSON) as f:
        return json.load(f)[name]


# ------------------------------------------------------------------ init-time restatements (numpy)
def S_skew(a):
    """geomutils.py:106-128"""
    return np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]], dtype=float)


def vehicle_matrices(v):
    """statespace.py:86-197 from a {tag: value} table."""
    g = lambda k: float(v.get(k, 0.0))  # noqa: E731
    m = g("m")
    I_g = np.array([[g("I_x"), -g("I_xy"), -g("I_xz")],
                    [-g("I_xy"), g("I_y"), -g("I_yz")],
                    [g("I_xz"), -g("I_yz"), g("I_z")]])                      # statespace.py:86-102 (sic: +I_xz)
    r_G = np.array([g("x_G"), g("y_G"), g("z_G")])
    r_B = np.array([g("x_B"), g("y_B"), g("z_B")])
    I_b = I_g + m * S_skew(r_G).dot(S_skew(r_G).T)                          # :105-117
    M_RB_CG = np.vstack([np.hstack([m * np.identity(3), np.zeros((3, 3))]),
                         np.hstack([np.zeros((3, 3)), I_g])])               # :138-161
    H = np.vstack([np.hstack([np.identity(3), S_skew(r_G).T]),
                   np.hstack([np.zeros((3, 3)), np.identity(3)])])          # geomutils.py:131-157
    M_RB = H.T.dot(M_RB_CG).dot(H)
    M_A = -np.diag([g("X_udot"), g("Y_vdot"), g("Z_wdot"), g("K_pdot"), g("M_qdot"), g("N_rdot")])  # :164-187
    M_inv = np.linalg.inv(M_RB + M_A)                                        # :190-197
    return dict(m=m, W=m * float(v.get("g", 9.81)), BY=g("BY"), r_G=r_G, r_B=r_B, I_b=I_b, M_RB=M_RB, M_A=M_A,
                M_inv=M_inv)


def damping_tables(v, vehicle):
    """statespace.py:337-351 (BlueROV2: diagonal) / LAUV.py:69-101 as three coefficient matrices."""
    g = lambda k: float(v.get(k, 0.0))  # noqa: E731
    D_lin = np.diag([g("X_u"), g("Y_v"), g("Z_w"), g("K_p"), g("M_q"), g("N_r")])
    D_quad = np.diag([g("X_uu"), g("Y_vv"), g("Z_ww"), g("K_pp"), g("M_qq"), g("N_rr")])
    L = np.zeros((6, 6))
    if vehicle == "LAUV":
        D_lin[1, 5], D_lin[2, 4], D_lin[4, 2], D_lin[5, 1] = g("Y_r"), g("Z_q"), g("M_w"), g("N_v")
        D_quad[1, 5], D_quad[2, 4], D_quad[4, 2], D_quad[5, 1] = g("Y_rr"), g("Z_qq"), g("M_ww"), g("N_vv")
        L[1, 1], L[1, 5] = g("Y_uvb") + g("Y_uvf"), g("Y_urf")
        L[2, 2], L[2, 4] = g("Z_uwb") + g("Z_uwf"), g("Z_uqf")
        L[4, 2], L[4, 4] = g("M_uwb") + g("M_uwf"), g("M_uqf")
        L[5, 1], L[5, 5] = g("N_uvb") + g("N_uvf"), g("N_urf")
    return D_lin, D_quad, L


def radar_table(alpha, beta, ray_per_deg, max_dist, blocksize_reduce=2, freq=1):
    """sensor.py:43-71 and docking3d.py:789-790 (beta_oa)."""
    tol = 10e-8
    a = np.arange(-alpha / 2, alpha / 2 + tol, ray_per_deg)
    n_v = a.shape[0]
    a = np.repeat(a, repeats=int((beta + tol) // ray_per_deg + 1), axis=0)
    b = np.arange(-beta / 2, beta / 2 + tol, ray_per_deg)
    n_h = b.shape[0]
    b = np.tile(b, (int((alpha + tol) // ray_per_deg + 1),))
    n = a.shape[0]
    rd_b = np.hstack([np.ones(n)[:, None], np.sin(b)[:, None], np.sin(a)[:, None]])
    rd_b = rd_b / np.linalg.norm(rd_b, axis=1)[:, None]
    beta_oa = (1 - np.abs(a) / (alpha / 2)) * (1 - np.abs(b) / (beta / 2)) + 0.01
    n_red = -(-n_v // blocksize_reduce) * -(-n_h // blocksize_reduce)
    return dict(n_rays=n, n_vert=n_v, n_horiz=n_h, rd_b=rd_b, beta_oa=beta_oa, alpha=a, beta=b,
                n_rays_reduced=n_red, max_dist=float(max_dist), block=int(blocksize_reduce))


def make_params(config, vehicle_key=None, cur_mu=0.005, cur_sigma=0.0):
    """env_config dict (config/env_config.py:20-91) + vehicle table -> OrcParams."""
    vehicle = config["vehicle"]
    v = vehicle_table(vehicle_key or vehicle)
    vm = vehicle_matrices(v)
    P = OrcParams()
    P.vehicle = 0 if vehicle == "BlueROV2" else 1
    u_bound = np.asarray(v["u_bound"], dtype=float)
    n_u = u_bound.shape[0]
    P.n_u = n_u
    P.m, P.W, P.BY = vm["m"], vm["W"], vm["BY"]
    P.r_G[:] = vm["r_G"].tolist()
    P.r_B[:] = vm["r_B"].tolist()
    P.I_b[:] = vm["I_b"].ravel().tolist()
    P.M_A[:] = vm["M_A"].ravel().tolist()
    P.M_inv[:] = vm["M_inv"].ravel().tolist()
    Dl, Dq, L = damping_tables(v, vehicle)
    P.D_lin[:] = Dl.ravel().tolist()
    P.D_quad[:] = Dq.ravel().tolist()
    P.L_lift[:] = L.ravel().tolist()
    if vehicle == "BlueROV2":
        B = np.asarray(v["B"], dtype=float)
        flat = B.ravel().tolist()
        for i, x in enumerate(flat):
            P.B_const[i] = x
    else:
        P.lauv_B[:] = [v["Y_uudr"], v["Z_uuds"], v["M_uuds"], v["N_uudr"]]
    for i in range(n_u):
        P.u_lo[i], P.u_hi[i] = u_bound[i, 0], u_bound[i, 1]
    h = float(config["t_step_size"])
    P.h = h
    P.lp_alpha = h / (h + v["lowpass_T1"])                               # lowpassfilter.py:27, auvsim.py:40,49-53
    P.safety_radius = v["safety_radius"]
    P.max_timesteps = int(config["max_timesteps"])
    P.reward_set = int(config["reward_set"])
    for k in ["max_dist_from_goal", "max_attitude", "dist_goal_reached_tol", "u_max", "v_max", "w_max", "p_max",
              "q_max", "r_max"]:
        setattr(P, k, float(config[k]))
    rf = config["reward_factors"]
    for k in ["w_d", "w_delta_psi", "w_delta_theta", "w_phi", "w_theta", "w_Thetadot", "w_oa"]:
        setattr(P, k, float(rf[k]))
    P.w_done[:] = [rf["w_goal"], rf["w_deltad_max"], rf["w_Theta_max"], rf["w_t_max"], rf["w_col"]]
    arf = config["action_reward_factors"]
    P.action_factor_is_scalar = int(np.isscalar(arf))
    arf = np.broadcast_to(np.asarray(arf, dtype=float), (n_u,))
    for i in range(n_u):
        P.action_reward_factors[i] = arf[i]
    P.cur_mu, P.cur_sigma = cur_mu, cur_sigma
    rc = config["radar"]
    rt = radar_table(rc["alpha"], rc["beta"], rc["ray_per_deg"], rc["max_dist"], rc.get("blocksize_reduce", 2))
    P.n_rays, P.n_vert, P.n_horiz, P.block = rt["n_rays"], rt["n_vert"], rt["n_horiz"], rt["block"]
    P.n_rays_reduced = rt["n_rays_reduced"]
    P.radar_max_dist = rt["max_dist"]
    flat = rt["rd_b"].ravel()
    C.memmove(P.rd_b, flat.ctypes.data, flat.nbytes)
    C.memmove(P.beta_oa, rt["beta_oa"].ctypes.data, rt["beta_oa"].nbytes)
    P.n_obs = 16 + rt["n_rays_reduced"]
    return P


def set_env(E, state, goal, heading_goal, capsules, spheres, current, u=None, t_steps=0):
    E.state[:] = np.asarray(state, dtype=float).tolist()
    for i in range(MAX_U):
        E.u[i] = 0.0 if u is None or i >= len(u) else float(u[i])
    E.goal[:] = np.asarray(goal, dtype=float).tolist()
    E.heading_goal = float(heading_goal)
    E.cur[:] = np.asarray(current, dtype=float).tolist()
    capsules = np.asarray(capsules, dtype=float).reshape(-1, 7)
    spheres = np.asarray(spheres, dtype=float).reshape(-1, 4)
    E.n_caps, E.n_sph = capsules.shape[0], spheres.shape[0]
    for k in range(E.n_caps):
        E.caps[k][:] = capsules[k].tolist()
    for k in range(E.n_sph):
        E.sph[k][:] = spheres[k].tolist()
    E.t_steps = int(t_steps)
    E.cum_reward = 0.0
    return E


def copy_env(E):
    """An independent copy of an OrcEnv (step() advances the env it is given)."""
    out = OrcEnv()
    C.memmove(C.byref(out), C.byref(E), C.sizeof(OrcEnv))
    return out


def rzyx(phi, theta, psi):
    """geomutils.py Rzyx as the oracle evaluates it: body -> NED rotation, 3 x 3."""
    R = np.zeros(9)
    lib().orc_Rzyx(float(phi), float(theta), float(psi), _dp(R))
    return R.reshape(3, 3)


def ray_directions(P, att):
    """World-frame unit ray directions [n_rays, 3] at attitude ``att`` (sensor.py:90-102), formed like orc_step forms
    them (each row R rd_b / |R rd_b|, summed in the same order)."""
    R = rzyx(*att)
    rd_b = np.ctypeslib.as_array(P.rd_b)[:3 * P.n_rays].reshape(-1, 3)
    v = R[:, 0] * rd_b[:, :1] + R[:, 1] * rd_b[:, 1:2] + R[:, 2] * rd_b[:, 2:3]
    return v / np.sqrt((v * v).sum(axis=1))[:, None]


def step(P, E, action, noise_w=0.0):
    """One env.step(); ``action`` dtype (float32 / float64) selects the reference's dtype-dependent branches."""
    a = np.ascontiguousarray(action)
    is_f32 = a.dtype == np.float32
    if not is_f32:
        a = a.astype(np.float64)
    out = OrcStepOut()
    lib().orc_step(C.byref(P), C.byref(E), a.ctypes.data_as(C.c_void_p), int(is_f32), float(noise_w), C.byref(out))
    return out


class BatchOracle:
    """N independent envs stepped by orc_step_batch (OpenMP) -- the CPU baseline of bench.py.  ``env_ids`` (optional,
    uint64 array of length n_envs) makes env i the env with that GLOBAL id of a larger batch: the reset stream is
    keyed by the global id, so an arbitrary sample of a 1M-env GPU batch can be followed on its own."""

    def __init__(self, config, scenario, n_envs, seed=0, n_extra_spheres=0, n_threads=0, env_id0=0, env_ids=None,
                 vehicle_key=None):
        self.P = make_params(config, vehicle_key=vehicle_key)
        self.n = int(n_envs)
        self.scenario = SCENARIOS[scenario] | (int(n_extra_spheres) << 8)
        self.seed, self.n_threads, self.env_id0 = int(seed), int(n_threads), int(env_id0)
        self.env_ids = None
        if env_ids is not None:
            self.env_ids = np.ascontiguousarray(env_ids, dtype=np.uint64)
            assert self.env_ids.shape == (self.n,)
        self.envs = (OrcEnv * self.n)()
        L = lib()
        for i in range(self.n):
            gid = int(self.env_ids[i]) if self.env_ids is not None else self.env_id0 + i
            L.orc_reset_env(C.byref(self.P), C.byref(self.envs[i]), self.scenario, self.seed, gid)
        self.obs = np.zeros((self.n, self.P.n_obs), dtype=np.float32)
        self.reward = np.zeros(self.n)
        self.done = np.zeros(self.n, dtype=np.uint8)
        self.cond_bits = np.zeros(self.n, dtype=np.uint8)      # bit k = done condition k of the last step
        # zero-copy numpy view of the env array (AoS) for field()
        self._raw = np.ctypeslib.as_array(C.cast(self.envs, C.POINTER(C.c_uint8)), shape=(self.n * C.sizeof(OrcEnv),))
        self._raw = self._raw.reshape(self.n, C.sizeof(OrcEnv))

    def step(self, actions):
        a = np.ascontiguousarray(actions)
        is_f32 = a.dtype == np.float32
        if not is_f32:
            a = a.astype(np.float64)
        ids = self.env_ids.ctypes.data_as(C.c_void_p) if self.env_ids is not None else None
        fin = lib().orc_step_batch_ids(C.byref(self.P), C.cast(self.envs, C.c_void_p), self.n,
                                       a.ctypes.data_as(C.c_void_p), int(is_f32), self.scenario, self.seed,
                                       self.env_id0, ids, self.obs.ctypes.data_as(C.c_void_p),
                                       self.reward.ctypes.data_as(C.c_void_p), self.done.ctypes.data_as(C.c_void_p),
                                       self.cond_bits.ctypes.data_as(C.c_void_p), self.n_threads)
        return self.obs, self.reward, self.done, fin

    def field(self, name):
        """Copy of one OrcEnv field over all envs ([n] or [n, k...]), read through a strided view of the AoS block."""
        f = getattr(OrcEnv, name)
        ctype = dict(OrcEnv._fields_)[name]
        base = ctype
        shape = []
        while hasattr(base, "_length_"):
            shape.append(base._length_)
            base = base._type_
        dt = np.dtype(base)
        count = int(np.prod(shape)) if shape else 1
        out = np.empty((self.n, count), dtype=dt)
        rows = self._raw[:, f.offset:f.offset + count * dt.itemsize]
        out.view(np.uint8).reshape(self.n, -1)[:] = rows
        return out.reshape([self.n] + shape) if shape else out[:, 0].copy()
