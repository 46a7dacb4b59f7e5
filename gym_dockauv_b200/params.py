"""env_config dict + vehicle table -> the flat DockauvParams block of include/dockauv.h.

Host-side counterpart of the reference's init-time work: StateSpace matrices (objects/statespace.py:86-197),
low-pass smoothing factor (utils/lowpassfilter.py:13-27), Radar ray table (objects/sensor.py:43-71) and the
obstacle-avoidance ray weights (envs/docking3d.py:789-790).  M_inv is computed with numpy.linalg.inv exactly
like the reference, everything else is plain arithmetic on the XML numbers.
"""
import ctypes as C

import numpy as np

from . import vehicles as _veh
from .config import validate

ABI_VERSION = 4
MAX_U, MAX_CAPSULES, MAX_SPHERES, MAX_RAYS, N_REWARDS, N_STATS = 8, 8, 8, 256, 13, 16
MAX_TAPS = 1024
F64, F32 = 0, 1
ACT_F64, ACT_F32 = 0, 1
LAYOUTS = {"auto": 0, "thread_per_env": 1, "warp_rays": 2, "pipeline": 4}
VEHICLE_IDS = {"BlueROV2": 0, "LAUV": 1}
SCENARIO_IDS = {"SimpleDocking3d": 0, "SimpleCurrentDocking3d": 1, "CapsuleDocking3d": 2,
                "CapsuleCurrentDocking3d": 3, "ObstaclesDocking3d": 4, "ObstaclesCurrentDocking3d": 5,
                "ObstaclesNoCapDocking3d": 6}
# capsules each scenario spawns (docking3d.py:860-965)
SCENARIO_CAPSULES = {0: 0, 1: 0, 2: 1, 3: 1, 4: 5, 5: 5, 6: 4}
STAT_NAMES = ("episodes", "sum_return", "sum_length", "done_goal_reached", "done_out_pos", "done_out_att",
              "done_max_t", "done_collision", "sum_final_delta_d", "nan_envs", "env_steps")

_d, _i = C.c_double, C.c_int32


class DockauvParams(C.Structure):
    """Mirror of `struct DockauvParams` (include/dockauv.h); the size is cross-checked against the library."""
    _fields_ = [
        ("abi_version", _i), ("precision", _i), ("vehicle", _i), ("n_u", _i), ("scenario", _i),
        ("n_capsules", _i), ("n_spheres", _i), ("n_synthetic_spheres", _i), ("max_timesteps", _i),
        ("reward_set", _i), ("n_rays", _i), ("n_vert", _i), ("n_horiz", _i), ("block_reduce", _i),
        ("action_factor_is_scalar", _i), ("layout", _i), ("force_current", _i), ("split_chunk_envs", _i),
        ("m", _d), ("r_G", _d * 3), ("I_b", _d * 9), ("MA_diag", _d * 6), ("M_inv", _d * 36),
        ("D_lin", _d * 10), ("D_quad", _d * 10), ("D_lift", _d * 10), ("G_WB", _d), ("G_r", _d * 3),
        ("B", _d * (6 * MAX_U)), ("lauv_B", _d * 4), ("u_lo", _d * MAX_U), ("u_hi", _d * MAX_U),
        ("lp_alpha", _d), ("h", _d), ("safety_radius", _d),
        ("max_dist_from_goal", _d), ("max_attitude", _d), ("dist_goal_reached_tol", _d),
        ("u_max", _d), ("v_max", _d), ("w_max", _d), ("p_max", _d), ("q_max", _d), ("r_max", _d),
        ("w_d", _d), ("w_delta_psi", _d), ("w_delta_theta", _d), ("w_phi", _d), ("w_theta", _d),
        ("w_Thetadot", _d), ("w_oa", _d), ("w_done", _d * 5), ("action_reward_factors", _d * MAX_U),
        ("cur_mu", _d), ("cur_sigma", _d), ("radar_max_dist", _d),
        ("rd_b", _d * (MAX_RAYS * 3)), ("beta_oa", _d * MAX_RAYS),
        ("seed", C.c_uint64), ("env_id0", C.c_uint64),
    ]


class DockauvBuffers(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("state", "u_prev", "goal", "heading_goal", "current", "capsules",
                                          "spheres", "ep_return", "t_steps", "episode")]


class DockauvStepOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("obs", "reward", "done", "cond_bits", "terminal_obs", "ep_return_out",
                                          "ep_len_out", "delta_d_out")]


class DockauvDebugOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("ray_dist", "reward_arr", "euler_dot", "nu_c", "nav", "obs_f64", "state_dot")]


class DockauvRolloutOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("obs", "reward", "done", "cond_bits", "terminal_obs", "ep_return_out",
                                          "ep_len_out", "delta_d_out")]


TAP_FIELDS = ("count", "pre_state", "pre_current", "pre_scene", "pre_t_steps", "pre_episode", "pre_ep_return", "state",
              "u", "state_dot", "nu_c", "ray_dist", "reward_arr", "obs", "reward", "done", "cond_bits")


class DockauvTapBuffers(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in TAP_FIELDS]


class DockauvReplayRing(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("obs", "terminal_obs", "actions", "reward", "done")]


class DockauvReplaySample(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("obs", "actions", "next_obs", "done", "reward", "index")]


SCENARIO_BANK_FIELDS = ("rows", "cdf", "row_of_env", "n_rows", "row_stride")


class DockauvScenarioBank(C.Structure):
    _fields_ = [("rows", C.c_void_p), ("cdf", C.c_void_p), ("row_of_env", C.c_void_p), ("n_rows", C.c_int64),
                ("row_stride", C.c_int64)]


class DockauvPolicy(C.Structure):
    _fields_ = [("pi_w", C.c_void_p * 3), ("pi_b", C.c_void_p * 3), ("vf_w", C.c_void_p * 3), ("vf_b", C.c_void_p * 3),
                ("log_std", C.c_void_p), ("hidden", C.c_int32), ("deterministic", C.c_int32)]


class DockauvPolicyOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("actions", "values", "log_probs", "last_values")]


# dockauv_rollout_policy: shared memory one CTA may hold (sm_100), and what both nets' f32 weights take there
# (gym_dockauv_b200/csrc/dockauv_policy.cuh: every piece padded to a multiple of 4 floats)
POLICY_MAX_SMEM = 232448


def policy_smem_bytes(n_obs, hidden, n_u):
    net = lambda n_out: n_obs * hidden + 2 * hidden + hidden * hidden + n_out * hidden + (n_out + 3) // 4 * 4  # noqa: E731
    return 4 * (net(n_u) + net(1) + (n_u + 3) // 4 * 4)


class DockauvSquashedActor(C.Structure):
    _fields_ = [("w", C.c_void_p * 2), ("b", C.c_void_p * 2), ("mu_w", C.c_void_p), ("mu_b", C.c_void_p),
                ("log_std_w", C.c_void_p), ("log_std_b", C.c_void_p), ("hidden", C.c_int32), ("deterministic", C.c_int32)]


# dockauv_replay_collect: what the SAC actor's bf16 weights, f32 biases and the per-warp epilogue tiles of its 8 warps
# take in shared memory (gym_dockauv_b200/csrc/dockauv_sac_actor.cuh: layer 0's columns padded to a multiple of 16,
# every bf16 row by 8 more; the two heads one 16-row block); n_u <= 8 does not change it
SAC_ACTOR_HIDDEN = (64, 128, 256)


def sac_actor_smem_bytes(n_obs, hidden, n_u):
    H, k0p = hidden, (n_obs + 15) // 16 * 16
    return 2 * (H * (k0p + 8) + H * (H + 8) + 16 * (H + 8)) + 4 * (2 * H + 16) + 4 * 8 * 16 * 16


def skew(a):
    """S(a) b = a x b (utils/geomutils.py:106-128)."""
    return np.array([[0.0, -a[2], a[1]], [a[2], 0.0, -a[0]], [-a[1], a[0], 0.0]])


def rigid_body_matrices(v):
    """Inertia about CO, rigid-body and added mass, and their inverse sum (statespace.py:86-197).
    Note the reference's I_g[2,0] = +I_xz (statespace.py:100) is kept as is."""
    m = v["m"]
    r_G = np.array([v["x_G"], v["y_G"], v["z_G"]])
    I_g = np.array([[v["I_x"], -v["I_xy"], -v["I_xz"]],
                    [-v["I_xy"], v["I_y"], -v["I_yz"]],
                    [v["I_xz"], -v["I_yz"], v["I_z"]]])
    S = skew(r_G)
    I_b = I_g + m * S.dot(S.T)
    M_CG = np.zeros((6, 6))
    M_CG[:3, :3] = m * np.identity(3)
    M_CG[3:, 3:] = I_g
    H = np.identity(6)
    H[:3, 3:] = S.T
    M_RB = H.T.dot(M_CG).dot(H)
    MA_diag = -np.array([v["X_udot"], v["Y_vdot"], v["Z_wdot"], v["K_pdot"], v["M_qdot"], v["N_rdot"]])
    M_inv = np.linalg.inv(M_RB + np.diag(MA_diag))
    return dict(r_G=r_G, I_b=I_b, M_RB=M_RB, MA_diag=MA_diag, M_inv=M_inv)


def damping_coefficients(v, vehicle):
    """(lin, quad, lift) in the 10-entry order of DockauvParams: diagonal, then [1,5], [2,4], [4,2], [5,1]
    (statespace.py:337-351 for BlueROV2, LAUV.py:69-101 for LAUV)."""
    g = lambda k: float(v.get(k, 0.0))  # noqa: E731
    lin = [g("X_u"), g("Y_v"), g("Z_w"), g("K_p"), g("M_q"), g("N_r"), 0, 0, 0, 0]
    quad = [g("X_uu"), g("Y_vv"), g("Z_ww"), g("K_pp"), g("M_qq"), g("N_rr"), 0, 0, 0, 0]
    lift = [0.0] * 10
    if vehicle == "LAUV":
        lin[6:] = [g("Y_r"), g("Z_q"), g("M_w"), g("N_v")]
        quad[6:] = [g("Y_rr"), g("Z_qq"), g("M_ww"), g("N_vv")]
        lift = [0.0, g("Y_uvb") + g("Y_uvf"), g("Z_uwb") + g("Z_uwf"), 0.0, g("M_uqf"), g("N_urf"),
                g("Y_urf"), g("Z_uqf"), g("M_uwb") + g("M_uwf"), g("N_uvb") + g("N_uvf")]
    return np.array(lin, float), np.array(quad, float), np.array(lift, float)


def radar_geometry(alpha, beta, ray_per_deg, max_dist=25, blocksize_reduce=2, freq=None):
    """Body-frame ray fan and pooled shape (sensor.py:43-71, 131-137) + OA weights (docking3d.py:789-790)."""
    tol = 10e-8
    if (alpha + tol) % ray_per_deg > 0.001 or (beta + tol) % ray_per_deg > 0.001:
        raise KeyError("Initialize the radar with valid ray_per_deg for alpha and beta.")
    va = np.arange(-alpha / 2, alpha / 2 + tol, ray_per_deg)
    hb = np.arange(-beta / 2, beta / 2 + tol, ray_per_deg)
    n_v, n_h = va.shape[0], hb.shape[0]
    a = np.repeat(va, n_h)
    b = np.tile(hb, n_v)
    rd_b = np.stack([np.ones(n_v * n_h), np.sin(b), np.sin(a)], axis=1)
    rd_b = rd_b / np.linalg.norm(rd_b, axis=1)[:, None]
    beta_oa = (1 - np.abs(a) / (alpha / 2)) * (1 - np.abs(b) / (beta / 2)) + 0.01
    blk = int(blocksize_reduce)
    n_red = -(-n_v // blk) * -(-n_h // blk)
    return dict(n_rays=n_v * n_h, n_vert=n_v, n_horiz=n_h, block=blk, n_rays_reduced=n_red, rd_b=rd_b,
                beta_oa=beta_oa, alpha=a, beta=b, max_dist=float(max_dist))


def pack_params(env_config, scenario, precision="f64", seed=0, env_id0=0, layout="auto", n_capsules=None,
                n_spheres=0, n_synthetic_spheres=0, vehicle_xml=None, control_mode="joystick", cur_mu=0.005,
                cur_sigma=0.0, force_current=False, split_chunk_envs=0):
    """Returns (DockauvParams, meta) where meta carries host-side derived values (n_obs, u_bound, radar table)."""
    cfg = validate(env_config)
    vname = cfg["vehicle"]
    v = _veh.load_vehicle(vname, xml_path=vehicle_xml, control_mode=control_mode)
    P = DockauvParams()
    P.abi_version = ABI_VERSION
    P.precision = {"f64": F64, "f32": F32}[precision]
    P.vehicle = VEHICLE_IDS[vname]
    n_u = v["n_u"]
    P.n_u = n_u
    scn = SCENARIO_IDS[scenario] if isinstance(scenario, str) else int(scenario)
    P.scenario = scn
    P.n_capsules = SCENARIO_CAPSULES[scn] if n_capsules is None else int(n_capsules)
    P.n_spheres = int(max(n_spheres, n_synthetic_spheres))
    P.n_synthetic_spheres = int(n_synthetic_spheres)
    if P.n_capsules > MAX_CAPSULES or P.n_spheres > MAX_SPHERES:
        raise ValueError("at most 8 capsules and 8 spheres per env")
    P.max_timesteps = int(cfg["max_timesteps"])
    P.reward_set = int(cfg["reward_set"])
    P.layout = LAYOUTS[layout]
    P.force_current = int(bool(force_current))
    P.split_chunk_envs = int(split_chunk_envs)
    rb = rigid_body_matrices(v)
    P.m = v["m"]
    P.r_G[:] = rb["r_G"].tolist()
    P.I_b[:] = rb["I_b"].ravel().tolist()
    P.MA_diag[:] = rb["MA_diag"].tolist()
    P.M_inv[:] = rb["M_inv"].ravel().tolist()
    lin, quad, lift = damping_coefficients(v, vname)
    P.D_lin[:] = lin.tolist()
    P.D_quad[:] = quad.tolist()
    P.D_lift[:] = lift.tolist()
    W = v["m"] * _veh.GRAVITY
    BY = v["BY"]
    P.G_WB = W - BY
    P.G_r[:] = [v["x_G"] * W - v["x_B"] * BY, v["y_G"] * W - v["y_B"] * BY, v["z_G"] * W - v["z_B"] * BY]
    if vname == "BlueROV2":
        flat = np.asarray(v["B"], dtype=float).ravel()
        for k, x in enumerate(flat):
            P.B[k] = x
    else:
        P.lauv_B[:] = [v["Y_uudr"], v["Z_uuds"], v["M_uuds"], v["N_uudr"]]
    u_bound = np.asarray(v["u_bound"], dtype=float)
    for k in range(n_u):
        P.u_lo[k], P.u_hi[k] = u_bound[k, 0], u_bound[k, 1]
    h = cfg["t_step_size"]
    P.h = h
    P.lp_alpha = h / (h + _veh.LOWPASS_T1)
    P.safety_radius = _veh.SAFETY_RADIUS
    for k in ("max_dist_from_goal", "max_attitude", "dist_goal_reached_tol", "u_max", "v_max", "w_max", "p_max",
              "q_max", "r_max"):
        setattr(P, k, float(cfg[k]))
    rf = cfg["reward_factors"]
    for k in ("w_d", "w_delta_psi", "w_delta_theta", "w_phi", "w_theta", "w_Thetadot", "w_oa"):
        setattr(P, k, float(rf[k]))
    P.w_done[:] = [float(rf[k]) for k in ("w_goal", "w_deltad_max", "w_Theta_max", "w_t_max", "w_col")]
    arf = cfg["action_reward_factors"]
    P.action_factor_is_scalar = int(np.isscalar(arf))
    arf = np.broadcast_to(np.asarray(arf, dtype=float), (n_u,))
    for k in range(n_u):
        P.action_reward_factors[k] = arf[k]
    P.cur_mu, P.cur_sigma = float(cur_mu), float(cur_sigma)
    rc = dict(cfg["radar"])
    rg = radar_geometry(rc["alpha"], rc["beta"], rc["ray_per_deg"], rc.get("max_dist", 25),
                        rc.get("blocksize_reduce", 2))
    if rg["n_rays"] > MAX_RAYS:
        raise ValueError(f"radar has {rg['n_rays']} rays; the kernels support at most {MAX_RAYS}")
    P.n_rays, P.n_vert, P.n_horiz, P.block_reduce = rg["n_rays"], rg["n_vert"], rg["n_horiz"], rg["block"]
    P.radar_max_dist = rg["max_dist"]
    flat = np.ascontiguousarray(rg["rd_b"].ravel())
    C.memmove(P.rd_b, flat.ctypes.data, flat.nbytes)
    bo = np.ascontiguousarray(rg["beta_oa"])
    C.memmove(P.beta_oa, bo.ctypes.data, bo.nbytes)
    P.seed = int(seed) & (2 ** 64 - 1)
    P.env_id0 = int(env_id0)
    meta = dict(n_obs=16 + rg["n_rays_reduced"], n_u=n_u, u_bound=u_bound, radar=rg, vehicle=v, rigid_body=rb,
                scenario=scn)
    return P, meta
