/* dockauv.h -- C ABI of the B200-native batched docking-AUV simulator (libdockauv_b200.so).
 *
 * This is the drop-in boundary for the `env.step()` hot path of Erikx3/gym_dockauv.  Every entry point
 * names the reference interface it replaces (paths relative to the reference repo root):
 *
 *   dockauv_create / dockauv_destroy   BaseDocking3d.__init__            gym_dockauv/envs/docking3d.py:48-220
 *                                      (vehicle + env_config + Radar constants frozen into one handle)
 *   dockauv_bind                       the per-env attributes that persist across steps (SURVEY.md 9.8):
 *                                      auv.state, auv.u, goal_location, heading_goal_reached, current,
 *                                      capsules / spheres, t_steps, cumulative_reward
 *   dockauv_reset                      BaseDocking3d.reset + <Scenario>.generate_environment
 *                                                                          docking3d.py:222-322, 803-988
 *   dockauv_step                       BaseDocking3d.step                 docking3d.py:346-402
 *                                      (Current.sim, AUVSim.step, Radar.update, update_radar_collision,
 *                                       update_body_collision, update_navigation_errors, observe, is_done,
 *                                       reward_step, and SB3-VecEnv style auto-reset)
 *   dockauv_step_host                  the same call with HOST buffers (what SB3's DummyVecEnv.step_wait
 *                                      hands over, train.py:64-71): H2D, kernel(s), D2H inside the call
 *   dockauv_get_stats / _clear_stats   FullDataStorage.update bookkeeping  utils/datastorage.py:65-74
 *   dockauv_rollout                    the step loop of the caller: model.learn() -> collect_rollouts of SB3's
 *                                      on-policy algorithms (train.py:64-71) and predict()'s while-loop
 *                                      (train.py:107-118), for action sequences that are known up front
 *   dockauv_rollout_policy             the same loops with SB3's MlpPolicy choosing the actions on the device
 *                                      (OnPolicyAlgorithm.collect_rollouts, predict(deterministic=True))
 *   dockauv_gae                        RolloutBuffer.compute_returns_and_advantage of the PPO caller
 *                                      (stable-baselines3 1.5.0, requirements.txt; selected at train.py:64)
 *   dockauv_replay_sample              ReplayBuffer.sample of the SAC caller (MODEL = SAC at train.py:64)
 *   dockauv_replay_collect             OffPolicyAlgorithm.collect_rollouts of the SAC caller: SAC's actor picks the
 *                                      actions on the device and the steps fill the replay ring
 *   DockauvDebugOut (state_dot, ...)   EpisodeDataStorage.update          utils/datastorage.py:268-288
 *   dockauv_set_taps                   the same, during training: every step of a few chosen envs recorded on
 *                                      the device (interval_datastorage, config.py; datastorage.py:268-288)
 *   dockauv_set_scenario_bank          a subclass's own generate_environment override (docking3d.py:795-988):
 *                                      resets draw caller-supplied initial conditions, uniformly or by weight
 *
 * Conventions
 *   - plain C types only; no torch / C++ types cross this boundary.
 *   - all `*_dev` pointers are device pointers on the handle's device.  The library never allocates, frees
 *     or keeps caller buffers beyond what dockauv_bind() registered; the caller (PyTorch) owns them.  The
 *     handle owns its ray table, the statistics vector, the buffers between the launches of a step
 *     (a 16-word record, the ray list entry and a float copy of the obstacles: ~350 bytes per env), lazily, device
 *     staging for dockauv_step_host and, while taps are set (dockauv_set_taps), shadow copies of the tapped envs.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Calls are asynchronous and
 *     stream-ordered; one handle must not be used from two threads at once.  Large batches (>= 131,072 envs)
 *     are stepped as two halves on two handle-owned streams that are forked from / joined to `stream` by
 *     events, so everything stays ordered with respect to `stream` (and capturable into a CUDA graph).
 *   - every function returns 0 on success, a negative DOCKAUV_E* code otherwise; dockauv_last_error()
 *     returns a human-readable description of the last failure on the calling thread.
 *   - there is NO CPU fallback: without a usable CUDA device dockauv_create fails with DOCKAUV_ECUDA.
 *
 * Memory layout (HBM): structure-of-arrays, component-major, env index fastest, e.g. state[c * n_envs + i].
 * `real` below is double for DOCKAUV_F64 handles and float for DOCKAUV_F32 handles.
 */
#ifndef DOCKAUV_H
#define DOCKAUV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DOCKAUV_ABI_VERSION 4

#if defined(__GNUC__)
#define DOCKAUV_API __attribute__((visibility("default")))
#else
#define DOCKAUV_API
#endif

#define DOCKAUV_MAX_U 8          /* control inputs: BlueROV2 joystick 6, direct 8; LAUV 3 */
#define DOCKAUV_MAX_CAPSULES 8
#define DOCKAUV_MAX_SPHERES 8
#define DOCKAUV_MAX_RAYS 256
#define DOCKAUV_N_REWARDS 13     /* docking3d.py:153 */
#define DOCKAUV_N_STATS 16

/* error codes */
#define DOCKAUV_OK 0
#define DOCKAUV_EINVAL (-1)      /* bad argument */
#define DOCKAUV_ECUDA (-2)       /* CUDA runtime error (see dockauv_last_error) */
#define DOCKAUV_ESTATE (-3)      /* call order (e.g. step before bind) */

/* precision of the persistent state and of the arithmetic */
#define DOCKAUV_F64 0
#define DOCKAUV_F32 1

/* vehicles (gym_dockauv/objects/vehicles/) */
#define DOCKAUV_VEHICLE_BLUEROV2 0
#define DOCKAUV_VEHICLE_LAUV 1

/* scenarios = the generate_environment() variants, docking3d.py:795-988 */
#define DOCKAUV_SCN_SIMPLE 0
#define DOCKAUV_SCN_SIMPLE_CURRENT 1
#define DOCKAUV_SCN_CAPSULE 2
#define DOCKAUV_SCN_CAPSULE_CURRENT 3
#define DOCKAUV_SCN_OBSTACLES 4
#define DOCKAUV_SCN_OBSTACLES_CURRENT 5
#define DOCKAUV_SCN_OBSTACLES_NOCAP 6

/* action dtypes accepted by dockauv_step (the reference's arithmetic depends on it, auvsim.py:74-75,
 * docking3d.py:584-585: a float32 action array keeps parts of the computation in float32) */
#define DOCKAUV_ACT_F64 0
#define DOCKAUV_ACT_F32 1

/* kernel layouts */
#define DOCKAUV_LAYOUT_AUTO 0
#define DOCKAUV_LAYOUT_THREAD_PER_ENV 1   /* one thread does everything for one env */
#define DOCKAUV_LAYOUT_WARP_RAYS 2        /* one launch: dynamics thread-per-env, radar one warp per env (lanes = rays) */
#define DOCKAUV_LAYOUT_PIPELINE 4         /* dynamics + cull + finish of the envs with nothing in view (thread per env), rays +
                                             finish (a thread or a warp per env that has an obstacle in view, from compact
                                             lists), episode end (per finished env, from a compact list) */

/* indices into the stats vector (sums since the last clear; reduce over ranks with one all-reduce) */
#define DOCKAUV_STAT_EPISODES 0
#define DOCKAUV_STAT_SUM_RETURN 1
#define DOCKAUV_STAT_SUM_LENGTH 2
#define DOCKAUV_STAT_COND0 3            /* ..COND0+4: Done-Goal_reached, out_pos, out_att, max_t, collision */
#define DOCKAUV_STAT_SUM_FINAL_DELTA_D 8
#define DOCKAUV_STAT_NAN_ENVS 9
#define DOCKAUV_STAT_ENV_STEPS 10

/* Everything that is constant for the lifetime of a handle.  Filled by the host side from the reference's
 * env_config dict (config/env_config.py:20-91) and vehicle XML (objects/vehicles/ *.xml). */
typedef struct DockauvParams {
    int32_t abi_version;         /* DOCKAUV_ABI_VERSION */
    int32_t precision;           /* DOCKAUV_F64 / DOCKAUV_F32 */
    int32_t vehicle;             /* DOCKAUV_VEHICLE_* */
    int32_t n_u;                 /* number of control inputs */
    int32_t scenario;            /* DOCKAUV_SCN_* (used by reset / auto-reset) */
    int32_t n_capsules;          /* capsules per env (0..8); row order = reference's self.capsules */
    int32_t n_spheres;           /* spheres per env (0..8) */
    int32_t n_synthetic_spheres; /* reset extension: random unit spheres per env (BASELINE config C4), <= n_spheres */
    int32_t max_timesteps;
    int32_t reward_set;          /* 1 or 2, docking3d.py:515-548 */
    int32_t n_rays, n_vert, n_horiz, block_reduce;   /* sensor.py:43-71; n_rays = n_vert * n_horiz */
    int32_t action_factor_is_scalar;   /* config "action_reward_factors" was a python scalar */
    int32_t layout;              /* DOCKAUV_LAYOUT_* */
    int32_t force_current;       /* evaluate the ocean current even if the scenario spawns none (injected currents) */
    int32_t split_chunk_envs;    /* DOCKAUV_LAYOUT_PIPELINE: 0 = library default: the whole batch, in two halves on two streams
                                    from 131,072 envs on; any other value: the whole batch as one launch group on the
                                    caller's stream */
    /* rigid body + hydrodynamics (statespace.py) */
    double m;
    double r_G[3];
    double I_b[9];               /* statespace.py:105-117, row-major */
    double MA_diag[6];           /* diag(M_A) = -(X_udot..N_rdot), statespace.py:164-187 */
    double M_inv[36];            /* inv(M_RB + M_A), statespace.py:190-197, row-major */
    double D_lin[10];            /* linear damping: 6 diagonal entries then [1,5],[2,4],[4,2],[5,1] (LAUV.py:78-83) */
    double D_quad[10];           /* quadratic damping, same order; entry [i,j] multiplies |nu_j| (LAUV.py:84-89) */
    double D_lift[10];           /* lift, same order; every entry multiplies |u| (LAUV.py:90-95,101) */
    double G_WB;                 /* W - BY */
    double G_r[3];               /* (x_G W - x_B BY, y_G W - y_B BY, z_G W - z_B BY), statespace.py:387-396 */
    double B[6 * DOCKAUV_MAX_U]; /* BlueROV2: constant 6 x n_u, row-major (BlueROV2.py:34-72) */
    double lauv_B[4];            /* LAUV: Y_uudr, Z_uuds, M_uuds, N_uudr (LAUV.py:59-67) */
    double u_lo[DOCKAUV_MAX_U], u_hi[DOCKAUV_MAX_U];   /* u_bound */
    double lp_alpha;             /* h / (h + T1), lowpassfilter.py:27 */
    double h;                    /* t_step_size */
    double safety_radius;        /* auvsim.py:43 */
    /* env_config */
    double max_dist_from_goal, max_attitude, dist_goal_reached_tol;
    double u_max, v_max, w_max, p_max, q_max, r_max;
    double w_d, w_delta_psi, w_delta_theta, w_phi, w_theta, w_Thetadot, w_oa;
    double w_done[5];            /* w_goal, w_deltad_max, w_Theta_max, w_t_max, w_col */
    double action_reward_factors[DOCKAUV_MAX_U];
    /* current (objects/current.py) */
    double cur_mu, cur_sigma;
    /* radar */
    double radar_max_dist;
    double rd_b[DOCKAUV_MAX_RAYS * 3];   /* body-frame unit ray directions, sensor.py:63-71 */
    double beta_oa[DOCKAUV_MAX_RAYS];    /* obstacle-avoidance ray weights, docking3d.py:789-790 */
    /* reset */
    uint64_t seed;               /* Philox key */
    uint64_t env_id0;            /* global id of local env 0 (rank offset when the batch is sharded) */
} DockauvParams;

/* Caller-owned persistent per-env state (device pointers). */
typedef struct DockauvBuffers {
    void *state;          /* real[12][N]: x y z phi theta psi | u v w p q r (relative velocity) */
    void *u_prev;         /* real[n_u][N]: low-passed command */
    void *goal;           /* real[3][N] */
    void *heading_goal;   /* real[N] */
    void *current;        /* real[5][N]: V_c, alpha, beta, V_min, V_max */
    void *capsules;       /* real[n_capsules*7][N]: vec_bot[3], vec_top[3], radius per capsule */
    void *spheres;        /* real[n_spheres*4][N]: centre[3], radius per sphere */
    void *ep_return;      /* real[N]: cumulative reward of the running episode */
    int32_t *t_steps;     /* int32[N] */
    int32_t *episode;     /* int32[N]: episodes started so far (Philox counter) */
} DockauvBuffers;

/* Per-step outputs (device pointers; nullable ones are skipped).  When n_obs is a multiple of 4 (every stock radar
 * geometry) observation rows are written with 128-bit stores: obs and terminal_obs must then be 16-byte aligned
 * (DOCKAUV_EINVAL otherwise). */
typedef struct DockauvStepOut {
    float *obs;            /* f32[N][n_obs] row-major; all-zero row when the env was auto-reset (docking3d.py:269,322) */
    void *reward;          /* real[N] */
    uint8_t *done;         /* u8[N] */
    uint8_t *cond_bits;    /* u8[N], nullable: bit k = done condition k (docking3d.py:606-617) */
    float *terminal_obs;   /* f32[N][n_obs], nullable: last observation of episodes that ended this step
                              (rows of envs that are not done are left untouched) */
    void *ep_return_out;   /* real[N], nullable: return of the episode that ended this step (Monitor 'r') */
    int32_t *ep_len_out;   /* int32[N], nullable: length of the episode that ended this step (Monitor 'l') */
    void *delta_d_out;     /* real[N], nullable: distance to the goal after the step = info["delta_d"] (docking3d.py:400) */
} DockauvStepOut;

/* Optional per-step intermediate values for the parity tests (device pointers, all nullable). */
typedef struct DockauvDebugOut {
    void *ray_dist;        /* real[n_rays][N], clamped distances (sensor.py:113-118) */
    void *reward_arr;      /* real[13][N] */
    void *euler_dot;       /* real[3][N], post-step Theta_dot (auvsim.py:108) */
    void *nu_c;            /* real[3][N], pre-step body-frame current (docking3d.py:349) */
    void *nav;             /* real[3][N]: delta_d, delta_theta, delta_psi */
    void *obs_f64;         /* real[n_obs][N]: observation before the float32 cast */
    void *state_dot;       /* real[12][N]: auv._state_dot = state_dot(post-step state, pre-step nu_c), auvsim.py:108
                              (the step itself only needs its Theta_dot part; the full vector is what
                              EpisodeDataStorage logs, datastorage.py:277) */
} DockauvDebugOut;

/* Outputs of dockauv_rollout: the per-step outputs stacked over T steps (device pointers). */
typedef struct DockauvRolloutOut {
    float *obs;            /* f32[T][N][n_obs]: row t = observation returned by step t */
    void *reward;          /* real[T][N] */
    uint8_t *done;         /* u8[T][N] */
    uint8_t *cond_bits;    /* u8[T][N], nullable */
    float *terminal_obs;   /* f32[T][N][n_obs], nullable: rows of episodes that ended at step t (others untouched) */
    void *ep_return_out;   /* real[T][N], nullable: only entries of episodes that ended at step t are written */
    int32_t *ep_len_out;   /* int32[T][N], nullable: same; the call zero-fills it first, so length > 0 marks an end */
    void *delta_d_out;     /* real[T][N], nullable */
} DockauvRolloutOut;

/* Ring of per-step records of the tapped envs (dockauv_set_taps): caller-owned device buffers.  S = capacity,
 * K = n_taps, real = handle precision; component-major inside a slot, tap index fastest. */
#define DOCKAUV_MAX_TAPS 1024
typedef struct DockauvTapBuffers {
    int64_t *count;        /* int64[1]: steps recorded since dockauv_set_taps; the next record goes to slot count % S */
    /* pre-step inputs of the tapped envs (what the real step read) */
    void *pre_state;       /* real[S][12][K] */
    void *pre_current;     /* real[S][5][K] */
    void *pre_scene;       /* real[S][4 + 7*n_capsules + 4*n_spheres][K]: goal[3], heading_goal, capsules, spheres */
    int32_t *pre_t_steps, *pre_episode;   /* int32[S][K] */
    void *pre_ep_return;   /* real[S][K] */
    /* post-step values, before any auto-reset */
    void *state, *u, *state_dot, *nu_c, *ray_dist, *reward_arr;   /* real[S][12|n_u|12|3|n_rays|13][K] */
    float *obs;            /* f32[S][K][n_obs]: the real observation, also for envs whose episode ended */
    void *reward;          /* real[S][K] */
    uint8_t *done, *cond_bits;            /* u8[S][K] */
} DockauvTapBuffers;

typedef struct DockauvHandle DockauvHandle;

DOCKAUV_API int dockauv_abi_version(void);
DOCKAUV_API const char *dockauv_last_error(void);
DOCKAUV_API size_t dockauv_sizeof_params(void);

/* n_obs = 16 + ceil(n_vert/block) * ceil(n_horiz/block) (docking3d.py:115, sensor.py:135-137) */
DOCKAUV_API int dockauv_n_obs(const DockauvParams *p);

DOCKAUV_API int dockauv_create(const DockauvParams *params, int64_t n_envs, int device, DockauvHandle **out);
DOCKAUV_API int dockauv_destroy(DockauvHandle *h);
DOCKAUV_API int dockauv_bind(DockauvHandle *h, const DockauvBuffers *buffers);

/* Re-key the counter-based random stream (gym's reset(seed=...), docking3d.py:296-298). */
DOCKAUV_API int dockauv_set_seed(DockauvHandle *h, uint64_t seed);

/* Re-initialise envs whose mask byte is non-zero (all envs if mask_dev == NULL). */
DOCKAUV_API int dockauv_reset(DockauvHandle *h, const uint8_t *mask_dev, void *stream);

/* The cull code reads a float copy of the obstacles relative to the goal, which the library keeps next to the bound
 * buffers: dockauv_bind and every reset (dockauv_reset, auto-reset inside a step) write it.  A caller that writes the
 * bound `capsules`, `spheres` or `goal` buffers ITSELF (exact-state injection: the reference's env.capsules = [...] /
 * env.goal_location = ..., docking3d.py:860-946) calls this afterwards, on the stream that did the writes. */
DOCKAUV_API int dockauv_refresh_obstacles(DockauvHandle *h, void *stream);

/* One batched env.step().  actions_dev: [N][n_u] row-major, float or double per action_dtype.
 * noise_dev (nullable): real[N] N(0, sigma) draws for Current.sim; when NULL and cur_sigma > 0 the draw
 * comes from the handle's Philox stream.  auto_reset != 0 re-initialises finished envs in the same launch. */
DOCKAUV_API int dockauv_step(DockauvHandle *h, const void *actions_dev, int action_dtype, const void *noise_dev,
                 const DockauvStepOut *out, const DockauvDebugOut *debug_or_null, int auto_reset, void *stream);

/* dockauv_step replays a CUDA graph of its launch sequence, captured once per set of pointers (actions, noise, outputs) and
 * cached per handle (96 sets; calls with debug outputs, with timing enabled, or on a stream that is itself being captured
 * issue plain launches).  On by default; dockauv_enable_step_graph(h, 0) switches to plain launches. */
DOCKAUV_API int dockauv_enable_step_graph(DockauvHandle *h, int enabled);
DOCKAUV_API int dockauv_step_graph_captures(DockauvHandle *h, int64_t *n_captures);

/* Same step with HOST buffers (pinned memory recommended): actions are copied in, obs/reward/done (and
 * cond_bits if non-NULL) are copied out, pipelined in chunks over the handle's internal streams; returns
 * after the results are in host memory.  The call is ordered after work already issued on the legacy default
 * stream; a caller that drives the handle from another stream synchronises that stream first.
 * reward_host is double[N] or float[N] per the handle precision.
 * aux_dev_or_null: optional DEVICE buffers for the per-episode extras (only terminal_obs, ep_return_out and
 * ep_len_out are read from it); they stay on the device, the caller fetches the few finished rows it needs. */
DOCKAUV_API int dockauv_step_host(DockauvHandle *h, const void *actions_host, int action_dtype, float *obs_host,
                      void *reward_host, uint8_t *done_host, uint8_t *cond_bits_host, int auto_reset,
                      const DockauvStepOut *aux_dev_or_null);

/* T consecutive batched steps with actions known up front (random-action rollouts, replayed action logs):
 * actions_dev is [T][N][n_u] row-major.  Equivalent to T dockauv_step calls writing into row t of `out`, but
 * issued from C (no per-step host round trip); with use_graph != 0 the launch sequence is captured once into a
 * CUDA graph per (pointers, T) and replayed, which is what makes small batches launch-bound no longer.
 * Stochastic-current handles draw their noise from the handle's Philox stream. */
DOCKAUV_API int dockauv_rollout(DockauvHandle *h, const void *actions_dev, int action_dtype, int n_steps,
                    const DockauvRolloutOut *out, int auto_reset, int use_graph, void *stream);

/* Closed-loop rollout: stable-baselines3's default MlpPolicy (separate pi and vf nets n_obs -> H -> H with Tanh,
 * action_net H -> n_u, value_net H -> 1, state-independent log_std, diagonal Gaussian) picks each step's actions on the
 * device.  H is a multiple of 32 in 32..128, and both nets' f32 weights must fit one CTA's shared memory (227 KB;
 * n_obs 36, H 64: 53 KB); DOCKAUV_EINVAL otherwise. */
typedef struct DockauvPolicy {        /* caller-owned f32 device tensors, nn.Linear layout: weight [out][in], bias [out] */
    const float *pi_w[3], *pi_b[3];   /* n_obs->H, H->H, H->n_u */
    const float *vf_w[3], *vf_b[3];   /* n_obs->H, H->H, H->1 */
    const float *log_std;             /* [n_u] */
    int32_t hidden, deterministic;
} DockauvPolicy;
typedef struct DockauvPolicyOut {     /* f32, device */
    float *actions;                   /* [T][N][n_u] raw samples (SB3 RolloutBuffer.actions) */
    float *values, *log_probs;        /* [T][N] */
    float *last_values;               /* [N], nullable: V(observation after step T-1), the GAE bootstrap */
} DockauvPolicyOut;

/* T steps of collect_rollouts (or, with deterministic != 0, of predict()'s loop) in one call.  Step t's policy reads
 * obs0_dev ([N][n_obs], f32) for t = 0 and row t-1 of out->obs otherwise, and writes, per env:
 *   actions   a = mu + sigma eps (deterministic: a = mu), as SB3's RolloutBuffer stores it
 *   values    V(obs)
 *   log_probs sum_k (-eps_k^2 / 2 - log sigma_k - log(2 pi) / 2)  (deterministic: eps = 0)
 * and the step reads a clipped to the action space [u_lo, u_hi] (np.clip in collect_rollouts) as float32 actions, from a
 * library-owned [N][n_u] buffer.  eps comes from the handle's Philox4x32-10 key at counter (global id lo, global id hi,
 * episode, 0xC0000000 | (t_steps mod 2^29) << 1 | j), j = 0, 1, with the env's episode and t_steps before the step;
 * Box-Muller on the 32-bit words (w >> 8) gives four normals per block (eps_{4j..4j+3}; DESIGN.md section 5.4).  So the
 * actions depend on (seed, global id, episode, t) only: they do not change with sharding, and a reset with the same seed
 * reproduces the rollout bit for bit.  With last_values set, one more policy evaluation writes V(row T-1 of out->obs).
 * Everything else is as in dockauv_rollout (ep_len_out zero-filled first, row alignment checked, taps recorded).  The
 * arguments are checked on the host first (the checks that need no handle before the null-handle check).
 * Graphs (use_graph != 0): one CUDA graph per (policy pointers, hidden, deterministic, obs0, outputs, T, auto_reset,
 * seed), a few cached per handle, so a training rollout and a deterministic evaluation rollout alternate without
 * re-capture.  Weights rewritten in place (optimizer.step()) are read by the next replay; re-allocated parameters (e.g.
 * .to()) are new pointers and are captured anew. */
DOCKAUV_API int dockauv_rollout_policy(DockauvHandle *h, const DockauvPolicy *pol, const float *obs0_dev, int n_steps,
                                       const DockauvRolloutOut *out, const DockauvPolicyOut *pout, int auto_reset,
                                       int use_graph, void *stream);

/* Record the envs env_ids_host[0..n_taps) (local indices, distinct, < n_envs, n_taps <= DOCKAUV_MAX_TAPS) on every
 * following dockauv_step / dockauv_rollout into the ring `bufs` (capacity slots); n_taps = 0 removes the taps (capacity
 * and bufs are then ignored).  Zeroes *bufs->count and drops the cached step and rollout graphs.
 * Each step first copies the tapped envs' pre-step state into the ring and into two handle-owned K-env shadows (one
 * launch on `stream`, before the step).  On a handle-owned side stream that joins `stream` before the call returns, one
 * shadow is stepped by the handle's own layout with the real step's inputs (so obs, reward, done, cond_bits, state and u
 * are exactly the real step's, before any auto-reset), the other by the single-launch kernel with debug outputs
 * (state_dot, nu_c, ray_dist, reward_arr); both without auto-reset.  Their results are copied to the ring slot, after
 * which *count is incremented on the device.  The real step and its outputs are left exactly as they are without taps.
 * dockauv_step_host refuses to run while taps are set (DOCKAUV_ESTATE): taps record device-driven steps. */
DOCKAUV_API int dockauv_set_taps(DockauvHandle *h, const int64_t *env_ids_host, int n_taps, int capacity,
                                 const DockauvTapBuffers *bufs);

/* Scenario bank: a caller-owned device table of K initial conditions that every reset draws from while it is set (the
 * in-step auto-reset of every layout and dockauv_reset), in place of the scenario's built-in distributions.  It stands
 * in for a subclass's own generate_environment (docking3d.py:795-988).
 *
 * A row holds W = 15 + 7 n_capsules + 4 n_spheres reals in the handle's precision:
 *   [0:6] pose x y z phi theta psi | [6:9] goal | [9] heading goal | [10:15] current V_c alpha beta V_min V_max |
 *   capsule slots (bot[3], top[3], r) | sphere slots (centre[3], r)
 * A reset from row r writes the pose and zeroes nu_r (auvsim.py:55-65), copies goal, heading goal, current and
 * obstacles (and the library's obstacle copies for the cull), zeroes u_prev, t_steps and ep_return, increments episode
 * and, when row_of_env is set, moves plane 0 to plane 1 and writes r to plane 0.  Unused obstacle slots take the form the
 * built-in reset gives them: radius 0 and every point at least 1e5 m from the goal.
 *
 * The row is drawn from Philox4x32-10 block (global id lo, global id hi, episode before the reset, 0x40000000): uniform
 * over K rows (high 64 bits of a 64-bit word times K), or, with cdf, the first r with cdf[r] > u cdf[K-1] for the block's
 * 53-bit uniform u (zero-weight rows are never drawn).  The draw depends on (seed, global id, episode) only: the same rows
 * whatever the sharding, and reset(seed=...) reproduces them. */
typedef struct DockauvScenarioBank {
    const void   *rows;        /* real[K][row_stride], caller-owned, 16-byte aligned */
    const double *cdf;         /* nullable: f64[K] running sum of non-negative row weights; NULL = uniform */
    int32_t      *row_of_env;  /* nullable: int32[2][N]; plane 0 = row of the running episode,
                                  plane 1 = row of the episode the env's most recent reset ended;
                                  -1 = none, the caller fills it before the first set */
    int64_t       n_rows;      /* K, 1 .. 2^31 - 1 */
    int64_t       row_stride;  /* in reals, >= W, row_stride * sizeof(real) a multiple of 16 */
} DockauvScenarioBank;

/* Set (bank_or_null non-NULL) or clear (NULL) the scenario bank.  The arguments are checked on the host first (rows,
 * K, alignment and stride: these checks need no handle and come before the null-handle check), then one validation
 * kernel reads the K rows and the cdf on `stream`, and the call synchronises `stream`.  A bank is refused
 * (DOCKAUV_EINVAL, the message names the first offending row and field) when a value is not finite, a radius is
 * negative, an obstacle is neither within 2 km of its row's goal at every defining point nor in the unused-slot form
 * (not checked on handles whose float cull is off anyway), a row has a non-zero current on a handle that does not
 * evaluate the current (force_current), or the cdf is not finite and non-decreasing from >= 0 with cdf[K-1] > 0.  A
 * refused bank leaves the previous setting in effect.
 * Graphs: the bank's pointers and K are baked into the captured step and rollout graphs.  A call with other pointers, K
 * or stride, and clearing, drops the cached graphs; a call with the SAME values only re-validates the contents and keeps
 * every graph.  That is how rows or weights rewritten in place are published (a curriculum update once per rollout).
 * Contents rewritten in place without this call are used unvalidated, like buffers written without
 * dockauv_refresh_obstacles. */
DOCKAUV_API int dockauv_set_scenario_bank(DockauvHandle *h, const DockauvScenarioBank *bank_or_null, void *stream);

/* Generalised advantage estimation over a stacked rollout, one thread per env walking t = T-1 .. 0
 * (float32 like the caller's RolloutBuffer):
 *   delta_t = r_t + gamma * V_{t+1} * (1 - done_t) - V_t ;  A_t = delta_t + gamma * lambda * (1 - done_t) * A_{t+1}
 * with V_T = last_values, returns = A + V.  rewards_dev is real[T][N] in the precision given by reward_precision
 * (DOCKAUV_F64 / DOCKAUV_F32), i.e. the `reward` rows dockauv_rollout / dockauv_step wrote; done_t is the done flag
 * returned by step t (the next observation starts a new episode).  Needs no handle. */
DOCKAUV_API int dockauv_gae(const void *rewards_dev, int reward_precision, const float *values_dev,
                const float *last_values_dev, const uint8_t *dones_dev, int n_steps, int64_t n_envs, float gamma,
                float gae_lambda, float *advantages_dev, float *returns_dev, void *stream);

/* Replay ring of an off-policy caller: S slots of the whole batch, written by dockauv_step (slot t % S holds the
 * observation acted on at step t, the action, the reward and done flag of step t, and the last real observation of the
 * envs whose episode ended at step t). */
typedef struct DockauvReplayRing {      /* caller-owned device buffers, S slots of N envs, env index fastest in a slot */
    const float *obs;                   /* f32[S][N][n_obs] */
    const float *terminal_obs;          /* f32[S][N][n_obs] (read only for rows whose done flag is set) */
    const float *actions;               /* f32[S][N][n_u] */
    const void *reward;                 /* real[S][N], precision per reward_precision */
    const uint8_t *done;                /* u8[S][N] */
} DockauvReplayRing;
typedef struct DockauvReplaySample {    /* f32 outputs, B rows, contiguous */
    float *obs, *actions, *next_obs, *done, *reward;
    int64_t *index;                     /* nullable: slot * N + env of each row (tests, prioritised callers) */
} DockauvReplaySample;

/* `batch` transitions drawn uniformly from the n_valid * n_envs (transition, env) pairs t_first .. t_first + n_valid - 1
 * (n_valid <= n_slots - 1: the slot the next step overwrites is never drawn).  Transition t lives in slot t % n_slots;
 * its next observation is terminal_obs of that slot where the done flag is set, else obs of slot (t + 1) % n_slots.
 * Row k is drawn from the Philox stream keyed by `seed` at counter (draw, k), so equal arguments give bit-identical
 * output.  Rewards are rounded to f32 once, done is written as 0.0 / 1.0.  One launch on `stream`, no host
 * synchronisation.  When n_obs is a multiple of 4 observation rows move in 16-byte pieces: ring and output
 * observation arrays must then be 16-byte aligned (DOCKAUV_EINVAL otherwise).  Needs no handle. */
DOCKAUV_API int dockauv_replay_sample(const DockauvReplayRing *ring, int reward_precision, int n_slots, int64_t n_envs,
                                      int n_obs, int n_u, int64_t t_first, int64_t n_valid, int64_t batch,
                                      uint64_t seed, uint64_t draw, const DockauvReplaySample *out, void *stream);

/* Off-policy collection on the device: stable-baselines3 1.5.0's SAC Actor (SAC's MlpPolicy, default H = 256) picks
 * each step's actions, and the steps write straight into a replay ring.
 *   latent_pi = Linear(n_obs, H), ReLU, Linear(H, H), ReLU;  mu = Linear(H, n_u);  log_std = Linear(H, n_u) clamped to
 *   [-20, 2];  a = tanh(mu + exp(log_std) eps), or a = tanh(mu) with deterministic != 0 (predict(deterministic=True)).
 * eps is the noise of dockauv_rollout_policy: Philox4x32-10 at (global id lo, global id hi, episode,
 * 0xC0000000 | (t_steps mod 2^29) << 1 | j) with the env's counters before the step, so the actions depend on (seed,
 * global id, episode, t) only.  H is 64, 128 or 256.  The actor runs on the tensor cores with bf16 operands: the
 * observation, every weight matrix and each hidden activation after bias and ReLU are rounded to bf16 (round to nearest
 * even); products are accumulated in f32; biases, the clamp, exp, the noise and tanh are f32.  The SAC update recomputes
 * log-probabilities and Q-values from the stored (observation, action) pairs, so only the stored action, which is
 * exactly what the step read, has to be exact.  The bf16 weights must fit one CTA's shared memory (227 KB; n_obs 36,
 * H 256: 178 KB); DOCKAUV_EINVAL otherwise. */
typedef struct DockauvSquashedActor {   /* caller-owned f32 device tensors, nn.Linear layout */
    const float *w[2], *b[2];           /* latent_pi: n_obs->H, H->H, ReLU after each */
    const float *mu_w, *mu_b;           /* H->n_u */
    const float *log_std_w, *log_std_b; /* H->n_u, clamped to [-20, 2] */
    int32_t hidden, deterministic;
} DockauvSquashedActor;

/* n_steps steps of SB3's OffPolicyAlgorithm.collect_rollouts in one call, writing THROUGH `ring` (its pointers are
 * const only because dockauv_replay_sample reads them).  With S = n_slots (2..64) and s0 = start_slot (0..S-1), step t
 * (0 <= t < n_steps):
 *   the actor reads obs[(s0 + t) % S] and writes actions[(s0 + t) % S] (f32, unclipped and unscaled);
 *   the step reads those actions as float32 and writes obs[(s0 + t + 1) % S], and reward, done and terminal_obs of slot
 *   (s0 + t) % S;
 * so the ring ends up as n_steps dockauv_step calls with the same actions would leave it.  reward is real[S][N] in the
 * handle's precision.  The arguments that need no handle are checked first, then the bind state and the shared-memory
 * limit, then the alignment of the ring's observation arrays.  Taps are recorded as in dockauv_rollout.
 * Graphs (use_graph != 0): one CUDA graph per (actor pointers, hidden, deterministic, ring, S, s0, n_steps, auto_reset,
 * seed), four cached per handle; with n_steps a multiple of S every call replays the same graph.  Weights rewritten in
 * place (optimizer.step()) are read by the next replay.  The steps run inside this launch chain and use none of the step
 * graphs of dockauv_step. */
DOCKAUV_API int dockauv_replay_collect(DockauvHandle *h, const DockauvSquashedActor *actor, const DockauvReplayRing *ring,
                                       int n_slots, int start_slot, int n_steps, int auto_reset, int use_graph,
                                       void *stream);

/* Episode statistics accumulated on the device since the last clear (DOCKAUV_STAT_*).  stats_dev points at
 * double[DOCKAUV_N_STATS] on the device: it is the send buffer of the per-rollout NCCL all-reduce.  The kernels
 * accumulate into DOCKAUV_STAT_COPIES replicas of the vector (same-address atomics of 10^4 warps per step would
 * serialise in one L2 slice); dockauv_fold_stats adds the replicas into the vector stats_dev points at -- call it on
 * the stream before reading through the pointer.  dockauv_get_stats folds by itself. */
#define DOCKAUV_STAT_COPIES 32
DOCKAUV_API int dockauv_stats_ptr(DockauvHandle *h, double **stats_dev);
DOCKAUV_API int dockauv_fold_stats(DockauvHandle *h, void *stream);
DOCKAUV_API int dockauv_get_stats(DockauvHandle *h, double *stats_host, void *stream);
DOCKAUV_API int dockauv_clear_stats(DockauvHandle *h, void *stream);

/* Micro-benchmarks for the roofline denominators (SURVEY.md 7, K4): sustained FP64 / FP32 FMA rate in
 * TFLOP/s and device copy bandwidth in GB/s, measured with CUDA events on `device`. */
DOCKAUV_API int dockauv_measure_peaks(int device, double *fp64_tflops, double *fp32_tflops, double *copy_gbs);

/* Kernel-level accounting for bench.py: number of kernels launched by this handle so far, and CUDA-event
 * time (ms) of the most recent dockauv_step launch when timing is enabled. */
DOCKAUV_API int dockauv_launch_count(DockauvHandle *h, int64_t *n_launches);
/* Work-list lengths of the most recent step of the pipeline layout, summed over the stepped env ranges: envs that had an
 * obstacle in view (the ray launch's work) and envs whose episode ended (the episode-end launch's work).  Synchronises
 * `stream`; diagnostics for bench.py (the counters are re-used by the next step). */
DOCKAUV_API int dockauv_last_list_counts(DockauvHandle *h, int64_t *n_listed, int64_t *n_ended, void *stream);
/* how many times dockauv_rollout(use_graph) had to capture its launch sequence (a replay with the same pointers does not) */
DOCKAUV_API int dockauv_rollout_captures(DockauvHandle *h, int64_t *n_captures);
/* the same for dockauv_rollout_policy(use_graph) */
DOCKAUV_API int dockauv_rollout_policy_captures(DockauvHandle *h, int64_t *n_captures);
/* the same for dockauv_replay_collect(use_graph) */
DOCKAUV_API int dockauv_replay_collect_captures(DockauvHandle *h, int64_t *n_captures);
DOCKAUV_API int dockauv_enable_timing(DockauvHandle *h, int enabled);
DOCKAUV_API int dockauv_last_step_ms(DockauvHandle *h, float *ms);
/* Per-launch CUDA-event times (ms) of the most recent timed dockauv_step of a multi-launch layout, in launch order
 * (DOCKAUV_LAYOUT_PIPELINE: dynamics + cull + finish, rays + finish (only with obstacles), episode end); *n_launches = 0
 * for the single-launch layouts. */
DOCKAUV_API int dockauv_last_step_launch_ms(DockauvHandle *h, float *ms, int capacity, int *n_launches);

#ifdef __cplusplus
}
#endif
#endif /* DOCKAUV_H */
