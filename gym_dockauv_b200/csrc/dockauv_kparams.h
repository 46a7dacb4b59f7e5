// dockauv_kparams.h -- device-side parameter block (passed by value as a __grid_constant__ kernel argument, so
// every field sits in the constant bank and uniform reads broadcast to the whole warp); ~2.7 KB.
#pragma once
#include <stdint.h>

#include <vector_types.h>

#include "../../include/dockauv.h"

namespace dockauv {

template <typename T>
struct KParams {
    // sizes / switches
    int64_t n_envs;
    int64_t env_begin, env_end;   // half-open range of envs this launch works on (chunked host pipeline)
    int32_t n_u, n_caps, n_sph, n_synth_sph, scenario;
    int32_t max_timesteps, reward_set;
    int32_t n_rays, n_vert, n_horiz, block, n_hr, n_rr, n_obs;   // n_hr = pooled columns, n_rr = pooled rays
    int32_t action_factor_is_scalar, auto_reset, has_current, has_noise, act_f32;
    uint64_t seed, env_id0;
    // vehicle
    T m, r_G[3], I_b[9], MA[6], M_inv[36];
    T D_lin[10], D_quad[10], D_lift[10];
    T G_WB, G_r[3];
    T B[6 * DOCKAUV_MAX_U];
    T lauv_B[4];
    T u_lo[DOCKAUV_MAX_U], u_span[DOCKAUV_MAX_U];   // u_span = u_hi - u_lo
    T lp_alpha, h, safety_radius;
    // env
    T max_dist_from_goal, max_attitude, dist_goal_reached_tol;
    T u_max, v_max, w_max, p_max, q_max, r_max;
    // reciprocals of the observation / reward normalisers (docking3d.py:467-483, 520-558): one multiply instead of a
    // ~25-instruction IEEE division each; the quotient may differ from numpy's by one ulp (1.1e-16 relative)
    T inv_u_max, inv_v_max, inv_w_max, inv_p_max, inv_q_max, inv_r_max, inv_max_attitude;
    T log_den_obs;    // log(dist_goal_reached_tol / max_dist_from_goal), docking3d.py:465-466
    T log_den_rew;    // log(max(tol, 1e-3) / max_dist), docking3d.py:723
    T inv_max_dist_from_goal, inv_log_den_obs, inv_log_den_rew;   // their reciprocals (same one-ulp caveat as above)
    T w_d, w_delta_psi, w_delta_theta, w_phi, w_theta, w_Thetadot, w_oa;
    T w_done[5];
    T arf[DOCKAUV_MAX_U];
    float arf_f32[DOCKAUV_MAX_U];
    T cur_mu, cur_sigma;
    T radar_max_dist, sum_beta_oa;
    // ray pyramid in the body frame: every ray direction satisfies x > 0, |y| <= fov_ty x, |z| <= fov_tz x;
    // fov_ny = sqrt(1 + ty^2), fov_nz = sqrt(1 + tz^2) (norms of the side-plane normals)
    T fov_ty, fov_tz, fov_ny, fov_nz;
    // persistent state (SoA, env fastest)
    T *state, *u_prev, *goal, *heading_goal, *current, *capsules, *spheres, *ep_return;
    int32_t *t_steps, *episode;
    // inputs
    const void *actions;
    const T *noise;
    // outputs
    float *obs, *terminal_obs;
    T *reward, *ep_return_out;
    uint8_t *done, *cond_bits;
    int32_t *ep_len_out;
    // debug outputs
    T *dbg_ray_dist, *dbg_reward_arr, *dbg_euler_dot, *dbg_nu_c, *dbg_nav, *dbg_obs, *dbg_state_dot;
    // pipeline layout (library-owned buffers):
    //   rec      T[n_envs][16], the 16-word record of an env, computed in registers by the dynamics launch (AoS: one
    //            128-byte line in f64): 0..5 sin/cos of the post-step attitude (sphi cphi sth cth spsi cpsi), 6..8
    //            post-step position relative to the goal, 9 (r0+r1)+(r2+r3), 10 r4+r5, 11 r7 (reward terms that need no
    //            radar, already combined in numpy's summation order), 12 log_precision(delta_d), 13 delta_d, 14
    //            done-condition bits 0..2 as a number, 15 NaN poison word (0 for a finite pose).  It is stored only for
    //            the LISTED envs, in the form the ray launch reads: everything that launch needs besides the obstacle
    //            rows, with words 6..8 the post-step position itself and word 14 the running return before this step
    //            (REC_POS, REC_EPR)
    //   obsf     float4[n_obsf][n_envs]: float copy of the obstacles RELATIVE TO THE GOAL for the cull (written by every
    //            reset and by dockauv_refresh_obstacles): capsule k -> slots 2k (bot - goal, radius), 2k+1 (unit axis
    //            (top - bot) / L, L); sphere s -> slot 2 n_caps + s (centre - goal, radius)
    //   obsd     T[n_envs][n_caps + n_sph][8]: env-major bit copy of the obstacles as stored, one 8-word row each
    //            (capsule: bot, top, radius, 0; sphere: centre, radius, 0, 0, 0), written wherever obsf is; the pipeline
    //            layout reads its obstacles in T from here (a row is one 64-byte piece in f64 instead of 7 planes)
    //   view_list / ended_list / view_count: work lists, one counter block per concurrently stepped range (running
    //            counts and their values at the start and end of the step, dockauv_launch.h): envs with something in
    //            view (local env index | in-view mask << 32 | condition bits << 48) for the ray launch, envs whose
    //            episode ended (local env index) for the episode-end launch
    T *rec;
    float4 *obsf;
    T *obsd;
    int32_t n_obsf, cull_exact;      // cull_exact: coordinates too large for the float cull -> decide everything in T (the step's copy then has n_obsf = 0: no float record is staged)
    int32_t tpe_rays;                // the thread-per-env ray launch covers this radar (2x2 pooling, <= 64 pooled cells)
    unsigned long long *view_list;
    uint32_t *ended_list;
    unsigned int *view_count;
    int32_t sm_count;
    int32_t sparse_minv;             // M_inv has only the z_G pattern (diagonal + [0,4] [4,0] [1,3] [3,1]) filled in
    T *delta_d_out;
    // stats accumulator (double[DOCKAUV_N_STATS])
    double *stats;
    // ray table in global memory (handle-owned): rd_b[3][n_rays] then beta_oa[n_rays].  It is not part of this block:
    // the block travels with every launch, and 8 KB of ray table made it 11 KB
    const T *ray_tab;
    // scenario bank (dockauv_set_scenario_bank), caller-owned; bank_rows == nullptr: the built-in reset.  Last in the
    // block so that every field above keeps its offset in the constant bank
    const T *bank_rows;              // real[bank_n][bank_stride], 16-byte aligned rows
    const double *bank_cdf;          // nullable: running sum of the row weights (weighted draw)
    int32_t *bank_row_of_env;        // nullable: int32[2][n_envs], row of the running / of the last ended episode
    int64_t bank_n, bank_stride;
};

}  // namespace dockauv
