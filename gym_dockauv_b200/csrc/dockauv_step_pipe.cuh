// dockauv_step_pipe.cuh -- layout DOCKAUV_LAYOUT_PIPELINE (default): one batched step as specialised launches.
//
//   1. dynamics     dynamics_kernel: thread per env.  Current, command filter, RKF45, angle wrap, navigation errors,
//      + cull        obs[0:16], done conditions 0..2, the reward terms that need no radar -- a 16-word record per env
//      + finish      (post-step attitude sines / cosines, position relative to the goal, the reward terms already combined
//                   in numpy's summation order, delta_d, condition bits) that stays in REGISTERS for the second half of the
//                   thread: the walk over the env's obstacles in FLOAT (float4 records relative to the goal, written at
//                   reset, waiting in shared memory since the start of the thread; cull_pair_rec): body collision
//                   (re-decided in T when within 2 mm of the threshold) and the range / field-of-view culls.
//                   Envs with something in view (24 % on the C4 workload) are appended to a compact list and their record
//                   goes to KParams::rec.  Done flag, condition bits and counters are final here for EVERY env (coalesced
//                   stores); an env with nothing in view is finished completely -- all ray cells read max_dist, r_oa = 0:
//                   reward, running return, statistics -- and goes on a second list if its episode ended.
//                   (Obstacle-free scenarios: the same code with no obstacle to walk over finishes every env.  Coordinates
//                   too large for float records: the same walk decides everything in T from the obstacle rows.)
//   2. rays+finish  rays_thread_kernel: persistent grid.  The listed envs with one or two obstacles in view with LANES =
//                   ENVS (tiles of 128), the others by one warp each (lanes = rays, next entry in flight while the current
//                   one is cast; radar_env, dockauv_rays.cuh) on the first CTAs of the same launch; then the reward with its
//                   obstacle-avoidance term and the running return.
//   3. episode end  episode_end_kernel: the ENDED envs (~1 % of the batch, compacted by launches 1 and 2): terminal-
//                   observation row, zero row, re-initialisation (warp = reset role, lane = env).
//
// Each launch has its own register budget and occupancy, the ray code never idles on envs with nothing in view, and no
// env is touched by a launch that has nothing to do for it.  Results are identical to the other layouts (same device
// functions, same order of operations per env; the ray tiles rotate obstacle records into the body frame instead of rays
// into NED, which moves ray distances in their last bits); debug outputs are served by the single-launch kernel.
#pragma once
#include "dockauv_step_warp.cuh"

namespace dockauv {

#ifndef DOCKAUV_DYN_THREADS
#define DOCKAUV_DYN_THREADS 256     // CTA size of the dynamics launch (measured at 1M envs, fused form: 64 or 128 threads 252 us, 256 threads 239 us, 512 threads 266 us: the warps of a CTA run in step and share their instruction-cache lines, a 512-thread CTA drains the whole SM at once)
#endif
#ifndef DOCKAUV_MINB_A
#define DOCKAUV_MINB_A 2            // its min-CTAs hint: (256, 2) = 128 registers, 16 warps per SM
#endif
constexpr int kDynThreads = DOCKAUV_DYN_THREADS;
#ifndef DOCKAUV_MINB_TPE
#define DOCKAUV_MINB_TPE 4          // thread-per-env ray launch: (128, 4) = 128 registers
#endif
#ifndef DOCKAUV_TPE_CTAS_PER_SM
#define DOCKAUV_TPE_CTAS_PER_SM 8   // persistent grid of the thread-per-env ray launch (twice what is resident: finer balance)
#endif
#ifndef DOCKAUV_TPE_WARP_CTAS_PER_SM
#define DOCKAUV_TPE_WARP_CTAS_PER_SM 1   // CTAs per SM of that launch that run the warp-per-env loop over class 3
#endif
#ifndef DOCKAUV_MINB_RAYS
#define DOCKAUV_MINB_RAYS 6         // ray launch: (128, 6) = 80 registers, 24 warps per SM
#endif
#ifndef DOCKAUV_RAY_CTAS_PER_SM
#define DOCKAUV_RAY_CTAS_PER_SM DOCKAUV_MINB_RAYS   // persistent grid of the ray launch, in 4-warp CTAs per SM (= what is resident)
#endif

// ---- the per-env record written by the dynamics launch (KParams::rec).  A listed env's record goes to the ray launch
//      with the words the ray launch does not read -- position relative to the goal, condition bits (they travel in the
//      list entry) -- replaced by the post-step position and the running return: with the obstacle rows, that launch then
//      reads nothing else of the env (the step counter only for the ~1 % whose episode ended)
constexpr int kRecWords = 16;
constexpr int REC_TRIG = 0, REC_PREL = 6, REC_A = 9, REC_B = 10, REC_R7 = 11, REC_LPD = 12, REC_DD = 13, REC_COND = 14,
              REC_POISON = 15;
constexpr int REC_POS = REC_PREL, REC_EPR = REC_COND;

// 16-byte vector access to a record: double -> 8 x double2, float -> 4 x float4
template <typename T>
struct RecIO;
template <>
struct RecIO<double> {
    static constexpr int kVecWords = 2;
    static __device__ __forceinline__ void store(double *dst, const double w[kRecWords]) {
        double2 *d = reinterpret_cast<double2 *>(dst);
#pragma unroll
        for (int c = 0; c < 8; c++) d[c] = make_double2(w[2 * c], w[2 * c + 1]);
    }
    // words [2 * first_vec, 2 * (first_vec + n_vec))
    template <int FIRST, int COUNT>
    static __device__ __forceinline__ void load(const double *src, double *w) {
        const double2 *s = reinterpret_cast<const double2 *>(src);
#pragma unroll
        for (int c = 0; c < COUNT; c++) {
            const double2 v = s[FIRST + c];
            w[2 * c] = v.x;
            w[2 * c + 1] = v.y;
        }
    }
};
template <>
struct RecIO<float> {
    static constexpr int kVecWords = 4;
    static __device__ __forceinline__ void store(float *dst, const float w[kRecWords]) {
        float4 *d = reinterpret_cast<float4 *>(dst);
#pragma unroll
        for (int c = 0; c < 4; c++) d[c] = make_float4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
    }
    // same word ranges as the double version: FIRST / COUNT are in units of two words
    template <int FIRST, int COUNT>
    static __device__ __forceinline__ void load(const float *src, float *w) {
        const float2 *s = reinterpret_cast<const float2 *>(src);
#pragma unroll
        for (int c = 0; c < COUNT; c++) {
            const float2 v = s[FIRST + c];
            w[2 * c] = v.x;
            w[2 * c + 1] = v.y;
        }
    }
};

// Launch as a PROGRAMMATIC DEPENDENT of the previous launch in the stream: the grid is set up while that launch drains and
// its threads wait in grid_dependency_wait() until everything the previous launch wrote is visible (no launch before it
// triggers early, so the wait is for its completion; an early trigger at the top of the launch before -- dependents set up
// during its last wave -- measured no faster).  What it saves is part of the launch-to-launch gap: 22.5 -> 22.3 us per
// 65,536-env SimpleDocking3d step, 0.391 -> 0.390 ms per 1M-env C4 step.
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// one word global -> shared without a register in between (completion: cp_async_wait_all); dst = shared-window address
template <typename T>
__device__ __forceinline__ void cp_async_word(unsigned dst_shared, const T *src) {
    if (sizeof(T) == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst_shared), "l"(src) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst_shared), "l"(src) : "memory");
}
// 16 bytes global -> shared past L1 (both addresses 16-byte aligned)
__device__ __forceinline__ void cp_async_16(unsigned dst_shared, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_shared), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------------- finish helpers
// is_done (docking3d.py:597-631): the five condition bits once the collision flag is known; t_steps is the counter before
// its increment (:612 is evaluated pre-increment, so max_timesteps = 1000 ends an episode at step 1001)
template <typename T>
__device__ __forceinline__ uint32_t done_conditions(const KParams<T> &p, uint32_t cond012, int32_t t_steps, bool collision) {
    return cond012 | ((t_steps >= p.max_timesteps) ? 8u : 0u) | (collision ? 16u : 0u);
}

// reward_step (docking3d.py:560-595) from the record words of the dynamics launch and the radar term r_oa
// (Reward.obstacle_avoidance, :767-792).  np.sum's order for 13 terms: ((r0+r1)+(r2+r3)) + ((r4+r5)+(r6+r7)) + r8 .. r12.
template <typename T>
__device__ __forceinline__ T step_reward(const KParams<T> &p, T A, T B, T r7, T lp_d, T r_oa, uint32_t cond) {
    T r6;
    if (p.reward_set == 1) r6 = -p.w_oa * r_oa;
    else r6 = -p.w_oa * cont_goal_constraints<T>(Mth<T>::abs_(r_oa), T(1), lp_d);
    T reward = A + (B + (r6 + r7));
    if (cond != 0u) {      // ~1 % of the env-steps; the other terms are exact zeros
#pragma unroll
        for (int k = 0; k < 5; k++) reward += ((cond >> k) & 1u) ? p.w_done[k] : T(0);
    }
    return reward;
}

// ------------------------------------------------------------------------------------------------------- 1. dynamics
// CUR: the ocean current is evaluated (scenario with a current, injected current or noise); SPM: sparse M_inv / C / G.
// The cull + finish code (section 2) runs in this launch, on the record while it is still in registers (scenarios without
// obstacles too: every ray reads max_dist and nothing can collide, so every env is finished here).

// shared memory of one dynamics CTA: park[kParkWords][kDynThreads] words of T that are only needed after the integration
// (position, goal, running return, step counter), filled by cp.async into the thread's own slots -- no register during
// the integration and no memory round trip after it
constexpr int kParkWords = 8;

// one env of the dynamics launch: the env's record is left in w[kRecWords] and its post-step position in pos[3]; its
// running return, step counter (park rows 6, 7) and float obstacle records (s_obs, [slot][kDynThreads]) are copied into
// shared memory for the cull + finish code (the cp.async wait after the integration covers them)
template <typename T, int VEH, int NU, bool CUR, bool SPM>
__device__ __forceinline__ void dynamics_env(const KParams<T> &p, const int64_t i, T *dyn_park, const float4 *s_obs,
                                             T w[kRecWords], T pos[3]) {
    const int64_t N = p.n_envs;
    // ---- what the integration starts from goes first: plain loads; the asynchronous copies of everything that is needed
    //      later queue up behind them (issued ahead of the loads, the 21 copies of a thread delayed its first use of a loaded
    //      value: 10 % of the fused launch's stall samples sat on that one wait)
    T y[9];
#pragma unroll
    for (int c = 0; c < 9; c++) y[c] = p.state[(int64_t)(3 + c) * N + i];
    CommandIn<T, NU> cin;
    load_command<T, NU>(p, i, cin);
    {
        const unsigned sa = (unsigned)__cvta_generic_to_shared(dyn_park + threadIdx.x);
        constexpr unsigned kPlane = kDynThreads * (unsigned)sizeof(T);
#pragma unroll
        for (int c = 0; c < 3; c++) cp_async_word<T>(sa + c * kPlane, p.state + (int64_t)c * N + i);
#pragma unroll
        for (int c = 0; c < 3; c++) cp_async_word<T>(sa + (3 + c) * kPlane, p.goal + (int64_t)c * N + i);
        cp_async_word<T>(sa + 6 * kPlane, p.ep_return + i);
        cp_async_word<int32_t>(sa + 7 * kPlane, p.t_steps + i);
        const unsigned so = (unsigned)__cvta_generic_to_shared(s_obs);
        for (int sl = 0; sl < p.n_obsf; sl++) cp_async_16(so + (unsigned)(sl * kDynThreads * 16), p.obsf + (int64_t)sl * N + i);
    }
    T tr0[6];
    Mth<T>::sincos_(y[0], &tr0[0], &tr0[1]);
    Mth<T>::sincos_(y[1], &tr0[2], &tr0[3]);
    Mth<T>::sincos_(y[2], &tr0[4], &tr0[5]);
    T nu_c[3] = {T(0), T(0), T(0)};
    if (CUR) dyn_current<T>(p, i, tr0, nu_c);
    T tau[6], penalty;
    {
        T u[NU];
        penalty = command_and_penalty<T, NU>(p, cin, u);
#pragma unroll
        for (int k = 0; k < NU; k++) p.u_prev[(int64_t)k * N + i] = u[k];
        dyn_tau<T, VEH, NU>(p, u, tau);
    }
    T pacc[3], tr1[6];
    rkf45_step<T, VEH, SPM, CUR>(p, y, tr0, tau, nu_c, pacc, tr1);
#pragma unroll
    for (int c = 0; c < 3; c++) y[c] = ssa<T>(y[c]);
    // position and goal are only needed from here on: they have been waiting in shared memory
    T goal[3];
    cp_async_wait_all();
#pragma unroll
    for (int c = 0; c < 3; c++) pos[c] = dyn_park[c * kDynThreads + threadIdx.x];
#pragma unroll
    for (int c = 0; c < 3; c++) goal[c] = dyn_park[(3 + c) * kDynThreads + threadIdx.x];
#pragma unroll
    for (int c = 0; c < 3; c++) pos[c] += pacc[c];
#pragma unroll
    for (int c = 0; c < 3; c++) p.state[(int64_t)c * N + i] = pos[c];
#pragma unroll
    for (int c = 0; c < 9; c++) p.state[(int64_t)(3 + c) * N + i] = y[c];

    DynOut<T> q;
    dyn_outputs<T>(p, pos, y, tr1, goal, nu_c, penalty, q);
    // a later launch zeroes the row if the env is reset
    store_obs_head<T>(p, i, q.o);
    // np.sum of the 13 reward terms is ((r0+r1)+(r2+r3)) + ((r4+r5)+(r6+r7)) + r8 + .. + r12 (reward_sum13): the two
    // sums that need no radar are formed here, in that order
    const T A = (q.r[0] + q.r[1]) + (q.r[2] + q.r[3]), B = q.r[4] + q.r[5];
#pragma unroll
    for (int c = 0; c < 6; c++) w[REC_TRIG + c] = tr1[c];
#pragma unroll
    for (int c = 0; c < 3; c++) w[REC_PREL + c] = pos[c] - goal[c];
    w[REC_A] = A;
    w[REC_B] = B;
    w[REC_R7] = q.r[7];
    w[REC_LPD] = q.r[6];
    w[REC_DD] = q.delta_d;
    w[REC_COND] = (T)q.cond;
    // envs with a non-finite pose take the warp-per-env ray path
    w[REC_POISON] = pose_poison<T>(pos, y);
}

// ------------------------------------------------------------------------------------------------------- 2. cull + finish
// One env through the float culls and everything that can be finished without rays; called by EVERY thread of a dynamics
// CTA (the list appends are warp-collective; `active` = the thread has an env).
//   w        the env's record (dynamics_env)
//   pos      post-step position (only for pairs within 2 mm of the collision threshold, and the exact culls)
//   s_obs    the env's float obstacle records in shared memory, [slot][kDynThreads] (KParams::obsf layout)
//   park     the thread's first park slot (running return in row 6, step counter in row 7), read after the obstacle loop
// Returns whether the env is on a view list (its record must then be in KParams::rec for the ray launch, with REC_POS
// and REC_EPR filled in).
template <typename T>
__device__ __forceinline__ bool cull_finish_env(const KParams<T> &p, const int64_t i, const int64_t i0, const bool active,
                                                const T w[kRecWords], const T pos[3], const float4 *s_obs, const T *park) {
    const int lane = threadIdx.x & 31;
    WarpStats bs;
    bool listed = false, ended = false;      // ended: episode over and nothing in view -> on the list of the episode-end launch
    bool poison_free = true;
    uint32_t info = 0;                       // bits 0..15 in-view mask (capsules first), 16 collision
    uint32_t cond = 0;
    if (active) {
        const int n_caps = p.n_caps, n_sph = p.n_sph, n_obst = n_caps + n_sph;
        const T *trig = w + REC_TRIG;
        if (n_obst > 0 && !p.cull_exact) {
            // ---- float culls + collision pre-test (cull_pair_rec)
            float Rf[9], prel[3];
            rzyx<float>((float)trig[0], (float)trig[1], (float)trig[2], (float)trig[3], (float)trig[4], (float)trig[5], Rf);
#pragma unroll
            for (int c = 0; c < 3; c++) prel[c] = (float)w[REC_PREL + c];
            // the next obstacle's record is requested before the current one is evaluated
            float4 q0 = s_obs[0], q1 = n_caps > 0 ? s_obs[kDynThreads] : make_float4(0.f, 0.f, 0.f, 0.f);
            int slot = n_caps > 0 ? 2 : 1;
#pragma unroll 1
            for (int k = 0; k < n_obst; k++) {
                const bool is_cap = k < n_caps;
                const float4 c0 = q0, c1 = q1;
                if (k + 1 < n_obst) {
                    q0 = s_obs[slot * kDynThreads];
                    if (k + 1 < n_caps) q1 = s_obs[(slot + 1) * kDynThreads];
                    slot += (k + 1 < n_caps) ? 2 : 1;
                }
                int hit3;
                bool view;
                cull_pair_rec<T>(p, prel, Rf, c0, c1, is_cap, hit3, view);
                bool hit = hit3 == 1;
                if (hit3 == 2) {      // within 2 mm of the collision threshold (or NaN): decided in T like the other layouts
                    T ob[kObstRowWords];
                    load_obstacle_row<T>(obstacle_row<T>(p, i, k), ob);
                    hit = obstacle_body_hit<T>(p, pos, ob, is_cap);
                }
                info |= view ? (1u << k) : 0u;
                info |= hit ? (1u << 16) : 0u;
            }
        } else if (n_obst > 0) {
            // ---- coordinates too large for float records: everything in T (obstacle_pair)
            T Rm[9];
            rzyx<T>(trig[0], trig[1], trig[2], trig[3], trig[4], trig[5], Rm);
#pragma unroll 1
            for (int k = 0; k < n_obst; k++) {
                const bool is_cap = k < n_caps;
                T ob[kObstRowWords];
                load_obstacle_row<T>(obstacle_row<T>(p, i, k), ob);
                bool hit, view;
                obstacle_pair<T, false>(p, pos, Rm, ob, is_cap, nullptr, hit, view);
                info |= view ? (1u << k) : 0u;
                info |= hit ? (1u << 16) : 0u;
            }
        }
        const T ep_return = park[6 * kDynThreads];
        const int32_t t_steps = reinterpret_cast<const int32_t *>(park + 7 * kDynThreads)[0];
        // a non-finite pose goes through the warp-per-env ray path, which reproduces the reference's treatment of it
        // (radar_env; without obstacles every ray reads max_dist whatever the pose, docking3d.py:441)
        poison_free = w[REC_POISON] == T(0);
        listed = (info & 0xffffu) != 0u || (n_obst > 0 && !poison_free);
        // ---- everything that does not depend on the rays is final for EVERY env: done, condition bits, counters.
        //      Stores of all lanes of the warp -> full sectors (a listed env only lacks its obstacle-avoidance term: its
        //      reward word is provisional here and rewritten by the ray launch together with the running return)
        cond = done_conditions<T>(p, (uint32_t)w[REC_COND], t_steps, (info >> 16) != 0u);
        const bool done = cond != 0;
        const int32_t t_new = t_steps + 1;
        const T r_oa = p.sum_beta_oa / p.sum_beta_oa - T(1);      // docking3d.py:792 with every ray at max_dist: exactly 0
        const T reward = step_reward<T>(p, w[REC_A], w[REC_B], w[REC_R7], w[REC_LPD], r_oa, cond);
        p.reward[i] = reward;
        p.done[i] = done ? 1 : 0;
        if (p.cond_bits) p.cond_bits[i] = (uint8_t)cond;
        if (p.delta_d_out) p.delta_d_out[i] = w[REC_DD];
        if (done && p.ep_len_out) p.ep_len_out[i] = t_new;
        if (listed) {
            p.t_steps[i] = t_new;        // the ray launch reads it back (and zeroes it if it re-initialises the env)
        } else {
            // ---- nothing in view: pooled cells all ones, r_oa = 0
            store_clear_cells<T>(p, i);
            const T ep_ret = ep_return + reward;
            if (done) {
                if (p.ep_return_out) p.ep_return_out[i] = ep_ret;
                bs.done = true;
                bs.cond = cond;
                bs.length = t_new;
                bs.ep_return = (double)ep_ret;
                bs.delta_d = (double)w[REC_DD];
                bs.nan = reward != reward;      // episodes that ended on a NaN reward
                ended = true;
            }
            if (!(done && p.auto_reset)) {
                p.ep_return[i] = ep_ret;
                p.t_steps[i] = t_new;
            }
        }
    }
    // ---- warp-aggregated appends to the work lists
    {
        int cls = 0;
        if (listed) {
            const int pc = __popc(info & 0xffffu);
            cls = (p.tpe_rays && pc >= 1 && pc <= 2 && poison_free) ? pc : 3;
        }
        const unsigned long long entry = (unsigned long long)(uint32_t)(i - p.env_begin) | ((unsigned long long)(info & 0xffffu) << 32) |
                                         ((unsigned long long)cond << 48);
        // the four appends of a warp (three view classes, ended list) reserve their slots with ONE atomic instruction: lane c
        // adds the warp's count to counter c, so the four round trips overlap (as four dependent atomics they were 15 % of
        // this launch's stall samples); the list's start, loaded beside the atomic, turns the ticket into a slot
        const unsigned m1 = __ballot_sync(0xffffffffu, cls == 1), m2 = __ballot_sync(0xffffffffu, cls == 2);
        const unsigned m3 = __ballot_sync(0xffffffffu, cls == 3), m4 = __ballot_sync(0xffffffffu, ended);
        const unsigned mine = lane == 0 ? m1 : (lane == 1 ? m2 : (lane == 2 ? m3 : (lane == 3 ? m4 : 0u)));
        unsigned base = 0;
        if (mine) {
            const unsigned first = p.view_count[kCounterNextStart + lane];
            base = atomicAdd(&p.view_count[lane], (unsigned)__popc(mine)) - first;
        }
        const unsigned b1 = __shfl_sync(0xffffffffu, base, 0), b2 = __shfl_sync(0xffffffffu, base, 1);
        const unsigned b3 = __shfl_sync(0xffffffffu, base, 2), b4 = __shfl_sync(0xffffffffu, base, 3);
        const unsigned below = (1u << lane) - 1u;
        if (cls == 1) p.view_list[b1 + __popc(m1 & below)] = entry;
        else if (cls == 2) p.view_list[p.n_envs + b2 + __popc(m2 & below)] = entry;
        else if (cls == 3) p.view_list[2 * p.n_envs + b3 + __popc(m3 & below)] = entry;
        if (ended) p.ended_list[b4 + __popc(m4 & below)] = (uint32_t)(i - p.env_begin);
    }
    bs.flush_direct(p.stats, threadIdx.x == 0 ? (int)min((int64_t)kDynThreads, p.env_end - i0) : 0);
    return listed;
}

// ---- the dynamics launch with the cull + finish code in it
// The env's running return, step counter and float obstacle records travel global -> shared by cp.async at the very start
// (records: [slot][thread], dynamic shared memory: 16 n_obsf bytes per thread) and wait there through the integration;
// the record never leaves the registers unless the env ends up on a view list.  Against a cull launch of its own this
// saves the record's round trip through HBM (128 B written for every env, 128 B read back) and every memory wait of the
// obstacle loop.
template <typename T, int VEH, int NU, bool CUR, bool SPM>
__global__ void __launch_bounds__(kDynThreads, DOCKAUV_MINB_A) dynamics_kernel(const __grid_constant__ KParams<T> p) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];      // float4 [n_obsf][kDynThreads]
    __shared__ __align__(8) T dyn_park[kParkWords * kDynThreads];
    const int64_t i0 = p.env_begin + (int64_t)blockIdx.x * kDynThreads;
    const int64_t i = i0 + threadIdx.x;
    const bool active = i < p.env_end;
    prefetch_dynamics_inputs<T, NU>(p, i, threadIdx.x & 31, true);
    T w[kRecWords], pos[3];
    // the lists of this step start where the previous step's ended (nobody reads the start words in this launch)
    if (blockIdx.x == 0 && threadIdx.x < kListCounters)
        p.view_count[kCounterStart + threadIdx.x] = p.view_count[kCounterNextStart + threadIdx.x];
    const float4 *s_obs = reinterpret_cast<const float4 *>(dyn_smem) + threadIdx.x;
    if (active) dynamics_env<T, VEH, NU, CUR, SPM>(p, i, dyn_park, s_obs, w, pos);
    const bool listed = cull_finish_env<T>(p, i, i0, active, w, pos, s_obs, dyn_park + threadIdx.x);
    if (listed) {      // the ray launch reads it
#pragma unroll
        for (int c = 0; c < 3; c++) w[REC_POS + c] = pos[c];
        w[REC_EPR] = dyn_park[6 * kDynThreads + threadIdx.x];
        RecIO<T>::store(p.rec + i * kRecWords, w);
    }
}

// ------------------------------------------------------------------------------------------------------- 3. rays + finish
// one append to the ended list by the ray launch (~1 % of the listed envs): the list's start is loaded beside the atomic,
// so the two round trips overlap (loaded once per thread, it stayed live through the ray loops: up to 3 more registers)
template <typename T>
__device__ __forceinline__ unsigned ended_slot(const KParams<T> &p) {
    const unsigned first = p.view_count[kCounterNextStart + 3];
    return atomicAdd(&p.view_count[3], 1u) - first;
}

// Shared memory of one warp of the ray launch (T words):
//   stage[2][kStageWords]   the data of two list entries (double buffer, filled by cp.async one entry ahead):
//                           0..15 the env's record (ray launch form), 16 + 8 k .. obstacle row k, k < 16
//   pre[16][kPreStride]     ray-test records of the in-view obstacles
//   ray[ray_stride]         clamped ray distances (pooling scratch)
//   lane[RayLaneShared]     per-lane ray constants
// Nothing of the software pipeline lives in registers (round 1 kept the next entry's 24 words there), and neither do the
// per-lane ray constants: 118 -> 80 registers, six CTAs of four warps per SM instead of four.  A warp's area is a whole
// number of 16-byte pieces (the stage is filled in 16-byte copies).
constexpr int kStageObst = kRecWords, kStageWords = kStageObst + 16 * kObstRowWords;
template <typename T, int RPL>
struct RaysSmem {
    int warp_words, ray_stride, pre_off, ray_off, lane_off;
    __host__ __device__ RaysSmem(int n_rays) {
        constexpr int kPiece = 16 / (int)sizeof(T);
        ray_stride = (n_rays + 2) & ~1;
        pre_off = 2 * kStageWords;
        ray_off = pre_off + 16 * kPreStride;
        lane_off = ray_off + ray_stride;
        warp_words = (lane_off + RayLaneShared<T, RPL>::words() + kPiece - 1) & ~(kPiece - 1);
    }
};

#ifndef DOCKAUV_RAY_WARPS
#define DOCKAUV_RAY_WARPS 4
#endif
constexpr int kRayWarps = DOCKAUV_RAY_WARPS;     // warps per CTA of the ray launch

// what the cull code left open for a listed env: the reward with its obstacle-avoidance term (oa_dot: the env's weighted
// sum, docking3d.py:767-792) and the running return, stored when `store`.  Returns the reward, the new return in ep_ret.
template <typename T>
__device__ __forceinline__ T finish_listed(const KParams<T> &p, int64_t ie, uint32_t cond, T oa_dot, T A, T B, T r7, T lp_d,
                                           T ep_before, bool store, T &ep_ret) {
    const T r_oa = p.sum_beta_oa / oa_dot - T(1);      // docking3d.py:792 (IEEE division: the other layouts' bits)
    const T reward = step_reward<T>(p, A, B, r7, lp_d, r_oa, cond);
    ep_ret = ep_before + reward;
    if (store) {
        const bool done = cond != 0;
        p.reward[ie] = reward;
        if (done && p.ep_return_out) p.ep_return_out[ie] = ep_ret;
        if (!(done && p.auto_reset)) p.ep_return[ie] = ep_ret;
    }
    return reward;
}

// the loop of ONE warp over the class-3 list: warp w_global of n_warps (called by all 32 lanes; smem_raw = the CTA's
// dynamic shared memory, kRayWarps * RaysSmem::warp_words words)
template <typename T, int RPL>
__device__ __forceinline__ void rays_warp_loop(const KParams<T> &p, unsigned char *smem_raw, unsigned w_global, unsigned n_warps) {
    const RaysSmem<T, RPL> L(p.n_rays);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T *s_warp = reinterpret_cast<T *>(smem_raw) + warp * L.warp_words;
    T *s_pre = s_warp + L.pre_off;
    T *s_ray = s_warp + L.ray_off;
    const unsigned count = p.view_count[2] - p.view_count[kCounterStart + 2];
    const unsigned long long *list = p.view_list + 2 * p.n_envs;
    unsigned idx = w_global;
    if (idx >= count) return;

    const int n_caps = p.n_caps, n_sph = p.n_sph, n_obst = n_caps + n_sph;
    RayLaneShared<T, RPL> rl;
    rl.init(p, lane, s_ray, s_warp + L.lane_off);

    // software pipeline over the list: the data of entry n + 1 is on its way into the other stage buffer while entry n is
    // cast.  What a lane fetches, in 16-byte pieces: lane c < kRecPieces piece c of the record, lane k < n_obst with bit k
    // of the mask the row of obstacle k.
    const bool lane_is_cap = lane < n_caps;
    constexpr int kPieceWords = 16 / (int)sizeof(T);
    constexpr int kRecPieces = kRecWords / kPieceWords, kRowPieces = kObstRowWords / kPieceWords;
    // shared-window addresses of this lane's slots in stage buffer 0 (buffer 1: + kStageWords words)
    const unsigned sa_rec = (unsigned)__cvta_generic_to_shared(s_warp + kPieceWords * (lane % kRecPieces));
    const unsigned sa_obst = (unsigned)__cvta_generic_to_shared(s_warp + kStageObst + kObstRowWords * (lane & 15));
    auto fetch = [&](uint64_t entry, int b) {
        const int64_t e = p.env_begin + (int64_t)(uint32_t)entry;
        const unsigned mask = (unsigned)(entry >> 32) & 0xffffu;
        const unsigned boff = b ? (unsigned)(kStageWords * sizeof(T)) : 0u;
        if (lane < kRecPieces) cp_async_16(sa_rec + boff, p.rec + e * kRecWords + kPieceWords * lane);
        if (lane < n_obst && ((mask >> lane) & 1u)) {
            const T *g = obstacle_row<T>(p, e, lane);
#pragma unroll
            for (int c = 0; c < kRowPieces; c++) cp_async_16(sa_obst + boff + 16u * c, g + kPieceWords * c);
        }
    };
    uint64_t cur = list[idx];
    uint64_t nxt = (idx + n_warps < count) ? list[idx + n_warps] : 0;
    fetch(cur, 0);
    double stat_acc = 0.0;       // lane k < DOCKAUV_STAT_ENV_STEPS accumulates statistic k of the episodes this warp ended
    int buf = 0;

    for (; idx < count; idx += n_warps, buf ^= 1) {
        const int64_t ie = p.env_begin + (int64_t)(uint32_t)cur;
        const unsigned mask = (unsigned)(cur >> 32) & 0xffffu;
        const uint32_t cond = (uint32_t)(cur >> 48) & 31u;
        const T *s_ent = s_warp + buf * kStageWords;
        // ---- the staged data of this entry is complete; start the next fetch into the other buffer (last read one
        //      iteration ago, before that iteration's closing __syncwarp)
        cp_async_wait_all();
        __syncwarp();
        const uint64_t nn = (idx + 2 * n_warps < count) ? list[idx + 2 * n_warps] : 0;
        if (idx + n_warps < count) fetch(nxt, buf ^ 1);
        const T pos[3] = {s_ent[REC_POS], s_ent[REC_POS + 1], s_ent[REC_POS + 2]};
        if (lane < n_obst && ((mask >> lane) & 1u))
            obstacle_ray_record<T>(pos, s_ent + kStageObst + kObstRowWords * lane, lane_is_cap, s_pre + lane * kPreStride);
        T R[9];
        rzyx<T>(s_ent[0], s_ent[1], s_ent[2], s_ent[3], s_ent[4], s_ent[5], R);
        const T poison = s_ent[REC_POISON];
        __syncwarp();

        // ---- cast rays against the in-view obstacles, pooled cells to the observation row
        const T oa_dot = radar_env<T, RPL, false, RayLaneShared<T, RPL>>(p, rl, R, poison, mask, s_pre, s_ray, lane, ie);

        // ---- reward and running return (every lane computes the same values from the staged record, lane 0 stores)
        T ep_ret;
        const T reward = finish_listed<T>(p, ie, cond, oa_dot, s_ent[REC_A], s_ent[REC_B], s_ent[REC_R7], s_ent[REC_LPD],
                                          s_ent[REC_EPR], lane == 0, ep_ret);
        const bool done = cond != 0;
        if (done) {       // warp-uniform, ~1 % of the listed envs
            double mine = 0.0;
            if (lane == DOCKAUV_STAT_EPISODES) mine = 1.0;
            else if (lane == DOCKAUV_STAT_SUM_RETURN) mine = (double)ep_ret;
            else if (lane == DOCKAUV_STAT_SUM_LENGTH) mine = (double)p.t_steps[ie];     // already incremented by the cull code
            else if (lane >= DOCKAUV_STAT_COND0 && lane < DOCKAUV_STAT_COND0 + 5) mine = ((cond >> (lane - DOCKAUV_STAT_COND0)) & 1u) ? 1.0 : 0.0;
            else if (lane == DOCKAUV_STAT_SUM_FINAL_DELTA_D) mine = (double)s_ent[REC_DD];
            else if (lane == DOCKAUV_STAT_NAN_ENVS) mine = (reward != reward) ? 1.0 : 0.0;
            stat_acc += mine;
            if (lane == 0) p.ended_list[ended_slot(p)] = (uint32_t)cur;
        }
        __syncwarp();
        cur = nxt;
        nxt = nn;
    }
    if (lane < DOCKAUV_STAT_ENV_STEPS && stat_acc != 0.0)
        atomicAdd(&p.stats[(blockIdx.x & (DOCKAUV_STAT_COPIES - 1)) * DOCKAUV_N_STATS + lane], stat_acc);
}

// the warp-per-env ray launch on its own (radars the thread mapping does not cover: every listed env is class 3)
template <typename T, int RPL>
__global__ void __launch_bounds__(kRayWarps * 32, DOCKAUV_MINB_RAYS * 4 / kRayWarps) rays_finish_kernel(const __grid_constant__ KParams<T> p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    rays_warp_loop<T, RPL>(p, smem_raw, blockIdx.x * kRayWarps + (threadIdx.x >> 5), gridDim.x * kRayWarps);
}

// ------------------------------------------------------------------------------------------------------- 3b. rays, thread per env
// The envs with exactly one or two obstacles in view -- nine in ten of the listed ones -- with LANES = ENVS: every lane
// walks over the rays of its own env, the ray-test records of its obstacles stay in registers.  Against the
// warp-per-env mapping, everything that is per-env scalar work there (list entry, record fetch, Rzyx, obstacle records,
// reward: ~450 of its ~600 warp instructions per env, done by 32 lanes redundantly) is amortised over the envs of a
// warp here.  The ray tests are straight-line code (cast_capsule_bf; spheres take the same path as degenerate capsules,
// so lanes never diverge on the obstacle type) and the four rays of a pooled cell are independent chains the compiler
// interleaves.  The body-frame ray table is walked in pooled-cell order (shared memory), so a cell's maximum is
// complete after four rays and goes straight into the observation row.  One persistent launch covers both classes:
// tiles of class 2 (the longer ones) first, then class 1.
constexpr int kTpeThreads = kRayWarps * 32;      // one CTA shape for both ray mappings of the launch
constexpr int kTpeMaxCells = 64;      // pooled cells the shared ray table holds
constexpr int kTpeTabWords = kTpeMaxCells * 4 * 4;

template <typename T, int NOB>
__device__ __forceinline__ void rays_thread_tile(const KParams<T> &p, const T *s_tab, unsigned tile, unsigned count) {
    const int64_t N = p.n_envs;
    const int n_rr = p.n_rr;
    const unsigned eidx = tile * kTpeThreads + threadIdx.x;
    const bool valid = eidx < count;
    const unsigned long long entry = valid ? p.view_list[(int64_t)(NOB - 1) * N + eidx] : 0ull;
    const int64_t ie = p.env_begin + (int64_t)(uint32_t)entry;
    unsigned mask = (unsigned)(entry >> 32) & 0xffffu;
    const uint32_t cond = (uint32_t)(entry >> 48) & 31u;
    const T *rec = p.rec + ie * kRecWords;
    // ---- pose and the ray-test records of the in-view obstacles (registers)
    T R[9], w[NOB][11];
    bool sph[NOB];
    {
        T w8[8];      // sin / cos of the attitude, position x, y
        RecIO<T>::template load<0, 4>(rec, w8);
        const T pos[3] = {w8[REC_POS], w8[REC_POS + 1], rec[REC_POS + 2]};
        rzyx<T>(w8[0], w8[1], w8[2], w8[3], w8[4], w8[5], R);
#pragma unroll
        for (int o = 0; o < NOB; o++) {
            const int k = mask ? __ffs(mask) - 1 : 0;
            mask &= mask - 1;
            const bool is_cap = k < p.n_caps;
            sph[o] = !is_cap;
            T ob[kObstRowWords];
            load_obstacle_row<T>(obstacle_row<T>(p, ie, k), ob);
#pragma unroll
            for (int c = 0; c < 11; c++) w[o][c] = T(0);
            obstacle_ray_record<T>(pos, ob, is_cap, w[o]);
            if (!is_cap) sphere_as_capsule<T>(w[o]);
            // the record's two vectors into the BODY frame (R^T v): a ray direction then is its table entry as it stands,
            // (R b) . v = b . (R^T v) -- 18 products per obstacle instead of 9 per ray
#pragma unroll
            for (int v = 0; v < 2; v++) {
                const T x = w[o][3 * v], y = w[o][3 * v + 1], z = w[o][3 * v + 2];
#pragma unroll
                for (int c = 0; c < 3; c++) w[o][3 * v + c] = R[c] * x + R[3 + c] * y + R[6 + c] * z;
            }
        }
    }
    T h_min[NOB];      // see cast_capsule_bf
#pragma unroll
    for (int o = 0; o < NOB; o++) h_min[o] = sph[o] ? -Mth<T>::min_normal() : T(0);
    const T dmax = p.radar_max_dist, inv_dmax = T(1) / dmax;
    float *orow = p.obs + ie * p.n_obs + 16;
    const bool vec_row = (p.n_obs & 3) == 0 && (n_rr & 3) == 0;      // the row is written in 16-byte pieces
    T oa_dot = T(0);
    float o4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    // (every lane runs all trips, valid or not: cast_capsule_bf contains a warp vote)
#pragma unroll 1
    for (int cell = 0; cell < n_rr; cell++) {
        T dq[4], bwq[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const T *tb = s_tab + 4 * (4 * cell + q);
            const T rd[3] = {tb[0], tb[1], tb[2]};
            bwq[q] = tb[3];
            T best = Mth<T>::inf();
#pragma unroll
            for (int o = 0; o < NOB; o++) {
                const T ba[3] = {w[o][0], w[o][1], w[o][2]}, oa[3] = {w[o][3], w[o][4], w[o][5]};
                best = cast_capsule_bf<T>(rd, ba, oa, w[o][6], w[o][7], w[o][8], w[o][9], w[o][10], h_min[o], best);
            }
            dq[q] = best > dmax ? dmax : best;        // clamp (sensor.py:117)
        }
        T mx = T(0);                                  // block_reduce pads with cval = 0 (sensor.py:131-137)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            if (bwq[q] < T(0)) continue;              // padding slot of the ray table: no ray
            // obstacle-avoidance sum (docking3d.py:767-792), 2x2 max-pool
            const T x = dq[q] * inv_dmax;
            const T qq = x * x;
            const T mq = !(qq <= T(0.001)) ? qq : T(0.001);     // np.maximum, NaN propagates
            oa_dot += mq * bwq[q];
            mx = !(dq[q] <= mx) ? dq[q] : mx;         // np.max, NaN propagates
        }
        T o = mx * inv_dmax;                          // clip(d / max_dist, 0, 1), docking3d.py:487
        o = o > T(1) ? T(1) : o;
        if (vec_row) {
            o4[cell & 3] = (float)o;
            if ((cell & 3) == 3 && valid) reinterpret_cast<float4 *>(orow)[cell >> 2] = make_float4(o4[0], o4[1], o4[2], o4[3]);
        } else if (valid) {
            orow[cell] = (float)o;
        }
    }
    if (valid) {
        T wf[8];
        RecIO<T>::template load<4, 4>(rec, wf);       // position z, A, B, r7, lp_d, delta_d, running return, poison
        T ep_ret;
        const T reward = finish_listed<T>(p, ie, cond, oa_dot, wf[1], wf[2], wf[3], wf[4], wf[6], true, ep_ret);
        if (cond != 0) {      // ~1 % of the listed envs
            WarpStats bs;
            bs.done = true;
            bs.cond = cond;
            bs.length = p.t_steps[ie];                // already incremented by the cull code
            bs.ep_return = (double)ep_ret;
            bs.delta_d = (double)wf[5];
            bs.nan = reward != reward;
            bs.flush_direct(p.stats, 0);
            p.ended_list[ended_slot(p)] = (uint32_t)entry;
        }
    }
}

// One launch for all three classes: the first `warp_ctas` CTAs run the warp-per-env loop over class 3 (few entries, each a
// long latency chain: started first, they run alongside the tiles instead of as a launch of their own that leaves the GPU
// 60 % idle for 11 us), the others are the persistent tile loop of classes 2 and 1.
template <typename T, int RPL>
__global__ void __launch_bounds__(kTpeThreads, DOCKAUV_MINB_TPE) rays_thread_kernel(const __grid_constant__ KParams<T> p, unsigned warp_ctas) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ __align__(16) T s_tab[kTpeTabWords];      // slot = 4 * cell + q: rb[3], bw; bw < 0 marks zero padding
    static_assert(kTpeThreads == kRayWarps * 32, "the two ray mappings share one CTA shape");
    grid_dependency_wait();
    if (blockIdx.x < warp_ctas) {
        rays_warp_loop<T, RPL>(p, smem_raw, blockIdx.x * kRayWarps + (threadIdx.x >> 5), warp_ctas * kRayWarps);
        return;
    }
    const unsigned bid = blockIdx.x - warp_ctas, n_ctas = gridDim.x - warp_ctas;
    const unsigned c1 = p.view_count[0] - p.view_count[kCounterStart], c2 = p.view_count[1] - p.view_count[kCounterStart + 1];
    const unsigned t2 = (c2 + kTpeThreads - 1) / kTpeThreads, t1 = (c1 + kTpeThreads - 1) / kTpeThreads;
    if (bid >= t1 + t2) return;
    const int n_rr = p.n_rr, n_r = p.n_rays;
    for (int t = threadIdx.x; t < 4 * n_rr; t += kTpeThreads) {
        const int cell = t >> 2, q = t & 3;
        const int pr = cell / p.n_hr, pcol = cell - pr * p.n_hr;
        const int rv = 2 * pr + (q >> 1), rh = 2 * pcol + (q & 1);
        const bool ok = rv < p.n_vert && rh < p.n_horiz;
        const int ir = ok ? rv * p.n_horiz + rh : 0;
#pragma unroll
        for (int c = 0; c < 3; c++) s_tab[4 * t + c] = ok ? p.ray_tab[c * n_r + ir] : T(0);
        s_tab[4 * t + 3] = ok ? p.ray_tab[3 * n_r + ir] : T(-1);
    }
    __syncthreads();
    for (unsigned tile = bid; tile < t1 + t2; tile += n_ctas) {
        if (tile < t2) rays_thread_tile<T, 2>(p, s_tab, tile, c2);
        else rays_thread_tile<T, 1>(p, s_tab, tile - t2, c1);
    }
}

// ------------------------------------------------------------------------------------------------------- 4. episode end
// The ENDED envs of the step (compact list, ~1 % of the batch): the last observation is kept as terminal_observation, the
// all-zero reset observation is handed back (docking3d.py:269,322) and the env is re-initialised.  One CTA of eight warps
// per 32 list entries: lane = env, warp = reset role (reset_envs_cta) and 16-byte piece of the observation row.
// Measured alternatives (1M-env step): one WARP per ended env (round 1, and the first version of this pipeline, inside the
// ray launch): ~4000 warp instructions per reset at 1..8 active lanes, 28 M per half batch, a third of the ray launch; one
// THREAD per ended env: 40x leaner but a 5500-instruction dependent chain, 70 us for a launch that occupies 5 % of the GPU;
// eight LANES per env: the roles serialise inside the warp, same 70 us.
//   BANK: finished envs are re-initialised from the scenario bank (KParams::bank_rows)
template <typename T, bool BANK>
__global__ void __launch_bounds__(kResetCta) episode_end_kernel(const __grid_constant__ KParams<T> p) {
    grid_dependency_wait();
    const unsigned n_ended = p.view_count[3] - p.view_count[kCounterStart + 3];
    const int n_obs = p.n_obs;
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    // every thread of a CTA runs the same number of trips (reset_envs_cta has a barrier)
    const unsigned trips = (n_ended + gridDim.x * 32 - 1) / (gridDim.x * 32);
    unsigned k = blockIdx.x * 32 + lane;
    for (unsigned trip = 0; trip < trips; trip++, k += gridDim.x * 32) {
        const bool valid = k < n_ended;
        int64_t ie = 0;
        if (valid) {
            ie = p.env_begin + (int64_t)p.ended_list[k];
            float *row = p.obs + ie * n_obs;
            float *trow = p.terminal_obs ? p.terminal_obs + ie * n_obs : nullptr;
            if ((n_obs & 3) == 0) {
                float4 *r4 = reinterpret_cast<float4 *>(row), *t4 = reinterpret_cast<float4 *>(trow);
                for (int c = role; c < (n_obs >> 2); c += kResetRoles) {
                    if (trow) t4[c] = r4[c];
                    if (p.auto_reset) r4[c] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                }
            } else {
                for (int c = role; c < n_obs; c += kResetRoles) {
                    if (trow) trow[c] = row[c];
                    if (p.auto_reset) row[c] = 0.0f;
                }
            }
        }
        if (p.auto_reset) reset_envs_cta<T, BANK>(p, ie, valid);
    }
    // every append of this step has completed (the wait above): the next step's lists start here (no CTA of this launch
    // reads these words)
    if (blockIdx.x == 0 && threadIdx.x < kListCounters)
        p.view_count[kCounterNextStart + threadIdx.x] = p.view_count[threadIdx.x];
}

// ------------------------------------------------------------------------------------------------------- launcher
template <typename... KArgs, typename... Args>
static cudaError_t launch_dependent(void (*kern)(KArgs...), unsigned blocks, unsigned threads, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

template <typename T, int VEH, int NU>
static cudaError_t launch_dynamics(const KParams<T> &k, unsigned blocks, cudaStream_t st) {
    const bool cur = k.has_current != 0, spm = k.sparse_minv != 0;
    const int smem = k.n_obsf * kDynThreads * 16;
    auto go = [&](auto kern) {
        const cudaError_t e = allow_dyn_smem(kern, smem, kParkWords * kDynThreads * (int)sizeof(T));
        if (e != cudaSuccess) return e;
        kern<<<blocks, kDynThreads, smem, st>>>(k);
        return cudaGetLastError();
    };
    if (cur && spm) return go(dynamics_kernel<T, VEH, NU, true, true>);
    if (cur) return go(dynamics_kernel<T, VEH, NU, true, false>);
    if (spm) return go(dynamics_kernel<T, VEH, NU, false, true>);
    return go(dynamics_kernel<T, VEH, NU, false, false>);
}

// the ray launch over the n envs of kc's range, RPL rays per lane
template <typename T, int RPL>
static cudaError_t launch_rays(const KParams<T> &kc, int64_t n, cudaStream_t st) {
    const int smem = kRayWarps * RaysSmem<T, RPL>(kc.n_rays).warp_words * (int)sizeof(T);
    const int64_t sms = kc.sm_count > 0 ? kc.sm_count : 148;
    cudaError_t e;
    if (kc.tpe_rays) {
        // ---- one launch; thread per env for the envs with one or two obstacles in view (persistent grid over tiles of
        //      128 lanes; the counts are only known on the device), warp per env for the rest on its first CTAs
        int64_t tb = (n + kTpeThreads - 1) / kTpeThreads;      // tiles if every env were listed
        if (tb > sms * DOCKAUV_TPE_CTAS_PER_SM) tb = sms * DOCKAUV_TPE_CTAS_PER_SM;
        int64_t wb = (n + kRayWarps - 1) / kRayWarps;
        if (wb > sms * DOCKAUV_TPE_WARP_CTAS_PER_SM) wb = sms * DOCKAUV_TPE_WARP_CTAS_PER_SM;
        auto kern = rays_thread_kernel<T, RPL>;
        if ((e = allow_dyn_smem(kern, smem, kTpeTabWords * (int)sizeof(T))) != cudaSuccess) return e;
        return launch_dependent(kern, (unsigned)(wb + tb), kTpeThreads, smem, st, kc, (unsigned)wb);
    }
    // ---- warp per env for every listed env (persistent grid)
    int64_t blocks = sms * (DOCKAUV_RAY_CTAS_PER_SM * 4 / kRayWarps);
    const int64_t most = (n + kRayWarps - 1) / kRayWarps;
    if (blocks > most) blocks = most;
    auto kern = rays_finish_kernel<T, RPL>;
    if ((e = allow_dyn_smem(kern, smem, 0)) != cudaSuccess) return e;
    kern<<<(unsigned)blocks, kRayWarps * 32, smem, st>>>(kc);
    return cudaGetLastError();
}

template <typename T, int VEH, int NU>
static cudaError_t launch_step_pipe(const KParams<T> &k, cudaStream_t st, int *n_launches, cudaEvent_t *marks, int *n_marks) {
    if (wants_debug(k) || k.rec == nullptr) {       // debug outputs: fused kernel
        *n_launches = 1;
        return launch_step_warp<T, VEH, NU>(k, st);
    }
    const int64_t n = k.env_end - k.env_begin;
    KParams<T> kc = k;
    kc.view_count = k.view_count + counter_block(k.env_begin);
    kc.view_list = k.view_list + k.env_begin;
    kc.ended_list = k.ended_list + k.env_begin;
    int n_mark = 0;      // one mark before the first launch and one after each
    auto mark = [&]() {
        if (marks) cudaEventRecord(marks[n_mark], st);
        n_mark++;
    };
    mark();
    if (k.cull_exact) kc.n_obsf = 0;      // the exact culls read no float record: the dynamics launch stages none
    cudaError_t e = launch_dynamics<T, VEH, NU>(kc, (unsigned)((n + kDynThreads - 1) / kDynThreads), st);
    if (e != cudaSuccess) return e;
    mark();
    if (pipe_has_obstacles(k)) {
        // rays per lane: 2 covers the stock 63-ray and the 64-ray radar; 8 covers everything up to DOCKAUV_MAX_RAYS
        e = k.n_rays <= 64 ? launch_rays<T, 2>(kc, n, st) : launch_rays<T, 8>(kc, n, st);
        if (e != cudaSuccess) return e;
        mark();
    }
    {
        // the list length is only known on the device: a grid for ~3 % of the range (32 entries per CTA), grid-stride beyond
        int64_t blocks = n / 1024 + 1;
        const int64_t cap = (int64_t)(k.sm_count > 0 ? k.sm_count : 148) * 4;
        if (blocks > cap) blocks = cap;
        auto kern = k.bank_rows != nullptr ? episode_end_kernel<T, true> : episode_end_kernel<T, false>;
        if ((e = launch_dependent(kern, (unsigned)blocks, kResetCta, 0, st, kc)) != cudaSuccess) return e;
        mark();
    }
    *n_launches = n_mark - 1;
    if (n_marks) *n_marks = marks ? n_mark : 0;
    return cudaGetLastError();
}

}  // namespace dockauv
