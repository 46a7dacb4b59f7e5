// dockauv_step_warp.cuh -- layout DOCKAUV_LAYOUT_WARP_RAYS: the whole step in ONE launch.
//
// One CTA of 128 threads owns 128 consecutive envs; each warp works only on the 32 envs of its own lanes, so the
// phases below are separated by __syncwarp() only.
//   phase A (thread per env) : current, command filter, RKF45, angle wrap, nav errors, obs[0:16], done bits 0..3 and
//                              the radar-independent reward terms; the post-step pose goes to shared memory.
//   phase B (warp per env)   : the 32 envs are taken in sub-batches of 32 / slots envs (slots = 8 or 16 obstacle
//                              slots per env).  Pass 1 of a sub-batch uses ALL lanes, one (env, obstacle) pair per
//                              lane: coalesced-by-sector obstacle loads, the ray-independent algebra, the
//                              body-collision test and the radar-range / field-of-view culls (in T, exact); two ballots
//                              publish the collision and in-view bits of the whole sub-batch.  Pass 2 walks over the
//                              envs of the sub-batch: radar_env (dockauv_rays.cuh).
//   phase C (thread per env) : reward, done, counters, statistics, auto-reset; then each warp moves the observation
//                              rows of finished envs.
// 168 registers: the radar's ~90 registers travel through the integrator, and a thread that finished an episode
// serialises a reset in front of its warp -- which is why the default layout is the pipeline (dockauv_step_pipe.cuh:
// 0.5 ms per 1M-env step against 0.9 ms).  This kernel serves every call that asks for debug outputs (DBG) and is the
// independently scheduled cross-check of the pipeline: same device functions, exact (T) culls instead of the float ones.
#pragma once
#include "dockauv_step_tpe.cuh"

namespace dockauv {

constexpr int kWarpEnvs = 128;       // envs (= threads) per CTA
constexpr int kPoseStride = 14;      // shared words per env: pos[3] R[9] poison pad

template <typename T>
struct WarpSmem {
    // layout of the dynamic shared memory block (offsets in bytes, computed on host and device alike)
    int pose_off, pre_off, ray_off, total;
    int ray_stride;     // T words per warp of ray-distance scratch (+1 zero slot for the pooling padding)
    __host__ __device__ WarpSmem(int n_rays) {
        int off = 0;
        pose_off = off; off += kWarpEnvs * kPoseStride * (int)sizeof(T);
        pre_off = off;  off += 4 * 32 * kPreStride * (int)sizeof(T);
        ray_stride = (n_rays + 2) & ~1;
        ray_off = off;  off += 4 * ray_stride * (int)sizeof(T);
        total = (off + 15) & ~15;
    }
};

#ifndef DOCKAUV_A_PREFETCH
#define DOCKAUV_A_PREFETCH 37      // CTAs ahead whose inputs the dynamics code prefetches into L2 (0 = off)
#endif

// CTAs are dispatched in blockIdx order: the inputs of a CTA a little further down the order are pulled into L2 now,
// while this one integrates (a third of a dynamics warp's lifetime was spent waiting for its own first HBM round trip:
// 31 % of the launch's stall samples).  Measured: distance 8..148 CTAs 218 us, 300 235 us, 592 (one resident wave) and
// beyond no gain, none 253 us.
template <typename T, int NU, int CTA = kWarpEnvs>
__device__ __forceinline__ void prefetch_dynamics_inputs(const KParams<T> &p, int64_t i, int lane, bool with_goal) {
#if DOCKAUV_A_PREFETCH > 0
    const int64_t N = p.n_envs;
    const int64_t j = i + (int64_t)DOCKAUV_A_PREFETCH * kWarpEnvs;      // distance in envs: 37 CTAs of 128
    if (j < p.env_end) {
        auto pf = [](const void *a) { asm volatile("prefetch.global.L2 [%0];" ::"l"(a)); };
#pragma unroll
        for (int c = 0; c < 12; c++) pf(p.state + (int64_t)c * N + j);
#pragma unroll
        for (int c = 0; c < NU; c++) pf(p.u_prev + (int64_t)c * N + j);
        if (with_goal) {
#pragma unroll
            for (int c = 0; c < 3; c++) pf(p.goal + (int64_t)c * N + j);
        }
        if ((lane & 3) == 0) pf((const char *)p.actions + (p.act_f32 ? 4 : 8) * NU * j);
        if ((lane & 7) == 0) pf(p.t_steps + j);
        if ((lane & 15) == 0) pf(p.ep_return + j);
    }
#endif
}

// no min-CTAs hint on purpose: __launch_bounds__(128, 3) ends at the same 168 registers but a 6 % slower schedule,
// (128, 4) and (128, 5) spill (measured on B200, profiles/r01/NOTES.md)
// DBG: debug outputs compiled in.
template <typename T, int VEH, int NU, int RPL, bool DBG>
__global__ void __launch_bounds__(kWarpEnvs) step_warp_kernel(const __grid_constant__ KParams<T> p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const WarpSmem<T> L(p.n_rays);
    T *s_pose = reinterpret_cast<T *>(smem_raw + L.pose_off);
    WarpStats bs;

    const int64_t N = p.n_envs;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t i0 = p.env_begin + (int64_t)blockIdx.x * kWarpEnvs;
    const int64_t i = i0 + tid;
    const bool active = i < p.env_end;
    int64_t left64 = p.env_end - i0;
    const int n_here = (int)(left64 < (int64_t)kWarpEnvs ? left64 : (int64_t)kWarpEnvs);
    const int e_warp = warp * 32;                         // first env (CTA-local) of this warp
    const int n_warp = max(0, min(32, n_here - e_warp));  // envs this warp really has

    prefetch_dynamics_inputs<T, NU>(p, i, lane, true);
    // ------------------------------------------------------------------ phase A
    StepCarry<T> cy;
    if (active) {
        T spsi, cpsi, att[3];
        float obs16[16];
        step_dynamics<T, VEH, NU, DBG>(p, i, cy, spsi, cpsi, obs16, att);
        T *ps = s_pose + tid * kPoseStride;
#pragma unroll
        for (int c = 0; c < 3; c++) ps[c] = cy.pos[c];
#pragma unroll
        for (int c = 0; c < 9; c++) ps[3 + c] = cy.R[c];
        ps[12] = pose_poison<T>(cy.pos, att);
        // obs[0:16] to its HBM row; phase C zeroes the row if the env is reset
        store_obs_head<T>(p, i, obs16);
    }
    __syncwarp();

    // ------------------------------------------------------------------ phase B
    T my_oa_dot = p.sum_beta_oa;     // owner-lane copies of the per-env radar results (neutral values: r_oa = 0)
    bool my_col = false;
    bool my_view_empty = true;       // nothing within range and view: the owner lane writes the all-ones ray cells
    const bool no_dbg = !DBG || (p.dbg_ray_dist == nullptr && p.dbg_obs == nullptr);
    {
        T *s_pre = reinterpret_cast<T *>(smem_raw + L.pre_off) + warp * 32 * kPreStride;
        T *s_ray = reinterpret_cast<T *>(smem_raw + L.ray_off) + warp * L.ray_stride;
        const int n_caps = p.n_caps, n_sph = p.n_sph, n_obst = n_caps + n_sph;
        RayLane<T, RPL> rl;
        rl.init(p, lane, s_ray);
        // obstacle slot of this lane in pass 1
        const int slots = n_obst <= 8 ? 8 : 16;
        const int epp = 32 / slots;                        // envs per sub-batch
        const unsigned slot_mask = (1u << slots) - 1u;
        const int my_slot = lane & (slots - 1), my_sub = lane / slots;
        const bool slot_is_cap = my_slot < n_caps, slot_used = my_slot < n_obst;
        const T *obst_row = slot_is_cap ? p.capsules + (int64_t)(my_slot * 7) * N
                                        : p.spheres + (int64_t)((my_slot - n_caps) * 4) * N;

        // raw obstacle of this lane's (env, slot) pair: loaded one sub-batch ahead so that the HBM latency of the
        // next pre-pass is covered by the ray loop of the current one
        auto load_obstacle = [&](int eb_, T ob[7]) {
            const int e_ = eb_ + my_sub;
            if (slot_used && e_ < n_warp) {
                const T *g = obst_row + (i0 + e_warp + e_);
                const int n_words = slot_is_cap ? 7 : 4;
#pragma unroll
                for (int c = 0; c < 7; c++)
                    if (c < n_words) ob[c] = g[(int64_t)c * N];
            }
        };
        T ob_next[7];
#pragma unroll
        for (int c = 0; c < 7; c++) ob_next[c] = T(0);
        load_obstacle(0, ob_next);

        for (int eb = 0; eb < n_warp; eb += epp) {
            T ob[7];
#pragma unroll
            for (int c = 0; c < 7; c++) ob[c] = ob_next[c];
            if (eb + epp < n_warp) load_obstacle(eb + epp, ob_next);
            // ---- pass 1: one (env, obstacle) pair per lane
            bool hit_body = false, in_range = false;
            {
                const int e = eb + my_sub;
                if (slot_used && e < n_warp) {
                    const T *pose = s_pose + (e_warp + e) * kPoseStride;
                    const T pos[3] = {pose[0], pose[1], pose[2]};
                    T *w = s_pre + lane * kPreStride;
                    obstacle_pair<T, true>(p, pos, pose + 3, ob, slot_is_cap, w, hit_body, in_range);
                }
            }
            const unsigned colb = __ballot_sync(0xffffffffu, hit_body);
            const unsigned nearb = __ballot_sync(0xffffffffu, in_range);
            {   // the owner lane of each env of this sub-batch keeps its collision flag for phase C
                const int s = lane - eb;
                if (s >= 0 && s < epp) {
                    my_col = ((colb >> (slots * s)) & slot_mask) != 0u;
                    my_view_empty = ((nearb >> (slots * s)) & slot_mask) == 0u;
                }
            }
            __syncwarp();

            // ---- pass 2: cast rays, env by env
            for (int s = 0; s < epp && eb + s < n_warp; s++) {
                const int e = eb + s;
                const T *pose = s_pose + (e_warp + e) * kPoseStride;
                const unsigned near_mask = (nearb >> (slots * s)) & slot_mask;
                const T poison = pose[12];
                if (near_mask == 0u && poison == T(0) && no_dbg) {
                    // nothing within range and view: every ray reads max_dist (sensor.py:113-117), the pooled
                    // observation is all ones (written by the owner lane in phase C) and the obstacle-avoidance
                    // sum keeps its neutral value sum(beta) (r_oa = 0)
                    continue;
                }
                T R[9];
#pragma unroll
                for (int c = 0; c < 9; c++) R[c] = pose[3 + c];
                const T oa_dot = radar_env<T, RPL, DBG, RayLane<T, RPL>>(p, rl, R, poison, near_mask, s_pre + (s * slots) * kPreStride, s_ray,
                                                        lane, i0 + e_warp + e);
                if (lane == e) my_oa_dot = oa_dot;
            }
        }
    }

    // ------------------------------------------------------------------ phase C
    bool done = false;
    if (active) {
        if (my_view_empty && no_dbg && s_pose[tid * kPoseStride + 12] == T(0)) store_clear_cells<T>(p, i);
        const T r_oa = p.sum_beta_oa / my_oa_dot - T(1);      // docking3d.py:792
        done = step_finish<T, DBG>(p, i, cy, r_oa, my_col, bs);
    }
    __syncwarp();     // orders the pooled-cell stores of the other lanes before the row fix-up below
    // ---- rows of envs whose episode ended (~1 % per step): keep the last observation as terminal_observation and
    //      hand back the all-zero reset observation (docking3d.py:269,322); the warp moves each such row together
    {
        unsigned dm = __ballot_sync(0xffffffffu, done);
        const int n_obs = p.n_obs;
        while (dm) {
            const int e = __ffs(dm) - 1;
            dm &= dm - 1;
            float *row = p.obs + (i0 + e_warp + e) * n_obs;
            float *trow = p.terminal_obs ? p.terminal_obs + (i0 + e_warp + e) * n_obs : nullptr;
            for (int c = lane; c < n_obs; c += 32) {
                if (trow) trow[c] = row[c];
                if (p.auto_reset) row[c] = 0.0f;
            }
        }
    }
    bs.flush(p.stats, warp == 0 ? n_here : 0);
}

// A kernel gets 48 KB of shared memory in all, its static arrays (static_bytes) included, unless it is allowed more
template <typename K>
static cudaError_t allow_dyn_smem(K kern, int smem, int static_bytes) {
    if (smem + static_bytes <= 48 * 1024) return cudaSuccess;
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

template <typename T, int VEH, int NU, int RPL, bool DBG>
static cudaError_t launch_step_warp_rpl(const KParams<T> &k, cudaStream_t st) {
    const int64_t n = k.env_end - k.env_begin;
    const WarpSmem<T> L(k.n_rays);
    const int smem = L.total;
    auto kern = step_warp_kernel<T, VEH, NU, RPL, DBG>;
    const cudaError_t e = allow_dyn_smem(kern, smem, 0);
    if (e != cudaSuccess) return e;
    const unsigned blocks = (unsigned)((n + kWarpEnvs - 1) / kWarpEnvs);
    kern<<<blocks, kWarpEnvs, smem, st>>>(k);
    return cudaGetLastError();
}

template <typename T>
static bool wants_debug(const KParams<T> &k) {
    return k.dbg_ray_dist || k.dbg_reward_arr || k.dbg_euler_dot || k.dbg_nu_c || k.dbg_nav || k.dbg_obs || k.dbg_state_dot;
}

// rays per lane: 2 covers the stock 63-ray and the 64-ray radar; 8 covers everything up to DOCKAUV_MAX_RAYS
template <typename T, int VEH, int NU>
static cudaError_t launch_step_warp(const KParams<T> &k, cudaStream_t st) {
    if (wants_debug(k))
        return k.n_rays <= 64 ? launch_step_warp_rpl<T, VEH, NU, 2, true>(k, st)
                              : launch_step_warp_rpl<T, VEH, NU, 8, true>(k, st);
    if (k.n_rays <= 64) return launch_step_warp_rpl<T, VEH, NU, 2, false>(k, st);
    return launch_step_warp_rpl<T, VEH, NU, 8, false>(k, st);
}

}  // namespace dockauv
