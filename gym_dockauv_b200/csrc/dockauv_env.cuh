// dockauv_env.cuh -- env-level pieces shared by the step kernels: reset, command filter, current, the
// non-radar part of observe / is_done / reward_step, episode statistics.
#pragma once
#include "dockauv_device.cuh"

namespace dockauv {

// ------------------------------------------------------------------------------------------- reset
// Env-major obstacle rows (KParams::obsd): obstacle k of env i (capsules first, then sphere k - n_caps) as stored,
// zero-filled to eight words, moved as 16-byte pieces (4 in f64, 2 in f32)
constexpr int kObstRowWords = 8;

template <typename T>
__device__ __forceinline__ T *obstacle_row(const KParams<T> &p, int64_t i, int k) {
    return p.obsd + (i * (p.n_caps + p.n_sph) + k) * kObstRowWords;
}

template <typename T>
__device__ __forceinline__ void load_obstacle_row(const T *row, T o[kObstRowWords]) {
    if constexpr (sizeof(T) == 8) {
        const double2 *s = reinterpret_cast<const double2 *>(row);
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const double2 v = s[c];
            o[2 * c] = v.x;
            o[2 * c + 1] = v.y;
        }
    } else {
        const float4 *s = reinterpret_cast<const float4 *>(row);
#pragma unroll
        for (int c = 0; c < 2; c++) {
            const float4 v = s[c];
            o[4 * c] = v.x;
            o[4 * c + 1] = v.y;
            o[4 * c + 2] = v.z;
            o[4 * c + 3] = v.w;
        }
    }
}

template <typename T>
__device__ __forceinline__ void store_obstacle_row(T *row, const T o[kObstRowWords]) {
    if constexpr (sizeof(T) == 8) {
        double2 *d = reinterpret_cast<double2 *>(row);
#pragma unroll
        for (int c = 0; c < 4; c++) d[c] = make_double2(o[2 * c], o[2 * c + 1]);
    } else {
        float4 *d = reinterpret_cast<float4 *>(row);
#pragma unroll
        for (int c = 0; c < 2; c++) d[c] = make_float4(o[4 * c], o[4 * c + 1], o[4 * c + 2], o[4 * c + 3]);
    }
}

// Obstacle k of env i (numbered as obstacle_row) as stored (T): a capsule bot[3] top[3] r (NW = 7) or a sphere
// centre[3] r (NW = 4).  The library keeps two copies of it, written here from the obstacle and the goal: the obstacle
// row (KParams::obsd) and the float record(s) for the cull code (KParams::obsf, see cull_pair_rec): capsule k -> slots
// 2k, 2k+1; sphere s = k - n_caps -> slot 2 n_caps + s.  The pipeline layout allocates both or neither.
template <typename T, int NW>
__device__ __forceinline__ void store_obstacle_copies(const KParams<T> &p, int64_t i, int k, const T (&ob)[NW],
                                                      const T goal[3]) {
    static_assert(NW == 7 || NW == 4, "capsule: 7 words, sphere: 4");
    constexpr bool is_cap = NW == 7;
    if (p.obsf == nullptr) return;
    const T *o = ob;       // a pointer: o[4..6] below are only read for a capsule
    {
        const T row[kObstRowWords] = {o[0], o[1], o[2], o[3], is_cap ? o[4] : T(0), is_cap ? o[5] : T(0),
                                      is_cap ? o[6] : T(0), T(0)};
        store_obstacle_row<T>(obstacle_row<T>(p, i, k), row);
    }
    const double obd[7] = {(double)o[0], (double)o[1], (double)o[2], (double)o[3], is_cap ? (double)o[4] : 0.0,
                           is_cap ? (double)o[5] : 0.0, is_cap ? (double)o[6] : 0.0};
    const double g[3] = {(double)goal[0], (double)goal[1], (double)goal[2]};
    float4 q0, q1;
    obstacle_record_f32(obd, g, is_cap, q0, q1);
    if (is_cap) {
        p.obsf[(int64_t)(2 * k) * p.n_envs + i] = q0;
        p.obsf[(int64_t)(2 * k + 1) * p.n_envs + i] = q1;
    } else {
        const int s = k - p.n_caps;
        p.obsf[(int64_t)(2 * p.n_caps + s) * p.n_envs + i] = q0;
    }
}

// Obstacle k of env i, in T or as drawn in double, rounded to T into the caller's planes (capsule k: capsules[k*7+j],
// sphere s = k - n_caps: spheres[s*4+j]) and into the library's copies
template <typename T, typename S, int NW>
__device__ __forceinline__ void store_obstacle(const KParams<T> &p, int64_t i, int k, const S (&ob)[NW], const T goal[3]) {
    const int64_t N = p.n_envs;
    T *plane = NW == 7 ? p.capsules + (int64_t)(k * 7) * N : p.spheres + (int64_t)((k - p.n_caps) * 4) * N;
    T o[NW];
#pragma unroll
    for (int j = 0; j < NW; j++) {
        o[j] = (T)ob[j];
        plane[(int64_t)j * N + i] = o[j];
    }
    store_obstacle_copies<T>(p, i, k, o, goal);
}

// Rebuilds the library's obstacle copies of env i from the bound buffers (after the caller wrote obstacles or goals
// itself: dockauv_refresh_obstacles).
template <typename T>
__global__ void refresh_obstacles_kernel(const __grid_constant__ KParams<T> p) {
    const int64_t N = p.n_envs;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const T goal[3] = {p.goal[i], p.goal[N + i], p.goal[2 * N + i]};
    for (int k = 0; k < p.n_caps; k++) {
        T cap[7];
#pragma unroll
        for (int j = 0; j < 7; j++) cap[j] = p.capsules[(int64_t)(k * 7 + j) * N + i];
        store_obstacle_copies<T>(p, i, k, cap, goal);
    }
    for (int s = 0; s < p.n_sph; s++) {
        T sph[4];
#pragma unroll
        for (int j = 0; j < 4; j++) sph[j] = p.spheres[(int64_t)(s * 4 + j) * N + i];
        store_obstacle_copies<T>(p, i, p.n_caps + s, sph, goal);
    }
}

// BaseDocking3d.reset (docking3d.py:222-322) + <Scenario>.generate_environment (:803-988) for env i.
// Distributions are the reference's; the random stream is Philox4x32-10 keyed by (seed, global env id,
// episode) instead of the reference's global MT19937 (DESIGN.md "reset").  Draw slots: 0 heading, 1-3
// position, 4-6 attitude, 7 goal angle, 8 goal depth, 9 pillar phase, 10-11 current direction, 12 current
// speed, 13+3s.. synthetic sphere s.
// The work of one reset is cut into kResetRoles independent ROLES so that eight warps can share it (a reset done by one
// thread is a ~5500-instruction dependent chain): 0 pose / goal / counters, 1..4 pillar k, 5 dock capsule + unused capsule
// slots + current + command, 6..7 spheres (s = role - 6, role - 4, ..).  Every role draws what it needs from the
// counter-based stream itself; roles never exchange values, so any mapping of roles to threads gives identical bits.
//   ep: the env's episode counter BEFORE this reset (the caller bumps it once all roles have read it)
constexpr int kResetRoles = 8;

template <typename T>
__device__ __forceinline__ void reset_env_role(const KParams<T> &p, int64_t i, int role, uint32_t ep) {
    const int64_t N = p.n_envs;
    const uint64_t gid = p.env_id0 + (uint64_t)i;
    const double PI = 3.141592653589793;
    // one Philox block yields two draws: the blocks a role needs are evaluated once each (role 0, the longest chain of the
    // eight, took nine block evaluations for its nine draws when every draw evaluated its own)
    auto U = [&](uint32_t idx) { return philox_uniform(p.seed, gid, ep, idx); };
    auto U2 = [&](uint32_t blk, double u[2]) { philox_uniform_pair(p.seed, gid, ep, blk, u); };
    const int scn = p.scenario;
    const bool has_goal_ring = scn >= DOCKAUV_SCN_CAPSULE;
    const bool has_dock = has_goal_ring && scn != DOCKAUV_SCN_OBSTACLES_NOCAP && p.n_caps > 0;
    const bool has_pillars = scn >= DOCKAUV_SCN_OBSTACLES;
    const int first_pillar = has_dock ? 1 : 0;
    const int n_pillars = has_pillars ? max(0, min(4, p.n_caps - first_pillar)) : 0;
    // the goal (draws 7 and 8): stored by role 0, and the origin of every float obstacle record
    double goal[3] = {0.0, 0.0, 0.0};
    double u67[2] = {0.0, 0.0}, u89[2] = {0.0, 0.0};      // draws 6..9: goal angle / depth here, yaw (role 0) and pillar phase below
    if (has_goal_ring || role == 0) U2(3, u67);
    if (has_goal_ring) {                                                       // :860-886
        U2(4, u89);
        double theta = u67[1] * 2 * PI;
        double radius = 1.0 + (double)p.safety_radius;
        double s, c;
        sincos(theta, &s, &c);
        goal[0] = c * radius;
        goal[1] = s * radius;
        goal[2] = (u89[0] - 0.5) * 4.0;
    }
    const T goal_t[3] = {(T)goal[0], (T)goal[1], (T)goal[2]};
    if (role == 0) {
        double u01[2], u23[2], u45[2];
        U2(0, u01);
        U2(1, u23);
        U2(2, u45);
        double heading = (u01[0] - 0.5) * PI;                                 // :814
        double r[3] = {u01[1] - 0.5, u23[0] - 0.5, u23[1] - 0.5};             // :694-696
        {
            double sg = (r[2] > 0.0) - (r[2] < 0.0);
            r[2] = fabs(r[0] + r[1]) / 3 * sg;
        }
        double sc = 15.0 / sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
        double pos[3] = {r[0] * sc, r[1] * sc, r[2] * sc};
        double max_att = (double)p.max_attitude;
        double att[3] = {(u45[0] - 0.5) * 2 * (max_att * 0.7), (u45[1] - 0.5) * 2 * (max_att * 0.7),
                         (u67[0] - 0.5) * 2 * PI};                             // :699-703
        // vec_line_point(goal, top=(0,0,-2), bot=(0,0,2)) = (-gx, -gy, 0)  (shape.py:420-433)
        if (has_goal_ring) heading = (double)ssa<double>(atan2(0.0 - goal[1], 0.0 - goal[0]));
#pragma unroll
        for (int c = 0; c < 3; c++) {
            p.state[(int64_t)c * N + i] = (T)pos[c];
            p.state[(int64_t)(3 + c) * N + i] = (T)att[c];
            p.goal[(int64_t)c * N + i] = goal_t[c];
        }
#pragma unroll
        for (int c = 6; c < 12; c++) p.state[(int64_t)c * N + i] = T(0);     // auvsim.py:55-65
        p.heading_goal[i] = (T)heading;
        p.t_steps[i] = 0;
        p.ep_return[i] = T(0);
    } else if (role <= 4) {                                                    // pillars, :919-946
        const int k = role - 1;
        if (k < n_pillars) {
            double theta = (has_goal_ring ? u89[1] : U(9)) * 2 * PI;
            for (int q = 0; q < k; q++) theta += 2 * PI / 4;
            const double half = 2.0 * (double)p.max_dist_from_goal / 2.0;
            double s, c;
            sincos(theta, &s, &c);
            const double x = c * 6, y = s * 6;
            const double cap[7] = {x, y, half, x, y, -half, 1.0};
            store_obstacle<T>(p, i, first_pillar + k, cap, goal_t);
        }
    } else if (role == 5) {
        if (has_dock) {
            const double cap[7] = {0, 0, 2.0, 0, 0, -2.0, 1.0};              // bot = 2*position - top, shape.py:105-108
            store_obstacle<T>(p, i, 0, cap, goal_t);
        }
        for (int kc = first_pillar + n_pillars; kc < p.n_caps; kc++) {         // unused slots: far away, zero radius
            const double cap[7] = {1e6, 1e6, 1e6, 1e6, 1e6, 1e6 + 1.0, 0.0};
            store_obstacle<T>(p, i, kc, cap, goal_t);
        }
        double cur[5] = {0, 0, 0, 0, 0};
        if (scn == DOCKAUV_SCN_SIMPLE_CURRENT || scn == DOCKAUV_SCN_CAPSULE_CURRENT || scn == DOCKAUV_SCN_OBSTACLES_CURRENT) {
            cur[1] = (U(10) - 0.5) * 2 * (PI / 2);                             // :843-848, :903-907, :983-987
            cur[2] = (U(11) - 0.5) * 2 * PI;
            double speed = (scn == DOCKAUV_SCN_SIMPLE_CURRENT) ? U(12) * 1.0 : 0.5;
            cur[0] = 0.5;
            cur[3] = cur[4] = speed;
        }
#pragma unroll
        for (int c = 0; c < 5; c++) p.current[(int64_t)c * N + i] = (T)cur[c];
        for (int k = 0; k < p.n_u; k++) p.u_prev[(int64_t)k * N + i] = T(0);
    } else {
        const int n_synth = min(p.n_synth_sph, p.n_sph);
        for (int ks = role - 6; ks < p.n_sph; ks += 2) {
            if (ks < n_synth) {                                                 // BASELINE C4 extension: random unit spheres
                double z = 2 * U(13 + 3 * ks) - 1;
                double az = 2 * PI * U(14 + 3 * ks);
                double rr = 4.0 + 6.0 * U(15 + 3 * ks);
                double q = sqrt(1 - z * z), s, c;
                sincos(az, &s, &c);
                const double sph[4] = {rr * q * c, rr * q * s, rr * z, 1.0};
                store_obstacle<T>(p, i, p.n_caps + ks, sph, goal_t);
            } else {
                const double sph[4] = {1e6, 1e6, 1e6, 0.0};
                store_obstacle<T>(p, i, p.n_caps + ks, sph, goal_t);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------- scenario bank reset
// Row layout (dockauv_set_scenario_bank): pose [0:6], goal [6:9], heading goal [9], current [10:15], then capsule slots
// (bot, top, r) and sphere slots (centre, r).  The row is drawn from Philox block (gid, episode, kBankCounter): the
// built-in reset uses blocks below 32 and the current noise 0x80000000 | t, so the three never share a block.
constexpr uint32_t kBankCounter = 0x40000000u;
constexpr int kBankPose = 0, kBankGoal = 6, kBankHeading = 9, kBankCurrent = 10, kBankObst = 15;

// the row of env gid's reset that starts episode ep + 1: uniform = high 64 bits of (64-bit word x K); weighted = the
// first r with cdf[r] > u cdf[K-1] (u the block's 53-bit uniform, so zero-weight rows are never drawn)
template <typename T>
__device__ __forceinline__ int64_t bank_draw(const KParams<T> &p, uint64_t gid, uint32_t ep) {
    uint32_t c[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), ep, kBankCounter};
    philox4x32_10(c, (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
    const double *cdf = p.bank_cdf;
    if (cdf == nullptr) return (int64_t)__umul64hi(((uint64_t)c[0] << 32) | c[1], (uint64_t)p.bank_n);
    const double x = ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6)) * (1.0 / 9007199254740992.0) * cdf[p.bank_n - 1];
    int64_t lo = 0, hi = p.bank_n - 1;         // x < cdf[K-1]: the answer lies in [lo, hi]
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (cdf[mid] > x) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}

// N reals of a row from offset o, read as the 16-byte pieces that cover them (rows and their stride are 16-byte
// multiples, so the pieces stay inside the row)
template <typename T, int N>
__device__ __forceinline__ void load_bank_span(const T *row, int o, T out[N]) {
    constexpr int V = 16 / (int)sizeof(T);
    constexpr int NP = (N + V - 1) / V + 1;           // pieces for N reals at any offset within a piece
    const int base = o & ~(V - 1), sh = o - base;
    T buf[NP * V];
#pragma unroll
    for (int c = 0; c < NP; c++) {
        if (base + c * V >= o + N) break;
        if constexpr (sizeof(T) == 8) {
            const double2 v = reinterpret_cast<const double2 *>(row + base)[c];
            buf[2 * c] = v.x;
            buf[2 * c + 1] = v.y;
        } else {
            const float4 v = reinterpret_cast<const float4 *>(row + base)[c];
            buf[4 * c] = v.x;
            buf[4 * c + 1] = v.y;
            buf[4 * c + 2] = v.z;
            buf[4 * c + 3] = v.w;
        }
    }
#pragma unroll
    for (int j = 0; j < N; j++) {
        T v = buf[j];
#pragma unroll
        for (int s = 1; s < V; s++)
            if (sh == s) v = buf[s + j];
        out[j] = v;
    }
}

// One role of a reset from the bank: the same eight-role split as reset_env_role and the same rule (every role draws the
// row itself, roles never exchange values).  0 pose, zero nu_r, goal, heading goal, counters, row_of_env; 1 current and
// u_prev; 2..7 obstacle slots role - 2, role + 4, .. (capsules first, then spheres).
//   ep: the env's episode counter BEFORE this reset
template <typename T>
__device__ __forceinline__ void bank_reset_role(const KParams<T> &p, int64_t i, int role, uint32_t ep) {
    const int64_t N = p.n_envs;
    const int n_slots = p.n_caps + p.n_sph;
    if (role >= 2 && role - 2 >= n_slots) return;
    const int64_t r = bank_draw<T>(p, p.env_id0 + (uint64_t)i, ep);
    const T *row = p.bank_rows + r * p.bank_stride;
    if (role == 0) {
        T a[10];
        load_bank_span<T, 10>(row, kBankPose, a);
#pragma unroll
        for (int c = 0; c < 6; c++) p.state[(int64_t)c * N + i] = a[c];
#pragma unroll
        for (int c = 6; c < 12; c++) p.state[(int64_t)c * N + i] = T(0);     // auvsim.py:55-65
#pragma unroll
        for (int c = 0; c < 3; c++) p.goal[(int64_t)c * N + i] = a[kBankGoal + c];
        p.heading_goal[i] = a[kBankHeading];
        p.t_steps[i] = 0;
        p.ep_return[i] = T(0);
        if (p.bank_row_of_env) {
            p.bank_row_of_env[N + i] = p.bank_row_of_env[i];
            p.bank_row_of_env[i] = (int32_t)r;
        }
    } else if (role == 1) {
        T cur[5];
        load_bank_span<T, 5>(row, kBankCurrent, cur);
#pragma unroll
        for (int c = 0; c < 5; c++) p.current[(int64_t)c * N + i] = cur[c];
        for (int k = 0; k < p.n_u; k++) p.u_prev[(int64_t)k * N + i] = T(0);
    } else {
        T goal[3];
        load_bank_span<T, 3>(row, kBankGoal, goal);
        for (int s = role - 2; s < n_slots; s += kResetRoles - 2) {
            if (s < p.n_caps) {
                T cap[7];
                load_bank_span<T, 7>(row, kBankObst + 7 * s, cap);
                store_obstacle<T>(p, i, s, cap, goal);
            } else {
                T sph[4];
                load_bank_span<T, 4>(row, kBankObst + 7 * p.n_caps + 4 * (s - p.n_caps), sph);
                store_obstacle<T>(p, i, s, sph, goal);
            }
        }
    }
}

// the whole bank reset by one thread, kept out of line: the single-launch step kernels reach it through one uniform branch
template <typename T>
static __device__ __noinline__ void bank_reset_env(const KParams<T> &p, int64_t i, uint32_t ep) {
#pragma unroll 1
    for (int role = 0; role < kResetRoles; role++) bank_reset_role<T>(p, i, role, ep);
}

// the whole reset by one thread (single-launch layouts: the env's own thread re-initialises it inside the step)
template <typename T>
static __device__ __noinline__ void reset_env(const KParams<T> &p, int64_t i) {
    const uint32_t ep = (uint32_t)p.episode[i];
    if (p.bank_rows != nullptr) {
        bank_reset_env<T>(p, i, ep);
    } else {
#pragma unroll 1
        for (int role = 0; role < kResetRoles; role++) reset_env_role<T>(p, i, role, ep);
    }
    p.episode[i] = (int32_t)(ep + 1);
}

// The reset of up to 32 envs by one CTA of kResetRoles warps: warp = role, lane = env.  Roles are different code paths,
// so they must not share a warp (eight roles on eight lanes of one warp run one after the other: measured, no faster than
// one thread per reset); as warps they run side by side and every lane of a warp does the same thing for another env.
//   valid: this lane has an env.  Must be called by all threads of the CTA.
//   BANK: reset from the scenario bank (KParams::bank_rows) instead of the built-in distributions
constexpr int kResetCta = 32 * kResetRoles;

template <typename T, bool BANK>
__device__ __forceinline__ void reset_envs_cta(const KParams<T> &p, int64_t i, bool valid) {
    const int role = threadIdx.x >> 5;
    uint32_t ep = 0;
    if (valid) ep = (uint32_t)p.episode[i];
    __syncthreads();                                 // every role has read the episode counter before role 0 bumps it
    if (valid) {
        if (BANK) bank_reset_role<T>(p, i, role, ep);
        else reset_env_role<T>(p, i, role, ep);
        if (role == 0) p.episode[i] = (int32_t)(ep + 1);
    }
}

// dockauv_reset: one CTA of kResetRoles warps per 32 envs
template <typename T, bool BANK>
__global__ void __launch_bounds__(kResetCta) reset_kernel(const __grid_constant__ KParams<T> p, const uint8_t *mask) {
    const int64_t i = p.env_begin + (int64_t)blockIdx.x * 32 + (threadIdx.x & 31);
    const bool valid = i < p.env_end && (mask == nullptr || mask[i] != 0);
    reset_envs_cta<T, BANK>(p, i, valid);
}

// ------------------------------------------------------------------------------------------- step pieces
// Everything the non-radar part of one step hands to the radar / finalisation part.
template <typename T>
struct StepCarry {
    T pos[3];          // post-step position
    T R[9];            // post-step Rzyx
    T partial_reward;  // reward terms that do not depend on the radar or the collision flag, summed later
    T rarr[13];        // reward_arr (only [0..5], [7] filled here)
    uint32_t cond;     // bits 0..3
    T delta_d;
    int32_t t_steps;   // episode step counter before this step
    T ep_return;       // cumulative reward before this step
};

// what command_and_penalty reads of one env: the raw action (float32 or float64, as the caller handed it over) and the
// previous low-passed command.  Loaded as one batch before anything is used: the float32 division of the penalty has a
// slow-path branch per actuator, loads are not moved across it, and with the loads inside the loop a thread paid NU memory
// round trips one after the other (ncu: 5 % of the dynamics launch's stall samples on these six waits)
template <typename T, int NU>
struct CommandIn {
    float a32[NU];
    double a64[NU];
    T up[NU];
};

template <typename T, int NU>
__device__ __forceinline__ void load_command(const KParams<T> &p, int64_t i, CommandIn<T, NU> &in) {
    const int64_t N = p.n_envs;
#pragma unroll
    for (int k = 0; k < NU; k++) in.up[k] = p.u_prev[(int64_t)k * N + i];
    if (p.act_f32) {
        const float *a = (const float *)p.actions + i * NU;
#pragma unroll
        for (int k = 0; k < NU; k++) in.a32[k] = a[k];
    } else {
        const double *a = (const double *)p.actions + i * NU;
#pragma unroll
        for (int k = 0; k < NU; k++) in.a64[k] = a[k];
    }
}

// action -> low-passed command (auvsim.py:67-87, lowpassfilter.py:29-42) and the action penalty
// (docking3d.py:584-585).  Returns -(sum((|a|/n_u)^2 * w)).
template <typename T, int NU>
__device__ __forceinline__ T command_and_penalty(const KParams<T> &p, const CommandIn<T, NU> &in, T u[NU]) {
    T pen;
    if (p.act_f32) {
        float pen32 = 0.0f;
        double pen64 = 0.0;
#pragma unroll
        for (int k = 0; k < NU; k++) {
            float ak = in.a32[k];
            float c = ak < -1.0f ? -1.0f : (ak > 1.0f ? 1.0f : ak);
            float frac = (c + 1.0f) / 2.0f;                       // numpy keeps this in float32
            T x = p.u_lo[k] + p.u_span[k] * (T)frac;
            u[k] = p.lp_alpha * x + (T(1) - p.lp_alpha) * in.up[k];
            // numpy evaluates (|a| / n_u) ** 2 * w and the sum in float32 with one rounding per operation:
            // explicit _rn intrinsics keep the compiler from contracting them into FMAs
            float q = __fdiv_rn(fabsf(ak), (float)NU);
            q = __fmul_rn(q, q);
            pen32 = __fadd_rn(pen32, __fmul_rn(q, p.arf_f32[k]));
            pen64 += (double)q * (double)p.arf[k];
        }
        pen = p.action_factor_is_scalar ? (T)pen32 : (T)pen64;
    } else {
        T s = T(0);
#pragma unroll
        for (int k = 0; k < NU; k++) {
            T ak = (T)in.a64[k];
            T frac = (clipv(ak, T(-1), T(1)) + T(1)) / T(2);
            T x = p.u_lo[k] + p.u_span[k] * frac;
            u[k] = p.lp_alpha * x + (T(1) - p.lp_alpha) * in.up[k];
            T q = Mth<T>::abs_(ak) / T(NU);
            s += (q * q) * p.arf[k];
        }
        pen = s;
    }
    return -pen;
}

template <typename T, int NU>
__device__ __forceinline__ T command_and_penalty(const KParams<T> &p, int64_t i, T u[NU]) {
    CommandIn<T, NU> in;
    load_command<T, NU>(p, i, in);
    return command_and_penalty<T, NU>(p, in, u);
}

// np.sum over the 13 reward terms in numpy's pairwise order for n = 13 (8 unrolled accumulators combined
// as a tree, then the 5 remaining terms added sequentially).
template <typename T>
__device__ __forceinline__ T reward_sum13(const T r[13]) {
    T s = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
#pragma unroll
    for (int k = 8; k < 13; k++) s += r[k];
    return s;
}

// obs[0:16] of env i straight to its HBM row (four 16-byte stores when n_obs allows them)
template <typename T, typename V>
__device__ __forceinline__ void store_obs_head(const KParams<T> &p, int64_t i, const V o[16]) {
    if ((p.n_obs & 3) == 0) {
        float4 *orow4 = reinterpret_cast<float4 *>(p.obs + i * p.n_obs);
#pragma unroll
        for (int c = 0; c < 4; c++)
            orow4[c] = make_float4((float)o[4 * c], (float)o[4 * c + 1], (float)o[4 * c + 2], (float)o[4 * c + 3]);
    } else {
        float *orow = p.obs + i * p.n_obs;
#pragma unroll
        for (int c = 0; c < 16; c++) orow[c] = (float)o[c];
    }
}

// 0 for a finite pose, NaN otherwise: radar_env poisons the ray distances with it where the reference's NaN propagation
// reaches them (envs without capsules)
template <typename T>
__device__ __forceinline__ T pose_poison(const T pos[3], const T att[3]) {
    return (((pos[0] + pos[1]) + (pos[2] + att[0])) + (att[1] + att[2])) * T(0);
}

// Episode statistics of one warp: each lane remembers the outcome of its env; if any episode of the warp ended,
// a shuffle reduction folds the contributions and lane 0 issues one global atomic per non-zero statistic.
struct WarpStats {
    bool done = false, nan = false;
    uint32_t cond = 0;
    int32_t length = 0;
    double ep_return = 0.0, delta_d = 0.0;

    // n_steps = env-steps to account for (callers pass the CTA's count from one warp only, 0 from the others:
    // one same-address atomic per CTA instead of one per warp)
    __device__ __forceinline__ void flush(double *g, int n_steps) const {
        const int lane = threadIdx.x & 31;
        g += (blockIdx.x & (DOCKAUV_STAT_COPIES - 1)) * DOCKAUV_N_STATS;   // replica of this CTA (dockauv_fold_stats)
        if (__any_sync(0xffffffffu, done)) {
            double v[DOCKAUV_STAT_ENV_STEPS];
            v[DOCKAUV_STAT_EPISODES] = done ? 1.0 : 0.0;
            v[DOCKAUV_STAT_SUM_RETURN] = done ? ep_return : 0.0;
            v[DOCKAUV_STAT_SUM_LENGTH] = done ? (double)length : 0.0;
#pragma unroll
            for (int k = 0; k < 5; k++) v[DOCKAUV_STAT_COND0 + k] = (done && ((cond >> k) & 1u)) ? 1.0 : 0.0;
            v[DOCKAUV_STAT_SUM_FINAL_DELTA_D] = done ? delta_d : 0.0;
            v[DOCKAUV_STAT_NAN_ENVS] = (done && nan) ? 1.0 : 0.0;
#pragma unroll
            for (int k = 0; k < DOCKAUV_STAT_ENV_STEPS; k++) {
                double x = v[k];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
                if (lane == 0 && x != 0.0) atomicAdd(&g[k], x);
            }
        }
        if (lane == 0 && n_steps > 0) atomicAdd(&g[DOCKAUV_STAT_ENV_STEPS], (double)n_steps);
    }

    // the same without the shuffle reduction: every lane whose episode ended adds its own contributions (fire-and-forget
    // atomics into the CTA's replica).  ~1 % of the lanes end an episode, but 27 % of the warps contain one: the reduction
    // costs those warps ~150 instructions, the direct form ~8 atomics per ended episode
    __device__ __forceinline__ void flush_direct(double *g, int n_steps) const {
        g += (blockIdx.x & (DOCKAUV_STAT_COPIES - 1)) * DOCKAUV_N_STATS;
        if (done) {
            atomicAdd(&g[DOCKAUV_STAT_EPISODES], 1.0);
            atomicAdd(&g[DOCKAUV_STAT_SUM_RETURN], ep_return);
            atomicAdd(&g[DOCKAUV_STAT_SUM_LENGTH], (double)length);
#pragma unroll
            for (int k = 0; k < 5; k++)
                if ((cond >> k) & 1u) atomicAdd(&g[DOCKAUV_STAT_COND0 + k], 1.0);
            atomicAdd(&g[DOCKAUV_STAT_SUM_FINAL_DELTA_D], delta_d);
            if (nan) atomicAdd(&g[DOCKAUV_STAT_NAN_ENVS], 1.0);
        }
        if (n_steps > 0) atomicAdd(&g[DOCKAUV_STAT_ENV_STEPS], (double)n_steps);
    }
};

}  // namespace dockauv
