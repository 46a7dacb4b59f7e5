// dockauv_capi.cu -- C ABI (include/dockauv.h) over the sm_100a step kernels.
//
// No torch types, no global state besides a thread-local error string.  All device memory that crosses the
// boundary is caller-owned; the handle owns only its small ray table, the statistics vector, (lazily) the
// device staging buffers + streams of the host-buffer entry point and, while taps are set, the K-env tap shadows and
// its side stream.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdint>
#include <cstring>
#include <algorithm>
#include <new>
#include <type_traits>
#include <utility>
#include <vector>

#include "dockauv_device.cuh"
#include "dockauv_launch.h"
#include "dockauv_policy.cuh"
#include "dockauv_sac_actor.cuh"

using namespace dockauv;

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            return fail(DOCKAUV_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                        __LINE__);                                                                       \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

#ifndef DOCKAUV_HOST_CHUNKS
#define DOCKAUV_HOST_CHUNKS 12     // chunks of dockauv_step_host (copies of chunk c + 1 overlap the launches of chunk c)
#endif
static const int kHostStreams = 3;
static const size_t kStatsBytes = sizeof(double) * DOCKAUV_N_STATS * DOCKAUV_STAT_COPIES;   // replica 0 = the public vector

// Captured launch sequences keyed by everything they bake in (pointers, switches, seed), up to `capacity` of them; once
// full, the oldest capture is replaced.  Keys are zero-filled and compared byte for byte, so a field added to a key
// struct takes part without further code.
template <typename Key>
struct GraphCache {
    static_assert(std::is_trivially_copyable<Key>::value && std::has_unique_object_representations<Key>::value &&
                      sizeof(Key) % 8 == 0,
                  "graph keys are compared byte for byte: plain data without padding, whole 64-bit words");
    struct Graph {
        Key key;
        cudaGraphExec_t exec = nullptr;
        int64_t launches = 0;              // kernels in the captured sequence
        std::vector<int64_t> begins;       // first env of every range its last step stepped (dockauv_last_list_counts)
    };
    size_t capacity;
    std::vector<Graph> graphs;
    size_t next = 0;                       // slot replaced next once the cache is full
    int64_t captures = 0;                  // how many sequences were captured (tests: replays must not re-capture)
    explicit GraphCache(size_t cap) : capacity(cap) {}
    // word by word, out at the first difference (an out-of-line memcmp per entry made a lookup in a 64-graph cache ~4x
    // slower on the host)
    static bool same(const Key &a, const Key &b) {
        const char *p = (const char *)&a, *q = (const char *)&b;
        for (size_t i = 0; i < sizeof(Key); i += 8) {
            uint64_t x, y;
            memcpy(&x, p + i, 8);
            memcpy(&y, q + i, 8);
            if (x != y) return false;
        }
        return true;
    }
    Graph *find(const Key &key) {
        for (auto &g : graphs)
            if (same(g.key, key)) return &g;
        return nullptr;
    }
    Graph *add(Graph &&fresh) {
        captures += 1;
        if (graphs.size() < capacity) {
            graphs.push_back(std::move(fresh));
            return &graphs.back();
        }
        Graph &victim = graphs[next];
        next = (next + 1) % graphs.size();
        cudaGraphExecDestroy(victim.exec);
        victim = std::move(fresh);
        return &victim;
    }
    void clear() {
        for (auto &g : graphs) cudaGraphExecDestroy(g.exec);
        graphs.clear();
        next = 0;
    }
};

#ifndef DOCKAUV_STEP_GRAPHS
#define DOCKAUV_STEP_GRAPHS 96     // cached step graphs per handle (a trainer alternates between a few tensors; bench.py's pool: 64)
#endif

struct DockauvHandle {
    DockauvParams params;
    int64_t n_envs = 0;
    int device = 0;
    int n_obs = 0;
    size_t esz = 0;                // bytes of one real: 8 (f64 handle) or 4 (f32)
    bool bound = false;
    KParams<double> kd;            // only the one of the handle's precision is filled and read (with_k)
    KParams<float> kf;
    void *ray_tab = nullptr;
    PipeBuffers pipe;              // pipeline layout: per-env records, float obstacle records and rows, work lists + counters
    void *pipe_buf = nullptr;
    double *stats = nullptr;
    int64_t launches = 0;
    bool timing = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool ev_valid = false;
    cudaEvent_t marks[kMaxStepLaunches + 1] = {};   // per-launch marks of the multi-launch layouts (timing enabled)
    int n_marks = 0;
    // host pipeline
    cudaStream_t hs[kHostStreams] = {nullptr, nullptr, nullptr};
    cudaEvent_t hev[kHostStreams] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr;   // device step in parts on the internal streams (see step_parts)
    void *st_actions = nullptr;
    size_t st_actions_bytes = 0;
    float *st_obs = nullptr;
    void *st_reward = nullptr;
    uint8_t *st_done = nullptr, *st_cond = nullptr;
    // a rollout's arguments (rollout_issue), which are also the key of its graph
    struct RolloutKey {
        DockauvPolicy pol;             // zero for an open-loop rollout
        const void *input;             // open loop: the actions [T][N][n_u]; closed loop: obs0 [N][n_obs]
        DockauvRolloutOut out;
        DockauvPolicyOut pout;         // zero for an open-loop rollout
        DockauvSquashedActor act;      // ring collection only (dockauv_replay_collect), else zero
        DockauvReplayRing ring;        // ring collection only: the ring the steps write into
        int64_t n_slots, start_slot;   // ring collection only: S and s0
        int64_t n_steps, action_dtype, auto_reset;
        uint64_t seed;
    };
    // open-loop rollout graphs (dockauv_rollout): one captured launch sequence, re-captured when the key changes
    GraphCache<RolloutKey> rg{1};
    // closed-loop rollout graphs (dockauv_rollout_policy): a trainer alternates a training and an evaluation rollout
    GraphCache<RolloutKey> pg{4};
    // ring collection graphs (dockauv_replay_collect): a training collection, an evaluation and a few start slots
    GraphCache<RolloutKey> cg{4};
    float *pol_actions = nullptr;  // f32[N][n_u]: the policy's clipped actions, read by the step (allocated on first use)
    // step graph cache: the launch sequence of ONE dockauv_step (launches of both halves, fork / join events) captured per
    // set of pointers and replayed; trainers alternate between a handful of action / output tensors
    struct StepKey {
        const void *actions, *noise;
        DockauvStepOut out;
        int64_t action_dtype, auto_reset;
        uint64_t seed;
    };
    GraphCache<StepKey> sg{DOCKAUV_STEP_GRAPHS};
    bool sg_enabled = true;
    std::vector<int64_t> last_begins;     // first env of every range the most recent device step stepped (their list counters)
    DockauvBuffers bound_bufs = {};
    // episode taps (dockauv_set_taps): two K-env shadows of the tapped envs, stepped on a side stream
    struct Taps {
        int n = 0;
        int64_t capacity = 0;
        DockauvTapBuffers ring = {};
        void *mem = nullptr;           // everything below that is a device pointer lives in this one allocation
        DockauvBuffers shadow = {};    // stepped by the real step's layout: outputs and post-step state (K-env SoA)
        DockauvBuffers dshadow = {};   // stepped by the single-launch kernel with debug outputs
        void *actions = nullptr, *noise = nullptr;
        DockauvStepOut out = {};       // obs, reward, done, cond_bits of `shadow`
        DockauvStepOut dout = {};      // the same of `dshadow` (not recorded)
        DockauvDebugOut dbg = {};      // ray_dist, reward_arr, nu_c, state_dot of `dshadow`
        // pipeline layout: the shadow's own pipeline buffers for K envs (pipe_buf null for the other layouts)
        PipeBuffers pipe;
        void *pipe_buf = nullptr;
        double *stats = nullptr;       // DOCKAUV_STAT_COPIES replicas nobody reads: the public statistics stay the real step's
        int64_t *ids = nullptr;
        unsigned int *sync = nullptr;
        TapRow *gather_rows = nullptr, *commit_rows = nullptr;
        int n_gather = 0, n_commit = 0;
        cudaStream_t st = nullptr, dst = nullptr;      // output shadow + commit; debug shadow (the two run side by side)
        cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_dbg = nullptr;
    } tap;
    // scenario bank (dockauv_set_scenario_bank): the caller's table as last accepted (rows == nullptr: none), and the
    // validation kernel's result word
    DockauvScenarioBank bank = {};
    unsigned long long *bank_check = nullptr;
};

static int pooled_dim(int n, int b) { return (n + b - 1) / b; }

static void drop_graphs(DockauvHandle *h) {      // captured launch sequences hold the old pointers / seed
    h->rg.clear();
    h->sg.clear();
    h->pg.clear();
    h->cg.clear();
}

// f(k) with the handle's KParams in its precision: the one place that chooses between kd and kf
template <typename F>
static auto with_k(DockauvHandle *h, F &&f) {
    return h->params.precision == DOCKAUV_F64 ? f(h->kd) : f(h->kf);
}

extern "C" int dockauv_abi_version(void) { return DOCKAUV_ABI_VERSION; }
extern "C" const char *dockauv_last_error(void) { return g_err; }
extern "C" size_t dockauv_sizeof_params(void) { return sizeof(DockauvParams); }

extern "C" int dockauv_n_obs(const DockauvParams *p) {
    if (!p || p->block_reduce <= 0) return DOCKAUV_EINVAL;
    return 16 + pooled_dim(p->n_vert, p->block_reduce) * pooled_dim(p->n_horiz, p->block_reduce);
}

template <typename T>
static void fill_kparams(const DockauvParams &s, int64_t n_envs, KParams<T> &k) {
    memset(&k, 0, sizeof(k));
    k.n_envs = n_envs;
    k.env_begin = 0;
    k.env_end = n_envs;
    k.n_u = s.n_u;
    k.n_caps = s.n_capsules;
    k.n_sph = s.n_spheres;
    k.n_synth_sph = s.n_synthetic_spheres;
    k.scenario = s.scenario;
    k.max_timesteps = s.max_timesteps;
    k.reward_set = s.reward_set;
    k.n_rays = s.n_rays;
    k.n_vert = s.n_vert;
    k.n_horiz = s.n_horiz;
    k.block = s.block_reduce;
    k.n_hr = pooled_dim(s.n_horiz, s.block_reduce);
    k.n_rr = pooled_dim(s.n_vert, s.block_reduce) * k.n_hr;
    k.n_obs = 16 + k.n_rr;
    k.action_factor_is_scalar = s.action_factor_is_scalar;
    k.seed = s.seed;
    k.env_id0 = s.env_id0;
    k.m = (T)s.m;
    for (int i = 0; i < 3; i++) k.r_G[i] = (T)s.r_G[i];
    for (int i = 0; i < 9; i++) k.I_b[i] = (T)s.I_b[i];
    for (int i = 0; i < 6; i++) k.MA[i] = (T)s.MA_diag[i];
    for (int i = 0; i < 36; i++) k.M_inv[i] = (T)s.M_inv[i];
    for (int i = 0; i < 10; i++) {
        k.D_lin[i] = (T)s.D_lin[i];
        k.D_quad[i] = (T)s.D_quad[i];
        k.D_lift[i] = (T)s.D_lift[i];
    }
    k.G_WB = (T)s.G_WB;
    for (int i = 0; i < 3; i++) k.G_r[i] = (T)s.G_r[i];
    for (int i = 0; i < 6 * DOCKAUV_MAX_U; i++) k.B[i] = (T)s.B[i];
    for (int i = 0; i < 4; i++) k.lauv_B[i] = (T)s.lauv_B[i];
    for (int i = 0; i < DOCKAUV_MAX_U; i++) {
        k.u_lo[i] = (T)s.u_lo[i];
        k.u_span[i] = (T)(s.u_hi[i] - s.u_lo[i]);
        k.arf[i] = (T)s.action_reward_factors[i];
        k.arf_f32[i] = (float)s.action_reward_factors[i];
    }
    k.lp_alpha = (T)s.lp_alpha;
    k.h = (T)s.h;
    k.safety_radius = (T)s.safety_radius;
    k.max_dist_from_goal = (T)s.max_dist_from_goal;
    k.max_attitude = (T)s.max_attitude;
    k.dist_goal_reached_tol = (T)s.dist_goal_reached_tol;
    k.u_max = (T)s.u_max; k.v_max = (T)s.v_max; k.w_max = (T)s.w_max;
    k.p_max = (T)s.p_max; k.q_max = (T)s.q_max; k.r_max = (T)s.r_max;
    k.inv_u_max = (T)(1.0 / s.u_max); k.inv_v_max = (T)(1.0 / s.v_max); k.inv_w_max = (T)(1.0 / s.w_max);
    k.inv_p_max = (T)(1.0 / s.p_max); k.inv_q_max = (T)(1.0 / s.q_max); k.inv_r_max = (T)(1.0 / s.r_max);
    k.inv_max_attitude = (T)(1.0 / s.max_attitude);
    k.log_den_obs = (T)std::log(s.dist_goal_reached_tol / s.max_dist_from_goal);
    k.log_den_rew = (T)std::log(std::fmax(s.dist_goal_reached_tol, 0.001) / s.max_dist_from_goal);
    k.inv_max_dist_from_goal = (T)(1.0 / s.max_dist_from_goal);
    k.inv_log_den_obs = (T)(1.0 / std::log(s.dist_goal_reached_tol / s.max_dist_from_goal));
    k.inv_log_den_rew = (T)(1.0 / std::log(std::fmax(s.dist_goal_reached_tol, 0.001) / s.max_dist_from_goal));
    k.w_d = (T)s.w_d; k.w_delta_psi = (T)s.w_delta_psi; k.w_delta_theta = (T)s.w_delta_theta;
    k.w_phi = (T)s.w_phi; k.w_theta = (T)s.w_theta; k.w_Thetadot = (T)s.w_Thetadot; k.w_oa = (T)s.w_oa;
    for (int i = 0; i < 5; i++) k.w_done[i] = (T)s.w_done[i];
    k.cur_mu = (T)s.cur_mu;
    k.cur_sigma = (T)s.cur_sigma;
    k.has_noise = s.cur_sigma > 0.0;
    k.radar_max_dist = (T)s.radar_max_dist;
    double sb = 0.0;
    for (int i = 0; i < s.n_rays; i++) sb += s.beta_oa[i];
    k.sum_beta_oa = (T)sb;
    // bounding pyramid of the ray fan (used by the warp layout's field-of-view cull); a ray with x <= 0 disables it
    double ty = 0.0, tz = 0.0;
    bool fan_ok = true;
    for (int i = 0; i < s.n_rays; i++) {
        const double x = s.rd_b[3 * i];
        if (!(x > 1e-6)) {
            fan_ok = false;
            break;
        }
        ty = std::fmax(ty, std::fabs(s.rd_b[3 * i + 1]) / x);
        tz = std::fmax(tz, std::fabs(s.rd_b[3 * i + 2]) / x);
    }
    if (!fan_ok) ty = tz = 1e30;
    ty *= 1.0 + 1e-9;
    tz *= 1.0 + 1e-9;
    // M_inv with nothing outside the diagonal and [0,4] [4,0] [1,3] [3,1] (centre of gravity offset along z only: both
    // stock vehicles): the kernels then skip the 26 exact zeros of the dense product
    bool sparse = true;
    for (int r = 0; r < 6; r++)
        for (int c = 0; c < 6; c++) {
            const bool allowed = r == c || (r == 0 && c == 4) || (r == 4 && c == 0) || (r == 1 && c == 3) || (r == 3 && c == 1);
            if (!allowed && s.M_inv[6 * r + c] != 0.0) sparse = false;
        }
    // ... and the same structure in C(nu) and G(eta): r_G and the buoyancy lever on the z axis, I_b diagonal
    if (s.r_G[0] != 0.0 || s.r_G[1] != 0.0 || s.G_r[0] != 0.0 || s.G_r[1] != 0.0) sparse = false;
    for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++)
            if (r != c && s.I_b[3 * r + c] != 0.0) sparse = false;
    k.sparse_minv = sparse ? 1 : 0;
    // the cull code works on float records relative to the goal: every coordinate that matters is within
    // max_dist_from_goal + max_dist of it; beyond ~2 km the float rounding would eat the 2 mm slack -> exact culls
    k.cull_exact = (s.max_dist_from_goal + s.radar_max_dist > 2000.0) ? 1 : 0;
    k.fov_ty = (T)ty;
    k.fov_tz = (T)tz;
    k.fov_ny = (T)std::sqrt(1.0 + ty * ty);
    k.fov_nz = (T)std::sqrt(1.0 + tz * tz);
}

extern "C" int dockauv_create(const DockauvParams *p, int64_t n_envs, int device, DockauvHandle **out) {
    if (!p || !out) return fail(DOCKAUV_EINVAL, "null argument");
    *out = nullptr;
    if (p->abi_version != DOCKAUV_ABI_VERSION)
        return fail(DOCKAUV_EINVAL, "ABI version mismatch: caller %d, library %d", p->abi_version, DOCKAUV_ABI_VERSION);
    if (n_envs <= 0) return fail(DOCKAUV_EINVAL, "n_envs must be positive");
    if (p->precision != DOCKAUV_F64 && p->precision != DOCKAUV_F32) return fail(DOCKAUV_EINVAL, "bad precision");
    if (p->vehicle == DOCKAUV_VEHICLE_BLUEROV2) {
        if (p->n_u != 6 && p->n_u != 8) return fail(DOCKAUV_EINVAL, "BlueROV2 needs n_u = 6 (joystick) or 8 (direct)");
    } else if (p->vehicle == DOCKAUV_VEHICLE_LAUV) {
        if (p->n_u != 3) return fail(DOCKAUV_EINVAL, "LAUV needs n_u = 3");
    } else {
        return fail(DOCKAUV_EINVAL, "unknown vehicle %d", p->vehicle);
    }
    if (p->n_capsules < 0 || p->n_capsules > DOCKAUV_MAX_CAPSULES || p->n_spheres < 0 ||
        p->n_spheres > DOCKAUV_MAX_SPHERES)
        return fail(DOCKAUV_EINVAL, "obstacle counts out of range");
    if (p->n_rays <= 0 || p->n_rays > DOCKAUV_MAX_RAYS || p->n_rays != p->n_vert * p->n_horiz || p->block_reduce <= 0)
        return fail(DOCKAUV_EINVAL, "bad radar geometry (n_rays=%d, %d x %d, block %d)", p->n_rays, p->n_vert,
                    p->n_horiz, p->block_reduce);
    if (p->n_synthetic_spheres < 0 || p->n_synthetic_spheres > p->n_spheres)
        return fail(DOCKAUV_EINVAL, "n_synthetic_spheres must be in 0..n_spheres");
    if (!(p->h > 0.0)) return fail(DOCKAUV_EINVAL, "t_step_size must be positive");
    if (p->max_timesteps <= 0) return fail(DOCKAUV_EINVAL, "max_timesteps must be positive");
    if (!(p->u_max > 0.0) || !(p->v_max > 0.0) || !(p->w_max > 0.0) || !(p->p_max > 0.0) || !(p->q_max > 0.0) ||
        !(p->r_max > 0.0) || !(p->max_attitude > 0.0))
        return fail(DOCKAUV_EINVAL, "u_max .. r_max and max_attitude must be positive (they normalise the observation)");
    if (!(p->max_dist_from_goal > 0.0) || !(p->dist_goal_reached_tol > 0.0) || !(p->radar_max_dist > 0.0))
        return fail(DOCKAUV_EINVAL, "max_dist_from_goal, dist_goal_reached_tol and the radar's max_dist must be positive");
    if (p->reward_set != 1 && p->reward_set != 2) return fail(DOCKAUV_EINVAL, "reward_set must be 1 or 2");
    if (p->scenario < 0 || p->scenario > DOCKAUV_SCN_OBSTACLES_NOCAP) return fail(DOCKAUV_EINVAL, "bad scenario");
    if (p->layout != DOCKAUV_LAYOUT_AUTO && p->layout != DOCKAUV_LAYOUT_THREAD_PER_ENV && p->layout != DOCKAUV_LAYOUT_WARP_RAYS &&
        p->layout != DOCKAUV_LAYOUT_PIPELINE)
        return fail(DOCKAUV_EINVAL, "unknown layout %d", p->layout);
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0)
        return fail(DOCKAUV_ECUDA, "no usable CUDA device (%s); this library has no CPU fallback",
                    cudaGetErrorString(e));
    if (device < 0 || device >= n_dev) return fail(DOCKAUV_EINVAL, "device %d out of range (0..%d)", device, n_dev - 1);
    DeviceGuard guard(device);
    DockauvHandle *h = new (std::nothrow) DockauvHandle();
    if (!h) return fail(DOCKAUV_EINVAL, "out of host memory");
    h->params = *p;
    h->n_envs = n_envs;
    h->device = device;
    h->n_obs = dockauv_n_obs(p);
    h->esz = with_k(h, [](auto &k) { return sizeof(k.m); });
    // ray table in global memory: rd_b[3][n_rays] then beta_oa[n_rays], in the handle's precision
    const int n = p->n_rays;
    std::vector<char> tab(h->esz * 4 * n);
    with_k(h, [&](auto &k) {
        fill_kparams(*p, n_envs, k);
        for (int i = 0; i < n; i++)
            for (int c = 0; c < 4; c++)
                ((decltype(k.m) *)tab.data())[c * n + i] = (decltype(k.m))(c < 3 ? p->rd_b[3 * i + c] : p->beta_oa[i]);
    });
    cudaError_t e1 = cudaMalloc(&h->ray_tab, tab.size());
    if (e1 == cudaSuccess) e1 = cudaMemcpy(h->ray_tab, tab.data(), tab.size(), cudaMemcpyHostToDevice);
    if (e1 == cudaSuccess) e1 = cudaMalloc((void **)&h->stats, kStatsBytes);
    if (e1 == cudaSuccess) e1 = cudaMemset(h->stats, 0, kStatsBytes);
    if (e1 != cudaSuccess) {
        dockauv_destroy(h);
        return fail(DOCKAUV_ECUDA, "device allocation failed: %s", cudaGetErrorString(e1));
    }
    with_k(h, [&](auto &k) {
        k.ray_tab = (decltype(k.ray_tab))h->ray_tab;
        k.stats = h->stats;
    });
    if (p->layout == DOCKAUV_LAYOUT_PIPELINE || p->layout == DOCKAUV_LAYOUT_AUTO) {
        h->pipe = pipe_buffers(n_envs, h->esz, p->n_capsules, p->n_spheres);
        cudaError_t e2 = cudaMalloc(&h->pipe_buf, h->pipe.bytes);
        if (e2 == cudaSuccess) e2 = cudaMemset(h->pipe_buf, 0, h->pipe.bytes);
        // list counters start all ones (any start works while the words of a block are equal): the first step wraps them
        if (e2 == cudaSuccess) e2 = cudaMemset((char *)h->pipe_buf + h->pipe.counters, 0xff, 4 * h->pipe.n_counters);
        if (e2 != cudaSuccess) {
            dockauv_destroy(h);
            return fail(DOCKAUV_ECUDA, "device allocation of the pipeline buffers failed: %s", cudaGetErrorString(e2));
        }
        int sms = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        with_k(h, [&](auto &k) {
            point_pipe(k, h->pipe, h->pipe_buf);
            k.sm_count = sms;
            k.tpe_rays = (p->block_reduce == 2 && k.n_rr <= 64) ? 1 : 0;
        });
    }
    *out = h;
    return DOCKAUV_OK;
}

extern "C" int dockauv_destroy(DockauvHandle *h) {
    if (!h) return DOCKAUV_OK;
    DeviceGuard guard(h->device);
    cudaDeviceSynchronize();
    if (h->ray_tab) cudaFree(h->ray_tab);
    if (h->pipe_buf) cudaFree(h->pipe_buf);
    if (h->stats) cudaFree(h->stats);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    for (cudaEvent_t m : h->marks)
        if (m) cudaEventDestroy(m);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    for (int s = 0; s < kHostStreams; s++) {
        if (h->hs[s]) cudaStreamDestroy(h->hs[s]);
        if (h->hev[s]) cudaEventDestroy(h->hev[s]);
    }
    if (h->st_actions) cudaFree(h->st_actions);
    if (h->st_obs) cudaFree(h->st_obs);
    if (h->st_reward) cudaFree(h->st_reward);
    if (h->st_done) cudaFree(h->st_done);
    if (h->st_cond) cudaFree(h->st_cond);
    if (h->tap.mem) cudaFree(h->tap.mem);
    if (h->tap.st) cudaStreamDestroy(h->tap.st);
    if (h->tap.ev_fork) cudaEventDestroy(h->tap.ev_fork);
    if (h->tap.ev_join) cudaEventDestroy(h->tap.ev_join);
    if (h->tap.dst) cudaStreamDestroy(h->tap.dst);
    if (h->tap.ev_dbg) cudaEventDestroy(h->tap.ev_dbg);
    if (h->bank_check) cudaFree(h->bank_check);
    if (h->pol_actions) cudaFree(h->pol_actions);
    drop_graphs(h);
    delete h;
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- episode taps: row tables
// The gather copies the pre-step rows of the tapped envs from the bound buffers into both shadows and the ring's pre_*
// fields; the commit copies the shadows' post-step rows into the ring's post-step fields.  One TapRow per component row.
static int build_tap_rows(DockauvHandle *h) {
    auto &tp = h->tap;
    const DockauvBuffers &b = h->bound_bufs;
    const DockauvTapBuffers &r = tp.ring;
    const int64_t N = h->n_envs, K = tp.n;
    const int esz = (int)h->esz;
    const int nu = h->params.n_u, nc = h->params.n_capsules, ns = h->params.n_spheres;
    const int n_scene = 4 + 7 * nc + 4 * ns, n_obs = h->n_obs, n_rays = h->params.n_rays;
    std::vector<TapRow> g, c;
    // one gathered row: component `comp` of a bound buffer (env-indexed) -> the same component of both shadows, and row
    // `ring_row` of a ring field with `ring_rows` rows per slot
    auto gather = [&](const void *src, void *shadow, void *dshadow, int comp, int e, void *ring, int ring_row, int ring_rows) {
        TapRow t;
        t.src = (const char *)src + (int64_t)comp * N * e;
        t.dst = (char *)shadow + (int64_t)comp * K * e;
        t.dst2 = dshadow ? (char *)dshadow + (int64_t)comp * K * e : nullptr;
        t.ring = ring ? (char *)ring + (int64_t)ring_row * K * e : nullptr;
        t.ring_slot = (int64_t)ring_rows * K * e;
        t.esz = e;
        t.src_step = t.dst_step = e;
        t.src_by_id = 1;
        g.push_back(t);
    };
    for (int k = 0; k < 12; k++) gather(b.state, tp.shadow.state, tp.dshadow.state, k, esz, r.pre_state, k, 12);
    for (int k = 0; k < nu; k++) gather(b.u_prev, tp.shadow.u_prev, tp.dshadow.u_prev, k, esz, nullptr, 0, 0);
    for (int k = 0; k < 3; k++) gather(b.goal, tp.shadow.goal, tp.dshadow.goal, k, esz, r.pre_scene, k, n_scene);
    gather(b.heading_goal, tp.shadow.heading_goal, tp.dshadow.heading_goal, 0, esz, r.pre_scene, 3, n_scene);
    for (int k = 0; k < 5; k++) gather(b.current, tp.shadow.current, tp.dshadow.current, k, esz, r.pre_current, k, 5);
    for (int k = 0; k < 7 * nc; k++) gather(b.capsules, tp.shadow.capsules, tp.dshadow.capsules, k, esz, r.pre_scene, 4 + k, n_scene);
    for (int k = 0; k < 4 * ns; k++) gather(b.spheres, tp.shadow.spheres, tp.dshadow.spheres, k, esz, r.pre_scene, 4 + 7 * nc + k, n_scene);
    gather(b.ep_return, tp.shadow.ep_return, tp.dshadow.ep_return, 0, esz, r.pre_ep_return, 0, 1);
    gather(b.t_steps, tp.shadow.t_steps, tp.dshadow.t_steps, 0, 4, r.pre_t_steps, 0, 1);
    gather(b.episode, tp.shadow.episode, tp.dshadow.episode, 0, 4, r.pre_episode, 0, 1);
    with_k(h, [&](auto &real) {
        auto shadow = real;
        point_pipe(shadow, tp.pipe, tp.pipe_buf);
        // the real step's float obstacle records (pipeline layout): the shadow culls exactly what the real step culls
        if (shadow.obsf)
            for (int k = 0; k < real.n_obsf; k++) gather(real.obsf, shadow.obsf, nullptr, k, 16, nullptr, 0, 0);
        // and its obstacle rows (env-major: 16-byte piece j of every tapped env's rows, one env's rows apart)
        if (shadow.obsd) {
            const int row_bytes = 8 * esz * (nc + ns);
            for (int j = 0; j < row_bytes / 16; j++) {
                TapRow t;
                t.src = (const char *)real.obsd + 16 * j;
                t.dst = (char *)shadow.obsd + 16 * j;
                t.dst2 = nullptr;
                t.ring = nullptr;
                t.ring_slot = 0;
                t.esz = 16;
                t.src_step = t.dst_step = row_bytes;
                t.src_by_id = 1;
                g.push_back(t);
            }
        }
    });
    // one committed row: row `comp` of a shadow field (tap-indexed, `step` bytes apart) -> row `comp` of a ring field
    auto commit = [&](const void *src, void *ring, int comp, int e, int rows, int step) {
        TapRow t;
        t.src = (const char *)src + (int64_t)comp * (step == e ? K * e : e);
        t.dst = t.dst2 = nullptr;
        t.ring = (char *)ring + (int64_t)comp * (step == e ? K * e : e);
        t.ring_slot = (int64_t)rows * K * e;
        t.esz = e;
        t.src_step = t.dst_step = step;
        t.src_by_id = 0;
        c.push_back(t);
    };
    for (int k = 0; k < 12; k++) commit(tp.shadow.state, r.state, k, esz, 12, esz);
    for (int k = 0; k < nu; k++) commit(tp.shadow.u_prev, r.u, k, esz, nu, esz);
    for (int k = 0; k < 12; k++) commit(tp.dbg.state_dot, r.state_dot, k, esz, 12, esz);
    for (int k = 0; k < 3; k++) commit(tp.dbg.nu_c, r.nu_c, k, esz, 3, esz);
    for (int k = 0; k < n_rays; k++) commit(tp.dbg.ray_dist, r.ray_dist, k, esz, n_rays, esz);
    for (int k = 0; k < 13; k++) commit(tp.dbg.reward_arr, r.reward_arr, k, esz, 13, esz);
    commit(tp.out.reward, r.reward, 0, esz, 1, esz);
    commit(tp.out.done, r.done, 0, 1, 1, 1);
    commit(tp.out.cond_bits, r.cond_bits, 0, 1, 1, 1);
    // observation rows are tap-major ([K][n_obs] in the shadow, [S][K][n_obs] in the ring): column k of every row
    for (int k = 0; k < n_obs; k++) commit(tp.out.obs, r.obs, k, 4, n_obs, 4 * n_obs);
    if ((int)g.size() != tp.n_gather || (int)c.size() != tp.n_commit)
        return fail(DOCKAUV_EINVAL, "internal: tap row tables have %zu / %zu rows, %d / %d reserved", g.size(), c.size(),
                    tp.n_gather, tp.n_commit);
    DeviceGuard guard(h->device);
    CUDA_TRY(cudaMemcpy(tp.gather_rows, g.data(), sizeof(TapRow) * g.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(tp.commit_rows, c.data(), sizeof(TapRow) * c.size(), cudaMemcpyHostToDevice));
    return DOCKAUV_OK;
}

template <typename T>
static void bind_k(KParams<T> &k, const DockauvBuffers &b) {
    k.state = (T *)b.state;
    k.u_prev = (T *)b.u_prev;
    k.goal = (T *)b.goal;
    k.heading_goal = (T *)b.heading_goal;
    k.current = (T *)b.current;
    k.capsules = (T *)b.capsules;
    k.spheres = (T *)b.spheres;
    k.ep_return = (T *)b.ep_return;
    k.t_steps = b.t_steps;
    k.episode = b.episode;
}

extern "C" int dockauv_bind(DockauvHandle *h, const DockauvBuffers *b) {
    if (!h || !b) return fail(DOCKAUV_EINVAL, "null argument");
    if (!b->state || !b->u_prev || !b->goal || !b->heading_goal || !b->current || !b->ep_return || !b->t_steps ||
        !b->episode)
        return fail(DOCKAUV_EINVAL, "a required state buffer is null");
    if ((h->params.n_capsules > 0 && !b->capsules) || (h->params.n_spheres > 0 && !b->spheres))
        return fail(DOCKAUV_EINVAL, "obstacle buffer is null but the handle has obstacles");
    with_k(h, [&](auto &k) { bind_k(k, *b); });
    h->bound_bufs = *b;
    h->bound = true;
    if (h->tap.n > 0) {
        const int rc = build_tap_rows(h);
        if (rc != DOCKAUV_OK) return rc;
    }
    {   // float obstacle records of whatever the buffers hold now (later writers: dockauv_reset, dockauv_refresh_obstacles)
        DeviceGuard guard(h->device);
        CUDA_TRY(with_k(h, [](auto &k) { return launch_refresh_obstacles(k, (cudaStream_t)0); }));
        CUDA_TRY(cudaStreamSynchronize((cudaStream_t)0));
    }
    drop_graphs(h);
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- launch dispatch
static bool scenario_has_current(int scn) {
    return scn == DOCKAUV_SCN_SIMPLE_CURRENT || scn == DOCKAUV_SCN_CAPSULE_CURRENT || scn == DOCKAUV_SCN_OBSTACLES_CURRENT;
}

static int resolve_layout(const DockauvHandle *h) {
    int layout = h->params.layout;
    // measured on B200 (1M envs of C4): fused kernel 0.91 ms, three-launch pipeline 0.5 ms; without obstacles the pipeline
    // is dynamics + finish only; thread-per-env stays as the independently written cross-check
    if (layout == DOCKAUV_LAYOUT_AUTO) layout = DOCKAUV_LAYOUT_PIPELINE;
    return layout;
}

// the current is "on" when the scenario spawns one, the caller asked for it, or noise is configured
static bool current_on(const DockauvHandle *h) {
    return scenario_has_current(h->params.scenario) || h->params.force_current != 0 || h->params.cur_sigma > 0.0;
}

template <typename T>
static void set_io(KParams<T> &k, const void *actions, bool act_f32, const void *noise, const DockauvStepOut &o,
                   const DockauvDebugOut *d, int auto_reset) {
    k.actions = actions;
    k.noise = (const T *)noise;
    k.obs = o.obs;
    k.terminal_obs = o.terminal_obs;
    k.reward = (T *)o.reward;
    k.ep_return_out = (T *)o.ep_return_out;
    k.done = o.done;
    k.cond_bits = o.cond_bits;
    k.ep_len_out = o.ep_len_out;
    k.delta_d_out = (T *)o.delta_d_out;
    k.auto_reset = auto_reset ? 1 : 0;
    k.act_f32 = act_f32 ? 1 : 0;
    k.dbg_ray_dist = d ? (T *)d->ray_dist : nullptr;
    k.dbg_reward_arr = d ? (T *)d->reward_arr : nullptr;
    k.dbg_euler_dot = d ? (T *)d->euler_dot : nullptr;
    k.dbg_nu_c = d ? (T *)d->nu_c : nullptr;
    k.dbg_nav = d ? (T *)d->nav : nullptr;
    k.dbg_obs = d ? (T *)d->obs_f64 : nullptr;
    k.dbg_state_dot = d ? (T *)d->state_dot : nullptr;
}

static int step_range(DockauvHandle *h, const void *actions, int action_dtype, const void *noise,
                      const DockauvStepOut *out, const DockauvDebugOut *dbg, int auto_reset, int64_t begin,
                      int64_t end, cudaStream_t st, bool with_marks = false) {
    int n = 0;
    const cudaError_t e = with_k(h, [&](auto &kh) {
        auto k = kh;
        set_io(k, actions, action_dtype == DOCKAUV_ACT_F32, noise, *out, dbg, auto_reset);
        k.env_begin = begin;
        k.env_end = end;
        k.has_current = current_on(h);
        return launch_step(k, h->params.vehicle, resolve_layout(h), st, &n, with_marks ? h->marks : nullptr,
                           with_marks ? &h->n_marks : nullptr);
    });
    if (e != cudaSuccess) return fail(DOCKAUV_ECUDA, "step kernel launch failed: %s", cudaGetErrorString(e));
    h->launches += n;
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- episode taps: launches
// With taps set, every step issues, besides its own launches, the gather on the caller's stream before the step's first
// launch (the only serial addition), then, on two tap streams forked after it, two shadow steps over K-env copies of the
// tapped envs side by side, and the commit once both are done.  The first shadow is stepped by the handle's own layout with the real step's inputs (state,
// float obstacle records, actions, noise), so its outputs and post-step state are those of the real step in either
// precision; the second by the single-launch kernel with debug outputs (the fields only that kernel has).  Neither
// touches a real env, output or statistic.  tap_end joins the tap stream back, so the next step's gather, which rewrites
// the shadows, is ordered after this step's commit.
static TapLaunch tap_launch(const DockauvHandle *h, bool gather, const void *actions, int action_dtype, const void *noise) {
    const auto &tp = h->tap;
    TapLaunch t;
    memset(&t, 0, sizeof(t));
    t.rows = gather ? tp.gather_rows : tp.commit_rows;
    t.n_rows = gather ? tp.n_gather : tp.n_commit;
    t.n_taps = tp.n;
    t.ids = tp.ids;
    t.count = tp.ring.count;
    t.capacity = tp.capacity;
    t.sync = tp.sync;
    t.actions = actions;
    t.act_f32 = action_dtype == DOCKAUV_ACT_F32 ? 1 : 0;
    t.n_u = h->params.n_u;
    t.shadow_actions = tp.actions;
    t.noise = noise;
    t.shadow_noise = tp.noise;
    return t;
}

// *n_launches receives the launches enqueued: gather, the shadow's step, the debug shadow's step, commit
template <typename T>
static cudaError_t tap_issue(DockauvHandle *h, const KParams<T> &real, const void *actions, int action_dtype,
                             const void *noise, cudaStream_t st, int *n_launches) {
    auto &tp = h->tap;
    cudaError_t e = launch_tap_gather<T>(real, tap_launch(h, true, actions, action_dtype, noise), st);
    if (e == cudaSuccess) e = cudaEventRecord(tp.ev_fork, st);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(tp.st, tp.ev_fork, 0);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(tp.dst, tp.ev_fork, 0);
    if (e != cudaSuccess) return e;
    // the shadow: the real step's own layout, so its outputs and post-step state are those of the real step
    KParams<T> k = real;
    k.n_envs = tp.n;
    k.env_begin = 0;
    k.env_end = tp.n;
    bind_k<T>(k, tp.shadow);
    set_io<T>(k, tp.actions, action_dtype == DOCKAUV_ACT_F32, tp.noise, tp.out, nullptr, 0);
    k.has_current = current_on(h);
    k.stats = tp.stats;
    k.bank_rows = nullptr;          // the shadows never reset (no auto-reset), and their env count is not the bank's N
    k.bank_cdf = nullptr;
    k.bank_row_of_env = nullptr;
    point_pipe(k, tp.pipe, tp.pipe_buf);
    int n_shadow = 0, n_dbg = 0;
    e = launch_step<T>(k, h->params.vehicle, resolve_layout(h), tp.st, &n_shadow);
    if (e != cudaSuccess) return e;
    // the debug shadow: the single-launch kernel with debug outputs (state_dot, nu_c, ray distances, reward terms)
    KParams<T> d = k;
    bind_k<T>(d, tp.dshadow);
    set_io<T>(d, tp.actions, action_dtype == DOCKAUV_ACT_F32, tp.noise, tp.dout, &tp.dbg, 0);
    point_pipe(d, tp.pipe, nullptr);
    e = launch_step<T>(d, h->params.vehicle, DOCKAUV_LAYOUT_WARP_RAYS, tp.dst, &n_dbg);
    if (e == cudaSuccess) e = cudaEventRecord(tp.ev_dbg, tp.dst);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(tp.st, tp.ev_dbg, 0);
    if (e == cudaSuccess) e = launch_tap_commit<T>(real, tap_launch(h, false, actions, action_dtype, noise), tp.st);
    if (e == cudaSuccess) e = cudaEventRecord(tp.ev_join, tp.st);
    *n_launches = 2 + n_shadow + n_dbg;
    return e;
}

static int tap_begin(DockauvHandle *h, const void *actions, int action_dtype, const void *noise, cudaStream_t st) {
    if (h->tap.n == 0) return DOCKAUV_OK;
    int n = 0;
    const cudaError_t e = with_k(h, [&](auto &k) { return tap_issue(h, k, actions, action_dtype, noise, st, &n); });
    if (e != cudaSuccess) return fail(DOCKAUV_ECUDA, "tap launch failed: %s", cudaGetErrorString(e));
    h->launches += n;
    return DOCKAUV_OK;
}

static int tap_end(DockauvHandle *h, cudaStream_t st) {
    if (h->tap.n > 0) CUDA_TRY(cudaStreamWaitEvent(st, h->tap.ev_join, 0));
    return DOCKAUV_OK;
}

extern "C" int dockauv_set_seed(DockauvHandle *h, uint64_t seed) {
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    h->params.seed = seed;
    with_k(h, [&](auto &k) { k.seed = seed; });
    return DOCKAUV_OK;
}

extern "C" int dockauv_reset(DockauvHandle *h, const uint8_t *mask_dev, void *stream) {
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    if (!h->bound) return fail(DOCKAUV_ESTATE, "dockauv_bind must be called before dockauv_reset");
    DeviceGuard guard(h->device);
    CUDA_TRY(with_k(h, [&](auto &k) { return launch_reset(k, mask_dev, (cudaStream_t)stream); }));
    h->launches += 1;
    return DOCKAUV_OK;
}

extern "C" int dockauv_refresh_obstacles(DockauvHandle *h, void *stream) {
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    if (!h->bound) return fail(DOCKAUV_ESTATE, "dockauv_bind must be called before dockauv_refresh_obstacles");
    DeviceGuard guard(h->device);
    return with_k(h, [&](auto &k) {
        if (k.obsf == nullptr) return DOCKAUV_OK;
        CUDA_TRY(launch_refresh_obstacles(k, (cudaStream_t)stream));
        h->launches += 1;
        return DOCKAUV_OK;
    });
}

static int ensure_streams(DockauvHandle *h) {
    for (int s = 0; s < kHostStreams; s++) {
        if (!h->hs[s]) CUDA_TRY(cudaStreamCreateWithFlags(&h->hs[s], cudaStreamNonBlocking));
        if (!h->hev[s]) CUDA_TRY(cudaEventCreateWithFlags(&h->hev[s], cudaEventDisableTiming));
    }
    if (!h->ev_fork) CUDA_TRY(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    return DOCKAUV_OK;
}

#ifndef DOCKAUV_PARTS_MIN_ENVS
#define DOCKAUV_PARTS_MIN_ENVS (1 << 17)   // smallest batch that is stepped in parts (262,144 envs: 0.164 ms in two parts, 0.182 ms in one)
#endif
#ifndef DOCKAUV_STEP_PARTS
#define DOCKAUV_STEP_PARTS 2      // 1 = the whole batch in the caller's stream; at most kHostStreams
#endif
// The whole batch as DOCKAUV_STEP_PARTS parts on internal streams, forked from / joined to the caller's stream by
// events: each launch of one part fills the tail waves of the other parts' launches (a four-launch step has four
// partially filled last waves; in one stream the next launch cannot start before the last CTA of the previous one has
// finished).  Measured at 1M envs: 1 part 0.594 ms, 2 parts 0.566 ms.
static bool steps_in_parts(const DockauvHandle *h) {
    return DOCKAUV_STEP_PARTS > 1 && h->n_envs >= (int64_t)DOCKAUV_PARTS_MIN_ENVS && resolve_layout(h) == DOCKAUV_LAYOUT_PIPELINE &&
           h->params.split_chunk_envs == 0;
}

static bool misaligned16(const void *p) { return (((uintptr_t)p) & 15u) != 0; }

// obs / terminal_obs rows are written in 16-byte pieces when n_obs is a multiple of 4
static int check_rows(const DockauvHandle *h, const float *obs, const float *terminal_obs) {
    if ((h->n_obs & 3) == 0 && ((((uintptr_t)obs) & 15u) != 0 || (((uintptr_t)terminal_obs) & 15u) != 0))
        return fail(DOCKAUV_EINVAL, "obs and terminal_obs must be 16-byte aligned (n_obs = %d is a multiple of 4: rows are "
                                    "written with 128-bit stores)", h->n_obs);
    return DOCKAUV_OK;
}

// Issues issue(begin, end, stream) for every env range of a device step and records the ranges as those of the most
// recent step (their list counters).  The range is the whole batch on the caller's stream, or, for large batches of the
// pipeline layout (unless `whole`), DOCKAUV_STEP_PARTS ranges of a multiple of 4096 envs, each on an internal stream
// forked from / joined to the caller's stream by events.
template <typename F>
static int over_ranges(DockauvHandle *h, bool whole, cudaStream_t st, F &&issue) {
    const int64_t N = h->n_envs;
    h->last_begins.clear();
    if (whole || !steps_in_parts(h)) {
        h->last_begins.push_back(0);
        return issue((int64_t)0, N, st);
    }
    int rc = ensure_streams(h);
    if (rc != DOCKAUV_OK) return rc;
    const int64_t part = (((N + DOCKAUV_STEP_PARTS - 1) / DOCKAUV_STEP_PARTS + 4095) / 4096) * 4096;   // at most PARTS ranges
    CUDA_TRY(cudaEventRecord(h->ev_fork, st));
    int s = 0;
    for (int64_t b = 0; b < N; b += part, s++) {
        h->last_begins.push_back(b);
        CUDA_TRY(cudaStreamWaitEvent(h->hs[s], h->ev_fork, 0));
        rc = issue(b, b + part < N ? b + part : N, h->hs[s]);
        if (rc != DOCKAUV_OK) return rc;
        CUDA_TRY(cudaEventRecord(h->hev[s], h->hs[s]));
        CUDA_TRY(cudaStreamWaitEvent(st, h->hev[s], 0));
    }
    return DOCKAUV_OK;
}

// one batched step on the device: in parts for large batches of the pipeline layout, else one launch group
static int step_device(DockauvHandle *h, const void *actions, int action_dtype, const void *noise,
                       const DockauvStepOut *out, const DockauvDebugOut *dbg, int auto_reset, cudaStream_t st, bool timing) {
    return over_ranges(h, timing || dbg != nullptr, st, [&](int64_t b, int64_t e, cudaStream_t s) {
        return step_range(h, actions, action_dtype, noise, out, dbg, auto_reset, b, e, s, timing);
    });
}

// step_device with the tap branch around it (when taps are set)
static int step_call(DockauvHandle *h, const void *actions, int action_dtype, const void *noise, const DockauvStepOut *out,
                     const DockauvDebugOut *dbg, int auto_reset, cudaStream_t st, bool timing) {
    int rc = tap_begin(h, actions, action_dtype, noise, st);
    if (rc == DOCKAUV_OK) rc = step_device(h, actions, action_dtype, noise, out, dbg, auto_reset, st, timing);
    if (rc == DOCKAUV_OK) rc = tap_end(h, st);
    return rc;
}

// Replays the graph cached under `key`, first capturing what issue(stream) enqueues when there is none: on a private
// stream (the caller's may be the legacy default stream, which cannot be captured).  The captured launches count once
// per replay, and a replay restores the step ranges recorded during the capture.
template <typename Key, typename F>
static int graph_call(DockauvHandle *h, GraphCache<Key> &cache, const Key &key, const char *what, cudaStream_t st,
                      F &&issue) {
    auto *g = cache.find(key);
    if (g == nullptr) {
        typename GraphCache<Key>::Graph fresh;
        fresh.key = key;
        cudaStream_t cs = nullptr;
        CUDA_TRY(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        cudaGraph_t graph = nullptr;
        cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        int rc = DOCKAUV_OK;
        const int64_t before = h->launches;
        if (e == cudaSuccess) {
            rc = issue(cs);
            e = cudaStreamEndCapture(cs, &graph);
        }
        fresh.launches = h->launches - before;
        h->launches = before;       // captured, not launched
        fresh.begins = h->last_begins;
        if (e == cudaSuccess && rc == DOCKAUV_OK) e = cudaGraphInstantiate(&fresh.exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        cudaStreamDestroy(cs);
        if (rc != DOCKAUV_OK) return rc;
        if (e != cudaSuccess) return fail(DOCKAUV_ECUDA, "%s graph capture failed: %s", what, cudaGetErrorString(e));
        g = cache.add(std::move(fresh));
    }
    CUDA_TRY(cudaGraphLaunch(g->exec, st));
    h->launches += g->launches;
    h->last_begins = g->begins;
    return DOCKAUV_OK;
}

extern "C" int dockauv_step(DockauvHandle *h, const void *actions_dev, int action_dtype, const void *noise_dev,
                            const DockauvStepOut *out, const DockauvDebugOut *dbg, int auto_reset, void *stream) {
    if (!h || !actions_dev || !out) return fail(DOCKAUV_EINVAL, "null argument");
    if (!h->bound) return fail(DOCKAUV_ESTATE, "dockauv_bind must be called before dockauv_step");
    if (!out->obs || !out->reward || !out->done) return fail(DOCKAUV_EINVAL, "obs, reward and done outputs are required");
    if (action_dtype != DOCKAUV_ACT_F32 && action_dtype != DOCKAUV_ACT_F64) return fail(DOCKAUV_EINVAL, "bad action dtype");
    if (check_rows(h, out->obs, out->terminal_obs) != DOCKAUV_OK) return DOCKAUV_EINVAL;
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (h->timing) {
        if (!h->ev0) {
            CUDA_TRY(cudaEventCreate(&h->ev0));
            CUDA_TRY(cudaEventCreate(&h->ev1));
            for (cudaEvent_t &m : h->marks) CUDA_TRY(cudaEventCreate(&m));
        }
        CUDA_TRY(cudaEventRecord(h->ev0, st));
    }
    // One dockauv_step as a CUDA graph: the launch sequence (both halves, their fork / join events) is captured once per
    // set of pointers and replayed -- one graph launch instead of six kernel launches and four event operations, and no
    // launch-to-launch gaps on the device (what makes a 65,536-env step 24 us instead of 29).
    if (!h->timing && dbg == nullptr && h->sg_enabled) {
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone) {
            DockauvHandle::StepKey key;
            memset(&key, 0, sizeof(key));
            key.actions = actions_dev;
            key.noise = noise_dev;
            key.out = *out;
            key.action_dtype = action_dtype;
            key.auto_reset = auto_reset;
            key.seed = h->params.seed;
            return graph_call(h, h->sg, key, "step", st, [&](cudaStream_t cs) {
                return step_call(h, actions_dev, action_dtype, noise_dev, out, nullptr, auto_reset, cs, false);
            });
        }
    }
    int rc = step_call(h, actions_dev, action_dtype, noise_dev, out, dbg, auto_reset, st, h->timing);
    if (rc != DOCKAUV_OK) return rc;
    if (h->timing) {
        CUDA_TRY(cudaEventRecord(h->ev1, st));
        h->ev_valid = true;
    }
    return DOCKAUV_OK;
}

extern "C" int dockauv_enable_step_graph(DockauvHandle *h, int enabled) {
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    h->sg_enabled = enabled != 0;
    return DOCKAUV_OK;
}

extern "C" int dockauv_step_graph_captures(DockauvHandle *h, int64_t *n) {
    if (!h || !n) return fail(DOCKAUV_EINVAL, "null argument");
    *n = h->sg.captures;
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- host-buffer step
static int ensure_host_pipeline(DockauvHandle *h, size_t action_bytes) {
    int rc0 = ensure_streams(h);
    if (rc0 != DOCKAUV_OK) return rc0;
    if (h->st_actions_bytes < action_bytes) {
        if (h->st_actions) CUDA_TRY(cudaFree(h->st_actions));
        h->st_actions = nullptr;
        CUDA_TRY(cudaMalloc(&h->st_actions, action_bytes));
        h->st_actions_bytes = action_bytes;
    }
    if (!h->st_obs) CUDA_TRY(cudaMalloc((void **)&h->st_obs, sizeof(float) * h->n_obs * (size_t)h->n_envs));
    if (!h->st_reward) CUDA_TRY(cudaMalloc(&h->st_reward, h->esz * (size_t)h->n_envs));
    if (!h->st_done) CUDA_TRY(cudaMalloc((void **)&h->st_done, (size_t)h->n_envs));
    if (!h->st_cond) CUDA_TRY(cudaMalloc((void **)&h->st_cond, (size_t)h->n_envs));
    return DOCKAUV_OK;
}

extern "C" int dockauv_step_host(DockauvHandle *h, const void *actions_host, int action_dtype, float *obs_host,
                                 void *reward_host, uint8_t *done_host, uint8_t *cond_bits_host, int auto_reset,
                                 const DockauvStepOut *aux) {
    if (!h || !actions_host || !obs_host || !reward_host || !done_host) return fail(DOCKAUV_EINVAL, "null argument");
    if (!h->bound) return fail(DOCKAUV_ESTATE, "dockauv_bind must be called before dockauv_step_host");
    if (h->tap.n > 0)
        return fail(DOCKAUV_ESTATE, "taps are set: they record device-driven steps (dockauv_step, dockauv_rollout); remove "
                                    "them (dockauv_set_taps with n_taps = 0) before dockauv_step_host");
    if (action_dtype != DOCKAUV_ACT_F32 && action_dtype != DOCKAUV_ACT_F64) return fail(DOCKAUV_EINVAL, "bad action dtype");
    DeviceGuard guard(h->device);
    const int64_t N = h->n_envs;
    const size_t asz = (action_dtype == DOCKAUV_ACT_F32 ? 4 : 8) * (size_t)h->params.n_u;
    const size_t esz = h->esz;
    int rc = ensure_host_pipeline(h, asz * (size_t)N);
    if (rc != DOCKAUV_OK) return rc;
    h->last_begins.clear();
    // chunks: multiples of 4096 envs, at most 12 per call so copies of chunk c+1 overlap the kernel of chunk c
    int64_t chunk = (N + DOCKAUV_HOST_CHUNKS - 1) / DOCKAUV_HOST_CHUNKS;
    chunk = ((chunk + 4095) / 4096) * 4096;
    if (chunk < 16384) chunk = 16384;
    DockauvStepOut out;
    memset(&out, 0, sizeof(out));
    out.obs = h->st_obs;
    out.reward = h->st_reward;
    out.done = h->st_done;
    out.cond_bits = h->st_cond;
    if (aux) {
        out.terminal_obs = aux->terminal_obs;
        out.ep_return_out = aux->ep_return_out;
        out.ep_len_out = aux->ep_len_out;
        out.delta_d_out = aux->delta_d_out;
        if (check_rows(h, out.obs, out.terminal_obs) != DOCKAUV_OK) return DOCKAUV_EINVAL;
    }
    // Per chunk: actions in, the step's launches, the observation rows out (the bulk of the bytes, one copy).  The
    // small outputs (reward, done, cond_bits) leave once per group of 2 * kHostStreams consecutive chunks (waiting for a
    // group is one event per stream): 36 small copies per step cost ~0.3 ms of copy-engine overhead on top of the
    // 2.6 ms the bytes need.
    // work issued earlier on the legacy default stream (PyTorch's default current stream: a preceding dockauv_step,
    // reset or set_state) is ordered before the internal streams start; callers on other streams synchronise themselves
    CUDA_TRY(cudaEventRecord(h->ev_fork, (cudaStream_t)0));
    for (int s = 0; s < kHostStreams; s++) CUDA_TRY(cudaStreamWaitEvent(h->hs[s], h->ev_fork, 0));
    int c = 0;
    int64_t group_begin = 0;
    auto flush_small = [&](int64_t gb, int64_t ge, int last_stream) -> int {
        cudaStream_t st = h->hs[last_stream];
        for (int s = 0; s < kHostStreams; s++) {
            if (s == last_stream) continue;
            CUDA_TRY(cudaEventRecord(h->hev[s], h->hs[s]));
            CUDA_TRY(cudaStreamWaitEvent(st, h->hev[s], 0));
        }
        CUDA_TRY(cudaMemcpyAsync((char *)reward_host + esz * gb, (char *)h->st_reward + esz * gb, esz * (ge - gb),
                                 cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(done_host + gb, h->st_done + gb, (size_t)(ge - gb), cudaMemcpyDeviceToHost, st));
        if (cond_bits_host)
            CUDA_TRY(cudaMemcpyAsync(cond_bits_host + gb, h->st_cond + gb, (size_t)(ge - gb), cudaMemcpyDeviceToHost, st));
        return DOCKAUV_OK;
    };
    for (int64_t b = 0; b < N; b += chunk, c++) {
        const int64_t e = b + chunk < N ? b + chunk : N;
        const int si = c % kHostStreams;
        cudaStream_t st = h->hs[si];
        CUDA_TRY(cudaMemcpyAsync((char *)h->st_actions + asz * b, (const char *)actions_host + asz * b, asz * (e - b),
                                 cudaMemcpyHostToDevice, st));
        rc = step_range(h, h->st_actions, action_dtype, nullptr, &out, nullptr, auto_reset, b, e, st);
        if (rc != DOCKAUV_OK) return rc;
        h->last_begins.push_back(b);
        CUDA_TRY(cudaMemcpyAsync(obs_host + (size_t)h->n_obs * b, h->st_obs + (size_t)h->n_obs * b,
                                 sizeof(float) * h->n_obs * (e - b), cudaMemcpyDeviceToHost, st));
        if ((c + 1) % (2 * kHostStreams) == 0 || e == N) {
            rc = flush_small(group_begin, e, si);
            if (rc != DOCKAUV_OK) return rc;
            group_begin = e;
        }
    }
    for (int s = 0; s < kHostStreams; s++) CUDA_TRY(cudaStreamSynchronize(h->hs[s]));
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- policy launch
template <int H, int NU>
static cudaError_t launch_policy_hu(const PolicyLaunch &p, size_t smem, cudaStream_t st) {
    auto kernel = policy_kernel<H, NU>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int dev = 0, sms = 0, per_sm = 0;
    if (e == cudaSuccess) e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // one thread per env; the CTA shrinks (down to one warp) until the range fills every SM with at least one CTA, so a
    // small batch is spread over the whole GPU; persistent CTAs beyond that (each stages the weights once)
    const int64_t n = p.env_end - p.env_begin;
    int threads = 256;
    while (threads > 32 && (n + threads - 1) / threads < sms) threads /= 2;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
    if (e != cudaSuccess) return e;
    const int64_t blocks = std::min<int64_t>((n + threads - 1) / threads, (int64_t)std::max(per_sm, 1) * sms);
    kernel<<<(unsigned)blocks, threads, smem, st>>>(p);
    return cudaGetLastError();
}

template <int H>
static cudaError_t launch_policy_h(const PolicyLaunch &p, int n_u, size_t smem, cudaStream_t st) {
    switch (n_u) {
        case 3: return launch_policy_hu<H, 3>(p, smem, st);     // LAUV
        case 6: return launch_policy_hu<H, 6>(p, smem, st);     // BlueROV2 joystick
        case 8: return launch_policy_hu<H, 8>(p, smem, st);     // BlueROV2 direct
        default: return cudaErrorInvalidValue;
    }
}

// One policy evaluation over envs [b, e): the observations `obs` ([N][n_obs]) -> actions, values, log-probs of one
// rollout row (value_only: values only) and the clipped actions the next step reads.
static int policy_range(DockauvHandle *h, const DockauvPolicy &pol, const float *obs, float *actions, float *values,
                        float *log_probs, bool value_only, int64_t b, int64_t e, cudaStream_t st) {
    PolicyLaunch p;
    memset(&p, 0, sizeof(p));
    for (int k = 0; k < 3; k++) {
        p.pi_w[k] = pol.pi_w[k];
        p.pi_b[k] = pol.pi_b[k];
        p.vf_w[k] = pol.vf_w[k];
        p.vf_b[k] = pol.vf_b[k];
    }
    p.log_std = pol.log_std;
    p.obs = obs;
    p.actions = actions;
    p.act_clipped = h->pol_actions;
    p.values = values;
    p.log_probs = log_probs;
    const int n_u = h->params.n_u;
    for (int k = 0; k < n_u; k++) {      // the float32 bounds of action_space (envs.py), as np.clip sees them
        p.u_lo[k] = (float)h->params.u_lo[k];
        p.u_hi[k] = (float)h->params.u_hi[k];
    }
    p.seed = h->params.seed;
    p.env_id0 = h->params.env_id0;
    p.t_steps = h->bound_bufs.t_steps;
    p.episode = h->bound_bufs.episode;
    p.env_begin = b;
    p.env_end = e;
    p.n_obs = h->n_obs;
    p.deterministic = pol.deterministic != 0;
    p.value_only = value_only ? 1 : 0;
    const size_t smem = policy_smem_bytes(h->n_obs, pol.hidden, n_u);
    cudaError_t err = cudaErrorInvalidValue;
    switch (pol.hidden) {
        case 32: err = launch_policy_h<32>(p, n_u, smem, st); break;
        case 64: err = launch_policy_h<64>(p, n_u, smem, st); break;
        case 96: err = launch_policy_h<96>(p, n_u, smem, st); break;
        case 128: err = launch_policy_h<128>(p, n_u, smem, st); break;
    }
    if (err != cudaSuccess) return fail(DOCKAUV_ECUDA, "policy kernel launch failed: %s", cudaGetErrorString(err));
    h->launches += 1;
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- SAC actor launch
template <int H, int NU>
static cudaError_t launch_sac_actor_hu(const SacActorLaunch &p, size_t smem, cudaStream_t st) {
    auto kernel = sac_actor_kernel<H, NU>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int dev = 0, sms = 0, per_sm = 0;
    if (e == cudaSuccess) e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // a warp per 16-env tile, tiles dealt to the CTAs round robin: a small batch is spread over every SM, persistent
    // CTAs beyond that.  The CTA keeps all its warps even when some get no tile: staging the weights (each CTA reads
    // and converts all of them once) is what a small batch waits for, and it goes as fast as the CTA has threads.
    const int64_t tiles = (p.env_end - p.env_begin + 15) / 16;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 32 * kSacWarps, smem);
    if (e != cudaSuccess) return e;
    const int64_t blocks = std::min<int64_t>(tiles, (int64_t)std::max(per_sm, 1) * sms);
    kernel<<<(unsigned)blocks, 32 * kSacWarps, smem, st>>>(p);
    return cudaGetLastError();
}

template <int H>
static cudaError_t launch_sac_actor_h(const SacActorLaunch &p, int n_u, size_t smem, cudaStream_t st) {
    switch (n_u) {
        case 3: return launch_sac_actor_hu<H, 3>(p, smem, st);     // LAUV
        case 6: return launch_sac_actor_hu<H, 6>(p, smem, st);     // BlueROV2 joystick
        case 8: return launch_sac_actor_hu<H, 8>(p, smem, st);     // BlueROV2 direct
        default: return cudaErrorInvalidValue;
    }
}

// One actor evaluation over envs [b, e): the observations `obs` ([N][n_obs]) -> the squashed actions ([N][n_u]) the
// next step reads
static int actor_range(DockauvHandle *h, const DockauvSquashedActor &act, const float *obs, float *actions, int64_t b,
                       int64_t e, cudaStream_t st) {
    SacActorLaunch p;
    memset(&p, 0, sizeof(p));
    p.w0 = act.w[0];
    p.b0 = act.b[0];
    p.w1 = act.w[1];
    p.b1 = act.b[1];
    p.mu_w = act.mu_w;
    p.mu_b = act.mu_b;
    p.log_std_w = act.log_std_w;
    p.log_std_b = act.log_std_b;
    p.obs = obs;
    p.actions = actions;
    p.t_steps = h->bound_bufs.t_steps;
    p.episode = h->bound_bufs.episode;
    p.seed = h->params.seed;
    p.env_id0 = h->params.env_id0;
    p.env_begin = b;
    p.env_end = e;
    p.n_obs = h->n_obs;
    p.deterministic = act.deterministic != 0;
    const int n_u = h->params.n_u;
    const size_t smem = sac_actor_smem_bytes(h->n_obs, act.hidden, n_u);
    cudaError_t err = cudaErrorInvalidValue;
    switch (act.hidden) {
        case 64: err = launch_sac_actor_h<64>(p, n_u, smem, st); break;
        case 128: err = launch_sac_actor_h<128>(p, n_u, smem, st); break;
        case 256: err = launch_sac_actor_h<256>(p, n_u, smem, st); break;
    }
    if (err != cudaSuccess) return fail(DOCKAUV_ECUDA, "SAC actor kernel launch failed: %s", cudaGetErrorString(err));
    h->launches += 1;
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- stacked rollout
// row t of every output of a stacked rollout
static DockauvStepOut rollout_step_out(const DockauvHandle *h, const DockauvRolloutOut &o, int t) {
    const size_t N = (size_t)h->n_envs, esz = h->esz, orow = (size_t)h->n_obs * N;
    DockauvStepOut so;
    so.obs = o.obs + orow * t;
    so.reward = (char *)o.reward + esz * N * t;
    so.done = o.done + N * t;
    so.cond_bits = o.cond_bits ? o.cond_bits + N * t : nullptr;
    so.terminal_obs = o.terminal_obs ? o.terminal_obs + orow * t : nullptr;
    so.ep_return_out = o.ep_return_out ? (char *)o.ep_return_out + esz * N * t : nullptr;
    so.ep_len_out = o.ep_len_out ? o.ep_len_out + N * t : nullptr;
    so.delta_d_out = o.delta_d_out ? (char *)o.delta_d_out + esz * N * t : nullptr;
    return so;
}

// ring slot t of the replay ring as the outputs of one step: obs of slot t + 1, reward, done and terminal_obs of slot t
static DockauvStepOut ring_step_out(const DockauvHandle *h, const DockauvReplayRing &ring, int S, int slot) {
    const size_t N = (size_t)h->n_envs, orow = (size_t)h->n_obs * N;
    DockauvStepOut so;
    memset(&so, 0, sizeof(so));
    so.obs = (float *)ring.obs + orow * ((slot + 1) % S);
    so.reward = (char *)ring.reward + h->esz * N * slot;
    so.done = (uint8_t *)ring.done + N * slot;
    so.terminal_obs = (float *)ring.terminal_obs + orow * slot;
    return so;
}

// The launches of one rollout.  Open loop (pol and act null): step t reads row t of r.input, the caller's actions.
// Closed loop: before step t a policy launch reads r.input (obs0) for t = 0 and row t - 1 of r.out.obs after that, and
// writes the clipped actions that the step reads from h->pol_actions (r.action_dtype is DOCKAUV_ACT_F32); with
// r.pout.last_values set, one more launch after the last step writes V(row T - 1 of r.out.obs).  Ring collection (act):
// with slot = (s0 + t) % S, before step t an actor launch reads obs[slot] of r.ring and writes actions[slot], which the
// step reads as float32; the step writes obs[slot + 1] and reward, done, terminal_obs of the slot (ring_step_out).
static int rollout_issue(DockauvHandle *h, const DockauvPolicy *pol, const DockauvSquashedActor *act,
                         const DockauvHandle::RolloutKey &r, cudaStream_t st) {
    const size_t N = (size_t)h->n_envs, n_u = (size_t)h->params.n_u;
    const int n_steps = (int)r.n_steps, action_dtype = (int)r.action_dtype, auto_reset = (int)r.auto_reset;
    const DockauvRolloutOut &o = r.out;
    const DockauvPolicyOut &po = r.pout;
    const size_t arow = (action_dtype == DOCKAUV_ACT_F32 ? 4 : 8) * n_u * N;
    auto slot = [&](int t) { return (int)((r.start_slot + t) % r.n_slots); };
    auto ring_actions = [&](int t) { return (float *)r.ring.actions + n_u * N * slot(t); };
    auto actions_of_step = [&](int t) {
        return act ? (const void *)ring_actions(t) : pol ? (const void *)h->pol_actions : (const char *)r.input + arow * t;
    };
    auto obs_of_step = [&](int t) { return t == 0 ? (const float *)r.input : o.obs + (size_t)h->n_obs * N * (t - 1); };
    auto step_out = [&](int t) { return act ? ring_step_out(h, r.ring, (int)r.n_slots, slot(t)) : rollout_step_out(h, o, t); };
    auto policy = [&](int t, int64_t b, int64_t e, cudaStream_t s) {
        if (act) return actor_range(h, *act, r.ring.obs + (size_t)h->n_obs * N * slot(t), ring_actions(t), b, e, s);
        if (!pol) return DOCKAUV_OK;
        return policy_range(h, *pol, obs_of_step(t), po.actions + n_u * N * t, po.values + N * t, po.log_probs + N * t,
                            false, b, e, s);
    };
    auto bootstrap = [&](int64_t b, int64_t e, cudaStream_t s) {
        if (!pol || !po.last_values) return DOCKAUV_OK;
        return policy_range(h, *pol, obs_of_step(n_steps), nullptr, po.last_values, nullptr, true, b, e, s);
    };
    if (h->tap.n > 0) {
        // the taps need one pre-step snapshot per step, so every step is forked and joined on its own (the parts of a
        // batch stepped in parts cannot run their T steps as one chain each), and the policy covers the whole batch
        for (int t = 0; t < n_steps; t++) {
            const DockauvStepOut so = step_out(t);
            int rc = policy(t, 0, h->n_envs, st);
            if (rc == DOCKAUV_OK)
                rc = step_call(h, actions_of_step(t), action_dtype, nullptr, &so, nullptr, auto_reset, st, false);
            if (rc != DOCKAUV_OK) return rc;
        }
        return bootstrap(0, h->n_envs, st);
    }
    // without taps, envs never interact: each part of a batch stepped in parts runs its T (policy, step) pairs as ONE
    // chain on its own stream, forked from / joined to the caller's stream once per rollout instead of once per step
    return over_ranges(h, false, st, [&](int64_t b, int64_t e, cudaStream_t s) {
        for (int t = 0; t < n_steps; t++) {
            const DockauvStepOut so = step_out(t);
            int rc = policy(t, b, e, s);
            if (rc == DOCKAUV_OK)
                rc = step_range(h, actions_of_step(t), action_dtype, nullptr, &so, nullptr, auto_reset, b, e, s);
            if (rc != DOCKAUV_OK) return rc;
        }
        return bootstrap(b, e, s);
    });
}

// The rollout entry points after their own argument checks: ep_len_out zero-filled, then the launches issued directly
// or (use_graph) replayed from the graph cached under the rollout's key, open loop in h->rg, closed loop in h->pg, ring
// collection (act and ring set, out zero) in h->cg.
static int rollout_run(DockauvHandle *h, const DockauvPolicy *pol, const DockauvSquashedActor *act,
                       const DockauvReplayRing *ring, int n_slots, int start_slot, const void *input, int action_dtype,
                       int n_steps, const DockauvRolloutOut &out, const DockauvPolicyOut *pout, int auto_reset,
                       int use_graph, void *stream) {
    if (check_rows(h, ring ? ring->obs : out.obs, ring ? ring->terminal_obs : out.terminal_obs) != DOCKAUV_OK)
        return DOCKAUV_EINVAL;
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    // the closed loop's action buffer: allocated before any capture, its pointer is baked into every graph
    if (pol && !h->pol_actions)
        CUDA_TRY(cudaMalloc((void **)&h->pol_actions, sizeof(float) * h->params.n_u * (size_t)h->n_envs));
    if (out.ep_len_out)
        CUDA_TRY(cudaMemsetAsync(out.ep_len_out, 0, sizeof(int32_t) * (size_t)h->n_envs * (size_t)n_steps, st));
    DockauvHandle::RolloutKey key;
    memset(&key, 0, sizeof(key));
    if (pol) {
        key.pol = *pol;
        key.pout = *pout;
    }
    if (act) {
        key.act = *act;
        key.ring = *ring;
        key.n_slots = n_slots;
        key.start_slot = start_slot;
    }
    key.input = input;
    key.out = out;
    key.n_steps = n_steps;
    key.action_dtype = action_dtype;
    key.auto_reset = auto_reset;
    key.seed = h->params.seed;
    auto issue = [&](cudaStream_t s) { return rollout_issue(h, pol, act, key, s); };
    if (!use_graph) return issue(st);
    return graph_call(h, act ? h->cg : pol ? h->pg : h->rg, key,
                      act ? "ring collection" : pol ? "policy rollout" : "rollout", st, issue);
}

extern "C" int dockauv_rollout(DockauvHandle *h, const void *actions_dev, int action_dtype, int n_steps,
                               const DockauvRolloutOut *out, int auto_reset, int use_graph, void *stream) {
    if (!h || !actions_dev || !out) return fail(DOCKAUV_EINVAL, "null argument");
    if (!h->bound) return fail(DOCKAUV_ESTATE, "dockauv_bind must be called before dockauv_rollout");
    if (!out->obs || !out->reward || !out->done) return fail(DOCKAUV_EINVAL, "obs, reward and done outputs are required");
    if (action_dtype != DOCKAUV_ACT_F32 && action_dtype != DOCKAUV_ACT_F64) return fail(DOCKAUV_EINVAL, "bad action dtype");
    if (n_steps <= 0) return fail(DOCKAUV_EINVAL, "n_steps must be positive");
    return rollout_run(h, nullptr, nullptr, nullptr, 0, 0, actions_dev, action_dtype, n_steps, *out, nullptr, auto_reset,
                       use_graph, stream);
}

extern "C" int dockauv_rollout_policy(DockauvHandle *h, const DockauvPolicy *pol, const float *obs0_dev, int n_steps,
                                      const DockauvRolloutOut *out, const DockauvPolicyOut *pout, int auto_reset,
                                      int use_graph, void *stream) {
    // what needs no handle first
    if (!pol || !obs0_dev || !out || !pout) return fail(DOCKAUV_EINVAL, "null argument (policy, obs0, out and pout are required)");
    for (int k = 0; k < 3; k++)
        if (!pol->pi_w[k] || !pol->pi_b[k] || !pol->vf_w[k] || !pol->vf_b[k])
            return fail(DOCKAUV_EINVAL, "policy layer %d: a weight or bias pointer is null", k);
    if (!pol->log_std) return fail(DOCKAUV_EINVAL, "policy log_std is null");
    if (pol->hidden < 32 || pol->hidden > 128 || pol->hidden % 32 != 0)
        return fail(DOCKAUV_EINVAL, "policy hidden width must be a multiple of 32 in 32..128, got %d", pol->hidden);
    if (n_steps <= 0) return fail(DOCKAUV_EINVAL, "n_steps must be positive");
    if (!out->obs || !out->reward || !out->done) return fail(DOCKAUV_EINVAL, "obs, reward and done outputs are required");
    if (!pout->actions || !pout->values || !pout->log_probs)
        return fail(DOCKAUV_EINVAL, "policy outputs actions, values and log_probs are required");
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    if (!h->bound) return fail(DOCKAUV_ESTATE, "dockauv_bind must be called before dockauv_rollout_policy");
    const size_t smem = policy_smem_bytes(h->n_obs, pol->hidden, h->params.n_u);
    if (smem > kPolicyMaxSmem)
        return fail(DOCKAUV_EINVAL, "policy weights need %zu bytes of shared memory (n_obs %d, hidden %d, n_u %d); one CTA "
                                    "holds at most %zu", smem, h->n_obs, pol->hidden, h->params.n_u, kPolicyMaxSmem);
    return rollout_run(h, pol, nullptr, nullptr, 0, 0, obs0_dev, DOCKAUV_ACT_F32, n_steps, *out, pout, auto_reset,
                       use_graph, stream);
}

extern "C" int dockauv_replay_collect(DockauvHandle *h, const DockauvSquashedActor *actor, const DockauvReplayRing *ring,
                                      int n_slots, int start_slot, int n_steps, int auto_reset, int use_graph,
                                      void *stream) {
    // what needs no handle first
    if (!actor || !ring) return fail(DOCKAUV_EINVAL, "null argument (actor and ring are required)");
    for (int k = 0; k < 2; k++)
        if (!actor->w[k] || !actor->b[k])
            return fail(DOCKAUV_EINVAL, "actor latent_pi layer %d: a weight or bias pointer is null", k);
    if (!actor->mu_w || !actor->mu_b) return fail(DOCKAUV_EINVAL, "actor mu: a weight or bias pointer is null");
    if (!actor->log_std_w || !actor->log_std_b) return fail(DOCKAUV_EINVAL, "actor log_std: a weight or bias pointer is null");
    if (!ring->obs || !ring->terminal_obs || !ring->actions || !ring->reward || !ring->done)
        return fail(DOCKAUV_EINVAL, "a ring buffer is null (ring obs, terminal_obs, actions, reward, done are required)");
    if (actor->hidden != 64 && actor->hidden != 128 && actor->hidden != 256)
        return fail(DOCKAUV_EINVAL, "actor hidden width must be 64, 128 or 256, got %d", actor->hidden);
    if (n_steps <= 0) return fail(DOCKAUV_EINVAL, "n_steps must be positive");
    if (n_slots < 2 || n_slots > 64) return fail(DOCKAUV_EINVAL, "n_slots must be in 2..64, got %d", n_slots);
    if (start_slot < 0 || start_slot >= n_slots)
        return fail(DOCKAUV_EINVAL, "start_slot must be in 0..n_slots - 1 = %d, got %d", n_slots - 1, start_slot);
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    if (!h->bound) return fail(DOCKAUV_ESTATE, "dockauv_bind must be called before dockauv_replay_collect");
    const size_t smem = sac_actor_smem_bytes(h->n_obs, actor->hidden, h->params.n_u);
    if (smem > kPolicyMaxSmem)
        return fail(DOCKAUV_EINVAL, "actor weights need %zu bytes of shared memory (n_obs %d, hidden %d, n_u %d); one CTA "
                                    "holds at most %zu", smem, h->n_obs, actor->hidden, h->params.n_u, kPolicyMaxSmem);
    DockauvRolloutOut none;
    memset(&none, 0, sizeof(none));
    return rollout_run(h, nullptr, actor, ring, n_slots, start_slot, nullptr, DOCKAUV_ACT_F32, n_steps, none, nullptr,
                       auto_reset, use_graph, stream);
}

// ------------------------------------------------------------------------------------------- episode taps: setup
extern "C" int dockauv_set_taps(DockauvHandle *h, const int64_t *env_ids_host, int n_taps, int capacity,
                                const DockauvTapBuffers *bufs) {
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    if (!h->bound) return fail(DOCKAUV_ESTATE, "dockauv_bind must be called before dockauv_set_taps");
    if (n_taps < 0 || n_taps > DOCKAUV_MAX_TAPS)
        return fail(DOCKAUV_EINVAL, "n_taps must be in 0..%d, got %d", DOCKAUV_MAX_TAPS, n_taps);
    if (n_taps > 0) {
        if (capacity < 1) return fail(DOCKAUV_EINVAL, "capacity must be at least 1, got %d", capacity);
        if (!env_ids_host || !bufs) return fail(DOCKAUV_EINVAL, "null env ids or tap buffers");
        const DockauvTapBuffers &b = *bufs;
        const void *need[] = {b.count, b.pre_state, b.pre_current, b.pre_scene, b.pre_t_steps, b.pre_episode,
                              b.pre_ep_return, b.state, b.u, b.state_dot, b.nu_c, b.ray_dist, b.reward_arr, b.obs,
                              b.reward, b.done, b.cond_bits};
        for (const void *q : need)
            if (!q) return fail(DOCKAUV_EINVAL, "a tap buffer is null");
        std::vector<int64_t> ids(env_ids_host, env_ids_host + n_taps);
        for (int64_t i : ids)
            if (i < 0 || i >= h->n_envs)
                return fail(DOCKAUV_EINVAL, "tap env id %lld out of range 0..%lld", (long long)i, (long long)h->n_envs - 1);
        std::sort(ids.begin(), ids.end());
        for (size_t k = 1; k < ids.size(); k++)
            if (ids[k] == ids[k - 1]) return fail(DOCKAUV_EINVAL, "tap env id %lld given twice", (long long)ids[k]);
    }
    DeviceGuard guard(h->device);
    auto &tp = h->tap;
    CUDA_TRY(cudaDeviceSynchronize());      // the side branch of an earlier step may still read the old shadow
    drop_graphs(h);
    if (tp.mem) CUDA_TRY(cudaFree(tp.mem));
    tp.mem = nullptr;
    tp.n = 0;
    if (n_taps == 0) return DOCKAUV_OK;
    if (!tp.st) CUDA_TRY(cudaStreamCreateWithFlags(&tp.st, cudaStreamNonBlocking));
    if (!tp.ev_fork) CUDA_TRY(cudaEventCreateWithFlags(&tp.ev_fork, cudaEventDisableTiming));
    if (!tp.ev_join) CUDA_TRY(cudaEventCreateWithFlags(&tp.ev_join, cudaEventDisableTiming));
    if (!tp.dst) CUDA_TRY(cudaStreamCreateWithFlags(&tp.dst, cudaStreamNonBlocking));
    if (!tp.ev_dbg) CUDA_TRY(cudaEventCreateWithFlags(&tp.ev_dbg, cudaEventDisableTiming));
    const size_t K = (size_t)n_taps, esz = h->esz;
    const int nu = h->params.n_u, nc = h->params.n_capsules, ns = h->params.n_spheres, n_rays = h->params.n_rays;
    const bool pipe = h->pipe_buf != nullptr;
    // the pipeline layout's buffers for K envs, laid out as dockauv_create lays them out for n_envs
    tp.pipe = pipe ? pipe_buffers((int64_t)K, esz, nc, ns) : PipeBuffers();
    const int row_pieces = pipe ? (int)(8 * esz * (size_t)(nc + ns) / 16) : 0;      // 16-byte pieces of one env's obstacle rows
    tp.n_gather = 12 + nu + 3 + 1 + 5 + 7 * nc + 4 * ns + 3 + tp.pipe.n_obsf + row_pieces;
    tp.n_commit = 12 + nu + 12 + 3 + n_rays + 13 + 3 + h->n_obs;
    // one allocation, every piece 256-byte aligned (observation rows are written with 16-byte stores)
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t o = off;
        off += (bytes + 255) & ~(size_t)255;
        return o;
    };
    // one K-env set of persistent state (both shadows have one)
    struct Shadow {
        size_t state, u, goal, hg, cur, caps, sph, epr, ts, ep;
    };
    auto take_shadow = [&]() {
        Shadow o;
        o.state = take(12 * K * esz); o.u = take(nu * K * esz); o.goal = take(3 * K * esz); o.hg = take(K * esz);
        o.cur = take(5 * K * esz); o.caps = take((size_t)std::max(7 * nc, 1) * K * esz);
        o.sph = take((size_t)std::max(4 * ns, 1) * K * esz); o.epr = take(K * esz); o.ts = take(4 * K); o.ep = take(4 * K);
        return o;
    };
    const Shadow os = take_shadow(), od = take_shadow();
    const size_t o_noise = take(K * esz), o_act = take(8 * nu * K), o_obs = take(4 * K * h->n_obs),
                 o_rew = take(K * esz), o_done = take(K), o_cond = take(K), o_dobs = take(4 * K * h->n_obs),
                 o_drew = take(K * esz), o_ddone = take(K), o_dcond = take(K), o_ray = take(n_rays * K * esz),
                 o_rarr = take(13 * K * esz), o_nuc = take(3 * K * esz), o_sdot = take(12 * K * esz),
                 o_stats = take(kStatsBytes), o_ids = take(8 * K), o_sync = take(4),
                 o_grows = take(sizeof(TapRow) * tp.n_gather), o_crows = take(sizeof(TapRow) * tp.n_commit);
    const size_t o_pipe = take(tp.pipe.bytes);
    CUDA_TRY(cudaMalloc(&tp.mem, off));
    CUDA_TRY(cudaMemset(tp.mem, 0, off));
    char *m = (char *)tp.mem;
    if (pipe) CUDA_TRY(cudaMemset(m + o_pipe + tp.pipe.counters, 0xff, 4 * tp.pipe.n_counters));      // as dockauv_create
    auto place = [&](DockauvBuffers &b, const Shadow &o) {
        b.state = m + o.state; b.u_prev = m + o.u; b.goal = m + o.goal; b.heading_goal = m + o.hg; b.current = m + o.cur;
        b.capsules = m + o.caps; b.spheres = m + o.sph; b.ep_return = m + o.epr;
        b.t_steps = (int32_t *)(m + o.ts); b.episode = (int32_t *)(m + o.ep);
    };
    place(tp.shadow, os);
    place(tp.dshadow, od);
    tp.noise = m + o_noise;
    tp.actions = m + o_act;
    memset(&tp.out, 0, sizeof(tp.out));
    tp.out.obs = (float *)(m + o_obs);
    tp.out.reward = m + o_rew;
    tp.out.done = (uint8_t *)(m + o_done);
    tp.out.cond_bits = (uint8_t *)(m + o_cond);
    memset(&tp.dout, 0, sizeof(tp.dout));
    tp.dout.obs = (float *)(m + o_dobs);
    tp.dout.reward = m + o_drew;
    tp.dout.done = (uint8_t *)(m + o_ddone);
    tp.dout.cond_bits = (uint8_t *)(m + o_dcond);
    tp.pipe_buf = pipe ? m + o_pipe : nullptr;
    memset(&tp.dbg, 0, sizeof(tp.dbg));
    tp.dbg.ray_dist = m + o_ray;
    tp.dbg.reward_arr = m + o_rarr;
    tp.dbg.nu_c = m + o_nuc;
    tp.dbg.state_dot = m + o_sdot;
    tp.stats = (double *)(m + o_stats);
    tp.ids = (int64_t *)(m + o_ids);
    tp.sync = (unsigned int *)(m + o_sync);
    tp.gather_rows = (TapRow *)(m + o_grows);
    tp.commit_rows = (TapRow *)(m + o_crows);
    tp.n = n_taps;
    tp.capacity = capacity;
    tp.ring = *bufs;
    int rc = build_tap_rows(h);
    cudaError_t e = cudaSuccess;
    if (rc == DOCKAUV_OK) e = cudaMemcpy(tp.ids, env_ids_host, 8 * K, cudaMemcpyHostToDevice);
    if (rc == DOCKAUV_OK && e == cudaSuccess) e = cudaMemset(bufs->count, 0, sizeof(int64_t));
    if (rc == DOCKAUV_OK && e == cudaSuccess) e = cudaDeviceSynchronize();
    if (rc != DOCKAUV_OK || e != cudaSuccess) {
        cudaFree(tp.mem);
        tp.mem = nullptr;
        tp.n = 0;
        return rc != DOCKAUV_OK ? rc : fail(DOCKAUV_ECUDA, "tap setup failed: %s", cudaGetErrorString(e));
    }
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- scenario bank
// Reasons a bank row is refused, in the order they are checked per field
enum BankReason { kBankNonFinite = 1, kBankNegRadius, kBankFar, kBankCurrent, kBankCdf };
static const char *const kBankReasonText[] = {
    "", "value is not finite", "radius is negative",
    "obstacle is neither within 2 km of the row's goal at every defining point nor an unused slot (radius 0, every point "
    "at least 1e5 m from the goal)",
    "non-zero current on a handle that does not evaluate the current (set force_current)",
    "cdf must be finite and non-decreasing from >= 0, with cdf[K-1] > 0"};

// Thread per row: the first offending field of the row (field W = the cdf entry) goes into *first_bad as
// row << 24 | field << 8 | reason, the lowest value winning.
template <typename T>
__global__ void bank_validate_kernel(const T *rows, int64_t K, int64_t stride, int nc, int ns, int check_far,
                                     int current_on, const double *cdf, unsigned long long *first_bad) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= K) return;
    const T *row = rows + r * stride;
    const int W = 15 + 7 * nc + 4 * ns;
    int field = -1, reason = 0;
    auto flag = [&](int f, int why) {
        if (field < 0) {
            field = f;
            reason = why;
        }
    };
    for (int f = 0; f < W && field < 0; f++)
        if (!isfinite((double)row[f])) flag(f, kBankNonFinite);
    if (field < 0 && !current_on)
        for (int c = 0; c < 5; c++)
            if (row[10 + c] != T(0)) flag(10 + c, kBankCurrent);
    const double g[3] = {(double)row[6], (double)row[7], (double)row[8]};
    auto dist = [&](const T *q) {
        const double dx = (double)q[0] - g[0], dy = (double)q[1] - g[1], dz = (double)q[2] - g[2];
        return sqrt(dx * dx + dy * dy + dz * dz);
    };
    for (int s = 0; s < nc + ns && field < 0; s++) {
        const bool cap = s < nc;
        const int o = cap ? 15 + 7 * s : 15 + 7 * nc + 4 * (s - nc);
        const int ri = o + (cap ? 6 : 3);
        const T *q = row + o;
        if (row[ri] < T(0)) {
            flag(ri, kBankNegRadius);
            break;
        }
        if (!check_far) continue;
        const double d0 = dist(q), d1 = cap ? dist(q + 3) : d0;
        const bool near = d0 <= 2000.0 && d1 <= 2000.0;
        const bool unused = row[ri] == T(0) && d0 >= 1e5 && d1 >= 1e5;
        if (!near && !unused) flag(o, kBankFar);
    }
    if (field < 0 && cdf != nullptr) {
        const double c = cdf[r], prev = r > 0 ? cdf[r - 1] : 0.0;
        if (!isfinite(c) || !(c >= prev) || (r == K - 1 && !(c > 0.0))) flag(W, kBankCdf);
    }
    if (field >= 0) atomicMin(first_bad, ((unsigned long long)r << 24) | ((unsigned long long)field << 8) | (unsigned)reason);
}

// name of field f of a row (f == W: the cdf entry)
static void bank_field_name(const DockauvParams &p, int f, char *out, size_t n) {
    static const char *const head[] = {"pose x", "pose y", "pose z", "pose phi", "pose theta", "pose psi", "goal x",
                                       "goal y", "goal z", "heading goal", "current V_c", "current alpha",
                                       "current beta", "current V_min", "current V_max"};
    static const char *const cap[] = {"bot x", "bot y", "bot z", "top x", "top y", "top z", "r"};
    static const char *const sph[] = {"centre x", "centre y", "centre z", "r"};
    const int nc = p.n_capsules, ns = p.n_spheres;
    if (f < 15) snprintf(out, n, "%s", head[f]);
    else if (f < 15 + 7 * nc) snprintf(out, n, "capsule %d %s", (f - 15) / 7, cap[(f - 15) % 7]);
    else if (f < 15 + 7 * nc + 4 * ns) snprintf(out, n, "sphere %d %s", (f - 15 - 7 * nc) / 4, sph[(f - 15 - 7 * nc) % 4]);
    else snprintf(out, n, "cdf");
}

extern "C" int dockauv_set_scenario_bank(DockauvHandle *h, const DockauvScenarioBank *b, void *stream) {
    // what needs no handle first (W >= 15 for every handle: the row without obstacles)
    if (b) {
        if (!b->rows) return fail(DOCKAUV_EINVAL, "scenario bank: rows is null (pass a null bank to clear it)");
        if (b->n_rows < 1 || b->n_rows > (int64_t)INT32_MAX)
            return fail(DOCKAUV_EINVAL, "scenario bank: n_rows (K) must be in 1..2^31 - 1, got %lld", (long long)b->n_rows);
        if (misaligned16(b->rows)) return fail(DOCKAUV_EINVAL, "scenario bank: rows must be 16-byte aligned");
        if (b->row_stride < 15)
            return fail(DOCKAUV_EINVAL, "scenario bank: row_stride %lld is below the row width W (at least 15 reals)",
                        (long long)b->row_stride);
        if ((((uintptr_t)b->cdf) & 7u) != 0 || (((uintptr_t)b->row_of_env) & 3u) != 0)
            return fail(DOCKAUV_EINVAL, "scenario bank: cdf must be 8-byte and row_of_env 4-byte aligned");
    }
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    if (!b) {
        if (h->bank.rows) drop_graphs(h);
        h->bank = DockauvScenarioBank{};
        with_k(h, [](auto &k) {
            k.bank_rows = nullptr;
            k.bank_cdf = nullptr;
            k.bank_row_of_env = nullptr;
            k.bank_n = k.bank_stride = 0;
        });
        return DOCKAUV_OK;
    }
    const int nc = h->params.n_capsules, ns = h->params.n_spheres, W = 15 + 7 * nc + 4 * ns;
    if (b->row_stride < W)
        return fail(DOCKAUV_EINVAL, "scenario bank: row_stride %lld is below the row width W = 15 + 7 n_capsules + 4 n_spheres "
                                    "= %d", (long long)b->row_stride, W);
    if ((b->row_stride * (int64_t)h->esz) % 16 != 0)
        return fail(DOCKAUV_EINVAL, "scenario bank: row_stride * sizeof(real) = %lld bytes must be a multiple of 16",
                    (long long)(b->row_stride * (int64_t)h->esz));
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (!h->bank_check) CUDA_TRY(cudaMalloc((void **)&h->bank_check, sizeof(unsigned long long)));
    CUDA_TRY(cudaMemsetAsync(h->bank_check, 0xff, sizeof(unsigned long long), st));
    const int check_far = with_k(h, [](auto &k) { return k.cull_exact ? 0 : 1; });
    const unsigned blocks = (unsigned)((b->n_rows + 255) / 256);
    if (h->params.precision == DOCKAUV_F64)
        bank_validate_kernel<double><<<blocks, 256, 0, st>>>((const double *)b->rows, b->n_rows, b->row_stride, nc, ns,
                                                             check_far, current_on(h) ? 1 : 0, b->cdf, h->bank_check);
    else
        bank_validate_kernel<float><<<blocks, 256, 0, st>>>((const float *)b->rows, b->n_rows, b->row_stride, nc, ns,
                                                            check_far, current_on(h) ? 1 : 0, b->cdf, h->bank_check);
    CUDA_TRY(cudaGetLastError());
    unsigned long long bad = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad, h->bank_check, sizeof(bad), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (bad != ~0ull) {
        char name[64];
        const int field = (int)((bad >> 8) & 0xffff), reason = (int)(bad & 0xff);
        bank_field_name(h->params, field, name, sizeof(name));
        return fail(DOCKAUV_EINVAL, "scenario bank refused: row %lld, %s: %s", (long long)(bad >> 24), name,
                    kBankReasonText[reason]);
    }
    const DockauvScenarioBank &o = h->bank;
    if (o.rows != b->rows || o.cdf != b->cdf || o.row_of_env != b->row_of_env || o.n_rows != b->n_rows ||
        o.row_stride != b->row_stride)
        drop_graphs(h);          // captured sequences hold the old pointers; the same pointers keep every graph
    h->bank = *b;
    with_k(h, [&](auto &k) {
        k.bank_rows = (decltype(k.bank_rows))b->rows;
        k.bank_cdf = b->cdf;
        k.bank_row_of_env = b->row_of_env;
        k.bank_n = b->n_rows;
        k.bank_stride = b->row_stride;
    });
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- GAE
template <typename R>
__global__ void gae_kernel(const R *__restrict__ rewards, const float *__restrict__ values,
                           const float *__restrict__ last_values, const uint8_t *__restrict__ dones, int T, int64_t N,
                           float gamma, float lam, float *__restrict__ adv, float *__restrict__ ret) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    float next_v = last_values[i], a = 0.0f;
    // rows are env-fastest, so each step is one coalesced request per warp; the next rows are in flight while the
    // recurrence of the current one (3 dependent FMAs) resolves
#pragma unroll 4
    for (int t = T - 1; t >= 0; t--) {
        const int64_t k = (int64_t)t * N + i;
        const float nt = dones[k] ? 0.0f : 1.0f;
        const float v = values[k];
        const float delta = (float)rewards[k] + gamma * next_v * nt - v;
        a = delta + gamma * lam * nt * a;
        adv[k] = a;
        ret[k] = a + v;
        next_v = v;
    }
}

extern "C" int dockauv_gae(const void *rewards_dev, int reward_precision, const float *values_dev,
                           const float *last_values_dev, const uint8_t *dones_dev, int n_steps, int64_t n_envs,
                           float gamma, float gae_lambda, float *advantages_dev, float *returns_dev, void *stream) {
    if (!rewards_dev || !values_dev || !last_values_dev || !dones_dev || !advantages_dev || !returns_dev)
        return fail(DOCKAUV_EINVAL, "null argument");
    if (n_steps <= 0 || n_envs <= 0) return fail(DOCKAUV_EINVAL, "n_steps and n_envs must be positive");
    if (reward_precision != DOCKAUV_F64 && reward_precision != DOCKAUV_F32) return fail(DOCKAUV_EINVAL, "bad reward precision");
    cudaStream_t st = (cudaStream_t)stream;
    const int threads = 256;
    const unsigned blocks = (unsigned)((n_envs + threads - 1) / threads);
    if (reward_precision == DOCKAUV_F64)
        gae_kernel<double><<<blocks, threads, 0, st>>>((const double *)rewards_dev, values_dev, last_values_dev, dones_dev,
                                                       n_steps, n_envs, gamma, gae_lambda, advantages_dev, returns_dev);
    else
        gae_kernel<float><<<blocks, threads, 0, st>>>((const float *)rewards_dev, values_dev, last_values_dev, dones_dev,
                                                      n_steps, n_envs, gamma, gae_lambda, advantages_dev, returns_dev);
    CUDA_TRY(cudaGetLastError());
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- replay sampling
// The warp's 32 rows are copied together: element e of the warp's output block is element e % n of row e / n, so
// every store instruction writes 32 consecutive elements, and each lane's source row pointer is fetched with a shuffle.
// Every lane runs the same n iterations (the shuffle needs the whole warp); lanes past the batch store nothing.
template <typename V>
__device__ __forceinline__ void copy_warp_rows(const float *src, float *__restrict__ dst, int n, int rows, int lane) {
#pragma unroll 4
    for (int e = lane; e < 32 * n; e += 32) {
        const int r = e / n;
        const V *s = (const V *)__shfl_sync(0xffffffffu, (unsigned long long)src, r);
        if (r < rows) ((V *)dst)[e] = __ldg(s + (e - r * n));
    }
}

// One thread draws one row from Philox4x32-10 at counter (row, draw): 64 bits scaled onto the n_valid transitions and 64
// onto the N envs, each by a 64 x 64 -> high-64 multiply (relative bias below n / 2^64, no division); then the warp
// copies observation, next observation and action rows.  V = float4 when n_obs % 4 == 0, else float.
template <typename R, typename V>
__global__ void replay_sample_kernel(DockauvReplayRing ring, int S, int64_t N, int n_obs, int n_u, int slot0, int n_valid,
                                     int64_t B, uint64_t seed, uint64_t draw, DockauvReplaySample out) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, row0 = row - lane;
    if (row0 >= B) return;      // whole warps only
    const int rows = (int)min((int64_t)32, B - row0);
    const float *o = ring.obs, *nx = ring.obs, *a = ring.actions;
    if (row < B) {
        uint32_t c[4] = {(uint32_t)row, (uint32_t)(row >> 32), (uint32_t)draw, (uint32_t)(draw >> 32)};
        philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        // (transition, env) uniform over n_valid * N pairs = transition and env independent and uniform
        const int k = (int)__umul64hi(((uint64_t)c[2] << 32) | c[3], (uint64_t)n_valid);   // transition t_first + k
        const int64_t env = (int64_t)__umul64hi(((uint64_t)c[0] << 32) | c[1], (uint64_t)N);
        const int slot = slot0 + k < S ? slot0 + k : slot0 + k - S, next = slot + 1 == S ? 0 : slot + 1;
        const int64_t at = (int64_t)slot * N + env;
        const bool d = ring.done[at] != 0;
        o = ring.obs + at * n_obs;
        nx = d ? ring.terminal_obs + at * n_obs : ring.obs + ((int64_t)next * N + env) * n_obs;
        a = ring.actions + at * n_u;
        out.reward[row] = (float)((const R *)ring.reward)[at];
        out.done[row] = d ? 1.0f : 0.0f;
        if (out.index) out.index[row] = at;
    }
    const int vw = (int)(sizeof(V) / sizeof(float));
    copy_warp_rows<V>(o, out.obs + row0 * n_obs, n_obs / vw, rows, lane);
    copy_warp_rows<V>(nx, out.next_obs + row0 * n_obs, n_obs / vw, rows, lane);
    copy_warp_rows<float>(a, out.actions + row0 * n_u, n_u, rows, lane);
}

template <typename R>
static void launch_replay_sample(bool vec4, unsigned blocks, cudaStream_t st, const DockauvReplayRing &ring, int S,
                                 int64_t N, int n_obs, int n_u, int slot0, int n_valid, int64_t B, uint64_t seed,
                                 uint64_t draw, const DockauvReplaySample &out) {
    if (vec4)
        replay_sample_kernel<R, float4><<<blocks, 256, 0, st>>>(ring, S, N, n_obs, n_u, slot0, n_valid, B, seed, draw, out);
    else
        replay_sample_kernel<R, float><<<blocks, 256, 0, st>>>(ring, S, N, n_obs, n_u, slot0, n_valid, B, seed, draw, out);
}

extern "C" int dockauv_replay_sample(const DockauvReplayRing *ring, int reward_precision, int n_slots, int64_t n_envs,
                                     int n_obs, int n_u, int64_t t_first, int64_t n_valid, int64_t batch, uint64_t seed,
                                     uint64_t draw, const DockauvReplaySample *out, void *stream) {
    if (!ring) return fail(DOCKAUV_EINVAL, "null ring");
    if (!out) return fail(DOCKAUV_EINVAL, "null out");
    if (!ring->obs || !ring->terminal_obs || !ring->actions || !ring->reward || !ring->done)
        return fail(DOCKAUV_EINVAL, "a ring buffer is null (ring obs, terminal_obs, actions, reward, done are required)");
    if (!out->obs || !out->actions || !out->next_obs || !out->done || !out->reward)
        return fail(DOCKAUV_EINVAL, "an out buffer is null (out obs, actions, next_obs, done, reward are required)");
    if (reward_precision != DOCKAUV_F64 && reward_precision != DOCKAUV_F32)
        return fail(DOCKAUV_EINVAL, "bad reward_precision %d", reward_precision);
    if (n_slots < 2 || n_slots > (1 << 30)) return fail(DOCKAUV_EINVAL, "n_slots must be in 2..2^30, got %d", n_slots);
    if (n_envs <= 0 || n_envs > ((int64_t)1 << 32))
        return fail(DOCKAUV_EINVAL, "n_envs must be in 1..2^32, got %lld", (long long)n_envs);
    if (n_obs < 1 || n_obs > 16 + DOCKAUV_MAX_RAYS)
        return fail(DOCKAUV_EINVAL, "n_obs must be in 1..%d, got %d", 16 + DOCKAUV_MAX_RAYS, n_obs);
    if (n_u < 1 || n_u > DOCKAUV_MAX_U) return fail(DOCKAUV_EINVAL, "n_u must be in 1..%d, got %d", DOCKAUV_MAX_U, n_u);
    if (t_first < 0) return fail(DOCKAUV_EINVAL, "t_first must not be negative, got %lld", (long long)t_first);
    if (n_valid < 1 || n_valid > n_slots - 1)
        return fail(DOCKAUV_EINVAL, "n_valid must be in 1..n_slots - 1 = %d (the slot the next step overwrites is never valid), "
                                    "got %lld", n_slots - 1, (long long)n_valid);
    if (batch <= 0 || batch > (int64_t)INT32_MAX)
        return fail(DOCKAUV_EINVAL, "batch must be in 1..2^31 - 1, got %lld", (long long)batch);
    const bool vec4 = (n_obs & 3) == 0;
    if (vec4 && (misaligned16(ring->obs) || misaligned16(ring->terminal_obs) || misaligned16(out->obs) ||
                 misaligned16(out->next_obs)))
        return fail(DOCKAUV_EINVAL, "ring obs / terminal_obs and out obs / next_obs must be 16-byte aligned (n_obs = %d is a "
                                    "multiple of 4: rows move as 128-bit loads and stores)", n_obs);
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)((batch + 255) / 256);
    const int slot0 = (int)(t_first % n_slots);
    if (reward_precision == DOCKAUV_F64)
        launch_replay_sample<double>(vec4, blocks, st, *ring, n_slots, n_envs, n_obs, n_u, slot0, (int)n_valid, batch, seed,
                                     draw, *out);
    else
        launch_replay_sample<float>(vec4, blocks, st, *ring, n_slots, n_envs, n_obs, n_u, slot0, (int)n_valid, batch, seed,
                                    draw, *out);
    CUDA_TRY(cudaGetLastError());
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- statistics
extern "C" int dockauv_stats_ptr(DockauvHandle *h, double **stats_dev) {
    if (!h || !stats_dev) return fail(DOCKAUV_EINVAL, "null argument");
    *stats_dev = h->stats;
    return DOCKAUV_OK;
}

__global__ void fold_stats_kernel(double *stats) {
    const int k = threadIdx.x;
    if (k >= DOCKAUV_N_STATS) return;
    // atomic swap / add: a step kernel on another stream may be accumulating while the replicas are folded
    double s = 0.0;
    for (int c = 1; c < DOCKAUV_STAT_COPIES; c++)
        s += __longlong_as_double((long long)atomicExch((unsigned long long *)&stats[c * DOCKAUV_N_STATS + k], 0ull));
    if (s != 0.0) atomicAdd(&stats[k], s);
}

extern "C" int dockauv_fold_stats(DockauvHandle *h, void *stream) {
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    DeviceGuard guard(h->device);
    fold_stats_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->stats);
    CUDA_TRY(cudaGetLastError());
    return DOCKAUV_OK;
}

extern "C" int dockauv_get_stats(DockauvHandle *h, double *stats_host, void *stream) {
    if (!h || !stats_host) return fail(DOCKAUV_EINVAL, "null argument");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = dockauv_fold_stats(h, stream);
    if (rc != DOCKAUV_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(stats_host, h->stats, sizeof(double) * DOCKAUV_N_STATS, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return DOCKAUV_OK;
}

extern "C" int dockauv_clear_stats(DockauvHandle *h, void *stream) {
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    DeviceGuard guard(h->device);
    CUDA_TRY(cudaMemsetAsync(h->stats, 0, kStatsBytes, (cudaStream_t)stream));
    return DOCKAUV_OK;
}

extern "C" int dockauv_launch_count(DockauvHandle *h, int64_t *n) {
    if (!h || !n) return fail(DOCKAUV_EINVAL, "null argument");
    *n = h->launches;
    return DOCKAUV_OK;
}

extern "C" int dockauv_last_list_counts(DockauvHandle *h, int64_t *n_listed, int64_t *n_ended, void *stream) {
    if (!h || !n_listed || !n_ended) return fail(DOCKAUV_EINVAL, "null argument");
    *n_listed = *n_ended = 0;
    if (!h->pipe_buf) return DOCKAUV_OK;
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    // one counter block per env range the most recent step call stepped (parts of the batch, chunks of step_host)
    const size_t n_cnt = h->pipe.n_counters;
    std::vector<unsigned int> host(n_cnt);
    return with_k(h, [&](auto &k) {
        CUDA_TRY(cudaMemcpyAsync(host.data(), k.view_count, n_cnt * sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        for (int64_t b : h->last_begins) {
            const size_t w = (size_t)counter_block(b);
            if (w + kCounterWords > n_cnt) continue;
            auto length = [&](int c) { return (int64_t)(host[w + c] - host[w + kCounterStart + c]); };      // mod 2^32
            *n_listed += length(0) + length(1) + length(2);
            *n_ended += length(3);
        }
        return DOCKAUV_OK;
    });
}

extern "C" int dockauv_rollout_captures(DockauvHandle *h, int64_t *n) {
    if (!h || !n) return fail(DOCKAUV_EINVAL, "null argument");
    *n = h->rg.captures;
    return DOCKAUV_OK;
}

extern "C" int dockauv_rollout_policy_captures(DockauvHandle *h, int64_t *n) {
    if (!h || !n) return fail(DOCKAUV_EINVAL, "null argument");
    *n = h->pg.captures;
    return DOCKAUV_OK;
}

extern "C" int dockauv_replay_collect_captures(DockauvHandle *h, int64_t *n) {
    if (!h || !n) return fail(DOCKAUV_EINVAL, "null argument");
    *n = h->cg.captures;
    return DOCKAUV_OK;
}

extern "C" int dockauv_enable_timing(DockauvHandle *h, int enabled) {
    if (!h) return fail(DOCKAUV_EINVAL, "null handle");
    h->timing = enabled != 0;
    h->ev_valid = false;
    return DOCKAUV_OK;
}

extern "C" int dockauv_last_step_ms(DockauvHandle *h, float *ms) {
    if (!h || !ms) return fail(DOCKAUV_EINVAL, "null argument");
    if (!h->ev_valid) return fail(DOCKAUV_ESTATE, "no timed step recorded (dockauv_enable_timing + dockauv_step first)");
    DeviceGuard guard(h->device);
    CUDA_TRY(cudaEventSynchronize(h->ev1));
    CUDA_TRY(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    return DOCKAUV_OK;
}

extern "C" int dockauv_last_step_launch_ms(DockauvHandle *h, float *ms, int capacity, int *n_launches) {
    if (!h || !ms || !n_launches) return fail(DOCKAUV_EINVAL, "null argument");
    if (!h->ev_valid) return fail(DOCKAUV_ESTATE, "no timed step recorded (dockauv_enable_timing + dockauv_step first)");
    DeviceGuard guard(h->device);
    CUDA_TRY(cudaEventSynchronize(h->ev1));
    const int n = h->n_marks > 0 ? h->n_marks - 1 : 0;
    *n_launches = n;
    for (int k = 0; k < n && k < capacity; k++) CUDA_TRY(cudaEventElapsedTime(&ms[k], h->marks[k], h->marks[k + 1]));
    return DOCKAUV_OK;
}

// ------------------------------------------------------------------------------------------- roofline denominators
template <typename T>
__global__ void fma_peak_kernel(T *out, int iters, T a, T b) {
    T x0 = (T)threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
            x0 = x0 * a + b; x1 = x1 * a + b; x2 = x2 * a + b; x3 = x3 * a + b;
            x4 = x4 * a + b; x5 = x5 * a + b; x6 = x6 * a + b; x7 = x7 * a + b;
        }
    }
    T s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == (T)123456.789) out[0] = s;   // keeps the chains alive, never true in practice
}

template <typename T>
static int measure_fma(double *tflops) {
    int dev = 0, sms = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    T *out = nullptr;
    CUDA_TRY(cudaMalloc((void **)&out, sizeof(T)));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int threads = 256, blocks = sms * 8, iters = 4096;
    fma_peak_kernel<T><<<blocks, threads>>>(out, 64, (T)1.0000001, (T)1e-9);   // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 5; rep++) {
        CUDA_TRY(cudaEventRecord(e0));
        fma_peak_kernel<T><<<blocks, threads>>>(out, iters, (T)1.0000001, (T)1e-9);
        CUDA_TRY(cudaEventRecord(e1));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        double flops = 2.0 * 64.0 * (double)iters * (double)threads * (double)blocks;
        double tf = flops / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    *tflops = best;
    return DOCKAUV_OK;
}

extern "C" int dockauv_measure_peaks(int device, double *fp64_tflops, double *fp32_tflops, double *copy_gbs) {
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev)
        return fail(DOCKAUV_ECUDA, "no usable CUDA device %d", device);
    DeviceGuard guard(device);
    int rc;
    if (fp64_tflops && (rc = measure_fma<double>(fp64_tflops)) != DOCKAUV_OK) return rc;
    if (fp32_tflops && (rc = measure_fma<float>(fp32_tflops)) != DOCKAUV_OK) return rc;
    if (copy_gbs) {
        const size_t bytes = (size_t)1 << 30;
        void *a = nullptr, *b = nullptr;
        CUDA_TRY(cudaMalloc(&a, bytes));
        CUDA_TRY(cudaMalloc(&b, bytes));
        CUDA_TRY(cudaMemset(a, 1, bytes));
        cudaEvent_t e0, e1;
        CUDA_TRY(cudaEventCreate(&e0));
        CUDA_TRY(cudaEventCreate(&e1));
        double best = 0.0;
        for (int rep = 0; rep < 6; rep++) {
            CUDA_TRY(cudaEventRecord(e0));
            CUDA_TRY(cudaMemcpyAsync(b, a, bytes, cudaMemcpyDeviceToDevice));
            CUDA_TRY(cudaEventRecord(e1));
            CUDA_TRY(cudaEventSynchronize(e1));
            float ms = 0;
            CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
            double gbs = 2.0 * (double)bytes / (ms * 1e-3) / 1e9;
            if (rep > 0 && gbs > best) best = gbs;
        }
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        cudaFree(a);
        cudaFree(b);
        *copy_gbs = best;
    }
    return DOCKAUV_OK;
}
