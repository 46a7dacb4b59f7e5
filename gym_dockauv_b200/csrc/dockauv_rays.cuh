// dockauv_rays.cuh -- the radar of ONE env done by one warp (lanes = rays): Radar.update / update_intersec /
// intersec_dist_reduced (objects/sensor.py:90-137), update_radar_collision (envs/docking3d.py:415-442) with the ray
// tests of objects/shape.py:235-264, 327-390 and the sum of Reward.obstacle_avoidance (docking3d.py:767-792).
// Shared by the fused warp kernel (dockauv_step_warp.cuh) and the ray launch of the pipeline (dockauv_step_pipe.cuh).
#pragma once
#include "dockauv_env.cuh"

namespace dockauv {

constexpr int kPreStride = 14;       // shared words per (env, obstacle) record, 16-byte aligned for 128-bit reads
                                     // capsule: ba[3] oa[3] baba baoa c c2a c2b ; sphere: oc[3] c

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// two shared words with one 128-bit (double) / 64-bit (float) load
template <typename T>
struct Pair;
template <>
struct Pair<double> {
    using type = double2;
};
template <>
struct Pair<float> {
    using type = float2;
};

// What a lane needs for the whole kernel: its rays (ray = lane + 32 j) and its pooled cell.  Two homes: registers
// (RayLane, fused warp kernel) or the warp's shared memory (RayLaneShared, ray launch of the pipeline: 24 registers less
// per thread decide whether five or six CTAs fit an SM there).
template <typename T, int RPL>
struct RayLane {
    T rb_[RPL][3], bw_[RPL];   // body-frame direction (sensor.py:63-71), obstacle-avoidance weight (docking3d.py:789-790)
    int pidx_[4];              // 2x2 pooling fast path: the four source slots of this lane's cell
    bool fast_pool;            // 2x2 blocks and at most one pooled cell per lane
    T dmax, inv_dmax;

    __device__ __forceinline__ T rb(int j, int c) const { return rb_[j][c]; }
    __device__ __forceinline__ T bw(int j) const { return bw_[j]; }
    __device__ __forceinline__ int pidx(int q) const { return pidx_[q]; }

    // s_ray: the warp's ray-distance scratch (n_rays + 2 words; slot n_rays holds the zero that block_reduce pads with)
    __device__ __forceinline__ void init(const KParams<T> &p, int lane, T *s_ray) {
        const int n_r = p.n_rays;
#pragma unroll
        for (int j = 0; j < RPL; j++) {
            const int ir = lane + 32 * j;
            const bool ok = ir < n_r;
#pragma unroll
            for (int c = 0; c < 3; c++) rb_[j][c] = ok ? p.ray_tab[c * n_r + ir] : T(0);
            bw_[j] = ok ? p.ray_tab[3 * n_r + ir] : T(0);
        }
        fast_pool = (p.block == 2) && (p.n_rr <= 32);
#pragma unroll
        for (int q = 0; q < 4; q++) pidx_[q] = n_r;
        if (fast_pool && lane < p.n_rr) {
            const int pr = lane / p.n_hr, pcol = lane - pr * p.n_hr;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int rv = 2 * pr + (q >> 1), rh = 2 * pcol + (q & 1);
                if (rv < p.n_vert && rh < p.n_horiz) pidx_[q] = rv * p.n_horiz + rh;
            }
        }
        if (lane == 0) s_ray[n_r] = T(0);
        dmax = p.radar_max_dist;
        inv_dmax = T(1) / dmax;
    }
};

// the same constants in shared memory: words [4 RPL][32] of T (rb, bw) followed by int [4][32] (pidx), this lane's column;
// read through volatile so that the compiler does not pull them back into registers for the whole loop
template <typename T, int RPL>
struct RayLaneShared {
    const T *w;        // + lane
    const int *pi;     // + lane
    bool fast_pool;
    T dmax, inv_dmax;

    static __host__ __device__ constexpr int words() { return 4 * RPL * 32 + 4 * 32 * (int)sizeof(int) / (int)sizeof(T); }
    __device__ __forceinline__ T rb(int j, int c) const { return reinterpret_cast<const volatile T *>(w)[(4 * j + c) * 32]; }
    __device__ __forceinline__ T bw(int j) const { return reinterpret_cast<const volatile T *>(w)[(4 * j + 3) * 32]; }
    __device__ __forceinline__ int pidx(int q) const { return reinterpret_cast<const volatile int *>(pi)[q * 32]; }

    __device__ __forceinline__ void init(const KParams<T> &p, int lane, T *s_ray, T *s_lane) {
        RayLane<T, RPL> r;
        r.init(p, lane, s_ray);
        T *wl = s_lane + lane;
        int *pl = reinterpret_cast<int *>(s_lane + 4 * RPL * 32) + lane;
#pragma unroll
        for (int j = 0; j < RPL; j++) {
#pragma unroll
            for (int c = 0; c < 3; c++) wl[(4 * j + c) * 32] = r.rb_[j][c];
            wl[(4 * j + 3) * 32] = r.bw_[j];
        }
#pragma unroll
        for (int q = 0; q < 4; q++) pl[q * 32] = r.pidx_[q];
        w = wl;
        pi = pl;
        fast_pool = r.fast_pool;
        dmax = r.dmax;
        inv_dmax = r.inv_dmax;
        __syncwarp();
    }
};

// One ray against one capsule record (shape.py:341-390: cylinder root, body hit if 0 < y < baba, else end cap) / one
// sphere record (shape.py:252-263: nearest root): returns min(best, distance) over the POSITIVE distances
// (docking3d.py:438-439).  Branch-free sqrt / reciprocal in the hit path.  Shared by every radar mapping -> same bits.
template <typename T>
__device__ __forceinline__ T cast_capsule(const T rd[3], const T ba[3], const T oa[3], T baba, T baoa, T cc, T c2a, T c2b, T best) {
    const T bard = rd[0] * ba[0] + rd[1] * ba[1] + rd[2] * ba[2];
    const T rdoa = rd[0] * oa[0] + rd[1] * oa[1] + rd[2] * oa[2];
    const T a = baba - bard * bard;
    const T b = baba * rdoa - baoa * bard;
    const T h = b * b - a * cc;
    if (h > T(0)) {
        const T t = (-b - Mth<T>::sqrt_pos(h)) * Mth<T>::rcp_(a);
        const T y = baoa + t * bard;
        T v = t;
        if (!(y > T(0) && y < baba)) {
            const bool far_end = y >= T(0);
            const T b2 = far_end ? rdoa - bard : rdoa;     // rd . (pos - cap end)
            const T h2 = b2 * b2 - (far_end ? c2b : c2a);
            v = (h2 > T(0)) ? (-b2 - Mth<T>::sqrt_pos(h2 > T(0) ? h2 : T(1))) : T(-1);
        }
        if (v > T(0) && v < best) best = v;
    }
    return best;
}

// cast_capsule for mappings where the lanes of a warp are different envs (some lane always hits, so the hit path runs
// anyway): straight-line code, which lets the compiler interleave the independent rays of a lane; only the end-cap root
// (second square root) sits behind a warp vote.  Every value is formed by the same expression as in cast_capsule /
// cast_sphere, so hits give identical bits.  Must be called by all 32 lanes.
//   A SPHERE goes through the same code as a capsule whose cylinder quadratic IS the sphere quadratic (sphere_as_capsule:
//   ba = 0, baba = 1, baoa = 1/2, cc = |oc|^2 - r^2 -> a = 1, b = rd . oc, h = b^2 - cc, y = 1/2: always a "body" hit);
//   h_min of such a record is minus the smallest normal number: a tangent ray (h == 0) counts as a hit there (shape.py:258
//   tests h < 0 for "miss"); a = 1 makes the rest of the capsule path the sphere's arithmetic bit for bit.
template <typename T>
__device__ __forceinline__ T cast_capsule_bf(const T rd[3], const T ba[3], const T oa[3], T baba, T baoa, T cc, T c2a, T c2b,
                                             T h_min, T best) {
    const T bard = rd[0] * ba[0] + rd[1] * ba[1] + rd[2] * ba[2];
    const T rdoa = rd[0] * oa[0] + rd[1] * oa[1] + rd[2] * oa[2];
    const T a = baba - bard * bard;
    const T b = baba * rdoa - baoa * bard;
    // (a sphere record has a = 1 exactly: a cc = cc, 1 / a = 1, so this is the sphere's fma(b, b, -c) and its root as it is --
    // no per-lane select on the obstacle type, which was a tenth of this launch's instructions)
    const T h = Mth<T>::fma_(b, b, -Mth<T>::mul_(a, cc));
    const T sq = Mth<T>::sqrt_pos(h > T(0) ? h : T(1));
    const T root = -b - (h > T(0) ? sq : T(0));
    const T t = root * Mth<T>::rcp_(a);
    const T y = baoa + t * bard;
    const bool cand = h > h_min;      // h_min = 0: capsule (shape.py:352 h > 0); -min_normal: sphere (shape.py:258 misses on h < 0 only)
    const bool body = y > T(0) && y < baba;
    T v = t;
    bool okv = cand && body;
    if (__any_sync(0xffffffffu, cand && !body)) {      // an end cap is in play for some env of the warp
        const bool far_end = y >= T(0);
        const T b2 = far_end ? rdoa - bard : rdoa;     // rd . (pos - cap end)
        const T h2 = b2 * b2 - (far_end ? c2b : c2a);
        const T v2 = -b2 - Mth<T>::sqrt_pos(h2 > T(0) ? h2 : T(1));
        if (!body) {
            v = v2;
            okv = cand && (h2 > T(0));
        }
    }
    return (okv && v > T(0) && v < best) ? v : best;
}

// the capsule-shaped record of a sphere for cast_capsule_bf: w = ba[3] oa[3] baba baoa c c2a c2b (obstacle_ray_record layout),
// from the sphere record oc[3], c
template <typename T>
__device__ __forceinline__ void sphere_as_capsule(T w[11]) {
    const T oc0 = w[0], oc1 = w[1], oc2 = w[2], c = w[3];
    w[0] = w[1] = w[2] = T(0);
    w[3] = oc0; w[4] = oc1; w[5] = oc2;
    w[6] = T(1); w[7] = T(0.5); w[8] = c; w[9] = c; w[10] = c;
}

template <typename T>
__device__ __forceinline__ T cast_sphere(const T rd[3], T ocx, T ocy, T ocz, T c, T best) {
    const T b = ocx * rd[0] + ocy * rd[1] + ocz * rd[2];
    const T h = b * b - c;
    if (h >= T(0)) {
        const T v = -b - (h > T(0) ? Mth<T>::sqrt_pos(h) : T(0));
        if (v > T(0) && v < best) best = v;
    }
    return best;
}

// Casts this lane's rays against the obstacles of `mask` (bit k = obstacle k, capsules first; records in shared memory
// at pre_env + k * kPreStride), clamps (sensor.py:117), writes the 2x2 zero-padded max-pool of the distances straight into
// the env's observation row (obs[16:], docking3d.py:487) and returns sum(max((d/d_max)^2, eps_c) * beta) on every lane.
//   R: post-step Rzyx (row-major); poison: 0, or NaN for a non-finite pose.  Must be called by all 32 lanes.
// A non-finite pose makes every capsule test return -inf and every sphere test NaN; where no distance is positive the
// reference takes the value of its FIRST obstacle column (docking3d.py:438-439), which is a capsule whenever the env has
// one (-inf -> max_dist, sensor.py:117) and the sphere column otherwise (NaN).  So the poison is added to every distance
// of sphere-only envs and to none of envs with capsules.
template <typename T, int RPL, bool DBG, typename LANE>
__device__ __forceinline__ T radar_env(const KParams<T> &p, const LANE &rl, const T R[9], T poison, unsigned mask,
                                       const T *pre_env, T *s_ray, int lane, int64_t ie) {
    using P2 = typename Pair<T>::type;
    const int n_caps = p.n_caps, n_sph = p.n_sph, n_r = p.n_rays;
    const T dmax = rl.dmax, inv_dmax = rl.inv_dmax;
    if (n_caps > 0 || n_sph == 0) poison = T(0);
    T best[RPL];
#pragma unroll
    for (int j = 0; j < RPL; j++) best[j] = Mth<T>::inf();
    if (mask) {
        T rd[RPL][3];
#pragma unroll
        for (int j = 0; j < RPL; j++) {
            const T b0 = rl.rb(j, 0), b1 = rl.rb(j, 1), b2 = rl.rb(j, 2);
#pragma unroll
            for (int c = 0; c < 3; c++) rd[j][c] = R[3 * c] * b0 + R[3 * c + 1] * b1 + R[3 * c + 2] * b2;
        }
        unsigned cap_mask = mask & ((1u << n_caps) - 1u);
        unsigned sph_mask = (mask >> n_caps) & ((1u << n_sph) - 1u);
        while (cap_mask) {
            const int k = __ffs(cap_mask) - 1;
            cap_mask &= cap_mask - 1;
            const P2 *w2 = reinterpret_cast<const P2 *>(pre_env + k * kPreStride);
            const P2 v0 = w2[0], v1 = w2[1], v2 = w2[2], v3 = w2[3], v4 = w2[4], v5 = w2[5];
            const T ba[3] = {v0.x, v0.y, v1.x}, oa[3] = {v1.y, v2.x, v2.y};
            const T baba = v3.x, baoa = v3.y, cc = v4.x, c2a = v4.y, c2b = v5.x;
#pragma unroll
            for (int j = 0; j < RPL; j++) best[j] = cast_capsule<T>(rd[j], ba, oa, baba, baoa, cc, c2a, c2b, best[j]);
        }
        while (sph_mask) {
            const int k = __ffs(sph_mask) - 1;
            sph_mask &= sph_mask - 1;
            const P2 *w2 = reinterpret_cast<const P2 *>(pre_env + (n_caps + k) * kPreStride);
            const P2 v0 = w2[0], v1 = w2[1];
#pragma unroll
            for (int j = 0; j < RPL; j++) best[j] = cast_sphere<T>(rd[j], v0.x, v0.y, v1.x, v1.y, best[j]);
        }
    }
    // ---- clamp (sensor.py:117), obstacle-avoidance partial sum (docking3d.py:767-792), stash for pooling
    T oa_part = T(0);
#pragma unroll
    for (int j = 0; j < RPL; j++) {
        const int ir = lane + 32 * j;
        if (ir < n_r) {
            // min positive distance over obstacles (docking3d.py:438-439), max_dist if none or farther
            const T d = (best[j] > dmax ? dmax : best[j]) + poison;
            s_ray[ir] = d;
            if (DBG && p.dbg_ray_dist) p.dbg_ray_dist[(int64_t)ir * p.n_envs + ie] = d;
            // (gamma_c (1 - c))^2 with c = clip(1 - d/d_max, 0, 1): 1 - c = d/d_max for d in [0, d_max]
            const T x = d * inv_dmax;
            const T qq = x * x;
            const T mx = !(qq <= T(0.001)) ? qq : T(0.001);     // np.maximum, NaN propagates
            oa_part += mx * rl.bw(j);
        }
    }
    const T oa_dot = warp_sum<T>(oa_part);
    __syncwarp();
    // ---- 2x2 max-pool with zero padding (sensor.py:131-137) -> obs[16:]
    float *orow = p.obs + ie * p.n_obs + 16;
    if (rl.fast_pool) {
        if (lane < p.n_rr) {
            T mx = s_ray[rl.pidx(0)];
#pragma unroll
            for (int q = 1; q < 4; q++) {
                const T v = s_ray[rl.pidx(q)];
                mx = !(v <= mx) ? v : mx;            // np.max, NaN propagates
            }
            T o = mx * inv_dmax;                     // clip(d / max_dist, 0, 1), docking3d.py:487
            o = o > T(1) ? T(1) : o;
            orow[lane] = (float)o;
            if (DBG && p.dbg_obs) p.dbg_obs[(int64_t)(16 + lane) * p.n_envs + ie] = o;
        }
    } else {
        for (int pc = lane; pc < p.n_rr; pc += 32) {
            const int pr = pc / p.n_hr, pcol = pc - pr * p.n_hr;
            T mx = T(0);
            for (int dv = 0; dv < p.block; dv++)
                for (int dh = 0; dh < p.block; dh++) {
                    const int rv = pr * p.block + dv, rh = pcol * p.block + dh;
                    if (rv < p.n_vert && rh < p.n_horiz) {
                        const T v = s_ray[rv * p.n_horiz + rh];
                        mx = !(v <= mx) ? v : mx;
                    }
                }
            T o = mx * inv_dmax;
            o = o > T(1) ? T(1) : o;
            orow[pc] = (float)o;
            if (DBG && p.dbg_obs) p.dbg_obs[(int64_t)(16 + pc) * p.n_envs + ie] = o;
        }
    }
    __syncwarp();
    return oa_dot;
}

// env i with nothing in view: every ray reads max_dist (sensor.py:113-117), so its pooled cells are all ones
template <typename T>
__device__ __forceinline__ void store_clear_cells(const KParams<T> &p, int64_t i) {
    float *cells = p.obs + i * p.n_obs + 16;
    if ((p.n_obs & 3) == 0 && (p.n_rr & 3) == 0) {
        float4 *c4 = reinterpret_cast<float4 *>(cells);
        for (int c = 0; c < (p.n_rr >> 2); c++) c4[c] = make_float4(1.0f, 1.0f, 1.0f, 1.0f);
    } else {
        for (int c = 0; c < p.n_rr; c++) cells[c] = 1.0f;
    }
}

}  // namespace dockauv
