// dockauv_device.cuh -- per-env device functions of the docking-AUV step (sm_100a).
//
// Formulation is matrix-free (SURVEY.md 9): the 6x6 Coriolis and damping matrices of the reference
// (gym_dockauv/objects/statespace.py:199-351) are never materialised, C(nu) nu is four cross products, D(nu) nu
// is a handful of FMAs, and the dead sixth Runge-Kutta stage (utils/odesolver45.py:23-27) is not evaluated.
// Position does not feed back into the ODE right-hand side, so only Theta (3) and nu_r (6) carry stage
// vectors; position is accumulated straight into the 4th-order result.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "dockauv_kparams.h"

namespace dockauv {

// ------------------------------------------------------------------------------------------- math traits
template <typename T>
struct Mth;

// The library sincos() carries a large Payne-Hanek slow path; inlining it at every call site made the step kernels
// > 170 KB of SASS (instruction-cache misses were 11 % of the stall samples).  One out-of-line copy instead.
static __device__ __noinline__ double2 sincos_outlined(double x) {
    double s, c;
    sincos(x, &s, &c);
    return make_double2(s, c);
}

template <>
struct Mth<double> {
    static constexpr double pi = 3.141592653589793;
    static constexpr double two_pi = 6.283185307179586;
    static constexpr double half_pi = 1.5707963267948966;
    static constexpr double inv_pi = 0.3183098861837907, inv_half_pi = 0.6366197723675814;
    static __device__ __forceinline__ double inf() { return CUDART_INF; }
    static __device__ __forceinline__ double min_normal() { return 2.2250738585072014e-308; }
    static __device__ __forceinline__ double nan() { return CUDART_NAN; }
    static __device__ __forceinline__ void sincos_(double x, double *s, double *c) {
        const double2 r = sincos_outlined(x);
        *s = r.x;
        *c = r.y;
    }
    static __device__ __forceinline__ double fma_(double a, double b, double c) { return __fma_rn(a, b, c); }
    static __device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }   // never contracted
    static __device__ __forceinline__ double sqrt_(double x) { return sqrt(x); }
    static __device__ __forceinline__ double abs_(double x) { return fabs(x); }
    static __device__ __forceinline__ double atan2_(double y, double x) { return atan2(y, x); }
    static __device__ __forceinline__ double log_(double x) { return log(x); }
    static __device__ __forceinline__ double fmod_(double x, double y) { return fmod(x, y); }
    static __device__ __forceinline__ double hypot_(double x, double y) { return hypot(x, y); }
    static __device__ __forceinline__ double cos_(double x) { return cos(x); }
    static __device__ __forceinline__ double sin_(double x) { return sin(x); }
    // Branch-free sqrt / reciprocal for the ray hit path (a handful of lanes per warp get there, so every instruction
    // of the library versions -- ~20 + ~25 with their slow-path checks -- is paid at 1/6 lane utilisation): hardware
    // seed (upper ~20 mantissa bits, full double range) + Newton steps; relative error ~2e-16, NaN / inf for
    // non-positive or non-finite input like the library versions.
    // (seed: >= 20 good bits; one Newton step for 1 / sqrt(x) -> 2^-40, then the correction s + r/2 (x - s^2) squares the
    // error again: 1 ulp, checked numerically for seeds of 20 and 22 bits)
    static __device__ __forceinline__ double sqrt_pos(double x) {
        double r;
        asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
        const double hx = 0.5 * x;
        r = r * fma(-hx * r, r, 1.5);
        double s = x * r;
        s = fma(0.5 * r, fma(-s, s, x), s);
        return s;
    }
    static __device__ __forceinline__ double rsqrt_pos(double x) {      // 1 / sqrt(x), x > 0
        double r;
        asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
        const double hx = 0.5 * x;
        r = r * fma(-hx * r, r, 1.5);
        r = r * fma(-hx * r, r, 1.5);
        return r;
    }
    static __device__ __forceinline__ double rcp_(double x) {
        double y;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
        y = fma(y, fma(-x, y, 1.0), y);
        y = fma(y, fma(-x, y, 1.0), y);
        return y;
    }
};

template <>
struct Mth<float> {
    static constexpr float pi = 3.14159265358979f;
    static constexpr float two_pi = 6.28318530717959f;
    static constexpr float half_pi = 1.57079632679490f;
    static constexpr float inv_pi = 0.318309886183791f, inv_half_pi = 0.636619772367581f;
    static __device__ __forceinline__ float inf() { return CUDART_INF_F; }
    static __device__ __forceinline__ float min_normal() { return 1.17549435e-38f; }
    static __device__ __forceinline__ float nan() { return CUDART_NAN_F; }
    static __device__ __forceinline__ void sincos_(float x, float *s, float *c) { sincosf(x, s, c); }
    static __device__ __forceinline__ float fma_(float a, float b, float c) { return __fmaf_rn(a, b, c); }
    static __device__ __forceinline__ float mul_(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float sqrt_(float x) { return sqrtf(x); }
    static __device__ __forceinline__ float abs_(float x) { return fabsf(x); }
    static __device__ __forceinline__ float atan2_(float y, float x) { return atan2f(y, x); }
    static __device__ __forceinline__ float log_(float x) { return logf(x); }
    static __device__ __forceinline__ float fmod_(float x, float y) { return fmodf(x, y); }
    static __device__ __forceinline__ float hypot_(float x, float y) { return hypotf(x, y); }
    static __device__ __forceinline__ float cos_(float x) { return cosf(x); }
    static __device__ __forceinline__ float sin_(float x) { return sinf(x); }
    static __device__ __forceinline__ float sqrt_pos(float x) { return sqrtf(x); }
    static __device__ __forceinline__ float rsqrt_pos(float x) { return 1.0f / sqrtf(x); }
    static __device__ __forceinline__ float rcp_(float x) { return 1.0f / x; }
};

// np.clip: minimum(maximum(x, lo), hi) -- NaN propagates
template <typename T>
__device__ __forceinline__ T clipv(T x, T lo, T hi) {
    return x < lo ? lo : (x > hi ? hi : x);
}

// general path of ssa (numpy floor-mod via fmod); cold: only angles beyond +-3 pi (blown-up LAUV states) get here
template <typename T>
static __device__ __noinline__ T ssa_general(T x) {
    const T pi = Mth<T>::pi, two_pi = Mth<T>::two_pi;
    T mod = Mth<T>::fmod_(x + pi, two_pi);
    if (mod != T(0)) {
        if (mod < T(0)) mod += two_pi;
    } else {
        mod = T(0);
    }
    return mod - pi;
}

// geomutils.py:4-11  ssa(x) = (x + pi) % (2 pi) - pi with numpy's floor-mod.  For |x| < 3 pi the modulo is a
// single conditional add/subtract (bit-identical to fmod there); the general path handles anything else.
template <typename T>
__device__ __forceinline__ T ssa(T x) {
    const T pi = Mth<T>::pi, two_pi = Mth<T>::two_pi;
    if (Mth<T>::abs_(x) < T(9.0)) {
        T a = x + pi;
        if (a >= two_pi) a -= two_pi;
        else if (a < T(0)) a += two_pi;
        return a - pi;
    }
    return ssa_general<T>(x);
}

// sin / cos of (a + d) from (sin a, cos a) by angle addition.  The Runge-Kutta stage angles and the post-step
// attitude are small shifts of the pre-step attitude (d = h * sum(a_ij k_j), |d| ~ h |Theta_dot|), so for
// |d| <= 0.5 sin d and cos d - 1 are short Taylor polynomials (truncation < 5e-17 relative) instead of a library
// sincos (~150 instructions with its range reduction); larger shifts and NaN / inf take the library call.
// The result differs from sincos(a + d) by ~1 ulp, three orders of magnitude inside the 1e-9 budget (SURVEY.md 8c).
// (Measured and not kept: a first tier |d| <= 1/4 with one coefficient less per polynomial and everything else out of
// line -- 28 DFMAs less per step, no faster; with the first tier at 1/8 one env in four of the C4 workload, whose roll
// and yaw rates reach 2.5 rad/s, fell through to the library call: 8 % slower.)
// Taylor coefficients of sin d / d - 1 and cos d - 1 in d^2, in constant memory: a 64-bit literal costs two UMOVs in
// front of every DFMA that uses it, a constant-bank word one load (or none)
__constant__ double kTaylorSin[6] = {1.0 / 6227020800.0, -1.0 / 39916800.0, 1.0 / 362880.0, -1.0 / 5040.0, 1.0 / 120.0, -1.0 / 6.0};
__constant__ double kTaylorCos[7] = {-1.0 / 87178291200.0, 1.0 / 479001600.0, -1.0 / 3628800.0, 1.0 / 40320.0, -1.0 / 720.0,
                                     1.0 / 24.0, -0.5};

template <typename T>
__device__ __forceinline__ void sincos_shift(T s0, T c0, T d, T *s, T *c) {
    T sd, cm1;
    if (Mth<T>::abs_(d) <= T(0.5)) {
        const T d2 = d * d;
        T ps = (T)kTaylorSin[0];
#pragma unroll
        for (int k = 1; k < 6; k++) ps = ps * d2 + (T)kTaylorSin[k];
        sd = (d * d2) * ps + d;
        T pc = (T)kTaylorCos[0];
#pragma unroll
        for (int k = 1; k < 7; k++) pc = pc * d2 + (T)kTaylorCos[k];
        cm1 = d2 * pc;
    } else {
        T cd;
        Mth<T>::sincos_(d, &sd, &cd);
        cm1 = cd - T(1);
    }
    *s = s0 + (s0 * cm1 + c0 * sd);
    *c = c0 + (c0 * cm1 - s0 * sd);
}

// cold-path logarithm (epsilon guards that practically never trigger): out of line to keep the hot code small
template <typename T>
static __device__ __noinline__ T log_cold(T x) {
    return Mth<T>::log_(x);
}

// ------------------------------------------------------------------------------------------- Philox4x32-10
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

// uniform double in [0,1): draw `idx` of the stream keyed by (seed, global env id, episode); one Philox block
// yields two draws (even idx -> words 0,1; odd idx -> words 2,3).
__device__ __forceinline__ double philox_uniform(uint64_t seed, uint64_t env_id, uint32_t episode, uint32_t idx) {
    uint32_t c[4] = {(uint32_t)env_id, (uint32_t)(env_id >> 32), episode, idx >> 1};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    uint32_t hi = (idx & 1) ? c[2] : c[0], lo = (idx & 1) ? c[3] : c[1];
    return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) * (1.0 / 9007199254740992.0);
}

// both uniforms of Philox block `blk` of the stream (seed, env id, episode): u[0] = draw 2*blk, u[1] = draw 2*blk+1
__device__ __forceinline__ void philox_uniform_pair(uint64_t seed, uint64_t env_id, uint32_t episode, uint32_t blk,
                                                    double u[2]) {
    uint32_t c[4] = {(uint32_t)env_id, (uint32_t)(env_id >> 32), episode, blk};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    u[0] = ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6)) * (1.0 / 9007199254740992.0);
    u[1] = ((double)(c[2] >> 5) * 67108864.0 + (double)(c[3] >> 6)) * (1.0 / 9007199254740992.0);
}

// standard normal from the per-step stream (Box-Muller); counter word 3 = 0x80000000 | t_steps keeps it apart
// from the reset stream of the same episode.
__device__ __forceinline__ double philox_normal(uint64_t seed, uint64_t env_id, uint32_t episode, uint32_t t_steps) {
    uint32_t c[4] = {(uint32_t)env_id, (uint32_t)(env_id >> 32), episode, 0x80000000u | t_steps};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    double u1 = ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6) + 1.0) * (1.0 / 9007199254740992.0);
    double u2 = ((double)(c[2] >> 5) * 67108864.0 + (double)(c[3] >> 6)) * (1.0 / 9007199254740992.0);
    return sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
}

// ------------------------------------------------------------------------------------------- dynamics
template <typename T>
__device__ __forceinline__ void cross3(const T a[3], const T b[3], T o[3]) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}

// Kinetic part of auvsim.py:152-158:  nu_dot = M^-1 (B(nu) u - D(nu) nu - C(nu) nu - G(eta)).
//   tau : BlueROV2 -> precomputed B u (B is constant, BlueROV2.py:74-75); LAUV -> the low-passed command u[3]
//   sphi, cphi, sth, cth : sin/cos of roll and pitch
template <typename T, int VEH, bool SPM = false>
__device__ __forceinline__ void nu_dot(const KParams<T> &p, const T nu[6], const T tau[6], T sphi, T cphi, T sth,
                                       T cth, T out[6]) {
    const T *n1 = nu, *n2 = nu + 3;
    T f[6];
    // control forces
    if (VEH == DOCKAUV_VEHICLE_BLUEROV2) {
#pragma unroll
        for (int i = 0; i < 6; i++) f[i] = tau[i];
    } else {   // LAUV.py:59-67
        T u2 = nu[0] * nu[0];
        f[0] = tau[0];
        f[1] = p.lauv_B[0] * u2 * tau[1];
        f[2] = p.lauv_B[1] * u2 * tau[2];
        f[3] = T(0);
        f[4] = p.lauv_B[2] * u2 * tau[2];
        f[5] = p.lauv_B[3] * u2 * tau[1];
    }
    // D(nu) nu, statespace.py:337-351 / LAUV.py:69-101.  D[i][j] = -(lin + quad |nu_j| + lift |u|)
    {
        T an[6];
#pragma unroll
        for (int i = 0; i < 6; i++) an[i] = Mth<T>::abs_(nu[i]);
        T d[6];
        if (VEH == DOCKAUV_VEHICLE_BLUEROV2) {
#pragma unroll
            for (int i = 0; i < 6; i++) d[i] = -(p.D_lin[i] + p.D_quad[i] * an[i]) * nu[i];
        } else {
            T au = an[0];
#pragma unroll
            for (int i = 0; i < 6; i++) d[i] = -(p.D_lin[i] + p.D_quad[i] * an[i] + p.D_lift[i] * au) * nu[i];
            d[1] += -(p.D_lin[6] + p.D_quad[6] * an[5] + p.D_lift[6] * au) * nu[5];
            d[2] += -(p.D_lin[7] + p.D_quad[7] * an[4] + p.D_lift[7] * au) * nu[4];
            d[4] += -(p.D_lin[8] + p.D_quad[8] * an[2] + p.D_lift[8] * au) * nu[2];
            d[5] += -(p.D_lin[9] + p.D_quad[9] * an[1] + p.D_lift[9] * au) * nu[1];
        }
#pragma unroll
        for (int i = 0; i < 6; i++) f[i] -= d[i];
    }
    // C(nu) nu = C_RB nu + C_A nu, statespace.py:224-227, 271-274
    {
        T c1[3], rgn2[3], t[3], rgc1[3], ibn2[3], t2[3];
        cross3(n2, n1, c1);                 // nu2 x nu1
        if (SPM) {
            // centre of gravity on the z axis and a diagonal I_b (what SPM stands for, checked on the host): the products
            // with the exact zeros of r_G and I_b are left out.  Every term that remains is rounded exactly as in the
            // general form (x * y - 0 * w and 0 * w + x * y are x * y), so finite results are identical bit for bit; a
            // non-finite velocity still makes some f[i] non-finite through D(nu) nu and the poison term below does the rest
            const T zg = p.r_G[2];
            rgn2[0] = -(zg * n2[1]); rgn2[1] = zg * n2[0]; rgn2[2] = T(0);             // r_G x nu2
            t[0] = -Mth<T>::mul_(n2[2], rgn2[1]); t[1] = Mth<T>::mul_(n2[2], rgn2[0]);  // nu2 x (r_G x nu2); never fused into c1 - t
            t[2] = n2[0] * rgn2[1] - n2[1] * rgn2[0];
            rgc1[0] = -(zg * c1[1]); rgc1[1] = zg * c1[0]; rgc1[2] = T(0);             // r_G x (nu2 x nu1)
            ibn2[0] = p.I_b[0] * n2[0]; ibn2[1] = p.I_b[4] * n2[1]; ibn2[2] = p.I_b[8] * n2[2];
        } else {
            cross3(p.r_G, n2, rgn2);            // r_G x nu2
            cross3(n2, rgn2, t);                // nu2 x (r_G x nu2)
            cross3(p.r_G, c1, rgc1);            // r_G x (nu2 x nu1)
#pragma unroll
            for (int i = 0; i < 3; i++) ibn2[i] = p.I_b[3 * i] * n2[0] + p.I_b[3 * i + 1] * n2[1] + p.I_b[3 * i + 2] * n2[2];
        }
        cross3(ibn2, n2, t2);               // (I_b nu2) x nu2
        T a1[3] = {p.MA[0] * n1[0], p.MA[1] * n1[1], p.MA[2] * n1[2]};
        T a2[3] = {p.MA[3] * n2[0], p.MA[4] * n2[1], p.MA[5] * n2[2]};
        T a1n2[3], a1n1[3], a2n2[3];
        cross3(a1, n2, a1n2);
        cross3(a1, n1, a1n1);
        cross3(a2, n2, a2n2);
#pragma unroll
        for (int i = 0; i < 3; i++) {
            f[i] -= p.m * (c1[i] - t[i]) - a1n2[i];
            f[3 + i] -= p.m * rgc1[i] - t2[i] - a1n1[i] - a2n2[i];
        }
    }
    // G(eta), statespace.py:387-396
    {
        T cc = cth * cphi, cs = cth * sphi;
        f[0] -= p.G_WB * sth;
        f[1] -= -p.G_WB * cs;
        f[2] -= -p.G_WB * cc;
        if (SPM) {      // centres of gravity and buoyancy on the z axis: G_r[0] = G_r[1] = 0 (host-checked), same bits as below
            f[3] -= Mth<T>::mul_(p.G_r[2], cs);
            f[4] -= Mth<T>::mul_(p.G_r[2], sth);
        } else {
            f[3] -= -p.G_r[1] * cc + p.G_r[2] * cs;
            f[4] -= p.G_r[2] * sth + p.G_r[0] * cc;
            f[5] -= -p.G_r[0] * cs - p.G_r[1] * sth;
        }
    }
    if (SPM) {
        // M_inv of a vehicle whose centre of gravity is offset along z only (both stock vehicles): ten non-zeros, the
        // diagonal and [0,4] [4,0] [1,3] [3,1].  The dense product adds exact zeros for the other 26 entries -- unless
        // a component of f is inf / NaN, in which case 0 * f poisons EVERY row; `z` keeps that behaviour.
        const T z = (((f[0] + f[1]) + (f[2] + f[3])) + (f[4] + f[5])) * T(0);
        // same operation order as the dense loop below (first product rounded, the second one fused into it), so the two
        // forms give identical bits for finite f
        out[0] = Mth<T>::fma_(p.M_inv[4], f[4], Mth<T>::mul_(p.M_inv[0], f[0])) + z;
        out[1] = Mth<T>::fma_(p.M_inv[9], f[3], Mth<T>::mul_(p.M_inv[7], f[1])) + z;
        out[2] = Mth<T>::mul_(p.M_inv[14], f[2]) + z;
        out[3] = Mth<T>::fma_(p.M_inv[21], f[3], Mth<T>::mul_(p.M_inv[19], f[1])) + z;
        out[4] = Mth<T>::fma_(p.M_inv[28], f[4], Mth<T>::mul_(p.M_inv[24], f[0])) + z;
        out[5] = Mth<T>::mul_(p.M_inv[35], f[5]) + z;
    } else {
#pragma unroll
        for (int i = 0; i < 6; i++) {
            T s = p.M_inv[6 * i] * f[0];
#pragma unroll
            for (int k = 1; k < 6; k++) s += p.M_inv[6 * i + k] * f[k];
            out[i] = s;
        }
    }
}

// Rzyx (geomutils.py:40-43) from precomputed sines / cosines, row-major
template <typename T>
__device__ __forceinline__ void rzyx(T sphi, T cphi, T sth, T cth, T spsi, T cpsi, T R[9]) {
    R[0] = cpsi * cth; R[1] = -spsi * cphi + cpsi * sth * sphi; R[2] = spsi * sphi + cpsi * cphi * sth;
    R[3] = spsi * cth; R[4] = cpsi * cphi + sphi * sth * spsi;  R[5] = -cpsi * sphi + sth * spsi * cphi;
    R[6] = -sth;       R[7] = cth * sphi;                       R[8] = cth * cphi;
}

// parked values (shared memory, stride ST != 1) are read through volatile: ptxas otherwise hoists the loads to the top
// of the integration and spills exactly as before
template <int ST, typename T>
__device__ __forceinline__ T parked(const T *q, int i) {
    if (ST == 1) return q[i];
    return reinterpret_cast<const volatile T *>(q)[i * ST];
}

// One evaluation of the reduced right-hand side (auvsim.py:110-160) at y = (Theta, nu_r).
//   tr = sin/cos of (phi, theta, psi) at y: {sphi, cphi, sth, cth, spsi, cpsi} (psi only read if WPOS)
//   k[0:3] = T(phi, theta) nu2 (geomutils.py:72-75), k[3:9] = nu_dot;  if WPOS, pacc += wpos * R(Theta) (nu1 + nu_c).
//   CUR = false: no ocean current (nu_c is not read).
template <typename T, int VEH, bool WPOS, bool SPM = false, bool CUR = true, int ST = 1>
__device__ __forceinline__ void rhs9(const KParams<T> &p, const T y[9], const T tr[6], const T *tau_s, const T nu_c[3],
                                     T wpos, T pacc[3], T k[9]) {
    T tau[6];
#pragma unroll
    for (int i = 0; i < 6; i++) tau[i] = parked<ST>(tau_s, i);
    const T sphi = tr[0], cphi = tr[1], sth = tr[2], cth = tr[3];
    const T *nu = y + 3;
    T inv_cth = Mth<T>::rcp_(cth);      // reciprocal by two Newton steps (~2e-16 relative): a fifth of the IEEE division's instructions
    T tth = sth * inv_cth;
    T qs = sphi * nu[4] + cphi * nu[5];
    k[0] = nu[3] + tth * qs;
    k[1] = cphi * nu[4] - sphi * nu[5];
    k[2] = qs * inv_cth;
    if (WPOS) {
        T R[9];
        rzyx(sphi, cphi, sth, cth, tr[4], tr[5], R);
        T v[3];
        if (CUR) {
            v[0] = nu[0] + nu_c[0]; v[1] = nu[1] + nu_c[1]; v[2] = nu[2] + nu_c[2];
        } else {
            v[0] = nu[0]; v[1] = nu[1]; v[2] = nu[2];
        }
#pragma unroll
        for (int i = 0; i < 3; i++) pacc[i] += wpos * (R[3 * i] * v[0] + R[3 * i + 1] * v[1] + R[3 * i + 2] * v[2]);
    }
    nu_dot<T, VEH, SPM>(p, nu, tau, sphi, cphi, sth, cth, k + 3);
}

// sin/cos of the stage attitude Theta0 + d from the pre-step values tr0 (psi skipped when the stage has no position weight)
template <typename T, bool WPSI, int ST = 1>
__device__ __forceinline__ void stage_trig(const T *tr0, const T d[3], T tr[6]) {
    sincos_shift<T>(parked<ST>(tr0, 0), parked<ST>(tr0, 1), d[0], &tr[0], &tr[1]);
    sincos_shift<T>(parked<ST>(tr0, 2), parked<ST>(tr0, 3), d[1], &tr[2], &tr[3]);
    if (WPSI) sincos_shift<T>(parked<ST>(tr0, 4), parked<ST>(tr0, 5), d[2], &tr[4], &tr[5]);
}

// utils/odesolver45.py:18-26 on the reduced state y = (Theta, nu_r); the 4th-order result is written back to y and the
// position increment h sum(b_i R(Theta_i)(nu1_i + nu_c)) is returned in pacc (position does not feed back).
//   tr0: sin/cos of the pre-step attitude y[0:3]; tr1 (out): sin/cos of the post-step attitude (before ssa, which
//   does not change them).
// Register pressure decides the speed of this function (the dynamics launch is latency-bound at 16 warps per SM), so
// the stage derivatives are not kept until they are last used: as soon as k3 exists, the partial sums of the two
// combinations that still need k1..k3 (the stage-5 input and the result) are formed and k1..k3 die; the sums are
// continued with k4 / k5 in the same left-to-right order as written in the tableau, so nothing changes numerically.
//   ST: stride of y / tr0 / tau (1 = plain arrays; the dynamics launch can park them in shared memory, [word][thread])
template <typename T, int VEH, bool SPM = false, bool CUR = true, int ST = 1>
__device__ __forceinline__ void rkf45_step(const KParams<T> &p, T *y, const T *tr0, const T *tau, const T nu_c[3],
                                           T pacc[3], T tr1[6]) {
    const T h = p.h;
    T yt[9], dy[9], tr[6];
    T d5[9], dw[9];      // running sums: stage-5 input increment, result increment
    pacc[0] = pacc[1] = pacc[2] = T(0);
    {
        T k1[9], k2[9], k3[9];
        T y0[9], tr0r[6];
#pragma unroll
        for (int i = 0; i < 9; i++) y0[i] = parked<ST>(y, i);
#pragma unroll
        for (int i = 0; i < 6; i++) tr0r[i] = parked<ST>(tr0, i);
        rhs9<T, VEH, true, SPM, CUR, ST>(p, y0, tr0r, tau, nu_c, h * T(25.0 / 216.0), pacc, k1);
        {
            const T a = h * T(0.25);
#pragma unroll
            for (int i = 0; i < 9; i++) {
                dy[i] = a * k1[i];
                yt[i] = parked<ST>(y, i) + dy[i];
            }
        }
        stage_trig<T, false, ST>(tr0, dy, tr);
        rhs9<T, VEH, false, SPM, CUR, ST>(p, yt, tr, tau, nu_c, T(0), pacc, k2);   // b2 = 0: no position contribution
        {
            const T a = h * T(3.0 / 32.0), b = h * T(9.0 / 32.0);
#pragma unroll
            for (int i = 0; i < 9; i++) {
                dy[i] = a * k1[i] + b * k2[i];
                yt[i] = parked<ST>(y, i) + dy[i];
            }
        }
        stage_trig<T, true, ST>(tr0, dy, tr);
        rhs9<T, VEH, true, SPM, CUR, ST>(p, yt, tr, tau, nu_c, h * T(1408.0 / 2565.0), pacc, k3);
        {
            const T a = h * T(1932.0 / 2197.0), b = h * T(-7200.0 / 2197.0), c = h * T(7296.0 / 2197.0);
            const T a5 = h * T(439.0 / 216.0), b5 = h * T(-8.0), c5 = h * T(3680.0 / 513.0);
            const T aw = h * T(25.0 / 216.0), cw = h * T(1408.0 / 2565.0);
#pragma unroll
            for (int i = 0; i < 9; i++) {
                dy[i] = a * k1[i] + b * k2[i] + c * k3[i];
                yt[i] = parked<ST>(y, i) + dy[i];
                d5[i] = a5 * k1[i] + b5 * k2[i] + c5 * k3[i];
                dw[i] = aw * k1[i] + cw * k3[i];
            }
        }
    }
    stage_trig<T, true, ST>(tr0, dy, tr);
    {
        T k4[9];
        rhs9<T, VEH, true, SPM, CUR, ST>(p, yt, tr, tau, nu_c, h * T(2197.0 / 4104.0), pacc, k4);
        const T d = h * T(-845.0 / 4104.0), dwc = h * T(2197.0 / 4104.0);
#pragma unroll
        for (int i = 0; i < 9; i++) {
            d5[i] = d5[i] + d * k4[i];
            yt[i] = parked<ST>(y, i) + d5[i];
            dw[i] = dw[i] + dwc * k4[i];
        }
    }
    stage_trig<T, true, ST>(tr0, d5, tr);
    {
        T k5[9];
        rhs9<T, VEH, true, SPM, CUR, ST>(p, yt, tr, tau, nu_c, h * T(-1.0 / 5.0), pacc, k5);
        const T e = h * T(-1.0 / 5.0);
#pragma unroll
        for (int i = 0; i < 9; i++) {
            dw[i] = dw[i] + e * k5[i];
            y[i * ST] = parked<ST>(y, i) + dw[i];
        }
    }
    stage_trig<T, true, ST>(tr0, dw, tr1);
}

// ------------------------------------------------------------------------------------------- radar geometry
// Ray-independent part of the ray/capsule test (all rays of one env share the origin, sensor.py:123-129).
template <typename T>
struct CapPre {
    T ba[3], oa[3], oc2[3];   // top-bot, pos-bot, pos-top
    T baba, baoa, c, c2a, c2b, r;
};

template <typename T>
__device__ __forceinline__ void capsule_pre(const T pos[3], const T bot[3], const T top[3], T r, CapPre<T> &q) {
#pragma unroll
    for (int i = 0; i < 3; i++) {
        q.ba[i] = top[i] - bot[i];
        q.oa[i] = pos[i] - bot[i];
        q.oc2[i] = pos[i] - top[i];
    }
    q.baba = q.ba[0] * q.ba[0] + q.ba[1] * q.ba[1] + q.ba[2] * q.ba[2];
    q.baoa = q.oa[0] * q.ba[0] + q.oa[1] * q.ba[1] + q.oa[2] * q.ba[2];
    T oaoa = q.oa[0] * q.oa[0] + q.oa[1] * q.oa[1] + q.oa[2] * q.oa[2];
    T r2 = r * r;
    q.c = q.baba * oaoa - q.baoa * q.baoa - r2 * q.baba;
    q.c2a = oaoa - r2;
    q.c2b = q.oc2[0] * q.oc2[0] + q.oc2[1] * q.oc2[1] + q.oc2[2] * q.oc2[2] - r2;
    q.r = r;
}

// sphere centre to vehicle: oc = pos - c, d2 = |oc|^2
template <typename T>
__device__ __forceinline__ void sphere_offset(const T pos[3], const T c[3], T oc[3], T &d2) {
    d2 = T(0);
#pragma unroll
    for (int k = 0; k < 3; k++) {
        oc[k] = pos[k] - c[k];
        d2 += oc[k] * oc[k];
    }
}

// The record the ray tests read -- capsule: ba[3] oa[3] baba baoa c c2a c2b, sphere: oc[3] c
template <typename T>
__device__ __forceinline__ void capsule_ray_record(const CapPre<T> &q, T *w) {
    w[0] = q.ba[0]; w[1] = q.ba[1]; w[2] = q.ba[2];
    w[3] = q.oa[0]; w[4] = q.oa[1]; w[5] = q.oa[2];
    w[6] = q.baba; w[7] = q.baoa; w[8] = q.c; w[9] = q.c2a; w[10] = q.c2b;
}

template <typename T>
__device__ __forceinline__ void sphere_ray_record(const T oc[3], T d2, T rad, T *w) {
    w[0] = oc[0]; w[1] = oc[1]; w[2] = oc[2]; w[3] = d2 - rad * rad;
}

// a length from its square: 0 stays 0, NaN stays NaN
template <typename T>
__device__ __forceinline__ T length_from_sq(T d2) {
    return d2 > T(0) ? Mth<T>::sqrt_pos(d2) : d2;
}

// Distance from the vehicle to the capsule's axis segment: dist_line_point (shape.py:393-417) with one reciprocal instead
// of three divisions and hypot.  inv_n (out): 1 / |top - bot|
template <typename T>
__device__ __forceinline__ T capsule_axis_dist(const CapPre<T> &q, T &inv_n) {
    inv_n = Mth<T>::rsqrt_pos(q.baba);
    const T sp = -q.baoa * inv_n;                                                         // (bot - pos) . d
    const T tp = (q.oc2[0] * q.ba[0] + q.oc2[1] * q.ba[1] + q.oc2[2] * q.ba[2]) * inv_n;  // (pos - top) . d
    T hh = sp;
    if (tp > hh || tp != tp) hh = tp;
    if (T(0) > hh) hh = T(0);
    T cr[3];
    cross3(q.oa, q.ba, cr);
    const T perp2 = (cr[0] * cr[0] + cr[1] * cr[1] + cr[2] * cr[2]) * (inv_n * inv_n);
    return length_from_sq(hh * hh + perp2);
}

// Ray-independent work for one (env, obstacle) pair, shared by every radar layout:
//   * the ray-test record (written if REC);
//   * the body-collision test (shape.py:182-210 with the safety radius of auvsim.py:43);
//   * two exact radar culls.  A culled obstacle can only yield "no positive distance" or a distance beyond max_dist,
//     both of which end as max_dist (sensor.py:117):
//       - range: nearest surface point farther than max_dist;
//       - field of view: the part of the obstacle a ray can reach lies entirely outside one of the five planes of the
//         ray pyramid {x >= 0, |y| <= ty x, |z| <= tz x} (body frame), in which every ray direction lies.  Only axis
//         points within max_dist + r of the vehicle can carry reachable surface points, so a capsule axis is first
//         clipped to that ball (a 40 m pillar seen under roll / pitch otherwise has its far ends on both sides of every
//         plane):  |bot + s ba - pos|^2 <= Rr^2  <=>  s in [(baoa - sqrt(D)) / baba, (baoa + sqrt(D)) / baba].
//   pos: vehicle position, Rm: Rzyx row-major (9 words), ob: raw obstacle (capsule: bot[3] top[3] r; sphere: c[3] r)
template <typename T, bool REC>
__device__ __forceinline__ void obstacle_pair(const KParams<T> &p, const T pos[3], const T *Rm, const T ob[7], bool is_cap,
                                              T *w, bool &hit_body, bool &in_view) {
    const T cull = p.radar_max_dist * T(1.000001);
    T rad, dist;
    T q0[3], q1[3];     // end points of the reachable part of the obstacle axis relative to the vehicle, NED
    bool axis_out = false;
    if (is_cap) {
        const T bot[3] = {ob[0], ob[1], ob[2]}, top[3] = {ob[3], ob[4], ob[5]};
        rad = ob[6];
        CapPre<T> q;
        capsule_pre<T>(pos, bot, top, rad, q);
        if (REC) capsule_ray_record<T>(q, w);
        T inv_n;
        dist = capsule_axis_dist<T>(q, inv_n);
        const T Rr = (cull + rad) * T(1.000001);
        const T oaoa = q.c2a + rad * rad;
        const T D = q.baoa * q.baoa - q.baba * (oaoa - Rr * Rr);
        const T sq = D > T(0) ? Mth<T>::sqrt_pos(D) : T(0);
        const T inv_baba = inv_n * inv_n;
        T s_lo = (q.baoa - sq) * inv_baba, s_hi = (q.baoa + sq) * inv_baba;
        s_lo = s_lo > T(0) ? s_lo : T(0);
        s_hi = s_hi < T(1) ? s_hi : T(1);
        axis_out = (D < T(0)) || (s_lo > s_hi);
#pragma unroll
        for (int c = 0; c < 3; c++) {
            q0[c] = s_lo * q.ba[c] - q.oa[c];
            q1[c] = s_hi * q.ba[c] - q.oa[c];
        }
    } else {
        T oc[3], d2;
        sphere_offset<T>(pos, ob, oc, d2);
        rad = ob[3];
        if (REC) sphere_ray_record<T>(oc, d2, rad, w);
        dist = length_from_sq(d2);
#pragma unroll
        for (int c = 0; c < 3; c++) q0[c] = q1[c] = -oc[c];
    }
    hit_body = dist <= rad + p.safety_radius;
    bool outside = (dist - rad > cull) || axis_out;
    {
        T a0[3], a1[3];    // body-frame coordinates R^T q
#pragma unroll
        for (int c = 0; c < 3; c++) {
            a0[c] = Rm[c] * q0[0] + Rm[3 + c] * q0[1] + Rm[6 + c] * q0[2];
            a1[c] = Rm[c] * q1[0] + Rm[3 + c] * q1[1] + Rm[6 + c] * q1[2];
        }
        // (clipping the segment against all five planes at once -- exact for segments that leave the pyramid through
        // different planes -- lists 24 % instead of 28 % of the C4 envs but costs more in the cull than it saves in the
        // ray launch: measured, profiles/r01/NOTES.md)
        const T rm = rad * T(1.000001) + T(1e-9);
        const T ry = rm * p.fov_ny, rz = rm * p.fov_nz;
        const T ty = p.fov_ty, tz = p.fov_tz;
        outside |= (a0[0] < -rm) && (a1[0] < -rm);
        outside |= (a0[1] - ty * a0[0] > ry) && (a1[1] - ty * a1[0] > ry);
        outside |= (-a0[1] - ty * a0[0] > ry) && (-a1[1] - ty * a1[0] > ry);
        outside |= (a0[2] - tz * a0[0] > rz) && (a1[2] - tz * a1[0] > rz);
        outside |= (-a0[2] - tz * a0[0] > rz) && (-a1[2] - tz * a1[0] > rz);
    }
    in_view = !outside;
}

// Just the ray-test record of obstacle_pair: what the ray launch needs once the cull code has decided collision and
// visibility.
template <typename T>
__device__ __forceinline__ void obstacle_ray_record(const T pos[3], const T ob[7], bool is_cap, T *w) {
    if (is_cap) {
        const T bot[3] = {ob[0], ob[1], ob[2]}, top[3] = {ob[3], ob[4], ob[5]};
        CapPre<T> q;
        capsule_pre<T>(pos, bot, top, ob[6], q);
        capsule_ray_record<T>(q, w);
    } else {
        T oc[3], d2;
        sphere_offset<T>(pos, ob, oc, d2);
        sphere_ray_record<T>(oc, d2, ob[3], w);
    }
}

// Just the body-collision decision of obstacle_pair: used by the cull code for the pairs its float pre-test leaves
// undecided.
template <typename T>
__device__ __forceinline__ bool obstacle_body_hit(const KParams<T> &p, const T pos[3], const T ob[7], bool is_cap) {
    T rad, dist;
    if (is_cap) {
        const T bot[3] = {ob[0], ob[1], ob[2]}, top[3] = {ob[3], ob[4], ob[5]};
        rad = ob[6];
        CapPre<T> q;
        capsule_pre<T>(pos, bot, top, rad, q);
        T inv_n;
        dist = capsule_axis_dist<T>(q, inv_n);
    } else {
        T oc[3], d2;
        sphere_offset<T>(pos, ob, oc, d2);
        rad = ob[3];
        dist = length_from_sq(d2);
    }
    return dist <= rad + p.safety_radius;
}

// The culls and the body-collision pre-test of obstacle_pair in FLOAT, for the cull code (FP64 runs at half rate, and
// the launch is bound by the instructions it issues: this function is written for instruction count).  Inputs are the
// float obstacle record (KParams::obsf, relative to the goal, written by every reset) and the vehicle position relative to
// the goal (formed in T by the dynamics launch, rounded once): every coordinate that matters is within
// max_dist_from_goal + max_dist of the origin, so the float rounding error of a position difference is a few 1e-6 m and
// that of a squared length below ~5e-4 m^2.  Every decision carries explicit slack far beyond that, so the result can
// only err on the safe side:
//   * in_view = false implies "culled" in exact arithmetic: lengths are widened by eps = 2e-3 m (+1e-4 relative),
//     discriminants by 1e-5 relative, clipped axis parameters by 1e-3 m;
//   * hit: 0 = clear, 1 = collision, 2 = within eps of the threshold (or NaN) -- the caller decides those in T.
//   q0: capsule (bot - goal, radius) / sphere (centre - goal, radius);  q1: capsule (unit axis d = (top - bot) / L, L)
// Geometry (capsule): with s = (pos - bot) . d the foot point, perp^2 = |pos - bot|^2 - s^2, the distance to the segment
// is hypot(max(-s, s - L, 0), perp); only axis points within Rr = max_dist + r of the vehicle can carry a surface point a
// ray reaches: t in [s - sqrt(Rr^2 - perp^2), s + sqrt(..)] clipped to [0, L] (a 40 m pillar seen under roll / pitch
// otherwise has its far ends on both sides of every plane).  Field of view: a surface point hit by a ray lies inside the
// ray pyramid {x >= 0, |y| <= ty x, |z| <= tz x} (body frame), so some axis point of that range lies within r of the
// inner side of ALL five planes; each signed distance g_k(t) = alpha_k t - beta_k is linear along the axis, each plane
// keeps an interval {t : alpha_k t <= beta_k}, and the obstacle is out of view when the intersection is empty (this also
// catches segments that leave the pyramid through different planes).
template <typename T>
__device__ __forceinline__ void cull_pair_rec(const KParams<T> &p, const float prel[3], const float Rm[9], float4 q0,
                                              float4 q1, bool is_cap, int &hit, bool &in_view) {
    const float eps = 2e-3f;
    const float cull = (float)p.radar_max_dist * 1.0001f + eps;
    const float rad = q0.w;
    const float oa[3] = {prel[0] - q0.x, prel[1] - q0.y, prel[2] - q0.z};
    const float oaoa = oa[0] * oa[0] + oa[1] * oa[1] + oa[2] * oa[2];
    const float Rr = cull + rad;
    // body-frame coordinates R^T v of the vehicle-to-obstacle offset
    float ob_[3];
#pragma unroll
    for (int c = 0; c < 3; c++) ob_[c] = Rm[c] * oa[0] + Rm[3 + c] * oa[1] + Rm[6 + c] * oa[2];
    const float rm = rad * 1.0001f + eps;
    const float ty = (float)p.fov_ty, tz = (float)p.fov_tz;
    const float ry = rm * (float)p.fov_ny, rz = rm * (float)p.fov_nz;
    const float vy = ty * ob_[0], vz = tz * ob_[0];
    // beta_k: the five plane offsets at t = 0 (the point bot, or the sphere centre): inside plane k iff beta_k >= 0
    const float b1 = rm - ob_[0], b2 = ry + ob_[1] - vy, b3 = ry - ob_[1] - vy, b4 = rz + ob_[2] - vz, b5 = rz - ob_[2] - vz;
    float dist2;
    bool outside;
    if (is_cap) {
        const float d[3] = {q1.x, q1.y, q1.z}, L = q1.w;
        const float s = oa[0] * d[0] + oa[1] * d[1] + oa[2] * d[2];
        float perp2 = oaoa - s * s;
        perp2 = perp2 < 0.0f ? 0.0f : perp2;           // NaN stays NaN (fmaxf would drop it)
        const float hh = fmaxf(fmaxf(-s, s - L), 0.0f);
        dist2 = hh * hh + perp2;                       // a NaN pose gives NaN here: hit = 2, not culled
        const float D = Rr * Rr - perp2, tolD = 1e-5f * (oaoa + s * s);
        const float sq = sqrtf(fmaxf(D, 0.0f) + tolD);
        float t_lo = fmaxf(s - sq - 1e-3f, 0.0f), t_hi = fminf(s + sq + 1e-3f, L);
        bool empty = D < -tolD;
        float db[3];
#pragma unroll
        for (int c = 0; c < 3; c++) db[c] = Rm[c] * d[0] + Rm[3 + c] * d[1] + Rm[6 + c] * d[2];
        const float uy = ty * db[0], uz = tz * db[0];
        auto clip = [&](float alpha, float beta) {        // keep { t : alpha t <= beta }
            // one MUFU instead of __fdividef's six instructions (25 quotients per env): q only decides with 1e-3 of slack, and
            // where alpha flushes to zero the plane simply does not clip (the conservative direction: more stays in view)
            float ra;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ra) : "f"(alpha));
            const float q = beta * ra;
            t_hi = fminf(t_hi, alpha > 0.0f ? q + 1e-3f : 3.0e38f);
            t_lo = fmaxf(t_lo, alpha < 0.0f ? q - 1e-3f : -3.0e38f);
            empty |= (alpha == 0.0f) && (beta < 0.0f);
        };
        clip(-db[0], b1);
        clip(db[1] - uy, b2);
        clip(-db[1] - uy, b3);
        clip(db[2] - uz, b4);
        clip(-db[2] - uz, b5);
        outside = empty || (t_lo > t_hi);
    } else {
        dist2 = oaoa;
        outside = (b1 < 0.0f) || (b2 < 0.0f) || (b3 < 0.0f) || (b4 < 0.0f) || (b5 < 0.0f);
    }
    const float thr = rad + (float)p.safety_radius;
    const float lo = thr - eps, hi = thr + eps;
    hit = (dist2 <= lo * lo) ? 1 : ((dist2 > hi * hi) ? 0 : 2);        // NaN -> 2
    outside |= dist2 > Rr * Rr;                                         // range: nearest surface point beyond max_dist
    in_view = !outside;
}

// The float obstacle record of cull_pair_rec from an obstacle as stored (capsule: bot[3] top[3] r; sphere: c[3] r) and
// the goal; differences are formed in double and rounded once.
__device__ __forceinline__ void obstacle_record_f32(const double ob[7], const double goal[3], bool is_cap, float4 &q0,
                                                    float4 &q1) {
    q0 = make_float4((float)(ob[0] - goal[0]), (float)(ob[1] - goal[1]), (float)(ob[2] - goal[2]), (float)(is_cap ? ob[6] : ob[3]));
    if (is_cap) {
        const double b[3] = {ob[3] - ob[0], ob[4] - ob[1], ob[5] - ob[2]};
        const double L = sqrt(b[0] * b[0] + b[1] * b[1] + b[2] * b[2]);
        q1 = make_float4((float)(b[0] / L), (float)(b[1] / L), (float)(b[2] / L), (float)L);
    } else {
        q1 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
}

// shape.py:341-390 for one ray: infinite-cylinder root, body hit if 0 < y < baba, else end-cap sphere.
// Returns -inf for "no intersection" and a negative distance for "behind" exactly like the reference.
template <typename T>
__device__ __forceinline__ T ray_capsule(const CapPre<T> &q, const T rd[3]) {
    T bard = rd[0] * q.ba[0] + rd[1] * q.ba[1] + rd[2] * q.ba[2];
    T rdoa = rd[0] * q.oa[0] + rd[1] * q.oa[1] + rd[2] * q.oa[2];
    T a = q.baba - bard * bard;
    T b = q.baba * rdoa - q.baoa * bard;
    T h = b * b - a * q.c;
    T res = -Mth<T>::inf();
    if (h > T(0)) {
        T t = (-b - Mth<T>::sqrt_(h)) / a;
        T y = q.baoa + t * bard;
        if (y > T(0) && y < q.baba) {
            res = t;
        } else {
            T b2, c2;
            if (y >= T(0)) {
                b2 = rd[0] * q.oc2[0] + rd[1] * q.oc2[1] + rd[2] * q.oc2[2];
                c2 = q.c2b;
            } else if (y <= T(0)) {
                b2 = rdoa;
                c2 = q.c2a;
            } else {   // y is NaN: the reference leaves oc = 0
                b2 = T(0);
                c2 = -q.r * q.r;
            }
            T h2 = b2 * b2 - c2;
            res = (h2 > T(0)) ? (-b2 - Mth<T>::sqrt_(h2)) : T(0);
        }
        if (res == T(0)) res = -Mth<T>::inf();
    }
    return res;
}

// shape.py:252-263 for one ray and one sphere: nearest root, -inf if the line misses
template <typename T>
__device__ __forceinline__ T ray_sphere(const T oc[3], T c, const T rd[3]) {
    T b = oc[0] * rd[0] + oc[1] * rd[1] + oc[2] * rd[2];
    T h = b * b - c;
    // the square root is evaluated for every lane (the select is if-converted); feeding it 1 instead of a negative
    // h keeps misses off the library's slow path (sqrt of a negative goes through the out-of-line NaN handler)
    T r = -b - Mth<T>::sqrt_(h < T(0) ? T(1) : h);
    return (h < T(0)) ? -Mth<T>::inf() : r;
}

// shape.py:393-417 dist_line_point(po, l1, l2) with l1 = bot, l2 = top
template <typename T>
__device__ __forceinline__ T dist_segment_point(const T pos[3], const T bot[3], const T top[3]) {
    T l[3] = {top[0] - bot[0], top[1] - bot[1], top[2] - bot[2]};
    T n = Mth<T>::sqrt_(l[0] * l[0] + l[1] * l[1] + l[2] * l[2]);
    // axis-aligned capsules have zero components; 0 / n is exact but takes the library's slow division path
    T d[3] = {l[0] == T(0) ? l[0] : l[0] / n, l[1] == T(0) ? l[1] : l[1] / n, l[2] == T(0) ? l[2] : l[2] / n};
    T s = (bot[0] - pos[0]) * d[0] + (bot[1] - pos[1]) * d[1] + (bot[2] - pos[2]) * d[2];
    T t = (pos[0] - top[0]) * d[0] + (pos[1] - top[1]) * d[1] + (pos[2] - top[2]) * d[2];
    T hh = s;
    if (t > hh || t != t) hh = t;
    if (T(0) > hh) hh = T(0);
    T q[3] = {pos[0] - bot[0], pos[1] - bot[1], pos[2] - bot[2]};
    T c[3];
    cross3(q, d, c);
    return Mth<T>::hypot_(hh, Mth<T>::sqrt_(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]));
}

// docking3d.py:712-723 given lg = log(x / x_max) (shared with observe()) -- the epsilon guard only matters
// when x < 1e-3
template <typename T>
__device__ __forceinline__ T log_precision(T x, T x_max, T log_den) {
    T xx = (x != x) ? x : (x > T(0.001) ? x : T(0.001));
    return T(1) - clipv(Mth<T>::log_(xx / x_max) / log_den, T(0), T(1));
}

// docking3d.py:742-765 with x_des = 0, exponents 4, no reversal (call sites :523-548, :571-582)
template <typename T>
__device__ __forceinline__ T cont_goal_constraints(T x, T x_max, T lp_delta_d) {
    T log_den_x = Mth<T>::log_(T(0.001) / x_max);
    T rx = Mth<T>::abs_(T(0) - log_precision(x, x_max, log_den_x));
    T rd = Mth<T>::abs_(T(0) - lp_delta_d);
    T rx2 = rx * rx, rd2 = rd * rd;
    return (rx2 * rx2) * (rd2 * rd2);
}

}  // namespace dockauv
