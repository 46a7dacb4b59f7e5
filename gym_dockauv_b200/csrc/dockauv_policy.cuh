// dockauv_policy.cuh -- the actor-critic of stable-baselines3's default MlpPolicy, evaluated between the steps of
// dockauv_rollout_policy (included from dockauv_capi.cu).
//
// Separate pi and vf nets n_obs -> H -> H with Tanh after each hidden layer, action_net H -> n_u, value_net H -> 1, a
// state-independent log_std and a diagonal Gaussian.  One thread per env; the CTA stages both nets' weights in shared
// memory once and then walks its envs grid-stride, so a CTA reads the ~50 KB of weights once and not once per 256
// envs.  Every weight load is a broadcast (all lanes read the same word).  Arithmetic is f32 FMAs over the inputs in
// index order, starting from the bias, with tanhf (not tanh.approx.f32, whose ~2^-11 relative error would move the
// log-probs PPO divides by) and no tensor cores: the log-probs agree with the f32 PyTorch update that recomputes them.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "dockauv_device.cuh"

namespace dockauv {

// largest dynamic shared memory one CTA may opt into on sm_100
constexpr size_t kPolicyMaxSmem = 232448;

// Shared-memory layout of one net, in floats, every piece a multiple of 4 (float4 loads): layer 0 transposed
// ([n_obs][H]: the H accumulators of one input are contiguous), its bias, layer 1 as nn.Linear stores it ([H][H]), its
// bias, the output layer ([n_out][H]) and its bias padded to 4.  The pi net comes first, then the vf net, then log_std.
__host__ __device__ inline int policy_net_floats(int n_obs, int H, int n_out) {
    return n_obs * H + H + H * H + H + n_out * H + ((n_out + 3) & ~3);
}
__host__ __device__ inline size_t policy_smem_bytes(int n_obs, int H, int n_u) {
    return sizeof(float) * ((size_t)policy_net_floats(n_obs, H, n_u) + policy_net_floats(n_obs, H, 1) + ((n_u + 3) & ~3));
}

struct PolicyLaunch {
    const float *pi_w[3], *pi_b[3], *vf_w[3], *vf_b[3], *log_std;   // nn.Linear layout, caller-owned
    const float *obs;            // f32[N][n_obs]: the observations acted on
    const int32_t *t_steps, *episode;   // the env's counters before the step (noise counter)
    float *actions;              // f32[N][n_u]: raw samples
    float *act_clipped;          // f32[N][n_u]: the samples clipped to [u_lo, u_hi], read by the step
    float *values, *log_probs;   // f32[N]
    float u_lo[DOCKAUV_MAX_U], u_hi[DOCKAUV_MAX_U];
    uint64_t seed, env_id0;
    int64_t env_begin, env_end;
    int32_t n_obs, deterministic;
    int32_t value_only;          // values only (the GAE bootstrap): no pi net, noise or action outputs
};

// copies one net into shared memory at `s` (layer 0 transposed)
__device__ __forceinline__ void policy_stage_net(float *s, const float *const w[3], const float *const b[3], int n_obs,
                                                 int H, int n_out) {
    for (int e = threadIdx.x; e < H * n_obs; e += blockDim.x) s[(e % n_obs) * H + e / n_obs] = __ldg(w[0] + e);
    s += n_obs * H;
    for (int e = threadIdx.x; e < H; e += blockDim.x) s[e] = __ldg(b[0] + e);
    s += H;
    for (int e = threadIdx.x; e < H * H; e += blockDim.x) s[e] = __ldg(w[1] + e);
    s += H * H;
    for (int e = threadIdx.x; e < H; e += blockDim.x) s[e] = __ldg(b[1] + e);
    s += H;
    for (int e = threadIdx.x; e < n_out * H; e += blockDim.x) s[e] = __ldg(w[2] + e);
    s += n_out * H;
    for (int e = threadIdx.x; e < n_out; e += blockDim.x) s[e] = __ldg(b[2] + e);
}

// out[k] = layer 2 of tanh(layer 1 (tanh(layer 0 (obs)))).  The H activations of layer 0 live in registers; layer 1's
// outputs are produced R at a time (R independent FMA chains) and accumulated straight into out[] in index order, so no
// second activation array is live.  R = 2 keeps H = 64 within 128 registers without spills; R = 4 spills there.
template <int H, int NO, int R = (H > 64 ? 4 : 2)>
__device__ __forceinline__ void policy_mlp(const float *__restrict__ s, const float *__restrict__ obs, int n_obs,
                                           float out[NO]) {
    const float *w0 = s, *b0 = w0 + n_obs * H, *w1 = b0 + H, *b1 = w1 + H * H, *w2 = b1 + H, *b2 = w2 + NO * H;
    float h[H];
#pragma unroll
    for (int q = 0; q < H / 4; q++) {
        const float4 v = ((const float4 *)b0)[q];
        h[4 * q] = v.x; h[4 * q + 1] = v.y; h[4 * q + 2] = v.z; h[4 * q + 3] = v.w;
    }
    auto input = [&](float x, int i) {
        const float4 *w = (const float4 *)(w0 + i * H);
#pragma unroll
        for (int q = 0; q < H / 4; q++) {
            const float4 v = w[q];
            h[4 * q] = fmaf(v.x, x, h[4 * q]);
            h[4 * q + 1] = fmaf(v.y, x, h[4 * q + 1]);
            h[4 * q + 2] = fmaf(v.z, x, h[4 * q + 2]);
            h[4 * q + 3] = fmaf(v.w, x, h[4 * q + 3]);
        }
    };
#pragma unroll 1
    for (int i = 0; i < n_obs; i++) input(__ldg(obs + i), i);
#pragma unroll
    for (int j = 0; j < H; j++) h[j] = tanhf(h[j]);
#pragma unroll
    for (int k = 0; k < NO; k++) out[k] = b2[k];
#pragma unroll 1
    for (int j = 0; j < H; j += R) {
        float t[R];
#pragma unroll
        for (int r = 0; r < R; r++) t[r] = b1[j + r];
#pragma unroll
        for (int q = 0; q < H / 4; q++) {
            float4 a[R];
#pragma unroll
            for (int r = 0; r < R; r++) a[r] = ((const float4 *)(w1 + (j + r) * H))[q];
#pragma unroll
            for (int r = 0; r < R; r++) t[r] = fmaf(a[r].x, h[4 * q], t[r]);
#pragma unroll
            for (int r = 0; r < R; r++) t[r] = fmaf(a[r].y, h[4 * q + 1], t[r]);
#pragma unroll
            for (int r = 0; r < R; r++) t[r] = fmaf(a[r].z, h[4 * q + 2], t[r]);
#pragma unroll
            for (int r = 0; r < R; r++) t[r] = fmaf(a[r].w, h[4 * q + 3], t[r]);
        }
#pragma unroll
        for (int r = 0; r < R; r++) t[r] = tanhf(t[r]);
#pragma unroll
        for (int k = 0; k < NO; k++)
#pragma unroll
            for (int r = 0; r < R; r++) out[k] = fmaf(w2[k * H + j + r], t[r], out[k]);
    }
}

// eps[k], k < NU: standard normals from Philox4x32-10 block j = k / 4 at counter (global id lo, global id hi, episode,
// 0xC0000000 | (t_steps mod 2^29) << 1 | j), Box-Muller on its words: with u = ((w0 >> 8) + 1) 2^-24 in (0, 1] and
// v = (w1 >> 8) 2^-24 in [0, 1), eps[4j] = sqrt(-2 ln u) cos(2 pi v), eps[4j + 1] = sqrt(-2 ln u) sin(2 pi v); words 2
// and 3 give eps[4j + 2], eps[4j + 3] the same way.  Word 3 >= 0xC0000000 is used by no other draw (resets < 32, scenario
// bank 0x40000000, current noise 0x80000000 | t), so the actions depend on (seed, global id, episode, t) only.
template <int NU>
__device__ __forceinline__ void policy_noise(uint64_t seed, uint64_t gid, uint32_t episode, uint32_t t_steps, float eps[NU]) {
#pragma unroll
    for (int j = 0; j < (NU + 3) / 4; j++) {
        uint32_t c[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), episode, 0xC0000000u | (t_steps & 0x1FFFFFFFu) << 1 | (uint32_t)j};
        philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
        for (int m = 0; m < 2; m++) {
            const float u = (float)((c[2 * m] >> 8) + 1u) * 5.9604644775390625e-08f;
            const float v = (float)(c[2 * m + 1] >> 8) * 5.9604644775390625e-08f;
            const float r = sqrtf(-2.0f * logf(u));
            float sn, cs;
            sincospif(2.0f * v, &sn, &cs);
            if (4 * j + 2 * m < NU) eps[4 * j + 2 * m] = r * cs;
            if (4 * j + 2 * m + 1 < NU) eps[4 * j + 2 * m + 1] = r * sn;
        }
    }
}

// H <= 64 keeps to 128 registers (two 256-thread CTAs per SM); H > 64 holds more activations than that and gets up to 255
template <int H, int NU>
__global__ void __launch_bounds__(256, H <= 64 ? 2 : 1) policy_kernel(PolicyLaunch p) {
    extern __shared__ float4 policy_smem[];
    float *pi = (float *)policy_smem;
    float *vf = pi + policy_net_floats(p.n_obs, H, NU);
    float *log_std = vf + policy_net_floats(p.n_obs, H, 1);
    policy_stage_net(pi, p.pi_w, p.pi_b, p.n_obs, H, NU);
    policy_stage_net(vf, p.vf_w, p.vf_b, p.n_obs, H, 1);
    for (int k = threadIdx.x; k < NU; k += blockDim.x) log_std[k] = __ldg(p.log_std + k);
    __syncthreads();
    for (int64_t i = p.env_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.env_end;
         i += (int64_t)gridDim.x * blockDim.x) {
        const float *obs = p.obs + i * p.n_obs;
        if (!p.value_only) {
            float mu[NU], eps[NU];
            policy_mlp<H, NU>(pi, obs, p.n_obs, mu);
#pragma unroll
            for (int k = 0; k < NU; k++) eps[k] = 0.0f;
            if (!p.deterministic)
                policy_noise<NU>(p.seed, p.env_id0 + (uint64_t)i, (uint32_t)p.episode[i], (uint32_t)p.t_steps[i], eps);
            float lp = 0.0f;
#pragma unroll
            for (int k = 0; k < NU; k++) {
                const float a = fmaf(expf(log_std[k]), eps[k], mu[k]);
                p.actions[i * NU + k] = a;
                p.act_clipped[i * NU + k] = fminf(fmaxf(a, p.u_lo[k]), p.u_hi[k]);
                lp += -0.5f * eps[k] * eps[k] - log_std[k] - 0.918938533204672742f;     // 0.5 ln(2 pi)
            }
            p.log_probs[i] = lp;
        }
        float v[1];
        policy_mlp<H, 1>(vf, obs, p.n_obs, v);
        p.values[i] = v[0];
    }
}

}  // namespace dockauv
