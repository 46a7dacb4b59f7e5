// dockauv_sac_actor.cuh -- stable-baselines3 1.5.0's SAC Actor, evaluated on the tensor cores before each step of
// dockauv_replay_collect (included from dockauv_capi.cu).
//
// latent_pi = Linear(n_obs, H), ReLU, Linear(H, H), ReLU; mu = Linear(H, n_u); log_std = Linear(H, n_u) clamped to
// [-20, 2]; a = tanh(mu + exp(log_std) eps), or tanh(mu) when deterministic.  eps is policy_noise<NU> (dockauv_policy.cuh).
//
// Mapping: persistent CTAs of 8 warps stage the weights once per launch in shared memory as bf16 (round to nearest
// even; layer 0's columns zero-padded to a multiple of 16, every row padded by 8 bf16 so that the 8 row addresses of an
// ldmatrix fall in different banks); the biases stay f32.  nn.Linear's [out][in] rows are the column-major B operand of
// mma.sync.m16n8k16.row.col as they are.  The two heads form one 16-row block: mu in rows 0..7, log_std in rows 8..15,
// zero-padded, so mu_k and log_std_k of an env land in the same lane.  A warp takes 16 envs at a time (tile i goes to
// CTA i mod grid, so a small batch is spread over every SM):
//   layer 0: A fragments from the observation rows (rounded to bf16), accumulators started from the bias; after ReLU
//            each 16-column chunk is packed into the bf16 A fragment of layer 1 (the accumulator fragment of m16n8k16
//            has the layout of the next product's A fragment), so the whole layer-0 output stays in registers;
//   layer 1: 32 output columns at a time (four independent accumulator chains); after bias and ReLU each 16-column
//            chunk goes, as bf16, straight into the 16 x 16 head accumulator;
//   epilogue: the head block passes through a per-warp 16 x 16 f32 tile in shared memory, then one lane per env draws
//            eps, clamps log_std and stores tanh(fmaf(expf(log_std), eps, mu)) as float32.
// Numerics: the observation, every weight matrix and each hidden activation after bias and ReLU are rounded to bf16;
// products are accumulated in f32 by the tensor cores; biases and the epilogue are f32.  Each output row depends only on
// its own env's row, so an env's action does not depend on its position in a tile or on how the batch is split.
// Only the action the step reads must be exact, and it is what goes into the replay ring: the SAC update recomputes
// every log-probability and Q-value from the stored (observation, action) pairs in f32.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "dockauv_policy.cuh"

namespace dockauv {

constexpr int kSacWarps = 8;      // warps per CTA (the per-warp epilogue tiles are sized for this many)

__host__ __device__ inline int sac_pad16(int n) { return (n + 15) & ~15; }

// Shared-memory layout, in bytes: W0 bf16 [H][pad16(n_obs) + 8], W1 bf16 [H][H + 8], heads bf16 [16][H + 8], then f32
// b0 [H], b1 [H], head bias [16], then one f32 16 x 16 epilogue tile per warp.  n_u (<= 8) does not change the size.
__host__ __device__ inline size_t sac_actor_smem_bytes(int n_obs, int H, int n_u) {
    (void)n_u;
    return 2 * ((size_t)H * (sac_pad16(n_obs) + 8) + (size_t)H * (H + 8) + (size_t)16 * (H + 8)) +
           4 * ((size_t)2 * H + 16) + 4 * (size_t)kSacWarps * 16 * 16;
}

struct SacActorLaunch {
    const float *w0, *b0, *w1, *b1, *mu_w, *mu_b, *log_std_w, *log_std_b;   // nn.Linear layout, caller-owned
    const float *obs;                   // f32[N][n_obs]: the observations acted on
    const int32_t *t_steps, *episode;   // the env's counters before the step (noise counter)
    float *actions;                     // f32[N][n_u]: the squashed actions, read by the step
    uint64_t seed, env_id0;
    int64_t env_begin, env_end;
    int32_t n_obs, deterministic;
};

// rows x cols of f32 (row-major, caller's pointer) -> bf16 rows of `stride` elements; columns cols..kp-1 zero
__device__ __forceinline__ void sac_stage_matrix(__nv_bfloat16 *s, int stride, const float *w, int rows, int cols, int kp) {
    if ((cols & 3) == 0 && (((uintptr_t)w) & 15u) == 0) {
        const int q = cols >> 2;
#pragma unroll 8
        for (int e = threadIdx.x; e < rows * q; e += blockDim.x) {
            const int r = e / q, c = (e - r * q) * 4;
            const float4 v = __ldg((const float4 *)(w + (size_t)r * cols + c));
            __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
            uint2 p;
            p.x = *(uint32_t *)&lo;
            p.y = *(uint32_t *)&hi;
            *(uint2 *)(s + r * stride + c) = p;
        }
    } else {
#pragma unroll 4
        for (int e = threadIdx.x; e < rows * cols; e += blockDim.x) {
            const int r = e / cols, c = e - r * cols;
            s[r * stride + c] = __float2bfloat16_rn(__ldg(w + e));
        }
    }
    const int pad = kp - cols;
    for (int e = threadIdx.x; e < rows * pad; e += blockDim.x) {
        const int r = e / pad;
        s[r * stride + cols + (e - r * pad)] = __float2bfloat16_rn(0.0f);
    }
}

__device__ __forceinline__ uint32_t sac_pack(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *(uint32_t *)&v;
}

// B fragments of two n-tiles (rows n0..n0+15 of `s`) for the k chunk k0..k0+15: b[0], b[1] of rows n0..n0+7, b[2],
// b[3] of rows n0+8..n0+15
__device__ __forceinline__ void sac_ldmatrix_b(uint32_t b[4], const __nv_bfloat16 *s, int stride, int n0, int k0, int lane) {
    const __nv_bfloat16 *p = s + (n0 + (lane & 7) + ((lane >> 4) << 3)) * stride + k0 + (((lane >> 3) & 1) << 3);
    const unsigned a = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];\n"
                 : "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]) : "r"(a));
}

// c += A (16 x 16, bf16) * B (16 x 8, bf16), f32 accumulators
__device__ __forceinline__ void sac_mma(float c[4], const uint32_t a[4], uint32_t b0, uint32_t b1) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
        "{%0, %1, %2, %3};\n"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// ReLU of the accumulators of two adjacent n-tiles (16 columns), rounded to bf16, as the A fragment of the next product
__device__ __forceinline__ void sac_relu_pack(uint32_t a[4], const float c0[4], const float c1[4]) {
    a[0] = sac_pack(fmaxf(c0[0], 0.0f), fmaxf(c0[1], 0.0f));
    a[1] = sac_pack(fmaxf(c0[2], 0.0f), fmaxf(c0[3], 0.0f));
    a[2] = sac_pack(fmaxf(c1[0], 0.0f), fmaxf(c1[1], 0.0f));
    a[3] = sac_pack(fmaxf(c1[2], 0.0f), fmaxf(c1[3], 0.0f));
}

// the accumulator of one n-tile starting from bias[n0 .. n0 + 7] (the lane's two columns, both rows)
__device__ __forceinline__ void sac_bias(float c[4], const float *bias, int n0, int t) {
    c[0] = c[2] = bias[n0 + 2 * t];
    c[1] = c[3] = bias[n0 + 2 * t + 1];
}

// 8 warps fit 255 registers each (one CTA per SM: the weights take most of the shared memory)
template <int H, int NU>
__global__ void __launch_bounds__(32 * kSacWarps, 1) sac_actor_kernel(SacActorLaunch p) {
    static_assert(H % 32 == 0 && NU <= 8, "H a multiple of 32, at most 8 actions");
    extern __shared__ float4 sac_smem[];
    const int k0p = sac_pad16(p.n_obs), s0 = k0p + 8, s1 = H + 8;
    __nv_bfloat16 *w0 = (__nv_bfloat16 *)sac_smem;
    __nv_bfloat16 *w1 = w0 + H * s0;
    __nv_bfloat16 *wh = w1 + H * s1;
    float *b0 = (float *)(wh + 16 * s1);
    float *b1 = b0 + H, *bh = b1 + H;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    float *tile = bh + 16 + warp * 256;

    sac_stage_matrix(w0, s0, p.w0, H, p.n_obs, k0p);
    sac_stage_matrix(w1, s1, p.w1, H, H, H);
    sac_stage_matrix(wh, s1, p.mu_w, NU, H, H);
    sac_stage_matrix(wh + 8 * s1, s1, p.log_std_w, NU, H, H);
    for (int e = threadIdx.x; e < (8 - NU) * H; e += blockDim.x) {    // head rows NU..7 and 8+NU..15
        const int r = NU + e / H, c = e % H;
        wh[r * s1 + c] = wh[(r + 8) * s1 + c] = __float2bfloat16_rn(0.0f);
    }
    for (int e = threadIdx.x; e < H; e += blockDim.x) {
        b0[e] = __ldg(p.b0 + e);
        b1[e] = __ldg(p.b1 + e);
    }
    for (int e = threadIdx.x; e < 16; e += blockDim.x) {
        const int k = e & 7;
        bh[e] = k < NU ? __ldg((e < 8 ? p.mu_b : p.log_std_b) + k) : 0.0f;
    }
    __syncthreads();

    const int64_t n_tiles = (p.env_end - p.env_begin + 15) >> 4;
    for (int64_t tile_i = (int64_t)warp * gridDim.x + blockIdx.x; tile_i < n_tiles; tile_i += (int64_t)gridDim.x * kSacWarps) {
        const int64_t base = p.env_begin + tile_i * 16;
        const int64_t r0 = base + g, r1 = base + g + 8;
        const bool v0 = r0 < p.env_end, v1 = r1 < p.env_end;
        const float *x0 = p.obs + r0 * p.n_obs, *x1 = p.obs + r1 * p.n_obs;

        // layer 0: [16 x k0p] x [k0p x H], accumulators from the bias
        float acc0[H / 8][4];
#pragma unroll
        for (int j = 0; j < H / 8; j++) sac_bias(acc0[j], b0, 8 * j, t);
#pragma unroll 1
        for (int k0 = 0; k0 < k0p; k0 += 16) {
            auto ld = [&](const float *x, bool v, int k) { return v && k < p.n_obs ? __ldg(x + k) : 0.0f; };
            const int ka = k0 + 2 * t, kb = ka + 8;
            uint32_t a[4];
            a[0] = sac_pack(ld(x0, v0, ka), ld(x0, v0, ka + 1));
            a[1] = sac_pack(ld(x1, v1, ka), ld(x1, v1, ka + 1));
            a[2] = sac_pack(ld(x0, v0, kb), ld(x0, v0, kb + 1));
            a[3] = sac_pack(ld(x1, v1, kb), ld(x1, v1, kb + 1));
#pragma unroll
            for (int j = 0; j < H / 16; j++) {
                uint32_t b[4];
                sac_ldmatrix_b(b, w0, s0, 16 * j, k0, lane);
                sac_mma(acc0[2 * j], a, b[0], b[1]);
                sac_mma(acc0[2 * j + 1], a, b[2], b[3]);
            }
        }
        uint32_t h0[H / 16][4];
#pragma unroll
        for (int j = 0; j < H / 16; j++) sac_relu_pack(h0[j], acc0[2 * j], acc0[2 * j + 1]);

        // layer 1, 32 columns at a time, each 16-column chunk fed into the head block after bias and ReLU
        float head[2][4];
        sac_bias(head[0], bh, 0, t);
        sac_bias(head[1], bh, 8, t);
#pragma unroll 1
        for (int n0 = 0; n0 < H; n0 += 32) {
            float acc1[4][4];
#pragma unroll
            for (int q = 0; q < 4; q++) sac_bias(acc1[q], b1, n0 + 8 * q, t);
#pragma unroll
            for (int k = 0; k < H / 16; k++) {
                uint32_t b[4], c[4];
                sac_ldmatrix_b(b, w1, s1, n0, 16 * k, lane);
                sac_ldmatrix_b(c, w1, s1, n0 + 16, 16 * k, lane);
                sac_mma(acc1[0], h0[k], b[0], b[1]);
                sac_mma(acc1[1], h0[k], b[2], b[3]);
                sac_mma(acc1[2], h0[k], c[0], c[1]);
                sac_mma(acc1[3], h0[k], c[2], c[3]);
            }
#pragma unroll
            for (int q = 0; q < 2; q++) {
                uint32_t a[4], b[4];
                sac_relu_pack(a, acc1[2 * q], acc1[2 * q + 1]);
                sac_ldmatrix_b(b, wh, s1, 0, n0 + 16 * q, lane);
                sac_mma(head[0], a, b[0], b[1]);
                sac_mma(head[1], a, b[2], b[3]);
            }
        }

        // epilogue: columns 0..7 of the head block are mu, 8..15 log_std
#pragma unroll
        for (int q = 0; q < 2; q++) {
            tile[g * 16 + 8 * q + 2 * t] = head[q][0];
            tile[g * 16 + 8 * q + 2 * t + 1] = head[q][1];
            tile[(g + 8) * 16 + 8 * q + 2 * t] = head[q][2];
            tile[(g + 8) * 16 + 8 * q + 2 * t + 1] = head[q][3];
        }
        __syncwarp();
        const int64_t i = base + lane;
        if (lane < 16 && i < p.env_end) {
            const float *row = tile + lane * 16;
            float eps[NU];
#pragma unroll
            for (int k = 0; k < NU; k++) eps[k] = 0.0f;
            if (!p.deterministic)
                policy_noise<NU>(p.seed, p.env_id0 + (uint64_t)i, (uint32_t)p.episode[i], (uint32_t)p.t_steps[i], eps);
#pragma unroll
            for (int k = 0; k < NU; k++) {
                const float mu = row[k], log_std = fminf(fmaxf(row[8 + k], -20.0f), 2.0f);
                const float u = p.deterministic ? mu : fmaf(expf(log_std), eps[k], mu);
                p.actions[i * NU + k] = tanhf(u);
            }
        }
        __syncwarp();
    }
}

}  // namespace dockauv
