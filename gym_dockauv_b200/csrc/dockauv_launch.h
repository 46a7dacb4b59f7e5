// dockauv_launch.h -- host-side launch entry points; one translation unit per precision instantiates them
// (dockauv_kernels_f64.cu, dockauv_kernels_f32.cu) so the two compile in parallel.
#pragma once
#include <cuda_runtime.h>

#include "dockauv_kparams.h"

namespace dockauv {

// One step of k's env range.  *n_launches receives how many kernels it enqueued (valid when it returns cudaSuccess).
// marks (nullable): kMaxStepLaunches + 1 events; when given, the multi-launch layouts record one before their first
// launch and one after each launch, *n_marks receives how many were recorded (0 for single-launch layouts)
constexpr int kMaxStepLaunches = 3;
template <typename T>
cudaError_t launch_step(const KParams<T> &k, int vehicle, int layout, cudaStream_t st, int *n_launches,
                        cudaEvent_t *marks = nullptr, int *n_marks = nullptr);

template <typename T>
cudaError_t launch_reset(const KParams<T> &k, const uint8_t *mask_dev, cudaStream_t st);

// Work-list counters (KParams::view_count): one block of kCounterWords words per concurrently stepped env range; the
// range that starts at env b uses block b / kCounterEnvs.  Per list c (view lists of class 1, 2, 3, ended list):
//   word c                       count: running total of the appends (atomicAdd), never reset
//   word kCounterStart + c       its value when the current / most recent step began (block 0 of the dynamics launch
//                                copies it from the word below at the start of every step)
//   word kCounterNextStart + c   its value when the most recent step ended (block 0 of the episode-end launch, after the
//                                wait for the launches before it)
// A list's length is count - start, an append's slot its ticket - next start, both in modular uint32 arithmetic (the
// counters wrap; the buffers start all ones).  Every word is written in one launch and read by other CTAs only in later
// ones, so no CTA depends on another of its own launch (DESIGN.md section 3).
constexpr int kCounterWords = 16, kCounterEnvs = 128;
constexpr int kListCounters = 4, kCounterStart = 4, kCounterNextStart = 8;
inline int64_t counter_block(int64_t env_begin) { return kCounterWords * (env_begin / kCounterEnvs); }
template <typename T>
inline bool pipe_has_obstacles(const KParams<T> &k) { return k.n_caps + k.n_sph > 0; }

// The library-owned buffers of the pipeline layout for n envs, as byte offsets into one allocation (every piece 256-byte
// aligned): per-env records T[n][16], float obstacle records float4[n_obsf][n], obstacle rows T[n][n_obst][8], three view
// lists u64[n] and the ended list u32[n], and the counter blocks.
struct PipeBuffers {
    int n_obsf = 0, n_obst = 0;
    size_t rec = 0, obsf = 0, obsd = 0, view_list = 0, ended_list = 0, counters = 0;
    size_t n_counters = 0, bytes = 0;
};
inline PipeBuffers pipe_buffers(int64_t n_envs, size_t esz, int n_caps, int n_sph) {
    PipeBuffers b;
    const size_t n = (size_t)n_envs;
    b.n_obsf = 2 * n_caps + n_sph;
    b.n_obst = n_caps + n_sph;
    auto take = [&](size_t bytes) {
        const size_t o = b.bytes;
        b.bytes += (bytes + 255) & ~(size_t)255;
        return o;
    };
    b.rec = take(16 * esz * n);
    b.obsf = take(16 * (size_t)b.n_obsf * n);
    b.obsd = take(8 * esz * (size_t)b.n_obst * n);
    b.view_list = take(3 * 8 * n);
    b.ended_list = take(4 * n);
    b.n_counters = kCounterWords * (n / kCounterEnvs + 2);      // slack: a range may start at any multiple of 4096
    b.counters = take(4 * b.n_counters);
    return b;
}
// points k at such buffers at `base`, or at none (base == nullptr: the single-launch layouts)
template <typename T>
inline void point_pipe(KParams<T> &k, const PipeBuffers &b, void *base) {
    char *m = (char *)base;
    k.n_obsf = b.n_obsf;
    k.rec = m ? (T *)(m + b.rec) : nullptr;
    k.obsf = m && b.n_obsf > 0 ? (float4 *)(m + b.obsf) : nullptr;
    k.obsd = m && b.n_obst > 0 ? (T *)(m + b.obsd) : nullptr;
    k.view_list = m ? (unsigned long long *)(m + b.view_list) : nullptr;
    k.ended_list = m ? (uint32_t *)(m + b.ended_list) : nullptr;
    k.view_count = m ? (unsigned int *)(m + b.counters) : nullptr;
}

// float obstacle records of the cull code from the bound obstacle / goal buffers (no-op for handles without them)
template <typename T>
cudaError_t launch_refresh_obstacles(const KParams<T> &k, cudaStream_t st);

// Episode taps (dockauv_set_taps).  One TapRow copies one component row of K values: element k of `src` (at byte
// k * src_step, or env_id * src_step when src_by_id) goes to `dst` and `dst2` (byte k * dst_step, nullable) and to the
// ring slot `*count % capacity` of `ring` (byte slot * ring_slot + k * dst_step, nullable).  esz: 1, 4, 8 or 16 bytes.
struct TapRow {
    const char *src;
    char *dst, *dst2, *ring;
    int64_t ring_slot;
    int32_t esz, src_step, dst_step, src_by_id;
};
struct TapLaunch {
    const TapRow *rows;        // device table
    int32_t n_rows, n_taps;
    const int64_t *ids;        // local env ids of the taps (device)
    int64_t *count;            // caller's record counter
    int64_t capacity;
    unsigned int *sync;        // commit: CTAs done so far (the last one bumps *count and zeroes it)
    // gather only: the step's actions and current noise for the shadow
    const void *actions;
    int32_t act_f32, n_u;
    void *shadow_actions;      // [K][n_u] in the actions' dtype
    const void *noise;         // real[N] of the caller, nullable
    void *shadow_noise;        // real[K]
};
// pre-step rows of the tapped envs -> shadow + ring, and the shadow's actions and noise (the Philox draw of dyn_current
// for the real env id when the caller passes no noise)
template <typename T>
cudaError_t launch_tap_gather(const KParams<T> &k, const TapLaunch &t, cudaStream_t st);
// shadow results -> ring slot, then ++*count on the device
template <typename T>
cudaError_t launch_tap_commit(const KParams<T> &k, const TapLaunch &t, cudaStream_t st);

}  // namespace dockauv
