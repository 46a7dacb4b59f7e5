// dockauv_launch.h -- host-side launch entry points; one translation unit per precision instantiates them
// (dockauv_kernels_f64.cu, dockauv_kernels_f32.cu) so the two compile in parallel.
#pragma once
#include <cuda_runtime.h>

#include "dockauv_kparams.h"

namespace dockauv {

// marks (nullable): kMaxStepLaunches + 1 events; when given, the multi-launch layouts record one before their first
// launch and one after each launch, *n_marks receives how many were recorded (0 for single-launch layouts)
constexpr int kMaxStepLaunches = 6;
template <typename T>
cudaError_t launch_step(const KParams<T> &k, int vehicle, int layout, cudaStream_t st, cudaEvent_t *marks = nullptr,
                        int *n_marks = nullptr);

template <typename T>
cudaError_t launch_reset(const KParams<T> &k, const uint8_t *mask_dev, cudaStream_t st);

#ifndef DOCKAUV_FUSE_MAX_OBSF
#define DOCKAUV_FUSE_MAX_OBSF 20    // pipeline layout: the cull + finish code runs inside the dynamics launch when an env has at most this many float4 obstacle records: 80 KB of shared memory per 256-thread CTA, two CTAs per SM stay resident
#endif
// whether the dynamics launch of the pipeline layout takes the cull + finish code in, and how many launches one step over
// one env range is
template <typename T>
inline bool pipe_fuses_cull(const KParams<T> &k) {
    return k.n_caps + k.n_sph > 0 && !k.cull_exact && k.n_obsf > 0 && k.n_obsf <= DOCKAUV_FUSE_MAX_OBSF;
}
template <typename T>
inline int pipe_launches(const KParams<T> &k) {
    if (k.n_caps + k.n_sph == 0) return 2;      // dynamics (+ finish), episode end
    return pipe_fuses_cull(k) ? 3 : 4;          // dynamics (+ cull + finish) [, cull + finish], rays, episode end
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
