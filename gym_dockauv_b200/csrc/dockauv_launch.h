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

}  // namespace dockauv
