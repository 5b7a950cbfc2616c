// vr_kernels.h -- host-side launch interface of the march kernels (one TU per basis size).
#pragma once
#include <cuda_runtime.h>

#include "vr_types.h"

namespace vrb {

// variant = kind + 16 * tune; 0 = the default for the tree's basis size.
//   kind 7: persistent warps + warp-shared shading queue (vr_march_q.cuh), >= 4 basis functions
//   kind 8: kind 7 + ray pool (tails of tiles are parked and re-marched 32 at a time), >= 4 basis functions
//   kind 3, tune 193: persistent warps, inline shading (vr_march.cuh)
//   -DVR_EXPERIMENTS only: 1 tile kernel, 2 tile + TMA top grid, 3 persistent (+ tuning bits),
//   4 persistent + TMA top grid, 5 persistent + deferred shading, 6 same + TMA top grid
struct LaunchCfg {
    int variant;
    int max_ctas;    // > 0: cap the persistent grid (leaves SMs to a concurrent copy/collective kernel)
    bool count;      // instrumented build: accumulate vr_counters
    bool surface;    // write a cudaSurfaceObject instead of linear memory
    int num_sms;
    unsigned int* queue;  // persistent kernels: {work head, done CTAs}
    unsigned char* pool;  // kind 8: parked-ray stacks of this (tree, stream), pool_bytes large (see pool_bytes_for)
    size_t pool_bytes;
    const void* l2_window;   // optional persisting-L2 access window (the node table)
    size_t l2_window_bytes;  // 0 = none
    bool pdl;                // allow overlap with the previous launch of the stream (see vr_march.cuh)
    cudaStream_t stream;
};

template <int KBD>
cudaError_t launch_march(LaunchDev& P, const LaunchCfg& cfg);

template <int KBD>
bool variant_supported(int variant);

// Caller-supplied rays (P.ray_o / ray_d / ray_tmax, P.n_rays > 0, float4 output in P.rgbaf): variant 0 (the batch
// default, inline shading) or 7 (shading queue, >= 4 basis functions); cudaErrorNotSupported for any other variant.
template <int KBD>
cudaError_t launch_rays(LaunchDev& P, const LaunchCfg& cfg);

// vr_camera_rays: the rays the march generates for the pixels of tile (x0, y0, w, h) of `cam`, row-major:
// origins c2w[9..11], directions before normalisation (vr_march.cuh camera_ray_dir).  float [w*h][3] each.
cudaError_t launch_camera_rays(const CamDev& cam, int x0, int y0, int w, int h, float* origins, float* dirs,
                               cudaStream_t stream);

// bytes of parked-ray storage a kind-8 launch needs on a device with num_sms SMs (0 when KBD has no such kernel)
template <int KBD>
size_t pool_bytes_for(int num_sms, int max_depth);

extern template cudaError_t launch_march<-1>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_rays<-1>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_march<1>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_rays<1>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_march<4>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_rays<4>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_march<9>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_rays<9>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_march<16>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_rays<16>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_march<25>(LaunchDev&, const LaunchCfg&);
extern template cudaError_t launch_rays<25>(LaunchDev&, const LaunchCfg&);
extern template bool variant_supported<-1>(int);
extern template size_t pool_bytes_for<-1>(int, int);
extern template bool variant_supported<1>(int);
extern template size_t pool_bytes_for<1>(int, int);
extern template bool variant_supported<4>(int);
extern template size_t pool_bytes_for<4>(int, int);
extern template bool variant_supported<9>(int);
extern template size_t pool_bytes_for<9>(int, int);
extern template bool variant_supported<16>(int);
extern template size_t pool_bytes_for<16>(int, int);
extern template bool variant_supported<25>(int);
extern template size_t pool_bytes_for<25>(int, int);

}  // namespace vrb
