// vr_rays.cu -- vr_camera_rays: the rays of a camera as arrays, for vr_render_rays.
//
// The direction is computed by camera_ray_dir (vr_march.cuh), the same code the march kernels run for a pixel, and
// stored before the normalisation: vr_render_rays normalises it with the operations of screen2worlddir's
// _normalize, so a camera's rays fed back reproduce vr_render bit for bit.
#include "vr_kernels.h"
#include "vr_march.cuh"

namespace vrb {

namespace {

__global__ void camera_rays_kernel(const CamDev cam, int x0, int y0, int w, long long n, float* __restrict__ origins,
                                   float* __restrict__ dirs) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int ly = (int)(i / w), lx = (int)(i - (long long)ly * w);
    float dx, dy, dz;
    camera_ray_dir(cam, x0 + lx, y0 + ly, dx, dy, dz);
    origins[3 * i] = cam.c2w[9]; origins[3 * i + 1] = cam.c2w[10]; origins[3 * i + 2] = cam.c2w[11];
    dirs[3 * i] = dx; dirs[3 * i + 1] = dy; dirs[3 * i + 2] = dz;
}

}  // namespace

cudaError_t launch_camera_rays(const CamDev& cam, int x0, int y0, int w, int h, float* origins, float* dirs,
                               cudaStream_t stream) {
    const long long n = (long long)w * h;
    if (n <= 0) return cudaSuccess;
    constexpr int kThreads = 256;
    const long long blocks = (n + kThreads - 1) / kThreads;
    if (blocks > 0x7fffffffLL) return cudaErrorInvalidValue;
    camera_rays_kernel<<<(unsigned)blocks, kThreads, 0, stream>>>(cam, x0, y0, w, n, origins, dirs);
    return cudaGetLastError();
}

}  // namespace vrb
