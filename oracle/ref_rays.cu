// ref_rays.cu -- ray-batch tap of the UNMODIFIED reference CUDA renderer (test infrastructure, like ref_harness.cu).
//
// Built only where the reference sources exist (oracle/Makefile.rays), into oracle/_ref/libvolrend_ref_rays.so.  No
// reference source is copied: this TU #includes the reference's own src/cuda/volrend.cu, and the kernel below calls
// its _normalize, maybe_world2ndc, rodrigues and device::trace_ray in the order of render_kernel
// (volrend.cu:136-158, offscreen branch) with screen2worlddir replaced by a loaded ray.  The reference has no ray
// entry point; the degenerate-ray rule of vr_render_rays (non-finite values or a direction of fp32 length 0 or
// infinity: a miss) is applied before any reference code runs.
//
//   ref_render_rays_f32 -> float out[4] per ray
#include <cmath>
#include <cstdint>

#include "../src/cuda/volrend.cu"  // resolved through -I$(VOLREND_REF)/include/.. (see Makefile.ref)

#include "volrend/n3tree.hpp"

namespace volrend {
namespace device {
__global__ static void ray_tap_kernel(TreeSpec tree, RenderOptions opt, const float* origins, const float* dirs,
                                      const float* t_max, int n, float4* out4) {
    CUDA_GET_THREAD_ID(idx, n);
    float dir[3], cen[3], out[4];
    out[0] = out[1] = out[2] = out[3] = 0.f;
    for (int i = 0; i < 3; ++i) {
        cen[i] = origins[3 * idx + i];
        dir[i] = dirs[3 * idx + i];
    }
    const float len = sqrtf(fmaf(dir[2], dir[2], fmaf(dir[0], dir[0], dir[1] * dir[1])));
    bool ok = isfinite(len) && len > 0.f;
    for (int i = 0; i < 3; ++i) ok = ok && isfinite(cen[i]) && isfinite(dir[i]);
    if (!ok) {
        if (opt.render_depth) out[3] = 1.f;   // as a ray that misses the box (rt_core.cuh:90-91)
    } else if (tree.N > 0) {
        _normalize(dir);
        float vdir[3] = {dir[0], dir[1], dir[2]};
        maybe_world2ndc(tree, dir, cen);
        for (int i = 0; i < 3; ++i) {
            cen[i] = tree.offset[i] + tree.scale[i] * cen[i];
        }
        const float tl = t_max ? t_max[idx] : 1e9f;
        rodrigues(opt.rot_dirs, vdir);
        trace_ray(tree, dir, vdir, cen, opt, tl, out);
    }
    const float remain = opt.background_brightness * (1.f - out[3]);
    out4[idx] = make_float4(out[0] + remain, out[1] + remain, out[2] + remain, out[3]);
}
}  // namespace device
}  // namespace volrend

using namespace volrend;

extern "C" {

struct ref_ray_options {
    float step_size, sigma_thresh, stop_thresh, background_brightness;
    float render_bbox[6];
    int32_t basis_minmax[2];
    float rot_dirs[3];
    int32_t render_depth;
};

// tree: an N3Tree* of libvolrend_ref.so's ref_tree_open would live in another library; this one opens its own.
void* ref_rays_tree_open(const char* npz_path) {
    N3Tree* t = new N3Tree(std::string(npz_path));
    if (!t->is_data_loaded()) { delete t; return nullptr; }
    return t;
}
void ref_rays_tree_close(void* t) { delete static_cast<N3Tree*>(t); }

// origins/dirs host float [n][3], t_max host float [n] or NULL; out_host float [n][4]
int ref_render_rays_f32(void* tp, const float* origins, const float* dirs, const float* t_max, int n,
                        const ref_ray_options* o, float* out_host) {
    N3Tree& tree = *static_cast<N3Tree*>(tp);
    RenderOptions opt;
    opt.step_size = o->step_size; opt.sigma_thresh = o->sigma_thresh; opt.stop_thresh = o->stop_thresh;
    opt.background_brightness = o->background_brightness;
    for (int i = 0; i < 6; ++i) opt.render_bbox[i] = o->render_bbox[i];
    opt.basis_minmax[0] = o->basis_minmax[0]; opt.basis_minmax[1] = o->basis_minmax[1];
    for (int i = 0; i < 3; ++i) opt.rot_dirs[i] = o->rot_dirs[i];
    opt.render_depth = o->render_depth != 0;
    float *d_o = nullptr, *d_d = nullptr, *d_t = nullptr;
    float4* d_out = nullptr;
    cuda(Malloc((void**)&d_o, sizeof(float) * 3 * n));
    cuda(Malloc((void**)&d_d, sizeof(float) * 3 * n));
    cuda(Malloc((void**)&d_out, sizeof(float4) * n));
    cuda(Memcpy(d_o, origins, sizeof(float) * 3 * n, cudaMemcpyHostToDevice));
    cuda(Memcpy(d_d, dirs, sizeof(float) * 3 * n, cudaMemcpyHostToDevice));
    if (t_max) {
        cuda(Malloc((void**)&d_t, sizeof(float) * n));
        cuda(Memcpy(d_t, t_max, sizeof(float) * n, cudaMemcpyHostToDevice));
    }
    const int N_CUDA_THREADS = 320;
    device::ray_tap_kernel<<<N_BLOCKS_NEEDED(n, N_CUDA_THREADS), N_CUDA_THREADS>>>(tree, opt, d_o, d_d, d_t, n, d_out);
    cuda(Memcpy(out_host, d_out, sizeof(float4) * n, cudaMemcpyDeviceToHost));
    cudaError_t e = cudaGetLastError();
    cuda(Free(d_o)); cuda(Free(d_d)); cuda(Free(d_out));
    if (d_t) cuda(Free(d_t));
    return e == cudaSuccess ? 0 : -(int)e;
}

}  // extern "C"
