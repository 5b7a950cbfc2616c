/*
 * volrend_b200.h -- thin C-ABI of the B200-native PlenOctree ray-marcher.
 *
 * This is the drop-in boundary for volrend's CUDA backend (reference paths relative to
 * /root/reference).  Everything the reference's `src/cuda/*` exports is re-expressed
 * here with plain pointers and sizes -- no torch, glm, cnpy or CUDA types:
 *
 *   vr_tree_create / vr_tree_destroy   replace N3Tree::load_cuda / free_cuda
 *                                      (src/cuda/n3tree.cu:9-41, :43-49; the struct
 *                                      N3Tree::device, include/volrend/n3tree.hpp:72-78)
 *   vr_render                          replaces launch_renderer(..., offscreen=true)
 *                                      (include/volrend/cuda/renderer_kernel.hpp:9-12,
 *                                      src/cuda/volrend.cu:195-245) and the device side
 *                                      render_kernel (volrend.cu:78-173) + trace_ray
 *                                      (include/volrend/cuda/rt_core.cuh:66-196)
 *   vr_render_composite                replaces launch_renderer(..., offscreen=false):
 *                                      colour + depth inputs (volrend.cu:92-96,143-146)
 *   vr_render_batch                    the per-pose loop of main_headless.cpp:208-223 as
 *                                      one call (same per-view semantics)
 *   vr_render_rays / vr_camera_rays    caller-supplied ray batches (origins + directions in,
 *                                      float RGBA out) on the same march kernels
 *   vr_render_frames_host              main_headless.cpp:208-223 with `-o`: renders and
 *                                      copies every frame to host memory (:216-219)
 *   vr_probe_lumisphere                retrieve_cursor_lumisphere_kernel (volrend.cu:175-191)
 *   vr_last_error                      replaces the abort-on-error cuda_assert
 *                                      (src/cuda/common.cu:8-21) -- the C-ABI never aborts;
 *                                      the C++ shim (volrend_b200/csrc/shim) restores it.
 *
 * All calls return 0 on success or a negative VR_E* code; vr_last_error() gives the text.
 * Device buffers are caller-owned; rendering is asynchronous on the given CUDA stream
 * (passed as void* == cudaStream_t).  One vr_tree lives on the device that was current at
 * creation.  There is NO CPU fallback: without a CUDA device every call fails with
 * VR_ENODEVICE.
 */
#ifndef VOLREND_B200_H_
#define VOLREND_B200_H_
#include <stddef.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VR_BASIS_MAX 25 /* VOLREND_GLOBAL_BASIS_MAX, include/volrend/render_options.hpp:6 */

enum { VR_OK = 0, VR_EINVAL = -1, VR_ENODEVICE = -2, VR_ECUDA = -3, VR_ENOMEM = -4, VR_EUNSUPPORTED = -5 };

/* DataFormat::format, include/volrend/data_format.hpp:9-15 */
enum { VR_FMT_RGBA = 0, VR_FMT_SH = 1, VR_FMT_SG = 2, VR_FMT_ASG = 3 };

typedef struct vr_tree vr_tree; /* opaque: re-laid-out device copy of one N3Tree */

/* Host-side view of a loaded N3Tree (fields of include/volrend/n3tree.hpp:33-85). */
typedef struct {
    const int32_t* child;   /* N3Tree::child_  int32 [capacity*N^3], relative offsets, 0 = leaf */
    const uint16_t* data;   /* N3Tree::data_   fp16  [capacity*N^3*data_dim] */
    const float* extra;     /* N3Tree::extra_  SG: [basis_dim*4], ASG: [basis_dim*11], else NULL */
    int64_t capacity;       /* N3Tree::capacity */
    int32_t N;              /* N3Tree::N (only 2 is supported, as in the reference) */
    int32_t data_dim;       /* N3Tree::data_dim */
    int32_t format;         /* N3Tree::data_format.format (VR_FMT_*) */
    int32_t basis_dim;      /* N3Tree::data_format.basis_dim (-1 for RGBA) */
    float offset[3];        /* N3Tree::offset */
    float scale[3];         /* N3Tree::scale */
    int32_t use_ndc;        /* N3Tree::use_ndc */
    float ndc_width, ndc_height, ndc_focal;
} vr_tree_desc;

/* Camera (include/volrend/camera.hpp:31-48); c2w by value, no device copy needed. */
typedef struct {
    int32_t width, height;
    float fx, fy;
    float c2w[12];          /* glm::mat4x3 Camera::transform, column-major */
} vr_camera;

/* RenderOptions (include/volrend/render_options.hpp:11-53), ray-march subset. */
typedef struct {
    float step_size, sigma_thresh, stop_thresh, background_brightness;
    float render_bbox[6];
    int32_t basis_minmax[2];
    float rot_dirs[3];
    int32_t render_depth;
} vr_options;

typedef struct { int32_t x0, y0, w, h; } vr_rect;

/* Work counters (device-resident, accumulated with atomics when requested). */
typedef struct {
    unsigned long long samples;      /* S        march-loop iterations (rt_core.cuh:108) */
    unsigned long long child_loads;  /* sum d_s  child[] reads the reference algorithm makes */
    unsigned long long shaded;       /* S_shaded samples with sigma > sigma_thresh */
    unsigned long long rays_hit;     /* rays entering the march */
    unsigned long long node_fetches; /* node words this implementation actually loaded */
} vr_counters;

typedef struct {
    int64_t capacity;
    int32_t max_depth;               /* deepest leaf (root children = 1) */
    int32_t rec_bytes;               /* padded leaf-record stride */
    int64_t node_bytes, rec_total_bytes, top_bytes; /* slot-indexed layout (resident in -DVR_EXPERIMENTS builds only) */
    int32_t kernel_basis;            /* -1 RGBA, 1, 4, 9, 16, 25 */
    int32_t wide_parity;             /* v: internal nodes of depth d with (d + v) % 2 == 0 own a 64-entry table (+ the root);
                                        the v with fewer tables is chosen per tree (% 3 and 512 entries in VR_WIDE_LV=3 builds) */
    int64_t n_tables;
    int64_t wide_bytes, wrecs_bytes; /* 64-entry tables; colour records indexed by table entry */
    int64_t kernel_bytes;            /* what the march kernels can touch: wide_bytes + wrecs_bytes */
    int64_t device_bytes;            /* everything the tree keeps resident */
} vr_tree_info;

/* Compressed N3Tree as written by scripts/compress_octree.py:93-118 (keys quant_colors, quant_map,
 * sigma, data_retained).  The reference decodes it on the CPU with a scalar loop at load time
 * (src/n3tree.cpp:279-340); vr_tree_create_quantized uploads the compressed arrays and decodes on
 * the GPU straight into the device layout (same resulting tree, bit for bit). */
typedef struct {
    vr_tree_desc base;             /* child + header fields; base.data must be NULL */
    const uint16_t* quant_colors;  /* fp16 [n_quant][65536][3] codebooks */
    const uint16_t* quant_map;     /* u16  [n_quant][capacity*N^3] codebook indices */
    const uint16_t* sigma;         /* fp16 [capacity*N^3] */
    const uint16_t* data_retained; /* fp16 [n_retain][capacity*N^3][3] or NULL */
    int32_t n_quant;               /* quantised basis functions */
    int32_t n_retain;              /* un-quantised leading basis functions (n_quant+n_retain == basis_dim) */
} vr_tree_quant_desc;

void vr_default_options(vr_options* o);

int vr_tree_create(const vr_tree_desc* desc, vr_tree** out);
int vr_tree_create_quantized(const vr_tree_quant_desc* desc, vr_tree** out);
void vr_tree_destroy(vr_tree* tree);
int vr_tree_get_info(const vr_tree* tree, vr_tree_info* info);

/* Offscreen render of `tile` (NULL = full frame) of view `cam`.  rgba8_dev: tile-sized
 * linear RGBA8 (pitch 4*tile.w) or NULL; rgba32f_dev: tile-sized float4 or NULL;
 * counters_dev: device vr_counters to accumulate into, or NULL. */
int vr_render(const vr_tree* tree, const vr_camera* cam, const vr_options* opt, const vr_rect* tile,
              uint8_t* rgba8_dev, float* rgba32f_dev, vr_counters* counters_dev, void* stream);

/* n_views cameras (host array), outputs are n_views consecutive tile-sized images. */
int vr_render_batch(const vr_tree* tree, const vr_camera* cams, int n_views, const vr_options* opt,
                    const vr_rect* tile, uint8_t* rgba8_dev, float* rgba32f_dev,
                    vr_counters* counters_dev, void* stream);

/* launch_renderer(offscreen=false): rgba8_dev is read (existing colour) and overwritten;
 * depth_dev holds the per-pixel ray-distance limit (world units), both tile-sized. */
int vr_render_composite(const vr_tree* tree, const vr_camera* cam, const vr_options* opt,
                        const vr_rect* tile, uint8_t* rgba8_dev, const float* depth_dev,
                        float* rgba32f_dev, void* stream);

/* Same, writing a CUDA surface object over an RGBA8 cudaArray (what the reference's
 * caller owns, main_headless.cpp:190-199); depth_surf = 0 => offscreen. */
int vr_render_surface(const vr_tree* tree, const vr_camera* cam, const vr_options* opt,
                      unsigned long long rgba8_surf, unsigned long long depth_surf, void* stream);

/* Ray-tile sharding of one frame across n_parts GPUs (SURVEY.md 8e): this call renders every
 * n_parts-th band of band_h rows (bands part, part+n_parts, ...) of the full frame and writes them
 * compactly, band after band, into rgba8_dev / rgba32f_dev (vr_band_rows() rows of cam->width
 * pixels).  One launch per GPU per frame; the caller gathers the compact buffers. */
int vr_render_bands(const vr_tree* tree, const vr_camera* cam, const vr_options* opt, int band_h, int n_parts,
                    int part, uint8_t* rgba8_dev, float* rgba32f_dev, void* stream);
int vr_band_rows(int height, int band_h, int n_parts, int part);
/* Same for n_views cameras in ONE launch: view i's bands land at rgba8_dev + i * 4*width*vr_band_rows(). */
int vr_render_bands_batch(const vr_tree* tree, const vr_camera* cams, int n_views, const vr_options* opt, int band_h,
                          int n_parts, int part, uint8_t* rgba8_dev, float* rgba32f_dev, void* stream);

/* Ray batches: renders n_rays caller-supplied rays instead of the pixels of a camera.
 *   origins_dev, dirs_dev  device float32 [n_rays][3], world space; directions need not be unit length
 *   t_max_dev              device float32 [n_rays] depth limits, or NULL (= 1e9 for every ray)
 *   rgba32f_dev            device float4 [n_rays]: premultiplied RGB + background, alpha
 *   counters_dev           device vr_counters to accumulate into, or NULL
 * Ray i is rendered exactly as render_kernel renders a pixel (volrend.cu:136-158, offscreen branch) with
 * screen2worlddir replaced by the loaded ray: the direction is normalised with screen2worlddir's _normalize and kept
 * as the view direction of the basis, then maybe_world2ndc, the tree's offset/scale, rodrigues(rot_dirs) and trace_ray
 * with t_max[i] as depth limit -- the unit of the composite-mode depth (rt_core.cuh:77): for non-NDC trees the world
 * distance from the origin along the normalised direction.  The result is composited over background_brightness.
 * Every vr_options field applies.  A ray with a non-finite origin or direction component, or whose direction has
 * fp32 length 0 or infinity, is a miss: background with alpha 0 (alpha 1 under render_depth, as for every miss), not
 * counted in rays_hit.  Any leading shape of rays is the caller's; n_rays == 0 is a no-op.  Runs on the tree's batch
 * kernel variant (vr_tree_variant; vr_set_variant 7 selects the shading queue); other variants fail with
 * VR_EUNSUPPORTED.  The ray arrays may be written by the previous kernel on `stream` without synchronisation.
 *
 * vr_camera_rays writes the rays the march generates for `cam` (tile NULL = full frame), one per pixel, row-major
 * over the tile: origin c2w[9..11], direction the un-normalised _mv3(c2w, xyz) of screen2worlddir.  Fed to
 * vr_render_rays they reproduce vr_render's float output and work counters bit for bit. */
int vr_render_rays(const vr_tree* tree, const float* origins_dev, const float* dirs_dev, const float* t_max_dev,
                   int n_rays, const vr_options* opt, float* rgba32f_dev, vr_counters* counters_dev, void* stream);
int vr_camera_rays(const vr_camera* cam, const vr_rect* tile, float* origins_dev, float* dirs_dev, void* stream);

/* Host-buffer entry point: renders n_views full frames and copies each to
 * rgba8_host + i*4*w*h (pinned or pageable); returns after the last copy completed. */
int vr_render_frames_host(const vr_tree* tree, const vr_camera* cams, int n_views,
                          const vr_options* opt, uint8_t* rgba8_host);

/* Image egress (main_headless.cpp:216-222 with -o + src/imwrite.cpp:14-79): PNG files, 8-bit RGBA,
 * compression level 0 / filter NONE like the reference, written without libpng (stored deflate
 * blocks + CRC-32/Adler-32).  vr_render_frames_png renders, copies out and encodes n_views frames,
 * overlapping the three stages; paths[i] receives view i. */
int vr_write_png(const char* path, const uint8_t* rgba8_host, int width, int height);
int vr_render_frames_png(const vr_tree* tree, const vr_camera* cams, int n_views, const vr_options* opt,
                         const char* const* paths, int n_threads);

/* Copies the colour coefficients of the leaf containing world point xyz into out_dev as floats
 * (retrieve_cursor_lumisphere_kernel): min(data_dim-1, 3*basis_dim) values (3 for RGBA). */
int vr_probe_lumisphere(const vr_tree* tree, const float xyz_world[3], float* out_dev, void* stream);

/* Diagnostics: one full-frame render with the instrumented kernel that also records, per 8x4-pixel
 * work item (row-major tiles of 8x4), {start ns, end ns, SM id, global warp id} into
 * trace_dev[4 * n_items] (n_items = ceil(w/8)*ceil(h/4)). */
int vr_debug_trace(const vr_tree* tree, const vr_camera* cam, const vr_options* opt, uint8_t* rgba8_dev,
                   vr_counters* counters_dev, unsigned long long* trace_dev, void* stream);

/* Kernel variant selection for measurement.  0 = default: the inline-shading kernel (3 + 16*193) for batches, the
 * shading-queue kernel (7) for single-view launches on trees with 4, 9 or 16 basis functions (measured, DESIGN.md 4;
 * both produce identical bits).  vr_get_variant returns the process-wide setting (0 unless changed), vr_tree_variant
 * the variant a BATCH launch on `tree` resolves to (-1 if the setting is not available for its basis size), vr_variant_supported whether `variant` is
 * built into this library for a kernel basis of -1 (RGBA), 1, 4, 9, 16 or 25. */
int vr_set_variant(int variant);
int vr_get_variant(void);
int vr_tree_variant(const vr_tree* tree);
int vr_variant_supported(int kernel_basis, int variant);
/* Cap the grid of the persistent march kernels at `max_ctas` CTAs (0 = all resident CTAs).  Used by
 * multi-GPU drivers to leave a few SMs to a concurrently running peer copy. */
int vr_set_max_ctas(int max_ctas);
/* Multi-GPU plumbing without SM-resident collectives: finished RGBA8 frames / bands are moved to the
 * gathering GPU by the copy engines over NVLink (cudaMemcpyAsync between peer-mapped buffers), so the
 * persistent march kernel keeps every SM.  vr_dev_alloc returns plain cudaMalloc memory (the base
 * address an IPC handle needs); vr_ipc_export writes the 64-byte cudaIpcMemHandle_t of such a buffer,
 * vr_ipc_open maps a peer process's buffer into this process (enabling peer access when possible),
 * vr_copy_async is a stream-ordered device/peer/host copy (kind inferred from the pointers). */
int vr_dev_alloc(size_t bytes, void** ptr);
int vr_dev_free(void* ptr);
int vr_ipc_export(void* dev_ptr, unsigned char handle_out[64]);
int vr_ipc_open(const unsigned char handle[64], void** ptr_out);
int vr_ipc_close(void* ptr);
int vr_copy_async(void* dst, const void* src, size_t bytes, void* stream);
/* 2-D variant (cudaMemcpy2DAsync, kind inferred): scatters a rank's compact bands into their interleaved rows
 * of a frame that lives in a peer-mapped buffer. */
int vr_copy2d_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t width_bytes, size_t rows,
                    void* stream);

/* ---- multi-GPU, one process driving N devices (volrend_b200/csrc/vr_mg.cu) ------------------------------
 * What a multi-GPU main_headless.cpp needs (the reference is single-GPU: main_headless.cpp:118-121 picks ONE
 * device): the tree replicated on `devices`, poses or ray tiles sharded over them, finished RGBA8 frames
 * gathered on devices[0] by the copy engines over NVLink (peer copies, no SM-resident collective).
 *   VR_MG_VIEWS  view i -> device i % n            VR_MG_TILES  band b (band_h rows) of every frame -> device b % n
 * vr_mg_render is synchronous: on return n_views frames are in rgba8_dev0 (device memory on devices[0]; NULL =
 * an internal buffer, see vr_mg_frames_dev0) and, when rgba8_host != NULL, in host memory.  `batch` = views per
 * kernel launch per device (<= 0: all).  *ms_out = device time of the whole job, max over devices (CUDA events;
 * all devices start idle). */
typedef struct vr_mg vr_mg;
enum { VR_MG_VIEWS = 0, VR_MG_TILES = 1 };
int vr_mg_create(const vr_tree_desc* desc, const int* devices, int n_devices, vr_mg** out);
void vr_mg_destroy(vr_mg* mg);
int vr_mg_device_count(const vr_mg* mg);
int vr_mg_device(const vr_mg* mg, int index);
vr_tree* vr_mg_tree(const vr_mg* mg, int index);
int vr_mg_render(vr_mg* mg, const vr_camera* cams, int n_views, const vr_options* opt, int mode, int band_h, int batch,
                 uint8_t* rgba8_dev0, uint8_t* rgba8_host, float* ms_out);
const uint8_t* vr_mg_frames_dev0(const vr_mg* mg);
const char* vr_mg_last_error(const vr_mg* mg);
/* How many of this library's kernels were launched by this process. */
unsigned long long vr_launch_count(void);

const char* vr_last_error(void);
const char* vr_version(void);

#ifdef __cplusplus
}
#endif
#endif
