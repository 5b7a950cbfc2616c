// vr_types.h -- device-side parameter blocks shared by the C-ABI and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "volrend_b200.h"

namespace vrb {

// Leaf flag of a node word; the low 16 bits then hold sigma as fp16 bits.
constexpr uint32_t kLeafBit = 0x80000000u;
// Level of the dense top grid staged into shared memory (16^3 cells).
constexpr int kTopLevel = 4;
constexpr int kTopCells = 1 << (3 * kTopLevel);
// Deepest leaf we accept: positions are 24-bit fixed point (fp32 mantissa).
constexpr int kMaxTreeDepth = 23;
// Octree levels resolved per table fetch (2: 64-entry tables, 3: 512-entry tables).  Build-time choice so that entry
// indices are shifts by constants: make lib EXTRA=-DVR_WIDE_LV=3.
#ifndef VR_WIDE_LV
#define VR_WIDE_LV 2
#endif
constexpr int kWideLv = VR_WIDE_LV;
constexpr int kWideEntries = 1 << (3 * kWideLv);
static_assert(kWideLv == 2 || kWideLv == 3, "tables resolve two or three octree levels");
// tables on a root-to-leaf path (the ancestor stack of the march kernels)
inline __host__ __device__ int wide_table_levels(int max_depth) { return (max_depth + kWideLv - 2) / kWideLv + 1; }

// Device copy of one N3Tree, re-laid-out at upload (vr_tree_create):
//  nodes[node*8 + oct]  internal: absolute child node id (>0)
//                       leaf:     kLeafBit | sigma_fp16_bits
//  recs[(node*8+oct)*rec_bytes ...]  colour coefficients only (sigma moved into the
//                       node word), channel-major fp16, padded to a 16-byte multiple
//                       (8 bytes for one coefficient per channel)
//  top[cell]            16^3 dense grid: (depth<<28)|node of the deepest internal node
//                       (depth <= kTopLevel-1) on the path to that level-4 cell
struct TreeDev {
    const uint32_t* nodes;
    const unsigned char* recs;
    const uint32_t* top;
    // two-levels-per-step view of the same octree: one 64-entry table per internal node whose depth has
    // parity wide_p (plus the root); entry = table id of the grandchild, or leaf word:
    //   kLeafBit | (103 + leaf depth) << 23 | sigma   (bits 23..30 = fp32 exponent of the cube size)
    const uint32_t* wide;
    const uint32_t* wslot;   // parallel array: the leaf's slot (node*8+oct) for record lookup
    const unsigned char* wrecs;  // colour records re-indexed by wide entry (no wslot indirection)
    const float* extra;
    float offset[3];
    float scale[3];
    float ndc_width, ndc_height, ndc_focal;
    int32_t N;          // 0: nothing to draw (background only)
    int32_t format;     // VR_FMT_*
    int32_t basis_dim;  // reference basis_dim (-1 RGBA)
    int32_t kbd;        // kernel basis: -1 RGBA, 1, 4, 9, 16, 25 (others collapse to 1)
    int32_t rec_bytes;
    int32_t max_depth;
    int32_t wide_p;     // v in [0, kWideLv): internal nodes of depth d with (d + v) % kWideLv == 0 own a table (+ the root)
    uint32_t wide_entries;  // number of table entries (64 per table): bound of every record / table index
    // With wide_p = 1 the tables behave as if the octree hung one level below a virtual root (octant 0): leaf words
    // carry depth + wide_p, and the march keeps positions on a 2^(24 - wide_p) grid.  The three constants below are
    // all the kernel needs of the parity -- no per-sample arithmetic on it.
    float pos_scale;        // 2^(24 - wide_p)
    float pos_hi;           // (1 - 1e-6f) * pos_scale: upper clamp of a position (n3tree_query.hpp:17-19)
    uint32_t icube_bias;    // 0x73000000 + (wide_p << 23): 1/2^depth = bits(icube_bias - (w & 0x7f800000))
};

struct CamDev {
    int32_t width, height;
    float fx, fy;
    float c2w[12];
};

struct OptDev {
    float step_size, sigma_thresh, stop_thresh, background_brightness;
    float render_bbox[6];
    int32_t basis_min, basis_max;
    float rot_dirs[3];
    int32_t render_depth;
};

// Magic numbers for n / d, exact for 0 <= n < 2^31 (d >= 1): with 2^(s-1) < d <= 2^s and
// m = ceil(2^(31+s) / d) < 2^32, floor(n*m / 2^(31+s)) = floor(n/d) because the excess
// n*(m*d - 2^(31+s)) / (d*2^(31+s)) stays below 1/d.
inline void set_div(uint32_t d, uint32_t& mul, int32_t& shift) {
    if (d <= 1) { mul = 0; shift = -1; return; }
    int s = 0;
    while ((1ull << s) < d) ++s;
    mul = (uint32_t)(((1ull << (31 + s)) + d - 1) / d);
    shift = s - 1;
}

// Work queue of the persistent kernels.  One slot per launch in flight: {head, done CTAs}, then per SM id (mod 256) a
// 64-bit block state and a 32-bit lock (SM-local tile blocks, vr_march.cuh next_item).
#ifndef VR_BLK_W
#define VR_BLK_W 8
#endif
#ifndef VR_BLK_H
#define VR_BLK_H 8
#endif
constexpr int kBlkW = VR_BLK_W, kBlkH = VR_BLK_H, kBlkTiles = kBlkW * kBlkH;    // a block = 8x8 warp tiles = 32x64 pixels
constexpr uint32_t kBlkDone = 0xfffffffdu, kBlkInvalid = 0xffffffffu;
constexpr unsigned long long kBlkIdle = 0x80000000ull;             // low word of a state that holds no tiles
constexpr int kQueueSlotBytes = 4096, kQueueStateOff = 64, kQueueLockOff = 64 + 256 * 8;

struct LaunchDev {
    TreeDev tree;
    OptDev opt;
    CamDev cam;            // used when cams == nullptr
    const CamDev* cams;    // device array for batches
    int32_t n_views;
    int32_t x0, y0, w, h;  // tile inside the cam.width x cam.height frame (h = rows of the output buffer)
    int32_t band_h, band_parts, band_part;  // ray-tile sharding: output row r is frame row
                                            // y0 + ((r/band_h)*band_parts + band_part)*band_h + r%band_h
    uint8_t* rgba8;        // linear tile-sized RGBA8 per view (or nullptr)
    float4* rgbaf;         // linear tile-sized float4 per view (or nullptr)
    const float* depth_in; // composite mode: per-pixel t limit (world units)
    vr_counters* counters; // device counters (instrumented kernels only)
    cudaSurfaceObject_t surf, dsurf;
    int32_t composite;     // 1: read existing colour from rgba8/surf + depth limit
    int32_t tiles_x, tiles_y, n_tiles;  // persistent kernels: work decomposition
    // division of a tile index (< 2^31) by tiles_x*tiles_y and by tiles_x as multiply-high + shift
    // (set_div): q = shift < 0 ? n : umulhi(n, mul) >> shift
    uint32_t div_view_mul, div_row_mul;
    int32_t div_view_shift, div_row_shift;
    unsigned int* work_counter;         // persistent kernels: global work queue {head, done CTAs} (start of a queue slot)
    // SM-local tile blocks (batches, vr_march.cuh next_item): the queue hands out BLOCKS of 8x8 warp tiles, the warps of
    // one SM share a block, so that neighbouring tiles -- same tables, same records -- are marched at the same time on
    // the same L1.  blk_mode 0: one tile per queue item (single frames: finest balance).
    int32_t blk_mode, blocks_x, n_blocks;
    unsigned char* pool;                // ray-pool kernels: parked-ray stacks, one per CTA (vr_march_q.cuh); nullptr = no parking
    unsigned long long* trace;          // diagnostics: per work item {start ns, end ns, smid, warp}
    // Ray launches (OUT == kOutRays, vr_render_rays): work item k is the 32 rays 32k .. 32k+31, lane l marches ray
    // 32k + l (< n_rays) and writes rgbaf[ray].  World-space origins / directions [n_rays][3]; depth limits or nullptr.
    const float* ray_o;
    const float* ray_d;
    const float* ray_tmax;
    int32_t n_rays;
};

}  // namespace vrb
