// vr_kernels_inst.cu -- instantiates the march kernels for one basis size (-DVR_KBD=...).
// Compiled six times (RGBA, SH/SG/ASG 1, 4, 9, 16, 25) so the builds run in parallel.
//
// Product kernels:
//   kind 7           march_queue_kernel (vr_march_q.cuh): default for single-frame launches with 4, 9 or 16 basis
//                    functions (launch_renderer, the CLI), selectable for batches and for 25
//   kind 8           (VR_EXPERIMENTS) the same kernel with the ray pool (POOL = true): measured, slower
//   kind 3, tune 193 march_persistent_kernel with inline shading: default for batches and for RGBA / 1 / 25 basis
//                    functions, and the A/B partner of the queue kernel in the parity tests and the bench
// Both product kernels are also instantiated with OUT = kOutRays for caller-supplied rays (launch_rays).
// Built only with -DVR_EXPERIMENTS (make lib SUFFIX=_exp EXTRA=-DVR_EXPERIMENTS): the measured and
// rejected structures of round 1 -- CTA-per-tile kernel, TMA-staged top grid, deferred shading,
// software-pipelined march, tuning knobs (DESIGN.md 4).
#include <cstdlib>
#include <mutex>

#include "vr_kernels.h"
#include "vr_march_q.cuh"

#ifndef VR_KBD
#error "compile with -DVR_KBD=<-1|1|4|9|16|25>"
#endif

namespace vrb {

namespace {

// Resident CTAs of a persistent kernel, cached per (device, kernel, dynamic shared memory).
template <typename K>
int resident_ctas(K kernel, size_t smem, int num_sms) {
    struct Entry { int device; const void* fn; size_t smem; int per_sm; };
    static std::mutex mu;
    static Entry cache[32];
    static int n_cache = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    const void* fn = reinterpret_cast<const void*>(kernel);
    std::lock_guard<std::mutex> lk(mu);
    for (int i = 0; i < n_cache; ++i)
        if (cache[i].device == dev && cache[i].fn == fn && cache[i].smem == smem) return cache[i].per_sm * num_sms;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kBlock, smem) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 1;
    }
    if (n_cache < 32) cache[n_cache++] = Entry{dev, fn, smem, per_sm};
    return per_sm * num_sms;
}

// blocks: whether the kernel understands SM-local tile blocks (the product kernels do)
void set_work(LaunchDev& P, const LaunchCfg& cfg, bool blocks = true) {
    P.tiles_x = (P.w + kTW - 1) / kTW;
    P.tiles_y = (P.h + kTH - 1) / kTH;
    P.work_counter = cfg.queue;
    // Batches can have the queue hand out blocks of 8x8 tiles, the warps of an SM sharing a block (vr_march.cuh next_item).
    // Measured (profiles/r02_tuning_sweeps.txt): config 4 (SH25, 160-byte records, 1080p) 0.511 -> 0.498 ms/frame, config 2
    // (SH16) 0.0961 -> 0.0967: on by default for 25 basis functions only; VR_BLOCKS=0/1 forces it.  It needs enough blocks
    // per SM to balance (a block is ~20 us of an SM), so single frames always keep one tile per item.
    static const int force = getenv("VR_BLOCKS") ? atoi(getenv("VR_BLOCKS")) : -1;
    const long long bx = (P.tiles_x + kBlkW - 1) / kBlkW, by = (P.tiles_y + kBlkH - 1) / kBlkH, nb = bx * by * P.n_views;
    const bool want = force >= 0 ? force != 0 : (P.tree.kbd == 25 && P.n_views >= 2 && nb >= 16LL * cfg.num_sms);
    if (blocks && want && nb * kBlkTiles <= 0x7fffffffLL) {
        P.blk_mode = 1; P.blocks_x = (int)bx; P.n_blocks = (int)nb;
        P.n_tiles = (int)(nb * kBlkTiles);   // item ids (block * 64 + tile), incl. the tiles beyond the image edge
        set_div((uint32_t)(bx * by), P.div_view_mul, P.div_view_shift);
        set_div((uint32_t)bx, P.div_row_mul, P.div_row_shift);
        return;
    }
    P.blk_mode = 0; P.blocks_x = 0; P.n_blocks = 0;
    P.n_tiles = P.tiles_x * P.tiles_y * P.n_views;
    set_div((uint32_t)(P.tiles_x * P.tiles_y), P.div_view_mul, P.div_view_shift);
    set_div((uint32_t)P.tiles_x, P.div_row_mul, P.div_row_shift);
}

// Ray launches: work item k = rays 32k .. 32k+31, one item per queue pull (blocks of tiles are a 2-D pixel notion).
// The queue kernel carries an item as (lane << 26 | item): items of n_rays <= 2^31 - 1 rays stay below 2^26.
static_assert((0x7fffffffLL + 31) / 32 <= (1LL << 26), "ray items must fit the 26-bit item field");
void set_work_rays(LaunchDev& P, const LaunchCfg& cfg) {
    P.work_counter = cfg.queue;
    P.blk_mode = 0; P.blocks_x = 0; P.n_blocks = 0;
    P.n_tiles = (int)(((long long)P.n_rays + 31) / 32);
}

template <typename K>
cudaError_t launch_persistent_grid(K kernel, size_t smem, LaunchDev& P, const LaunchCfg& cfg, bool blocks = true) {
    if (P.n_rays > 0) set_work_rays(P, cfg);
    else set_work(P, cfg, blocks);
    int grid = resident_ctas(kernel, smem, cfg.num_sms);
    if (cfg.max_ctas > 0 && grid > cfg.max_ctas) grid = cfg.max_ctas;
    const int need = (P.n_tiles + (kBlock / 32) - 1) / (kBlock / 32);
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid); lc.blockDim = dim3(kBlock); lc.dynamicSmemBytes = smem; lc.stream = cfg.stream;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (cfg.pdl) {  // programmatic dependent launch: see pdl_wait_predecessor() in vr_march.cuh
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    if (cfg.l2_window_bytes) {  // keep the node table resident in the persisting part of L2
        attr[na].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[na].val.accessPolicyWindow.base_ptr = const_cast<void*>(cfg.l2_window);
        attr[na].val.accessPolicyWindow.num_bytes = cfg.l2_window_bytes;
        attr[na].val.accessPolicyWindow.hitRatio = 1.0f;
        attr[na].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr[na].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        ++na;
    }
    lc.attrs = attr; lc.numAttrs = na;
    return cudaLaunchKernelEx(&lc, kernel, P);
}

template <int KBD, bool TOP, bool COUNT, int OUT, int TUNE = 0>
cudaError_t launch_persistent(LaunchDev& P, const LaunchCfg& cfg) {
    const size_t smem = march_smem_bytes<TOP, (TUNE & kTuneWide) != 0 && !TOP>(P.tree.max_depth) + basis_smem_bytes<KBD>();
    return launch_persistent_grid(march_persistent_kernel<KBD, TOP, COUNT, OUT, TUNE>, smem, P, cfg);
}

template <int KBD, bool COUNT, int OUT, bool POOL = false>
cudaError_t launch_queue(LaunchDev& P, const LaunchCfg& cfg) {
    if constexpr (KBD >= 4) {
        // VR_EXTRA_SMEM: measurement knob -- pads the CTA's shared memory to move the L1/shared carve-out
        static const size_t extra = getenv("VR_EXTRA_SMEM") ? (size_t)atoi(getenv("VR_EXTRA_SMEM")) : 0;
        const size_t smem = queue_smem_bytes<KBD>(P.tree.max_depth) + extra;
        P.pool = nullptr;
        if (POOL) {   // parked-ray stacks: one per CTA of the persistent grid
            set_work(P, cfg, false);
            // a parked ray carries its pixel as (lane slot << 26 | tile index)
            if (P.n_tiles > (1 << 26)) return launch_queue<KBD, COUNT, OUT, false>(P, cfg);
            const size_t need = (size_t)resident_ctas(march_queue_kernel<KBD, COUNT, OUT, POOL>, smem, cfg.num_sms) * pool_bytes_per_cta<KBD>();
            if (cfg.pool && cfg.pool_bytes >= need) P.pool = cfg.pool;
        }
        return launch_persistent_grid(march_queue_kernel<KBD, COUNT, OUT, POOL>, smem, P, cfg, false);   // tile queue only
    } else {
        return cudaErrorInvalidValue;
    }
}

#ifdef VR_EXPERIMENTS
template <int KBD, bool TOP, bool COUNT, int OUT>
cudaError_t launch_tile(const LaunchDev& P, const LaunchCfg& cfg) {
    const size_t smem = march_smem_bytes<TOP>(P.tree.max_depth) + basis_smem_bytes<KBD>();
    dim3 grid((P.w + kTileW - 1) / kTileW, (P.h + kTileH - 1) / kTileH, P.n_views);
    march_tile_kernel<KBD, TOP, COUNT, OUT><<<grid, kBlock, smem, cfg.stream>>>(P);
    return cudaGetLastError();
}

template <int KBD, bool TOP, bool COUNT, int OUT>
cudaError_t launch_deferred(LaunchDev& P, const LaunchCfg& cfg) {
    const size_t smem = deferred_smem_bytes<TOP>(P.tree.max_depth);
    set_work(P, cfg, false);
    int grid = resident_ctas(march_deferred_kernel<KBD, TOP, COUNT, OUT>, smem, cfg.num_sms);
    const int need = (P.n_tiles + (kBlock / 32) - 1) / (kBlock / 32);
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    march_deferred_kernel<KBD, TOP, COUNT, OUT><<<grid, kBlock, smem, cfg.stream>>>(P);
    return cudaGetLastError();
}
#endif

constexpr int kInline = 193;  // cache hints + wide tables + table-indexed records

}  // namespace

// variant 0: the default for this basis size.  kind = variant & 15, tune = variant >> 4.
template <int KBD>
bool variant_supported(int variant) {
    if (variant == 0) return true;
    const int kind = variant & 15, tune = variant >> 4;
    if (kind == 7) return tune == 0 && KBD >= 4;
#ifdef VR_EXPERIMENTS
    if (kind == 8) return tune == 0 && KBD >= 4;
#endif
    if (kind == 3 && tune == kInline) return true;
#ifdef VR_EXPERIMENTS
    if (kind == 3) return tune == 0 || tune == 1 || tune == 2 || tune == 3 || tune == 8 || tune == 10 || tune == 16 ||
                          tune == 17 || tune == 64 || tune == 65;
    if (kind >= 1 && kind <= 6) return tune == 0;
#endif
    return false;
}

template <int KBD>
cudaError_t launch_march(LaunchDev& P, const LaunchCfg& cfg) {
    int variant = cfg.variant;
    if (!variant_supported<KBD>(variant)) return cudaErrorInvalidValue;
    // Default, from the measurements in DESIGN.md 4 (bench tree, ms/frame in 200-view batches / single-frame launches):
    //   SH4  inline 0.0849 / 0.152   queue 0.0919 / 0.146        SH9   inline 0.0866 / 0.159   queue 0.0936 / 0.149
    //   SH16 inline 0.0962 / 0.183   queue 0.0987 / 0.154        SH25  inline 0.1185 / 0.219   queue 0.3196 / 0.392
    // The queue pays ~30 instructions per march iteration (ballots, ring bookkeeping) for a 3x denser colour block: a
    // loss in batches, where other warps hide the inline block's latency, a win on single frames, where the long-ray
    // tail of the frame is what is waited for.  With 25 basis functions its per-ray basis values (112 B) push the CTA's
    // shared memory over the 8-CTA budget.  Both kernels produce identical bits.
    if (variant == 0) variant = (P.n_views == 1 && KBD >= 4 && KBD <= 16) ? 7 : 3 + 16 * kInline;
    const int kind = variant & 15, tune = variant >> 4;
    const bool queue = kind == 7 || kind == 8;
#ifdef VR_EXPERIMENTS
    if (kind == 8) {   // measured and rejected (DESIGN.md 4): the ray-pool form of the queue kernel
        if (cfg.surface) return launch_queue<KBD, false, kOutSurface, true>(P, cfg);
        if (cfg.count) return launch_queue<KBD, true, kOutLinear, true>(P, cfg);
        return launch_queue<KBD, false, kOutLinear, true>(P, cfg);
    }
#endif
    if (cfg.surface) {  // drop-in launch_renderer path writing the caller's cudaArray
        return queue ? launch_queue<KBD, false, kOutSurface>(P, cfg)
                     : launch_persistent<KBD, false, false, kOutSurface, kInline>(P, cfg);
    }
    if (cfg.count) {  // instrumented builds
        return queue ? launch_queue<KBD, true, kOutLinear>(P, cfg)
                     : launch_persistent<KBD, false, true, kOutLinear, kInline>(P, cfg);
    }
    if (queue) return launch_queue<KBD, false, kOutLinear>(P, cfg);
    if (kind == 3 && tune == kInline) return launch_persistent<KBD, false, false, kOutLinear, kInline>(P, cfg);
#ifdef VR_EXPERIMENTS
    if (kind == 3) {
        switch (tune) {
            case 0: return launch_persistent<KBD, false, false, kOutLinear>(P, cfg);
            case 1: return launch_persistent<KBD, false, false, kOutLinear, 1>(P, cfg);
            case 2: return launch_persistent<KBD, false, false, kOutLinear, 2>(P, cfg);
            case 3: return launch_persistent<KBD, false, false, kOutLinear, 3>(P, cfg);
            case 8: return launch_persistent<KBD, false, false, kOutLinear, 8>(P, cfg);
            case 10: return launch_persistent<KBD, false, false, kOutLinear, 10>(P, cfg);
            case 16: return launch_persistent<KBD, false, false, kOutLinear, 16>(P, cfg);
            case 17: return launch_persistent<KBD, false, false, kOutLinear, 17>(P, cfg);
            case 64: return launch_persistent<KBD, false, false, kOutLinear, 64>(P, cfg);
            case 65: return launch_persistent<KBD, false, false, kOutLinear, 65>(P, cfg);
            default: return cudaErrorInvalidValue;
        }
    }
    switch (kind) {
        case 1: return launch_tile<KBD, false, false, kOutLinear>(P, cfg);
        case 2: return launch_tile<KBD, true, false, kOutLinear>(P, cfg);
        case 4: return launch_persistent<KBD, true, false, kOutLinear>(P, cfg);
        case 5: return launch_deferred<KBD, false, false, kOutLinear>(P, cfg);
        case 6: return launch_deferred<KBD, true, false, kOutLinear>(P, cfg);
        default: break;
    }
#endif
    return cudaErrorInvalidValue;
}

// Ray launches (vr_render_rays): the two product kernels only.  Variant 0 resolves to the batch default, the inline
// kernel (vr_tree_variant); 7 selects the shading queue.  Anything else: cudaErrorNotSupported.
template <int KBD>
cudaError_t launch_rays(LaunchDev& P, const LaunchCfg& cfg) {
    const int variant = cfg.variant == 0 ? 3 + 16 * kInline : cfg.variant;
    if (P.n_rays <= 0 || cfg.surface) return cudaErrorInvalidValue;
    if (variant == 7 && KBD >= 4)
        return cfg.count ? launch_queue<KBD, true, kOutRays>(P, cfg) : launch_queue<KBD, false, kOutRays>(P, cfg);
    if (variant == 3 + 16 * kInline)
        return cfg.count ? launch_persistent<KBD, false, true, kOutRays, kInline>(P, cfg)
                         : launch_persistent<KBD, false, false, kOutRays, kInline>(P, cfg);
    return cudaErrorNotSupported;
}

template <int KBD>
size_t pool_bytes_for(int num_sms, int max_depth) {
#ifndef VR_EXPERIMENTS
    (void)num_sms; (void)max_depth;
    return 0;
#else
    if constexpr (KBD >= 4) {
        const size_t smem = queue_smem_bytes<KBD>(max_depth);
        return (size_t)resident_ctas(march_queue_kernel<KBD, false, kOutLinear, true>, smem, num_sms) * pool_bytes_per_cta<KBD>();
    } else {
        return 0;
    }
#endif
}

template cudaError_t launch_march<VR_KBD>(LaunchDev&, const LaunchCfg&);
template cudaError_t launch_rays<VR_KBD>(LaunchDev&, const LaunchCfg&);
template size_t pool_bytes_for<VR_KBD>(int, int);
template bool variant_supported<VR_KBD>(int);

}  // namespace vrb
