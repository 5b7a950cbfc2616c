// vr_api.cu -- C-ABI of the B200 PlenOctree ray-marcher (declared in include/volrend_b200.h).
//
// Owns the device layout of a tree (the job of N3Tree::load_cuda, reference
// src/cuda/n3tree.cu:9-41) and the launch logic (launch_renderer, src/cuda/volrend.cu:195-245).
// There is no CPU path in this library: every entry point needs a CUDA device.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cub/device/device_scan.cuh>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "volrend_b200.h"
#include "vr_kernels.h"
#include "vr_types.h"

using namespace vrb;

// ------------------------------------------------------------------------------------ errors
namespace {
thread_local std::string g_err;
std::atomic<int> g_variant{0};
std::atomic<unsigned long long> g_launches{0};
std::atomic<int> g_max_ctas{0};
// Resolved default variants (vr_kernels.h): queue kernel for >= 4 basis functions, else inline shading
constexpr int kVariantQueue = 7, kVariantInline = 3 + 16 * 193;
constexpr int kQueueSlots = 256;
constexpr int kCamRing = 8192;  // device ring of per-view cameras for batched launches

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define VR_CUDA(expr)                                                                              \
    do {                                                                                           \
        cudaError_t e__ = (expr);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(e__ == cudaErrorMemoryAllocation ? VR_ENOMEM : VR_ECUDA, "%s: %s (%s:%d)", \
                        #expr, cudaGetErrorString(e__), __FILE__, __LINE__);                       \
    } while (0)

int kernel_basis(int format, int basis_dim) {
    if (format == VR_FMT_RGBA || basis_dim < 0) return -1;
    switch (basis_dim) {
        case 1: case 4: case 9: case 16: case 25: return basis_dim;
        default: return 1;  // rt_core.cuh:134-160: no switch case matches -> only coefficient 0
    }
}
int rec_bytes_for(int kbd) { return kbd <= 1 ? 8 : ((3 * kbd * 2 + 15) / 16) * 16; }
}  // namespace

// Per-stream launch resources of a tree.  Work-queue slots and the camera ring are recycled in
// stream order only: a launch that reuses a slot is ordered behind the launch that used it before, so
// no fence is needed, and launches on different streams never share a slot.
struct StreamRes {
    unsigned int* queues = nullptr;  // kQueueSlots slots of kQueueSlotBytes: {head, done}, per-SM block states and locks (vr_march.cuh)
    CamDev* cam_ring = nullptr;      // kCamRing entries; batches take consecutive slots
    unsigned int next_queue = 0, cam_pos = 0;
    unsigned char* pool = nullptr;   // parked-ray stacks of the ray-pool kernel (kind 8), allocated on first use
    size_t pool_bytes = 0;
};

struct vr_tree {
    int device = 0;
    int num_sms = 0;
    TreeDev dev{};
    uint32_t* wide = nullptr;
    unsigned char* wrecs = nullptr;
    float* extra = nullptr;
    // slot-indexed arrays: only the experiment kernels (-DVR_EXPERIMENTS) read them
    uint32_t* nodes = nullptr;
    unsigned char* recs = nullptr;
    uint32_t* top = nullptr;
    uint32_t* wslot = nullptr;
    long long n_tables = 0;
    std::mutex res_mu;
    std::unordered_map<cudaStream_t, StreamRes> res;
    // vr_render_frames_host: chunk ring, streams and events are created once and kept
    struct HostPath {
        static constexpr int kRing = 4;
        uint8_t* buf[kRing] = {};
        size_t buf_bytes = 0;
        cudaEvent_t rendered[kRing] = {}, copied[kRing] = {};
        cudaStream_t sr[2] = {nullptr, nullptr}, sc = nullptr;
        bool ready = false;
    } host;
    std::mutex host_mu;
    vr_tree_info info{};
    int data_dim = 0;
    size_t l2_window_bytes = 0;  // table window kept in persisting L2 (VR_L2_PERSIST=1)
};

// ------------------------------------------------------------------------------------ upload
namespace {

// Host -> device copy of a large pageable array at pinned-memory speed: a few worker threads copy
// chunks into process-wide pinned staging buffers and issue the DMA from there (the reference uploads
// with one synchronous pageable cudaMemcpy, src/cuda/n3tree.cu:20-33, ~12 GB/s).
class Uploader {
  public:
    static constexpr int kWorkers = 4;
    static constexpr size_t kChunk = 8u << 20;
    static Uploader& get() { static Uploader u; return u; }
    cudaError_t copy(void* dst, const void* src, size_t bytes) {
        if (bytes < 4 * kChunk || !ensure()) return cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice);
        std::lock_guard<std::mutex> lk(mu_);
        int dev = 0;
        cudaGetDevice(&dev);
        const size_t n_chunks = (bytes + kChunk - 1) / kChunk;
        std::atomic<int> err{0};
        std::vector<std::thread> th;
        for (int w = 0; w < kWorkers; ++w)
            th.emplace_back([&, w]() {
                cudaSetDevice(dev);
                cudaStream_t st = nullptr;
                cudaEvent_t ev[2] = {nullptr, nullptr};
                if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) { err = 1; return; }
                for (auto& e : ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
                int k = 0;
                for (size_t c = (size_t)w; c < n_chunks && !err; c += kWorkers, ++k) {
                    const size_t off = c * kChunk, n = bytes - off < kChunk ? bytes - off : kChunk;
                    unsigned char* stage = stage_[2 * w + (k & 1)];
                    if (k >= 2) cudaEventSynchronize(ev[k & 1]);   // the DMA that last read this buffer is done
                    memcpy(stage, (const unsigned char*)src + off, n);
                    if (cudaMemcpyAsync((unsigned char*)dst + off, stage, n, cudaMemcpyHostToDevice, st) != cudaSuccess) err = 1;
                    cudaEventRecord(ev[k & 1], st);
                }
                if (cudaStreamSynchronize(st) != cudaSuccess) err = 1;
                for (auto& e : ev) cudaEventDestroy(e);
                cudaStreamDestroy(st);
            });
        for (auto& t : th) t.join();
        return err ? cudaErrorUnknown : cudaSuccess;
    }

  private:
    bool ensure() {
        std::lock_guard<std::mutex> lk(mu_);
        if (ready_) return true;
        if (failed_) return false;
        for (int i = 0; i < 2 * kWorkers; ++i)
            if (cudaHostAlloc((void**)&stage_[i], kChunk, cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                failed_ = true;
                return false;
            }
        ready_ = true;
        return true;
    }
    std::mutex mu_;
    unsigned char* stage_[2 * kWorkers] = {};
    bool ready_ = false, failed_ = false;
};

}  // namespace

// ------------------------------------------------------------------------------------ re-layout kernels
namespace {

// Source of the fp16 leaf data: the plain [slot][data_dim] array, or a quantised tree
// (scripts/compress_octree.py; CPU decode in src/n3tree.cpp:309-340):
//   data[slot][j + n_retain + k*n_total] = quant_colors[j][quant_map[j][slot]][k]   j < n_quant
//   data[slot][j + k*n_total]            = data_retained[j][slot][k]                j < n_retain
//   data[slot][data_dim-1]               = sigma[slot]
struct LeafSrc {
    const unsigned short* data;      // plain
    const unsigned short* colors;    // quantised
    const unsigned short* qmap;
    const unsigned short* retained;
    const unsigned short* sigma;
    long long n_slots;
    int data_dim, basis_dim, kbd, n_total, n_retain;
};

__device__ __forceinline__ unsigned short leaf_sigma(const LeafSrc& S, long long slot) {
    return S.data ? S.data[(size_t)slot * S.data_dim + (S.data_dim - 1)] : S.sigma[slot];
}

// half c (= channel * kbd + j) of the padded colour record of `slot`
__device__ __forceinline__ unsigned short leaf_half(const LeafSrc& S, long long slot, int c) {
    if (S.kbd <= 1) {  // one coefficient per channel: RGBA -> halfs 0,1,2 ; basis -> k[0], k[bd], k[2bd]
        if (c >= 3) return 0;
        if (S.data) return S.data[(size_t)slot * S.data_dim + (S.kbd < 0 ? c : c * S.basis_dim)];
        const int j = 0, k = c;  // quantised trees are never RGBA
        if (j < S.n_retain) return S.retained[((size_t)j * S.n_slots + slot) * 3 + k];
        return S.colors[((size_t)(j - S.n_retain) * 65536 + S.qmap[(size_t)(j - S.n_retain) * S.n_slots + slot]) * 3 + k];
    }
    if (c >= 3 * S.kbd) return 0;
    if (S.data) return S.data[(size_t)slot * S.data_dim + c];
    const int j = c % S.n_total, k = c / S.n_total;   // kbd == n_total here
    if (j < S.n_retain) return S.retained[((size_t)j * S.n_slots + slot) * 3 + k];
    const int q = j - S.n_retain;
    return S.colors[((size_t)q * 65536 + S.qmap[(size_t)q * S.n_slots + slot]) * 3 + k];
}

// nodes[i]: absolute child id, or leaf bit | sigma.  Also validates child links.
__global__ void relayout_nodes_kernel(const int32_t* __restrict__ child, LeafSrc S, uint32_t* __restrict__ nodes,
                                      long long capacity, int* __restrict__ bad) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S.n_slots) return;
    const int32_t rel = child[i];
    if (rel != 0) {
        const long long tgt = (i >> 3) + rel;
        if (tgt <= 0 || tgt >= capacity) {
            atomicExch(bad, 1);
            nodes[i] = kLeafBit;
        } else {
            nodes[i] = (uint32_t)tgt;
        }
    } else {
        nodes[i] = kLeafBit | (uint32_t)leaf_sigma(S, i);
    }
}

// depth[n] of every node by level-synchronous relaxation from the root.  A node that is reached
// twice (two parents, or a cycle) makes the input a DAG, not a tree: rejected, because the table
// builder and the ancestor stacks assume one depth per node.
__global__ void node_depth_kernel(const uint32_t* __restrict__ nodes, int* __restrict__ depth, long long capacity,
                                  int level, int* __restrict__ flags) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= capacity || depth[n] != level) return;
#pragma unroll
    for (int s = 0; s < 8; ++s) {
        const uint32_t w = nodes[n * 8 + s];
        if (!(w & kLeafBit)) {
            if (atomicCAS(&depth[w], -1, level + 1) != -1) atomicExch(flags + 2, 1);
            flags[1] = 1;
        }
    }
}

// cnt[r]: number of internal nodes whose depth is r modulo kWideLv
__global__ void count_parity_kernel(const int* __restrict__ depth, long long capacity, unsigned long long* __restrict__ cnt) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int r = (n < capacity && depth[n] >= 0) ? depth[n] % kWideLv : -1;
#pragma unroll
    for (int k = 0; k < kWideLv; ++k) {
        const unsigned int c = __reduce_add_sync(0xffffffffu, r == k ? 1u : 0u);
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(cnt + k, (unsigned long long)c);
    }
}

// a node owns a table when it is the root or its depth d has (d + v) % kWideLv == 0
__global__ void table_flag_kernel(const int* __restrict__ depth, long long capacity, int v, uint32_t* __restrict__ flag) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= capacity) return;
    const int d = depth[n];
    flag[n] = (d >= 0 && (n == 0 || (d + v) % kWideLv == 0)) ? 1u : 0u;
}

// wide[table * E + e], E = 8^kWideLv: e = ex << 2*LV | ey << LV | ez holds kWideLv octree levels per axis, first level
// in the high bit.  The tree hangs v levels below a virtual root (octant 0 each time), so the root table resolves only
// kWideLv - v real levels: its entries with a non-zero virtual bit are never looked up.
__global__ void build_wide_kernel(const uint32_t* __restrict__ nodes, const int* __restrict__ depth,
                                  const uint32_t* __restrict__ tid, uint32_t* __restrict__ wide,
                                  uint32_t* __restrict__ wslot, long long capacity, int v) {
    constexpr int LV = kWideLv, M = (1 << LV) - 1;
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n = g >> (3 * LV);
    const int e = (int)(g & (kWideEntries - 1));
    if (n >= capacity) return;
    const int d = depth[n];
    if (d < 0 || (n != 0 && (d + v) % LV != 0)) return;   // unreachable, or folded into an ancestor's table
    // leaf entry = kLeafBit | (103 + leaf depth + v) << 23 | sigma: the exponent field of the cube size on the
    // 2^(24-v) position grid (vr_march.cuh)
    const uint32_t ex = (e >> (2 * LV)) & M, ey = (e >> LV) & M, ez = e & M;
    const size_t o = (size_t)tid[n] * kWideEntries + e;
    uint32_t node = (uint32_t)n;
    int dn = d;
    for (int k = (n == 0) ? v : 0; k < LV; ++k) {
        const int sh = LV - 1 - k;
        const uint32_t oct = (((ex >> sh) & 1u) << 2) | (((ey >> sh) & 1u) << 1) | ((ez >> sh) & 1u);
        const uint32_t s = node * 8u + oct;
        const uint32_t w = nodes[s];
        if (w & kLeafBit) {
            wide[o] = kLeafBit | ((uint32_t)(103 + dn + 1 + v) << 23) | (w & 0xffffu);
            wslot[o] = s;
            return;
        }
        node = w;
        ++dn;
    }
    wide[o] = tid[node];
    wslot[o] = 0xffffffffu;
}

// wrecs[entry]: padded colour record of the entry's leaf, straight from the source arrays
// (16-byte chunks; 8-byte records as one chunk).  Entries that are not leaves stay zero.
__global__ void build_wrecs_kernel(const uint32_t* __restrict__ wslot, LeafSrc S, unsigned char* __restrict__ wrecs,
                                   long long n_entries, int rec_bytes) {
    const int chunks = rec_bytes >= 16 ? rec_bytes / 16 : 1;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long e = gid / chunks;
    const int c = (int)(gid % chunks);
    if (e >= n_entries) return;
    const uint32_t slot = wslot[e];
    const bool leaf = slot != 0xffffffffu;
    if (rec_bytes == 8) {
        ushort4 v = make_ushort4(0, 0, 0, 0);
        if (leaf) { v.x = leaf_half(S, slot, 0); v.y = leaf_half(S, slot, 1); v.z = leaf_half(S, slot, 2); }
        reinterpret_cast<ushort4*>(wrecs)[e] = v;
        return;
    }
    unsigned short h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (leaf) {
#pragma unroll
        for (int j = 0; j < 8; ++j) h[j] = leaf_half(S, slot, c * 8 + j);
    }
    uint4 v;
    v.x = h[0] | ((uint32_t)h[1] << 16); v.y = h[2] | ((uint32_t)h[3] << 16);
    v.z = h[4] | ((uint32_t)h[5] << 16); v.w = h[6] | ((uint32_t)h[7] << 16);
    reinterpret_cast<uint4*>(wrecs + (size_t)e * rec_bytes)[c] = v;
}

#ifdef VR_EXPERIMENTS
// recs[i]: colour coefficients of slot i, padded.  One thread per (slot, 16-byte chunk).
__global__ void relayout_recs_kernel(LeafSrc S, unsigned char* __restrict__ recs, int rec_bytes) {
    const int chunks = rec_bytes >= 16 ? rec_bytes / 16 : 1;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long slot = gid / chunks;
    const int c = (int)(gid % chunks);
    if (slot >= S.n_slots) return;
    if (rec_bytes == 8) {
        ushort4 v;
        v.x = leaf_half(S, slot, 0); v.y = leaf_half(S, slot, 1); v.z = leaf_half(S, slot, 2); v.w = 0;
        reinterpret_cast<ushort4*>(recs)[slot] = v;
        return;
    }
    unsigned short h[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) h[j] = leaf_half(S, slot, c * 8 + j);
    uint4 v;
    v.x = h[0] | ((uint32_t)h[1] << 16); v.y = h[2] | ((uint32_t)h[3] << 16);
    v.z = h[4] | ((uint32_t)h[5] << 16); v.w = h[6] | ((uint32_t)h[7] << 16);
    reinterpret_cast<uint4*>(recs + (size_t)slot * rec_bytes)[c] = v;
}

// top[cell]: leaf word (bit31 | depth<<28 | sigma) or the depth-4 node id.
__global__ void build_top_kernel(const uint32_t* __restrict__ nodes, uint32_t* __restrict__ top) {
    const int cell = blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= kTopCells) return;
    const uint32_t cx = (cell >> 8) & 15, cy = (cell >> 4) & 15, cz = cell & 15;
    uint32_t node = 0;
    for (int l = 1; l <= kTopLevel; ++l) {
        const int sh = kTopLevel - l;
        const uint32_t oct = (((cx >> sh) & 1u) << 2) | (((cy >> sh) & 1u) << 1) | ((cz >> sh) & 1u);
        const uint32_t w = nodes[node * 8u + oct];
        if (w & kLeafBit) {
            top[cell] = kLeafBit | ((uint32_t)l << 28) | (w & 0xffffu);
            return;
        }
        node = w;
    }
    top[cell] = node;
}
#endif

// one block per queue slot: {head, done} = 0, every SM's block state = "no block", locks free (vr_march.cuh next_item)
__global__ void queue_init_kernel(unsigned char* slots) {
    unsigned char* slot = slots + (size_t)blockIdx.x * kQueueSlotBytes;
    const int i = threadIdx.x;
    if (i < 2) reinterpret_cast<unsigned int*>(slot)[i] = 0u;
    reinterpret_cast<unsigned long long*>(slot + kQueueStateOff)[i] = ((unsigned long long)kBlkInvalid << 32) | kBlkIdle;
    reinterpret_cast<unsigned int*>(slot + kQueueLockOff)[i] = 0u;
}

// retrieve_cursor_lumisphere_kernel (volrend.cu:175-191): descends the wide tables.
__global__ void probe_kernel(TreeDev tree, float x, float y, float z, int n_out, float* __restrict__ out) {
    float p[3] = {tree.offset[0] + tree.scale[0] * x, tree.offset[1] + tree.scale[1] * y,
                  tree.offset[2] + tree.scale[2] * z};
    uint32_t u[3];
    for (int i = 0; i < 3; ++i) {
        p[i] = fmaxf(fminf(p[i], 1.f - 1e-6f), 0.f);
        u[i] = __float2uint_rz(p[i] * tree.pos_scale);
    }
    uint32_t T = 0, eidx = 0;
    constexpr uint32_t M = (1u << kWideLv) - 1u;
    for (int j = 0; j < 16; ++j) {
        const int sh = (24 - kWideLv) - kWideLv * j;
        eidx = T * (uint32_t)kWideEntries + ((((u[0] >> sh) & M) << (2 * kWideLv)) | (((u[1] >> sh) & M) << kWideLv) | ((u[2] >> sh) & M));
        const uint32_t w = tree.wide[eidx];
        if (w & kLeafBit) break;
        T = w;
    }
    const unsigned short* rec = reinterpret_cast<const unsigned short*>(tree.wrecs + (size_t)eidx * tree.rec_bytes);
    for (int i = threadIdx.x; i < n_out; i += blockDim.x) out[i] = __half2float(__ushort_as_half(rec[i]));
}

}  // namespace

// ------------------------------------------------------------------------------------ C-ABI
extern "C" {

const char* vr_last_error(void) { return g_err.c_str(); }
const char* vr_version(void) { return "volrend_b200 0.2 (sm_100a)"; }
static bool variant_ok(int kbd, int variant) {
    switch (kbd) {
        case -1: return variant_supported<-1>(variant);
        case 1: return variant_supported<1>(variant);
        case 4: return variant_supported<4>(variant);
        case 9: return variant_supported<9>(variant);
        case 16: return variant_supported<16>(variant);
        case 25: return variant_supported<25>(variant);
        default: return false;
    }
}
int vr_variant_supported(int kernel_basis, int variant) { return variant >= 0 && variant_ok(kernel_basis, variant) ? 1 : 0; }
int vr_set_variant(int variant) {
    // accepted when at least one basis size has it; a tree whose basis size lacks it fails at launch
    bool any = false;
    for (int kbd : {-1, 1, 4, 9, 16, 25}) any = any || (variant >= 0 && variant_ok(kbd, variant));
    if (!any) return fail(VR_EINVAL, "kernel variant %d is not built into this library", variant);
    g_variant.store(variant);
    return VR_OK;
}
int vr_get_variant(void) { return g_variant.load(); }
int vr_set_max_ctas(int max_ctas) {
    if (max_ctas < 0) return fail(VR_EINVAL, "max_ctas < 0");
    g_max_ctas.store(max_ctas);
    return VR_OK;
}
int vr_tree_variant(const vr_tree* t) {
    if (!t) return -1;
    const int v = g_variant.load();
    if (v != 0) return variant_ok(t->dev.kbd, v) ? v : -1;
    (void)kVariantQueue;   // single-view launches of 4/9/16-basis trees use it (launch_march, vr_kernels_inst.cu)
    return kVariantInline;
}
unsigned long long vr_launch_count(void) { return g_launches.load(); }

void vr_default_options(vr_options* o) {
    if (!o) return;
    memset(o, 0, sizeof(*o));
    o->step_size = 1e-4f; o->sigma_thresh = 1e-2f; o->stop_thresh = 1e-2f;  // render_options.hpp:14-23
    o->background_brightness = 1.f;
    o->render_bbox[3] = o->render_bbox[4] = o->render_bbox[5] = 1.f;
    o->basis_minmax[0] = 0; o->basis_minmax[1] = VR_BASIS_MAX - 1;
}

void vr_tree_destroy(vr_tree* t) {
    if (!t) return;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(t->device);
    cudaFree(t->nodes); cudaFree(t->recs); cudaFree(t->top); cudaFree(t->extra);
    cudaFree(t->wide); cudaFree(t->wslot); cudaFree(t->wrecs);
    for (auto& kv : t->res) { cudaFree(kv.second.queues); cudaFree(kv.second.cam_ring); cudaFree(kv.second.pool); }
    for (int i = 0; i < vr_tree::HostPath::kRing; ++i) {
        cudaFree(t->host.buf[i]);
        if (t->host.rendered[i]) cudaEventDestroy(t->host.rendered[i]);
        if (t->host.copied[i]) cudaEventDestroy(t->host.copied[i]);
    }
    for (auto st : t->host.sr) if (st) cudaStreamDestroy(st);
    if (t->host.sc) cudaStreamDestroy(t->host.sc);
    cudaSetDevice(prev);
    delete t;
}

static int tree_create_impl(const vr_tree_desc* d, const vr_tree_quant_desc* q, vr_tree** out) {
    if (!d || !out) return fail(VR_EINVAL, "null argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(VR_ENODEVICE, "no CUDA device: volrend_b200 has no CPU fallback");
    }
    if (d->N != 2) return fail(VR_EUNSUPPORTED, "N=%d: only N=2 octrees are supported (as in the reference)", d->N);
    if (d->capacity < 1 || d->capacity >= (1ll << 28)) return fail(VR_EINVAL, "capacity %lld out of range", (long long)d->capacity);
    if (!d->child || (!q && !d->data)) return fail(VR_EINVAL, "child/data arrays missing");
    if (q) {
        if (!q->quant_colors || !q->quant_map || !q->sigma) return fail(VR_EINVAL, "quantised arrays missing");
        if (q->n_quant < 1 || q->n_retain < 0 || (q->n_retain > 0 && !q->data_retained))
            return fail(VR_EINVAL, "bad quantised basis counts");
        if (d->format == VR_FMT_RGBA || q->n_quant + q->n_retain != d->basis_dim)
            return fail(VR_EINVAL, "codebook and map basis numbers does not match");   // n3tree.cpp:296-299
    }
    if (d->format < VR_FMT_RGBA || d->format > VR_FMT_ASG) return fail(VR_EINVAL, "bad data format %d", d->format);
    const int kbd = kernel_basis(d->format, d->basis_dim);
    if (kbd < 0 ? d->data_dim < 4 : d->data_dim < 3 * d->basis_dim + 1)
        return fail(VR_EINVAL, "data_dim %d too small for format %d basis %d", d->data_dim, d->format, d->basis_dim);
    if ((d->format == VR_FMT_SG || d->format == VR_FMT_ASG) && !d->extra)
        return fail(VR_EINVAL, "SG/ASG trees need extra_data");
    if ((d->format == VR_FMT_SG || d->format == VR_FMT_ASG) && d->basis_dim > VR_BASIS_MAX)
        return fail(VR_EINVAL, "basis_dim %d > %d", d->basis_dim, VR_BASIS_MAX);

    vr_tree* t = new vr_tree();
    struct Guard { vr_tree*& t; bool ok = false; ~Guard() { if (!ok) { vr_tree_destroy(t); t = nullptr; } } } guard{t};
    VR_CUDA(cudaGetDevice(&t->device));
    cudaDeviceProp prop;
    VR_CUDA(cudaGetDeviceProperties(&prop, t->device));
    t->num_sms = prop.multiProcessorCount;
    t->data_dim = d->data_dim;
    const long long n_slots = d->capacity * 8;
    const int rec_bytes = rec_bytes_for(kbd);
    const int TB = 256;
    Uploader& up = Uploader::get();

    // device scratch, freed on every exit path
    std::vector<void*> scratch;
    struct Scratch { std::vector<void*>& v; ~Scratch() { for (void* p : v) cudaFree(p); } } scratch_guard{scratch};
    auto dalloc = [&](void** p, size_t bytes) -> cudaError_t {
        cudaError_t e = cudaMalloc(p, bytes ? bytes : 1);
        if (e == cudaSuccess) scratch.push_back(*p);
        return e;
    };
    auto release = [&](void* p) {
        for (auto& s : scratch) if (s == p) { cudaFree(p); s = nullptr; }
    };

    int32_t* raw_child = nullptr;
    int* flags = nullptr;   // {bad link, changed, node reached twice}
    int* depth = nullptr;
    LeafSrc S{};
    S.n_slots = n_slots; S.data_dim = d->data_dim; S.basis_dim = d->basis_dim; S.kbd = kbd;
    S.n_total = d->basis_dim; S.n_retain = q ? q->n_retain : 0;
    VR_CUDA(dalloc((void**)&raw_child, (size_t)n_slots * 4));
    VR_CUDA(dalloc((void**)&flags, 4 * sizeof(int)));
    VR_CUDA(dalloc((void**)&depth, (size_t)d->capacity * sizeof(int)));
    VR_CUDA(cudaMalloc(&t->nodes, (size_t)n_slots * 4));
    VR_CUDA(up.copy(raw_child, d->child, (size_t)n_slots * 4));
    if (!q) {
        unsigned short* raw = nullptr;
        const size_t data_bytes = (size_t)n_slots * d->data_dim * 2;
        VR_CUDA(dalloc((void**)&raw, data_bytes));
        VR_CUDA(up.copy(raw, d->data, data_bytes));
        S.data = raw;
    } else {
        const size_t cb = (size_t)q->n_quant * 65536 * 3 * 2, mb = (size_t)q->n_quant * n_slots * 2,
                     sb = (size_t)n_slots * 2, rb = (size_t)q->n_retain * n_slots * 3 * 2;
        unsigned short *qc = nullptr, *qm = nullptr, *qs = nullptr, *qr = nullptr;
        VR_CUDA(dalloc((void**)&qc, cb));
        VR_CUDA(dalloc((void**)&qm, mb));
        VR_CUDA(dalloc((void**)&qs, sb));
        VR_CUDA(up.copy(qc, q->quant_colors, cb));
        VR_CUDA(up.copy(qm, q->quant_map, mb));
        VR_CUDA(up.copy(qs, q->sigma, sb));
        if (q->n_retain > 0) {
            VR_CUDA(dalloc((void**)&qr, rb));
            VR_CUDA(up.copy(qr, q->data_retained, rb));
        }
        S.colors = qc; S.qmap = qm; S.sigma = qs; S.retained = qr;
    }
    VR_CUDA(cudaMemset(flags, 0, 4 * sizeof(int)));
    if (d->extra && (d->format == VR_FMT_SG || d->format == VR_FMT_ASG)) {
        const size_t nf = (size_t)d->basis_dim * (d->format == VR_FMT_SG ? 4 : 11);
        VR_CUDA(cudaMalloc(&t->extra, nf * sizeof(float)));
        VR_CUDA(cudaMemcpy(t->extra, d->extra, nf * sizeof(float), cudaMemcpyHostToDevice));
    }
    relayout_nodes_kernel<<<(unsigned)((n_slots + TB - 1) / TB), TB>>>(raw_child, S, t->nodes, d->capacity, flags);
    VR_CUDA(cudaGetLastError());
    release(raw_child);

    // node depths (level-synchronous sweep) -> max leaf depth; validates that the links form a tree
    VR_CUDA(cudaMemset(depth, 0xff, (size_t)d->capacity * sizeof(int)));
    VR_CUDA(cudaMemset(depth, 0, sizeof(int)));
    int max_node_depth = 0;
    int h_flags[3] = {0, 0, 0};
    for (int level = 0;; ++level) {
        if (level >= kMaxTreeDepth) return fail(VR_EUNSUPPORTED, "tree deeper than %d levels (or its child links form a cycle)", kMaxTreeDepth);
        VR_CUDA(cudaMemsetAsync(flags + 1, 0, sizeof(int)));
        node_depth_kernel<<<(unsigned)((d->capacity + TB - 1) / TB), TB>>>(t->nodes, depth, d->capacity, level, flags);
        VR_CUDA(cudaMemcpy(h_flags, flags, sizeof(h_flags), cudaMemcpyDeviceToHost));
        if (h_flags[0]) return fail(VR_EINVAL, "child array has links outside [1, capacity)");
        if (h_flags[2]) return fail(VR_EINVAL, "child array is not a tree: a node is reachable along two paths");
        if (!h_flags[1]) break;
        max_node_depth = level + 1;
    }

    // kWideLv-levels-per-step tables.  Which nodes own one: those whose depth d has (d + v) % kWideLv == 0, plus the
    // root; the v with the fewest tables wins -- with another one every table at the deepest internal level would
    // replicate its 8 leaves 8 (or 64) times (several times more colour-record memory).
    unsigned long long* pcnt = nullptr;
    VR_CUDA(dalloc((void**)&pcnt, 4 * sizeof(unsigned long long)));
    VR_CUDA(cudaMemset(pcnt, 0, 4 * sizeof(unsigned long long)));
    count_parity_kernel<<<(unsigned)((d->capacity + TB - 1) / TB), TB>>>(depth, d->capacity, pcnt);
    unsigned long long h_pcnt[4] = {0, 0, 0, 0};
    VR_CUDA(cudaMemcpy(h_pcnt, pcnt, sizeof(h_pcnt), cudaMemcpyDeviceToHost));
    int wp = 0;
    unsigned long long n_tab64 = ~0ull;
    for (int v = 0; v < kWideLv; ++v) {
        if (max_node_depth + 1 + v > 24) continue;   // leaf depth + v must fit the 24-bit position grid
        const unsigned long long nt = h_pcnt[(kWideLv - v) % kWideLv] + (v ? 1 : 0);
        if (nt + 1 < n_tab64 || n_tab64 == ~0ull) { n_tab64 = nt; wp = v; }
    }
    if (const char* e = getenv("VR_WIDE_PARITY")) {
        const int v = atoi(e);
        if (v >= 0 && v < kWideLv && max_node_depth + 1 + v <= 24) { wp = v; n_tab64 = h_pcnt[(kWideLv - v) % kWideLv] + (v ? 1 : 0); }
    }
    if (n_tab64 * (unsigned long long)kWideEntries >= (1ull << 32)) return fail(VR_EUNSUPPORTED, "too many nodes for the wide tables");
    const uint32_t n_tab = (uint32_t)n_tab64;
    const long long n_entries = (long long)n_tab * kWideEntries;
    {
        uint32_t *flag = nullptr, *tid = nullptr;
        void* tmp = nullptr;
        size_t tmp_bytes = 0;
        VR_CUDA(dalloc((void**)&flag, (size_t)d->capacity * 4));
        VR_CUDA(dalloc((void**)&tid, (size_t)d->capacity * 4));
        table_flag_kernel<<<(unsigned)((d->capacity + TB - 1) / TB), TB>>>(depth, d->capacity, wp, flag);
        VR_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, flag, tid, (int)d->capacity));
        VR_CUDA(dalloc(&tmp, tmp_bytes));
        VR_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, flag, tid, (int)d->capacity));
        VR_CUDA(cudaMalloc(&t->wide, (size_t)n_entries * 4));
        VR_CUDA(cudaMalloc(&t->wslot, (size_t)n_entries * 4));
        const long long work = d->capacity * (long long)kWideEntries;
        build_wide_kernel<<<(unsigned)((work + TB - 1) / TB), TB>>>(t->nodes, depth, tid, t->wide, t->wslot, d->capacity, wp);
        VR_CUDA(cudaGetLastError());
        release(flag); release(tid); release(tmp);
    }
    release(depth);
    {
        const size_t wrec_bytes = (size_t)n_entries * rec_bytes;
        cudaError_t e = cudaMalloc(&t->wrecs, wrec_bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(VR_ENOMEM, "colour records of the wide tables need %.2f GB (%lld entries x %d B): %s", wrec_bytes / 1e9,
                        n_entries, rec_bytes, cudaGetErrorString(e));
        }
        const long long rwork = n_entries * (rec_bytes >= 16 ? rec_bytes / 16 : 1);
        build_wrecs_kernel<<<(unsigned)((rwork + TB - 1) / TB), TB>>>(t->wslot, S, t->wrecs, n_entries, rec_bytes);
        VR_CUDA(cudaGetLastError());
    }
#ifdef VR_EXPERIMENTS
    {   // slot-indexed records and the dense top grid of the experiment kernels
        VR_CUDA(cudaMalloc(&t->recs, (size_t)n_slots * rec_bytes));
        VR_CUDA(cudaMalloc(&t->top, kTopCells * 4));
        const long long rec_work = n_slots * (rec_bytes >= 16 ? rec_bytes / 16 : 1);
        relayout_recs_kernel<<<(unsigned)((rec_work + TB - 1) / TB), TB>>>(S, t->recs, rec_bytes);
        build_top_kernel<<<(kTopCells + TB - 1) / TB, TB>>>(t->nodes, t->top);
        VR_CUDA(cudaGetLastError());
    }
    VR_CUDA(cudaDeviceSynchronize());
#else
    VR_CUDA(cudaDeviceSynchronize());
    // the product kernels read the tables and the table-indexed records only
    cudaFree(t->nodes); t->nodes = nullptr;
    cudaFree(t->wslot); t->wslot = nullptr;
#endif
    t->n_tables = n_tab;
    g_launches += 7;

    TreeDev& D = t->dev;
    D.nodes = t->nodes; D.recs = t->recs; D.top = t->top; D.extra = t->extra;
    D.wide = t->wide; D.wslot = t->wslot; D.wrecs = t->wrecs;
    for (int i = 0; i < 3; ++i) { D.offset[i] = d->offset[i]; D.scale[i] = d->scale[i]; }
    D.ndc_width = d->use_ndc ? d->ndc_width : -1.f;  // data_spec.hpp:47
    D.ndc_height = d->ndc_height; D.ndc_focal = d->ndc_focal;
    D.N = d->N; D.format = d->format; D.basis_dim = d->basis_dim; D.kbd = kbd;
    D.rec_bytes = rec_bytes; D.max_depth = max_node_depth + 1; D.wide_p = wp; D.wide_entries = (uint32_t)n_entries;
    D.pos_scale = (float)(1u << (24 - wp));
    D.pos_hi = (1.f - 1e-6f) * D.pos_scale;   // exact: a power-of-two multiple of 0x3F7FFFEF
    D.icube_bias = 0x73000000u + ((uint32_t)wp << 23);
    vr_tree_info& I = t->info;
    I.capacity = d->capacity; I.max_depth = D.max_depth; I.rec_bytes = rec_bytes;
    I.node_bytes = n_slots * 4; I.rec_total_bytes = n_slots * (long long)rec_bytes;
    I.top_bytes = kTopCells * 4;
    I.kernel_basis = kbd; I.wide_parity = wp; I.n_tables = n_tab;
    I.wide_bytes = n_entries * 4; I.wrecs_bytes = n_entries * (long long)rec_bytes;
    I.kernel_bytes = I.wide_bytes + I.wrecs_bytes;
    I.device_bytes = I.kernel_bytes + (t->nodes ? I.node_bytes : 0) + (t->recs ? I.rec_total_bytes : 0) +
                     (t->wslot ? I.wide_bytes : 0) + (t->top ? I.top_bytes : 0);
    if (const char* e = getenv("VR_L2_PERSIST")) {
        if (atoi(e) > 0) {
            int max_persist = 0, max_window = 0;
            cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, t->device);
            cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, t->device);
            size_t want = (size_t)n_entries * 4;
            if (want > (size_t)max_window) want = (size_t)max_window;
            size_t carve = want < (size_t)max_persist ? want : (size_t)max_persist;
            if (carve > 0 && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve) == cudaSuccess)
                t->l2_window_bytes = want;
            cudaGetLastError();
        }
    }
    guard.ok = true;
    *out = t;
    return VR_OK;
}

int vr_tree_create(const vr_tree_desc* d, vr_tree** out) { return tree_create_impl(d, nullptr, out); }

int vr_tree_create_quantized(const vr_tree_quant_desc* q, vr_tree** out) {
    if (!q) return fail(VR_EINVAL, "null argument");
    if (q->base.data) return fail(VR_EINVAL, "quantised descriptor must not carry decoded data");
    return tree_create_impl(&q->base, q, out);
}

int vr_tree_get_info(const vr_tree* t, vr_tree_info* info) {
    if (!t || !info) return fail(VR_EINVAL, "null argument");
    *info = t->info;
    return VR_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------ launch plumbing
namespace {

void fill_opt(OptDev& o, const vr_options* s) {
    o.step_size = s->step_size; o.sigma_thresh = s->sigma_thresh; o.stop_thresh = s->stop_thresh;
    o.background_brightness = s->background_brightness;
    for (int i = 0; i < 6; ++i) o.render_bbox[i] = s->render_bbox[i];
    o.basis_min = s->basis_minmax[0]; o.basis_max = s->basis_minmax[1];
    for (int i = 0; i < 3; ++i) o.rot_dirs[i] = s->rot_dirs[i];
    o.render_depth = s->render_depth;
}
void fill_cam(CamDev& c, const vr_camera* s) {
    c.width = s->width; c.height = s->height; c.fx = s->fx; c.fy = s->fy;
    memcpy(c.c2w, s->c2w, sizeof(c.c2w));
}

// Launch resources of (tree, stream); created on the first launch on that stream.
int stream_res(vr_tree* t, cudaStream_t stream, StreamRes*& out) {
    std::lock_guard<std::mutex> lk(t->res_mu);
    auto it = t->res.find(stream);
    if (it == t->res.end()) {
        StreamRes r;
        VR_CUDA(cudaMalloc(&r.queues, (size_t)kQueueSlots * kQueueSlotBytes));
        cudaError_t e = cudaMalloc(&r.cam_ring, kCamRing * sizeof(CamDev));
        if (e == cudaSuccess) {   // legacy stream: ordered before later launches
            queue_init_kernel<<<kQueueSlots, 256>>>(reinterpret_cast<unsigned char*>(r.queues));
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        if (e != cudaSuccess) {
            cudaFree(r.queues); cudaFree(r.cam_ring);
            return fail(VR_ECUDA, "stream resources: %s", cudaGetErrorString(e));
        }
        it = t->res.emplace(stream, r).first;
    }
    out = &it->second;
    return VR_OK;
}

// rays: P describes caller-supplied rays (launch_rays) instead of pixels of a camera (launch_march)
int dispatch(const vr_tree* t, LaunchDev& P, bool count, bool surface, cudaStream_t stream, bool rays = false) {
    LaunchCfg cfg;
    cfg.variant = vr_get_variant();
    if (!variant_ok(t->dev.kbd, cfg.variant))
        return fail(VR_EUNSUPPORTED, "kernel variant %d is not available for kernel basis %d", cfg.variant, t->dev.kbd);
    cfg.max_ctas = g_max_ctas.load();
    cfg.count = count; cfg.surface = surface; cfg.num_sms = t->num_sms; cfg.stream = stream;
    vr_tree* mt = const_cast<vr_tree*>(t);
    StreamRes* sr = nullptr;
    if (int rc = stream_res(mt, stream, sr)) return rc;
    {
        std::lock_guard<std::mutex> lk(mt->res_mu);
        cfg.queue = reinterpret_cast<unsigned int*>(reinterpret_cast<unsigned char*>(sr->queues) + (size_t)(sr->next_queue++ % kQueueSlots) * kQueueSlotBytes);
    }
    cfg.pool = nullptr; cfg.pool_bytes = 0;
    if ((cfg.variant & 15) == 8) {   // ray-pool kernel: its parked-ray stacks live with the (tree, stream) resources
        size_t need = 0;
        switch (t->dev.kbd) {
            case 4: need = pool_bytes_for<4>(t->num_sms, t->dev.max_depth); break;
            case 9: need = pool_bytes_for<9>(t->num_sms, t->dev.max_depth); break;
            case 16: need = pool_bytes_for<16>(t->num_sms, t->dev.max_depth); break;
            case 25: need = pool_bytes_for<25>(t->num_sms, t->dev.max_depth); break;
            default: break;
        }
        std::lock_guard<std::mutex> lk(mt->res_mu);
        if (need > sr->pool_bytes) {
            // a grow only happens before the first kind-8 launch on this stream (the size depends on the tree alone)
            if (sr->pool) { cudaStreamSynchronize(stream); cudaFree(sr->pool); sr->pool = nullptr; sr->pool_bytes = 0; }
            if (cudaMalloc(&sr->pool, need) == cudaSuccess) sr->pool_bytes = need;
            else { cudaGetLastError(); sr->pool = nullptr; }   // no memory: the kernel runs without parking
        }
        cfg.pool = sr->pool; cfg.pool_bytes = sr->pool_bytes;
    }
    cfg.l2_window = t->wide;
    cfg.l2_window_bytes = t->l2_window_bytes;
    static const bool no_pdl = getenv("VR_NO_PDL") != nullptr && atoi(getenv("VR_NO_PDL")) > 0;
    cfg.pdl = !no_pdl;
    cudaError_t e;
    switch (t->dev.kbd) {
        case -1: e = rays ? launch_rays<-1>(P, cfg) : launch_march<-1>(P, cfg); break;
        case 1: e = rays ? launch_rays<1>(P, cfg) : launch_march<1>(P, cfg); break;
        case 4: e = rays ? launch_rays<4>(P, cfg) : launch_march<4>(P, cfg); break;
        case 9: e = rays ? launch_rays<9>(P, cfg) : launch_march<9>(P, cfg); break;
        case 16: e = rays ? launch_rays<16>(P, cfg) : launch_march<16>(P, cfg); break;
        case 25: e = rays ? launch_rays<25>(P, cfg) : launch_march<25>(P, cfg); break;
        default: return fail(VR_EUNSUPPORTED, "unsupported kernel basis %d", t->dev.kbd);
    }
    if (e == cudaErrorNotSupported)
        return fail(VR_EUNSUPPORTED, "kernel variant %d has no ray-batch form (ray launches run on variants 0, 7 and %d)",
                    cfg.variant, kVariantInline);
    if (e != cudaSuccess) return fail(VR_ECUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    g_launches += 1;
    return VR_OK;
}

// Upper bound of the warp tiles of one view for every tile shape the kernels are built with
// (2x16, 4x8, 8x4 pixels): the persistent kernels index tiles of a whole batch with 31 bits.
long long tile_bound(const vr_rect& r) { return ((long long)r.w / 2 + 1) * ((long long)r.h / 4 + 1); }

int check_common(const vr_tree* t, const vr_camera* cam, const vr_options* opt, const vr_rect* tile, vr_rect& r) {
    if (!t || !cam || !opt) return fail(VR_EINVAL, "null argument");
    if (cam->width <= 0 || cam->height <= 0) return fail(VR_EINVAL, "bad camera size %dx%d", cam->width, cam->height);
    if (tile) {
        r = *tile;
        if (r.w < 0 || r.h < 0 || r.x0 < 0 || r.y0 < 0 || r.x0 + r.w > cam->width || r.y0 + r.h > cam->height)
            return fail(VR_EINVAL, "tile (%d,%d,%d,%d) outside %dx%d frame", r.x0, r.y0, r.w, r.h, cam->width, cam->height);
    } else {
        r.x0 = r.y0 = 0; r.w = cam->width; r.h = cam->height;
    }
    if (tile_bound(r) > 0x7fffffffLL)
        return fail(VR_EUNSUPPORTED, "%dx%d pixels: more tiles than the 31-bit work queue can index", r.w, r.h);
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return fail(VR_ENODEVICE, "no CUDA device");
    if (dev != t->device) return fail(VR_EINVAL, "tree lives on device %d but device %d is current", t->device, dev);
    return VR_OK;
}

}  // namespace

namespace {
// Cameras of a batch go through a device ring owned by (tree, stream): no allocation on the launch path (a
// stream-ordered pool would hand memory back to the OS at every synchronisation), and a slot is rewritten
// only by a copy that is stream-ordered behind the launch that read it.  n_views <= kCamRing.
int stage_cams(const vr_tree* t, const vr_camera* cams, int n_views, cudaStream_t stream, LaunchDev& P) {
    if (n_views <= 1) return VR_OK;
    vr_tree* mt = const_cast<vr_tree*>(t);
    StreamRes* sr = nullptr;
    if (int rc = stream_res(mt, stream, sr)) return rc;
    unsigned int slot;
    {
        std::lock_guard<std::mutex> lk(mt->res_mu);
        if (sr->cam_pos + (unsigned int)n_views > (unsigned int)kCamRing) sr->cam_pos = 0;  // no wrap inside a batch
        slot = sr->cam_pos;
        sr->cam_pos += (unsigned int)n_views;
    }
    std::vector<CamDev> h(n_views);
    for (int i = 0; i < n_views; ++i) fill_cam(h[i], &cams[i]);
    CamDev* dcams = sr->cam_ring + slot;
    VR_CUDA(cudaMemcpyAsync(dcams, h.data(), sizeof(CamDev) * n_views, cudaMemcpyHostToDevice, stream));
    // pageable source: the copy has been staged when cudaMemcpyAsync returns
    P.cams = dcams;
    return VR_OK;
}
}  // namespace

extern "C" {

int vr_render_batch(const vr_tree* t, const vr_camera* cams, int n_views, const vr_options* opt, const vr_rect* tile,
                    uint8_t* rgba8_dev, float* rgba32f_dev, vr_counters* counters_dev, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n_views < 0) return fail(VR_EINVAL, "n_views < 0");
    if (n_views == 0) return VR_OK;
    vr_rect r;
    int rc = check_common(t, cams, opt, tile, r);
    if (rc) return rc;
    for (int i = 1; i < n_views; ++i)
        if (cams[i].width != cams[0].width || cams[i].height != cams[0].height)
            return fail(VR_EINVAL, "all views of a batch must share one image size");
    if (r.w == 0 || r.h == 0) return VR_OK;
    LaunchDev P{};
    P.tree = t->dev;
    fill_opt(P.opt, opt);
    fill_cam(P.cam, &cams[0]);
    P.n_views = n_views;
    P.x0 = r.x0; P.y0 = r.y0; P.w = r.w; P.h = r.h;
    P.rgba8 = rgba8_dev; P.rgbaf = reinterpret_cast<float4*>(rgba32f_dev);
    P.counters = counters_dev;
    int max_views = kCamRing;  // split very large batches: camera ring size, 31-bit tile index
    if (tile_bound(r) * max_views > 0x7fffffffLL) max_views = (int)(0x7fffffffLL / tile_bound(r));
    if (n_views > max_views) {
        const size_t tile_px = (size_t)r.w * r.h;
        for (int v0 = 0; v0 < n_views; v0 += max_views) {
            const int nv = n_views - v0 < max_views ? n_views - v0 : max_views;
            rc = vr_render_batch(t, cams + v0, nv, opt, tile, rgba8_dev ? rgba8_dev + 4 * tile_px * v0 : nullptr,
                                 rgba32f_dev ? rgba32f_dev + 4 * tile_px * v0 : nullptr, counters_dev, stream_);
            if (rc) return rc;
        }
        return VR_OK;
    }
    if ((rc = stage_cams(t, cams, n_views, stream, P))) return rc;
    return dispatch(t, P, counters_dev != nullptr, false, stream);
}

int vr_render_bands_batch(const vr_tree* t, const vr_camera* cams, int n_views, const vr_options* opt, int band_h,
                          int n_parts, int part, uint8_t* rgba8_dev, float* rgba32f_dev, void* stream_) {
    if (n_views < 0) return fail(VR_EINVAL, "n_views < 0");
    if (n_views == 0) return VR_OK;
    vr_rect r;
    int rc = check_common(t, cams, opt, nullptr, r);
    if (rc) return rc;
    if (band_h < 4 || band_h % 4 || n_parts < 1 || part < 0 || part >= n_parts)
        return fail(VR_EINVAL, "bands: band_h must be a positive multiple of 4 and 0 <= part < n_parts");
    for (int i = 1; i < n_views; ++i)
        if (cams[i].width != cams[0].width || cams[i].height != cams[0].height)
            return fail(VR_EINVAL, "all views of a batch must share one image size");
    const int rows = vr_band_rows(cams[0].height, band_h, n_parts, part);
    if (rows == 0) return VR_OK;
    vr_rect rr = r;
    rr.h = rows;
    int max_views = kCamRing;  // camera ring size, 31-bit tile index
    if (tile_bound(rr) * max_views > 0x7fffffffLL) max_views = (int)(0x7fffffffLL / tile_bound(rr));
    if (n_views > max_views) {
        const size_t part_px = (size_t)r.w * rows;
        for (int v0 = 0; v0 < n_views; v0 += max_views) {
            const int nv = n_views - v0 < max_views ? n_views - v0 : max_views;
            rc = vr_render_bands_batch(t, cams + v0, nv, opt, band_h, n_parts, part, rgba8_dev ? rgba8_dev + 4 * part_px * v0 : nullptr,
                                       rgba32f_dev ? rgba32f_dev + 4 * part_px * v0 : nullptr, stream_);
            if (rc) return rc;
        }
        return VR_OK;
    }
    LaunchDev P{};
    P.tree = t->dev;
    fill_opt(P.opt, opt);
    fill_cam(P.cam, &cams[0]);
    P.n_views = n_views;
    P.x0 = 0; P.y0 = 0; P.w = r.w; P.h = rows;
    P.band_h = band_h; P.band_parts = n_parts; P.band_part = part;
    P.rgba8 = rgba8_dev; P.rgbaf = reinterpret_cast<float4*>(rgba32f_dev);
    if ((rc = stage_cams(t, cams, n_views, (cudaStream_t)stream_, P))) return rc;
    return dispatch(t, P, false, false, (cudaStream_t)stream_);
}

int vr_render_bands(const vr_tree* t, const vr_camera* cam, const vr_options* opt, int band_h, int n_parts,
                    int part, uint8_t* rgba8_dev, float* rgba32f_dev, void* stream_) {
    return vr_render_bands_batch(t, cam, 1, opt, band_h, n_parts, part, rgba8_dev, rgba32f_dev, stream_);
}

int vr_band_rows(int height, int band_h, int n_parts, int part) {
    if (height <= 0 || band_h <= 0 || n_parts <= 0 || part < 0 || part >= n_parts) return 0;
    const int n_bands = (height + band_h - 1) / band_h;
    int rows = 0;
    for (int b = part; b < n_bands; b += n_parts) {
        const int y = b * band_h;
        rows += (height - y < band_h) ? height - y : band_h;
    }
    return rows;
}

int vr_debug_trace(const vr_tree* t, const vr_camera* cam, const vr_options* opt, uint8_t* rgba8_dev,
                   vr_counters* counters_dev, unsigned long long* trace_dev, void* stream_) {
    vr_rect r;
    int rc = check_common(t, cam, opt, nullptr, r);
    if (rc) return rc;
    if (!counters_dev || !trace_dev) return fail(VR_EINVAL, "trace needs counters and a trace buffer");
    LaunchDev P{};
    P.tree = t->dev;
    fill_opt(P.opt, opt);
    fill_cam(P.cam, cam);
    P.n_views = 1;
    P.x0 = 0; P.y0 = 0; P.w = r.w; P.h = r.h;
    P.rgba8 = rgba8_dev; P.counters = counters_dev; P.trace = trace_dev;
    return dispatch(t, P, true, false, (cudaStream_t)stream_);
}

int vr_render_rays(const vr_tree* t, const float* origins_dev, const float* dirs_dev, const float* t_max_dev, int n_rays,
                   const vr_options* opt, float* rgba32f_dev, vr_counters* counters_dev, void* stream_) {
    if (!t || !opt) return fail(VR_EINVAL, "null argument");
    if (n_rays < 0) return fail(VR_EINVAL, "n_rays < 0");
    if (n_rays == 0) return VR_OK;
    if (!origins_dev || !dirs_dev || !rgba32f_dev) return fail(VR_EINVAL, "null ray or output array");
    int ndev = 0, dev = -1;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cudaGetDevice(&dev) != cudaSuccess) {
        cudaGetLastError();
        return fail(VR_ENODEVICE, "no CUDA device: volrend_b200 has no CPU fallback");
    }
    if (dev != t->device) return fail(VR_EINVAL, "tree lives on device %d but device %d is current", t->device, dev);
    // the product kernels only: the experiment kernels and the ray-pool kernel (kind 8) march pixels of a camera
    const int v = vr_get_variant();
    if (v != 0 && v != kVariantQueue && v != kVariantInline)
        return fail(VR_EUNSUPPORTED, "kernel variant %d has no ray-batch form (ray launches run on variants 0, 7 and %d)", v,
                    kVariantInline);
    LaunchDev P{};
    P.tree = t->dev;
    fill_opt(P.opt, opt);
    P.n_views = 1;
    P.rgbaf = reinterpret_cast<float4*>(rgba32f_dev);
    P.counters = counters_dev;
    P.ray_o = origins_dev; P.ray_d = dirs_dev; P.ray_tmax = t_max_dev; P.n_rays = n_rays;
    return dispatch(t, P, counters_dev != nullptr, false, (cudaStream_t)stream_, true);
}

int vr_camera_rays(const vr_camera* cam, const vr_rect* tile, float* origins_dev, float* dirs_dev, void* stream_) {
    if (!cam || !origins_dev || !dirs_dev) return fail(VR_EINVAL, "null argument");
    if (cam->width <= 0 || cam->height <= 0) return fail(VR_EINVAL, "bad camera size %dx%d", cam->width, cam->height);
    vr_rect r{0, 0, cam->width, cam->height};
    if (tile) {
        r = *tile;
        if (r.w < 0 || r.h < 0 || r.x0 < 0 || r.y0 < 0 || r.x0 + r.w > cam->width || r.y0 + r.h > cam->height)
            return fail(VR_EINVAL, "tile (%d,%d,%d,%d) outside %dx%d frame", r.x0, r.y0, r.w, r.h, cam->width, cam->height);
    }
    if (r.w == 0 || r.h == 0) return VR_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(VR_ENODEVICE, "no CUDA device: volrend_b200 has no CPU fallback");
    }
    CamDev c;
    fill_cam(c, cam);
    VR_CUDA(launch_camera_rays(c, r.x0, r.y0, r.w, r.h, origins_dev, dirs_dev, (cudaStream_t)stream_));
    g_launches += 1;
    return VR_OK;
}

int vr_render(const vr_tree* t, const vr_camera* cam, const vr_options* opt, const vr_rect* tile, uint8_t* rgba8_dev,
              float* rgba32f_dev, vr_counters* counters_dev, void* stream) {
    return vr_render_batch(t, cam, 1, opt, tile, rgba8_dev, rgba32f_dev, counters_dev, stream);
}

int vr_render_composite(const vr_tree* t, const vr_camera* cam, const vr_options* opt, const vr_rect* tile,
                        uint8_t* rgba8_dev, const float* depth_dev, float* rgba32f_dev, void* stream_) {
    vr_rect r;
    int rc = check_common(t, cam, opt, tile, r);
    if (rc) return rc;
    if (!rgba8_dev || !depth_dev) return fail(VR_EINVAL, "composite mode needs colour and depth inputs");
    if (r.w == 0 || r.h == 0) return VR_OK;
    LaunchDev P{};
    P.tree = t->dev;
    fill_opt(P.opt, opt);
    fill_cam(P.cam, cam);
    P.n_views = 1;
    P.x0 = r.x0; P.y0 = r.y0; P.w = r.w; P.h = r.h;
    P.rgba8 = rgba8_dev; P.rgbaf = reinterpret_cast<float4*>(rgba32f_dev);
    P.depth_in = depth_dev; P.composite = 1;
    return dispatch(t, P, false, false, (cudaStream_t)stream_);
}

int vr_render_surface(const vr_tree* t, const vr_camera* cam, const vr_options* opt, unsigned long long rgba8_surf,
                      unsigned long long depth_surf, void* stream_) {
    vr_rect r;
    int rc = check_common(t, cam, opt, nullptr, r);
    if (rc) return rc;
    if (!rgba8_surf) return fail(VR_EINVAL, "null surface");
    LaunchDev P{};
    P.tree = t->dev;
    fill_opt(P.opt, opt);
    fill_cam(P.cam, cam);
    P.n_views = 1;
    P.x0 = 0; P.y0 = 0; P.w = r.w; P.h = r.h;
    P.surf = (cudaSurfaceObject_t)rgba8_surf; P.dsurf = (cudaSurfaceObject_t)depth_surf;
    P.composite = depth_surf != 0;
    return dispatch(t, P, false, true, (cudaStream_t)stream_);
}

int vr_render_frames_host(const vr_tree* t, const vr_camera* cams, int n_views, const vr_options* opt,
                          uint8_t* rgba8_host) {
    // main_headless.cpp:208-223 with -o: every frame goes back to host memory.  Frames are
    // rendered in chunks of a few views per launch on two alternating streams (the tail of
    // one chunk overlaps the head of the next) and copied out on a third stream while the
    // following chunks render.
    if (n_views < 0) return fail(VR_EINVAL, "n_views < 0");
    if (n_views == 0) return VR_OK;
    if (!rgba8_host) return fail(VR_EINVAL, "null host buffer");
    vr_rect r;
    int rc = check_common(t, cams, opt, nullptr, r);
    if (rc) return rc;
    for (int i = 1; i < n_views; ++i)
        if (cams[i].width != cams[0].width || cams[i].height != cams[0].height)
            return fail(VR_EINVAL, "all views must share one image size");
    const size_t frame = (size_t)4 * r.w * r.h;
    int chunk = 8;
    if (const char* e = getenv("VR_HOST_CHUNK")) chunk = atoi(e) > 0 ? atoi(e) : chunk;
    if (chunk > n_views) chunk = n_views;
    vr_tree* mt = const_cast<vr_tree*>(t);
    std::lock_guard<std::mutex> host_lock(mt->host_mu);   // one host-path sweep per tree at a time
    vr_tree::HostPath& R = mt->host;
    constexpr int kRing = vr_tree::HostPath::kRing;
    if (!R.ready) {
        VR_CUDA(cudaStreamCreateWithFlags(&R.sr[0], cudaStreamNonBlocking));
        VR_CUDA(cudaStreamCreateWithFlags(&R.sr[1], cudaStreamNonBlocking));
        VR_CUDA(cudaStreamCreateWithFlags(&R.sc, cudaStreamNonBlocking));
        for (int i = 0; i < kRing; ++i) {
            VR_CUDA(cudaEventCreateWithFlags(&R.rendered[i], cudaEventDisableTiming));
            VR_CUDA(cudaEventCreateWithFlags(&R.copied[i], cudaEventDisableTiming));
        }
        R.ready = true;
    }
    if (R.buf_bytes < frame * chunk) {
        for (int i = 0; i < kRing; ++i) { cudaFree(R.buf[i]); R.buf[i] = nullptr; }
        R.buf_bytes = 0;
        for (int i = 0; i < kRing; ++i) VR_CUDA(cudaMalloc(&R.buf[i], frame * chunk));
        R.buf_bytes = frame * chunk;
    }
    int c = 0;
    for (int v0 = 0; v0 < n_views; v0 += chunk, ++c) {
        const int nv = n_views - v0 < chunk ? n_views - v0 : chunk;
        const int s = c % kRing;
        cudaStream_t sr = R.sr[c & 1];
        if (c >= kRing) VR_CUDA(cudaStreamWaitEvent(sr, R.copied[s], 0));
        rc = vr_render_batch(t, cams + v0, nv, opt, nullptr, R.buf[s], nullptr, nullptr, sr);
        if (rc) return rc;
        VR_CUDA(cudaEventRecord(R.rendered[s], sr));
        VR_CUDA(cudaStreamWaitEvent(R.sc, R.rendered[s], 0));
        VR_CUDA(cudaMemcpyAsync(rgba8_host + (size_t)v0 * frame, R.buf[s], frame * nv, cudaMemcpyDeviceToHost, R.sc));
        VR_CUDA(cudaEventRecord(R.copied[s], R.sc));
    }
    VR_CUDA(cudaStreamSynchronize(R.sc));
    VR_CUDA(cudaStreamSynchronize(R.sr[0]));
    VR_CUDA(cudaStreamSynchronize(R.sr[1]));
    return VR_OK;
}

int vr_dev_alloc(size_t bytes, void** ptr) {
    if (!ptr) return fail(VR_EINVAL, "null argument");
    *ptr = nullptr;
    VR_CUDA(cudaMalloc(ptr, bytes ? bytes : 1));
    return VR_OK;
}
int vr_dev_free(void* ptr) {
    VR_CUDA(cudaFree(ptr));
    return VR_OK;
}
int vr_ipc_export(void* dev_ptr, unsigned char handle_out[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    if (!dev_ptr || !handle_out) return fail(VR_EINVAL, "null argument");
    cudaIpcMemHandle_t h;
    VR_CUDA(cudaIpcGetMemHandle(&h, dev_ptr));
    memcpy(handle_out, &h, 64);
    return VR_OK;
}
int vr_ipc_open(const unsigned char handle[64], void** ptr_out) {
    if (!handle || !ptr_out) return fail(VR_EINVAL, "null argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    VR_CUDA(cudaIpcOpenMemHandle(ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return VR_OK;
}
int vr_ipc_close(void* ptr) {
    VR_CUDA(cudaIpcCloseMemHandle(ptr));
    return VR_OK;
}
int vr_copy_async(void* dst, const void* src, size_t bytes, void* stream) {
    if (bytes == 0) return VR_OK;
    if (!dst || !src) return fail(VR_EINVAL, "null argument");
    VR_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
    return VR_OK;
}

int vr_copy2d_async(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width_bytes, size_t rows, void* stream) {
    if (width_bytes == 0 || rows == 0) return VR_OK;
    if (!dst || !src) return fail(VR_EINVAL, "null argument");
    VR_CUDA(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width_bytes, rows, cudaMemcpyDefault, (cudaStream_t)stream));
    return VR_OK;
}

int vr_probe_lumisphere(const vr_tree* t, const float xyz[3], float* out_dev, void* stream_) {
    if (!t || !xyz || !out_dev) return fail(VR_EINVAL, "null argument");
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return fail(VR_ENODEVICE, "no CUDA device");
    if (dev != t->device) return fail(VR_EINVAL, "tree lives on device %d but device %d is current", t->device, dev);
    if (t->dev.kbd > 0 && t->dev.kbd != t->dev.basis_dim)
        return fail(VR_EUNSUPPORTED, "probe unavailable for basis_dim %d (only coefficient 0 is resident)", t->dev.basis_dim);
    // the resident record holds the colour coefficients only: 3 per RGBA leaf, 3*basis_dim otherwise
    // (extra trailing channels of an over-wide data_dim are not kept)
    const int resident = t->dev.kbd < 0 ? 3 : 3 * t->dev.kbd;
    const int n_out = t->data_dim - 1 < resident ? t->data_dim - 1 : resident;
    probe_kernel<<<1, 32, 0, (cudaStream_t)stream_>>>(t->dev, xyz[0], xyz[1], xyz[2], n_out, out_dev);
    VR_CUDA(cudaGetLastError());
    g_launches += 1;
    return VR_OK;
}

}  // extern "C"
