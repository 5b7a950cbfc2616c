// vr_march_q.cuh -- the march kernel with a WARP-SHARED SHADING QUEUE (warp-level compaction of the colour work):
// persistent warps + wide tables (vr_march.cuh) + a ballot/popc-compacted ring of shaded samples per warp.
// Default for single-view launches on trees with 4, 9 or 16 basis functions (launch_renderer, the CLI); batches
// default to the inline-shading kernel of vr_march.cuh (launch_march in vr_kernels_inst.cu has the numbers).
//
// Why (tools/lane_sim.c replays the exact sample sequence of the bench frames on the CPU and counts warp
// instructions per scheduling policy, profiles/r02_lane_sim.txt; ncu in profiles/r02_ncu_queue_*.txt):
//   * with inline shading the 190-instruction colour block of rt_core.cuh:125-165 runs whenever ANY lane of the
//     warp sits on a surface: 10.8 of 32 lanes active, 28 % of all issued instructions;
//   * a queue shared by the warp keeps the coherent 4x8 tiles for the traversal and compacts the shading work
//     across lanes AND iterations: 29.8 of 32 lanes in the colour block, and the 96-byte record fetch is waited
//     for once per 32 shaded samples instead of once per shaded warp-iteration;
//   * the price is ~30 instructions per march iteration (two votes, ring bookkeeping, a predicated body) and
//     12 KB more shared memory per CTA (less L1).  Measured: a tie to a small loss in 200-view batches, where other
//     warps hide the inline block's latency; 17 % faster on single frames, where the frame waits for its tail.
//
// How: the colour of a sample never feeds back into the traversal (transmittance, early stop and the
// next position depend on sigma and the cell geometry only, rt_core.cuh:116-120,174-187).  So the
// march loop only appends {record index, weight, owner lane} to a 64-slot ring in shared memory
// (ballot + popc compaction).  Whenever 32 items are pending, ALL lanes shade one item each -- any
// lane can shade any ray's sample because the per-ray basis values are parked in shared memory -- and
// write the three colour terms weight/(1+exp(-dot)) back into the slot.  Each owner then adds its
// terms to its own accumulators in slot order == sample order, so every ray performs exactly the
// additions of rt_core.cuh:163 in the reference's order: bit-identical output.
#pragma once
#include <cstdio>

#include "vr_march.cuh"

namespace vrb {

#ifndef VR_QPREFETCH
#define VR_QPREFETCH 0   // L2 prefetches of the colour record issued at enqueue time (0, 1 or 3 per record)
#endif

constexpr int kQSlots = 64;          // ring slots per warp (two 32-item windows)
constexpr int kQSlotBytes = 16;      // {idx, weight, owner, -} in; {r, g, b, -} out

template <int KBD>
struct BasisQ { static constexpr int n = (BasisCount<KBD>::n + 3) / 4; };   // float4 groups per ray

__host__ __device__ inline int wide_levels(int max_depth) {
    const int l = wide_table_levels(max_depth);
    return l < 1 ? 1 : l;
}

constexpr int kParkQ = 3;   // float4 groups of ray constants parked across a drain

// shared memory of one CTA: [ control | parked ray constants | basis values | shading queues | table-id stacks ]
template <int KBD>
__host__ __device__ inline size_t queue_smem_bytes(int max_depth) {
    return 16 /* control words, see kCtrlBytes */ + (size_t)wide_levels(max_depth) * kBlock * 4 + (size_t)kParkQ * kBlock * 16 +
           (size_t)BasisQ<KBD>::n * kBlock * 16 + (size_t)(kBlock / 32) * kQSlots * kQSlotBytes;
}

__device__ __forceinline__ void sts128_a(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" :: "r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void lds128_a(uint32_t addr, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
}

// One channel of rt_core.cuh:130-163: tmp = B0*k0 (+ s[16..24]) (+ s[9..15]) (+ s[4..8]) + s[1..3], every chain
// s[lo..hi] = fma(B_hi, k_hi, ... fma(B_lo, k_lo, B_{lo+1} * k_{lo+1})).  The basis values of the OWNER ray are
// read from shared memory one float4 group at a time and consumed immediately (4 live values instead of
// 16/25): the chains are independent, so visiting the coefficients in memory order and keeping one partial
// sum per chain performs exactly the reference's operations on exactly its operands.
template <int KBD, typename KF>
__device__ __forceinline__ float channel_dot(KF K, uint32_t bs_owner) {
    static_assert(KBD == 4 || KBD == 9 || KBD == 16 || KBD == 25, "queue kernel: 4, 9, 16 or 25 basis functions");
    float tmp0 = 0.f, s1 = 0.f, s4 = 0.f, s9 = 0.f, s16 = 0.f;
#pragma unroll
    for (int q = 0; q < BasisQ<KBD>::n; ++q) {
        uint32_t v[4];
        lds128_a(bs_owner + (uint32_t)q * (32u * 16u), v[0], v[1], v[2], v[3]);
        auto B = [&](int j) -> float { return __uint_as_float(v[j - 4 * q]); };
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int j = 4 * q + k;
            if (j >= KBD) continue;
            if (j == 0) { tmp0 = __fmul_rn(B(0), K(0)); continue; }
            // chain starts: the reference multiplies element lo+1 first, then fuses element lo
            if (j == 1)  { s1 = __fmaf_rn(B(1), K(1), __fmul_rn(B(2), K(2))); continue; }
            if (j == 4)  { s4 = __fmaf_rn(B(4), K(4), __fmul_rn(B(5), K(5))); continue; }
            if (j == 9)  { s9 = __fmaf_rn(B(9), K(9), __fmul_rn(B(10), K(10))); continue; }
            if (j == 16) { s16 = __fmaf_rn(B(16), K(16), __fmul_rn(B(17), K(17))); continue; }
            if (j == 2 || j == 5 || j == 10 || j == 17) continue;  // consumed by the chain start
            if (j <= 3) s1 = __fmaf_rn(B(j), K(j), s1);
            else if (j <= 8) s4 = __fmaf_rn(B(j), K(j), s4);
            else if (j <= 15) s9 = __fmaf_rn(B(j), K(j), s9);
            else s16 = __fmaf_rn(B(j), K(j), s16);
        }
    }
    float tmp = tmp0;
    if constexpr (KBD >= 25) tmp = __fadd_rn(tmp, s16);
    if constexpr (KBD >= 16) tmp = __fadd_rn(tmp, s9);
    if constexpr (KBD >= 9) tmp = __fadd_rn(tmp, s4);
    tmp = __fadd_rn(tmp, s1);
    return tmp;
}

// All lanes: lane i shades item i of the window at q_win (n items) and replaces it by its three colour
// terms weight / (1 + expf(-dot)) (rt_core.cuh:163).
template <int KBD>
__device__ __forceinline__ void drain_window(uint32_t q_win, uint32_t n, uint32_t bs_warp, const unsigned char* __restrict__ wrecs,
                                             uint32_t dbg_limit = 0u, int dbg_site = 0) {
    const uint32_t lane = threadIdx.x & 31u;
    if (lane < n) {
        const uint32_t slot = q_win + lane * kQSlotBytes;
        uint32_t idx, wbits, owner, pad;
        lds128_a(slot, idx, wbits, owner, pad);
#ifdef VR_POOL_DEBUG
        if (idx >= dbg_limit || owner > 31u) {
            printf("drain site %d: block %d warp %d lane %u n %u q_win %u: idx %u (limit %u) w %08x owner %u pad %u\n", dbg_site, blockIdx.x,
                   threadIdx.x >> 5, lane, n, q_win, idx, dbg_limit, wbits, owner, pad);
            idx = 0; owner = 0;
        }
#endif
        const unsigned char* rec = rec_addr(wrecs, idx, RecBytes<KBD>::n);
        const uint32_t bs_owner = bs_warp + owner * 16u;
        const float weight = __uint_as_float(wbits);
        float out[3];
        if constexpr (RecWords<KBD>::n <= 24) {
            // whole record in flight at once (3 x LDG.256 for SH16)
            uint32_t w[RecWords<KBD>::n];
            load_rec<KBD, kTuneHint | kTuneLd256>(rec, w);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                auto K = [&](int j) -> float {
                    const int h = c * KBD + j;
                    const uint32_t u = w[h >> 1];
                    return half_bits_to_float((h & 1) ? (u >> 16) : u);
                };
                out[c] = sigmoid_weighted(weight, channel_dot<KBD>(K, bs_owner));
            }
        } else {
            // SH25: 160-byte record, one channel (50 bytes inside four 16-byte chunks) at a time
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                constexpr int kHalfs = KBD;
                const int first = (c * kHalfs * 2) / 16;   // first 16-byte chunk of the channel
                uint32_t w[16];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    uint4 qv;
                    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(qv.x), "=r"(qv.y), "=r"(qv.z), "=r"(qv.w) : "l"(rec + 16 * (first + i)));
                    w[4 * i] = qv.x; w[4 * i + 1] = qv.y; w[4 * i + 2] = qv.z; w[4 * i + 3] = qv.w;
                }
                auto K = [&](int j) -> float {
                    const int h = c * kHalfs + j - first * 8;
                    const uint32_t u = w[h >> 1];
                    return half_bits_to_float((h & 1) ? (u >> 16) : u);
                };
                out[c] = sigmoid_weighted(weight, channel_dot<KBD>(K, bs_owner));
            }
        }
        sts128_a(slot, __float_as_uint(out[0]), __float_as_uint(out[1]), __float_as_uint(out[2]), 0u);
    }
    __syncwarp();
}

// ---------------------------------------------------------------- ray pool (tail compaction)
// Rays of a 4x8 tile end at different iterations: 21 % of the march iterations of the bench scene run with <= 8 of
// 32 lanes (tools/lane_sim.c).  POOL = true adds the compaction: when a warp is down to kPoolTheta live rays it
// flushes its shading queue, PARKS the survivors (complete ray state, 13..16 quads each) in a per-CTA stack in
// global memory and takes new work; a warp that finds >= 32 parked rays marches them as one dense pass.  A ray
// performs exactly the same operations whoever runs it, so the output stays bit-identical.
//   * the stack and its smem control words {lock, count, queue-exhausted flag} are per CTA: no inter-CTA traffic;
//   * parking is allowed only while the global tile queue still has work, and every warp returns to the work loop
//     after parking, so a parked ray is always picked up (at the latest by the warp that parked it);
//   * the pool memory belongs to (tree, stream) and is shared by consecutive launches, so a launch waits for its
//     predecessor (griddepcontrol.wait) before its first park.
constexpr int kPoolSlots = 128;   // parked rays per CTA
constexpr int kPoolStackQ = 3;    // quads reserved for the table-id stack (12 levels: depth <= 23)
#ifndef VR_POOL_THETA
#define VR_POOL_THETA 12
#endif
constexpr int kPoolTheta = VR_POOL_THETA;
#ifdef VR_POOL_NOPACK   // bisecting aid: previous depth in its own register instead of the top byte of W.pux (one register
                        // more in the march loop: the kernel then spills it); it must then travel with a parked ray
constexpr bool kPoolPack = false;
#else
constexpr bool kPoolPack = true;
#endif

template <int KBD>
struct PoolQuads { static constexpr int n = 3 + kParkQ + kPoolStackQ + BasisQ<KBD>::n; };   // quads per parked ray

template <int KBD>
__host__ __device__ inline size_t pool_bytes_per_cta() { return (size_t)PoolQuads<KBD>::n * kPoolSlots * 16; }

__device__ __forceinline__ void stg128_cg(uint4* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.global.cg.v4.u32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void ldg128_cg(const uint4* p, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ uint32_t lds_volatile(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
// A control word as ONE value for the whole warp (lane 0 reads, everybody gets its copy): the words change under
// the warp's feet (other warps park, pop, flag the end of the tile queue), and lanes that are not converged at
// the read would otherwise see different values and take different sides of warp-level branches.
__device__ __forceinline__ uint32_t lds_uniform(uint32_t addr) {
    uint32_t v = 0u;
    if ((threadIdx.x & 31) == 0) v = lds_volatile(addr);
    return __shfl_sync(0xffffffffu, v, 0);
}
__device__ __forceinline__ void sts_volatile(uint32_t addr, uint32_t v) {
    asm volatile("st.volatile.shared.u32 [%0], %1;" :: "r"(addr), "r"(v) : "memory");
}
// CTA-level spin lock in shared memory, taken by a whole warp (lane 0 spins)
__device__ __forceinline__ void pool_lock(uint32_t lock_addr) {
    if ((threadIdx.x & 31) == 0) {
        uint32_t old;
        do {
            asm volatile("atom.shared.acquire.cta.cas.b32 %0, [%1], 0, 1;" : "=r"(old) : "r"(lock_addr) : "memory");
            if (old) __nanosleep(32);
        } while (old);
    }
    __syncwarp();
}
__device__ __forceinline__ void pool_unlock(uint32_t lock_addr) {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) {
        uint32_t old;
        asm volatile("atom.shared.release.cta.exch.b32 %0, [%1], 0;" : "=r"(old) : "r"(lock_addr) : "memory");
    }
}

// shared memory of one CTA: [ control 16 B | parked ray constants | basis values | shading queues | table-id stacks ]
constexpr uint32_t kCtrlBytes = 16;

// Basis values of this lane's ray (view direction vd) -> shared memory, bs[q][lane].
template <int KBD>
__device__ __forceinline__ void park_basis_q(const LaunchDev& P, const float (&vd)[3], uint32_t bs_warp, int lane) {
    float B[BasisCount<KBD>::n];
    eval_basis<KBD>(P.tree, P.opt, vd, B);
#pragma unroll
    for (int q = 0; q < BasisQ<KBD>::n; ++q) {
        float v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = (4 * q + k < BasisCount<KBD>::n) ? B[4 * q + k] : 0.f;
        sts128_a(bs_warp + ((uint32_t)q * 32u + (uint32_t)lane) * 16u, __float_as_uint(v[0]), __float_as_uint(v[1]),
                 __float_as_uint(v[2]), __float_as_uint(v[3]));
    }
}

// ---------------------------------------------------------------- the kernel
template <int KBD, bool COUNT, int OUT, bool POOL = false>
__global__ void __launch_bounds__(kBlock, kMinBlocks) march_queue_kernel(const __grid_constant__ LaunchDev P) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int KQ = BasisQ<KBD>::n;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // every region but the last has a compile-time size, so all addresses are constants + f(threadIdx): nothing but
    // the stack pointer has to stay in a register across the march loop
    const uint32_t ctrl = smem_u32(smem);   // {lock, parked rays, tile queue exhausted, -}
    const uint32_t smem0 = ctrl + kCtrlBytes;
    const uint32_t levels = (uint32_t)wide_levels(P.tree.max_depth);
    // ray constants of this thread, parked across a drain: rs[quad][thread]
    const uint32_t rs = smem0 + threadIdx.x * 16u;
    const uint32_t bs0 = smem0 + kParkQ * (kBlock * 16u);
    const uint32_t bs_warp = bs0 + (uint32_t)warp * (KQ * 32u * 16u);
    const uint32_t q_warp = bs0 + (kBlock / 32) * (KQ * 32u * 16u) + (uint32_t)warp * (kQSlots * kQSlotBytes);
    // stack[level][thread]; opaque so that the address stays in one register (see march())
    uint32_t stack_a = bs0 + (kBlock / 32) * (KQ * 32u * 16u + kQSlots * kQSlotBytes) + threadIdx.x * 4u;
    asm volatile("mov.u32 %0, %0;" : "+r"(stack_a));
    uint32_t lt_mask;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt_mask));
    const bool pool_on = POOL && P.pool != nullptr;
    // this CTA's parked-ray stack (recomputed where it is used: two registers less in the march loop)
    auto pool_base = [&]() -> uint4* { return reinterpret_cast<uint4*>(P.pool) + (size_t)blockIdx.x * (PoolQuads<KBD>::n * kPoolSlots); };
    if (POOL) {
        if (threadIdx.x == 0) sts128_a(ctrl, 0u, 0u, 0u, 0u);
        __syncthreads();
    }

    pdl_launch_dependents();
    Counts cnt = {0, 0, 0, 0, 0};
    bool dep_done = false;
    // instrumented runs, batches (camera ring written by a copy) and ray launches (ray arrays usually written by the
    // previous kernel of the stream) do not overlap
    if (COUNT || P.cams || OUT == kOutRays) {
        pdl_wait_predecessor();
        dep_done = true;
    }
    const float step = P.opt.step_size, sthr = P.opt.sigma_thresh;
    const uint32_t* __restrict__ wide = P.tree.wide;
    const int wp = P.tree.wide_p;

    for (;;) {
        // ------------------------------------------------ acquire work: 32 parked rays, or the next tile
        // Which pixel a lane works on travels as ONE word, lane slot << 26 | tile index, in the spare word of the
        // parked ray constants (rs quad 2): nothing about the pixel is live across the march loop.
        uint32_t init = 0;
        Ray R;
        R.t = 0.f; R.tmax = -1.f;
        bool hit = false;
        float t = __int_as_float(0x7fc00000), T = 1.f, r = 0.f, g = 0.f, b = 0.f;   // NaN: no ray in this lane
        Walk W = {kPoolPack && POOL ? (104u << 24) : 0u, 0u, 0u, kWideDepthBias + 1};   // "previous leaf" of a fresh ray: depth 1
        bool can_park = false;    // park when 1 <= live rays <= kPoolTheta (warp-uniform)
        bool from_pool = false;
        unsigned long long t_begin = 0;
        unsigned int item = 0;

        if (POOL && pool_on) {
            const uint32_t pc = lds_uniform(ctrl + 4), ex = lds_uniform(ctrl + 8);
            if (pc >= 32u || (ex && pc)) {
                pool_lock(ctrl);
                const uint32_t have = lds_uniform(ctrl + 4);
                const uint32_t take = (have >= 32u || lds_uniform(ctrl + 8)) ? (have < 32u ? have : 32u) : 0u;
                const uint32_t base = have - take;
                if ((uint32_t)lane < take) {
                    const uint4* src = pool_base() + base + lane;   // quad q of slot s at pool[q * kPoolSlots + s]
                    uint32_t a0, a1, a2, a3;
                    ldg128_cg(src, a0, a1, a2, a3);
                    t = __uint_as_float(a0); T = __uint_as_float(a1); r = __uint_as_float(a2); g = __uint_as_float(a3);
                    ldg128_cg(src + kPoolSlots, a0, a1, a2, a3);
                    b = __uint_as_float(a0); W.pux = a1; W.puy = a2; W.puz = a3;   // (the depth rides in W.pux)
                    if (!kPoolPack) { ldg128_cg(src + 2 * kPoolSlots, a0, a1, a2, a3); W.pdepth = (int)a0; }
                    ldg128_cg(src + 3 * kPoolSlots, a0, a1, a2, a3);
                    sts128_a(rs, a0, a1, a2, a3);
                    R.dx = __uint_as_float(a0); R.dy = __uint_as_float(a1); R.dz = __uint_as_float(a2); R.cx = __uint_as_float(a3);
                    ldg128_cg(src + 4 * kPoolSlots, a0, a1, a2, a3);
                    sts128_a(rs + kBlock * 16u, a0, a1, a2, a3);
                    R.cy = __uint_as_float(a0); R.cz = __uint_as_float(a1); R.ix = __uint_as_float(a2); R.iy = __uint_as_float(a3);
                    ldg128_cg(src + 5 * kPoolSlots, a0, a1, a2, a3);
                    sts128_a(rs + 2u * kBlock * 16u, a0, a1, a2, a3);
                    R.iz = __uint_as_float(a0); R.tmax = __uint_as_float(a1); R.ds = __uint_as_float(a2);
                    R.ox = fmaxf(R.ix, 0.f); R.oy = fmaxf(R.iy, 0.f); R.oz = fmaxf(R.iz, 0.f);
                    for (uint32_t j = 0; j < levels; j += 4u) {   // table-id stack
                        ldg128_cg(src + (6u + (j >> 2)) * kPoolSlots, a0, a1, a2, a3);
                        asm volatile("st.shared.u32 [%0], %1;" :: "r"(stack_a + j * (kBlock * 4u)), "r"(a0) : "memory");
                        if (j + 1u < levels) asm volatile("st.shared.u32 [%0], %1;" :: "r"(stack_a + (j + 1u) * (kBlock * 4u)), "r"(a1) : "memory");
                        if (j + 2u < levels) asm volatile("st.shared.u32 [%0], %1;" :: "r"(stack_a + (j + 2u) * (kBlock * 4u)), "r"(a2) : "memory");
                        if (j + 3u < levels) asm volatile("st.shared.u32 [%0], %1;" :: "r"(stack_a + (j + 3u) * (kBlock * 4u)), "r"(a3) : "memory");
                    }
#pragma unroll
                    for (int q = 0; q < KQ; ++q) {
                        ldg128_cg(src + (6 + kPoolStackQ + q) * kPoolSlots, a0, a1, a2, a3);
                        sts128_a(bs_warp + ((uint32_t)q * 32u + (uint32_t)lane) * 16u, a0, a1, a2, a3);
                    }
                    hit = true;
                } else {   // no ray in this lane: the pixel word says so
                    asm volatile("st.shared.u32 [%0], %1;" :: "r"(rs + 2u * kBlock * 16u + 12u), "r"(0xffffffffu) : "memory");
                }
                __syncwarp();
                if (lane == 0 && take) sts_volatile(ctrl + 4, base);
                pool_unlock(ctrl);
                if (take == 0u) continue;     // another warp was faster
                from_pool = true;
                if (!hit) t = __int_as_float(0x7fc00000);
            } else if (ex) {
                break;                        // no tiles left and nothing parked
            }
        }
        if (!from_pool) {
            item = next_item<false>(P, lane);
            if (item == kNoItem) {
                if (POOL && pool_on) {        // tell the CTA, then look at the pool once more
                    if (lane == 0) sts_volatile(ctrl + 8, 1u);
                    __syncwarp();
                    continue;
                }
                break;
            }
            if constexpr (OUT == kOutRays) {   // lane l of item k: ray 32k + l
                const uint32_t ray = item * 32u + (uint32_t)lane;
                float c[3], d[3], tlim;
                if (ray < (uint32_t)P.n_rays && P.tree.N > 0 && load_ray(P, ray, c, d, tlim)) {
                    float vd[3];
                    hit = ray_geometry_world(P.tree, P.opt, d[0], d[1], d[2], c, tlim, R, vd, P.tree.pos_scale);
                    if (hit) park_basis_q<KBD>(P, vd, bs_warp, lane);
                }
            } else {
                int view, tx, ty;
                decode_item<false>(P, item, view, tx, ty);
                const int lx = tx * kTW + (lane % kTW), ly = ty * kTH + (lane / kTW);
                const bool inb = lx < P.w && ly < P.h;
                const CamDev& cam = P.cams ? P.cams[view] : P.cam;
                if (COUNT && P.trace) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_begin));

                const int px = P.x0 + lx, py = P.y0 + frame_row(P, ly);
                float tlim = 1e9f;
                if (P.composite && inb) {  // volrend.cu:92-96,143-146
                    if (!dep_done) { pdl_wait_predecessor(); dep_done = true; }  // reads the previous image
                    const size_t o = ((size_t)view * P.h + ly) * P.w + lx;
                    if (OUT == kOutSurface) {
                        init = surf2Dread<uint32_t>(P.surf, px * 4, py, cudaBoundaryModeZero);
                        if (P.dsurf) tlim = surf2Dread<float>(P.dsurf, px * 4, py, cudaBoundaryModeZero);
                    } else {
                        init = reinterpret_cast<const uint32_t*>(P.rgba8)[o];
                        if (P.depth_in) tlim = P.depth_in[o];
                    }
                }
                if (inb && P.tree.N > 0) {
                    float vd[3];
                    hit = ray_geometry(P.tree, P.opt, cam, px, py, tlim, R, vd, P.tree.pos_scale);
                    if (hit) park_basis_q<KBD>(P, vd, bs_warp, lane);
                }
            }
            if (COUNT && hit) ++cnt.hit;
            if (hit) {  // the drain needs the registers: the ray constants are reloaded after it (hand-made live-range split)
                sts128_a(rs, __float_as_uint(R.dx), __float_as_uint(R.dy), __float_as_uint(R.dz), __float_as_uint(R.cx));
                sts128_a(rs + kBlock * 16u, __float_as_uint(R.cy), __float_as_uint(R.cz), __float_as_uint(R.ix), __float_as_uint(R.iy));
                sts128_a(rs + 2u * kBlock * 16u, __float_as_uint(R.iz), __float_as_uint(R.tmax), __float_as_uint(R.ds), 0u);
            }
            asm volatile("st.shared.u32 [%0], %1;" :: "r"(rs + 2u * kBlock * 16u + 12u), "r"(((uint32_t)lane << 26) | item) : "memory");
            // Ray state.  A finished ray is encoded in t itself: t >= tmax at a normal end, t = +inf after an
            // early stop (rt_core.cuh:176), so no flag has to be carried through the loop.
            t = hit ? R.t : __int_as_float(0x7fc00000);   // NaN: t < tmax is false, and it is not the early-stop marker
            asm volatile("st.shared.u32 [%0], %1;" :: "r"(stack_a), "r"(0u) : "memory");
        }
        if (POOL && pool_on && !P.composite && !lds_uniform(ctrl + 8)) can_park = true;
        uint32_t mine_cur = 0u, mine_next = 0u;   // slots of the draining / the following window that hold this lane's samples
        uint32_t qhead = 0u, qcount = 0u;         // warp-uniform

        const bool want_colour = !P.opt.render_depth;
#ifdef VR_POOL_DEBUG
        uint32_t dbg_iter = 0u, dbg_flushes = 0u;
#endif
        uint32_t alive;
        for (;;) {   // march; left when no ray is alive, or with <= park_theta survivors to park them
        do {
            bool shaded = false;   // this lane produced a sample whose colour has to be evaluated
#ifdef VR_POOL_DEBUG
            ++dbg_iter;
#endif
            uint32_t eidx;
            float weight;
            // (taking 2 or 3 samples per lane between two rounds of votes was measured: +2 % time, profiles/r02_tuning_sweeps.txt)
            if (t < R.tmax) {   // rt_core.cuh:108
                float x, y, z;
                uint32_t ux, uy, uz, w;
                int depth;
                sample_pos(R, t, x, y, z, ux, uy, uz, P.tree.pos_hi);
                find_leaf_wide<COUNT, kTuneHint | kTuneWide | kTuneWideRecs | (kPoolPack && POOL ? kTunePackDepth : 0)>(wide, stack_a, W, ux, uy, uz, w, eidx, depth,
                                                                                                        cnt, 0, wp);
                if (COUNT) { ++cnt.samples; cnt.child_loads += depth; }
                const float dt = cell_delta_t<true, POOL>(R, x, y, z, ux, uy, uz, depth, step, w, P.tree.icube_bias);
                const float sigma = half_bits_to_float(w);
                bool stop = false;
                if (sigma > sthr) {                 // :118
                    const float att = expf_pinned(__fmul_rn(__fmul_rn(-dt, R.ds), sigma));  // :119
                    weight = __fmul_rn(T, __fsub_rn(1.f, att));                               // :120
                    if (COUNT) ++cnt.shaded;
                    if (!want_colour) r = __fmaf_rn(t, weight, r);  // :122-123
                    shaded = want_colour;
                    T = __fmul_rn(T, att);  // :174
                    stop = T < P.opt.stop_thresh;   // :176
                }
                t = stop ? __int_as_float(0x7f800000) : __fadd_rn(t, dt);        // :187, or the early-stop marker
            }
            const uint32_t bal = __ballot_sync(0xffffffffu, shaded);
            if (bal) {
                const uint32_t rel = qcount + (uint32_t)__popc(bal & lt_mask);   // position behind the ring head, < 64
                if (shaded) {
#ifdef VR_POOL_DEBUG
                    sts128_a(q_warp + ((qhead + rel) & (kQSlots - 1)) * kQSlotBytes, eidx, __float_as_uint(weight), (uint32_t)lane, 0x80000000u | dbg_iter);
#else
                    sts128_a(q_warp + ((qhead + rel) & (kQSlots - 1)) * kQSlotBytes, eidx, __float_as_uint(weight), (uint32_t)lane, 0u);
#endif
                    const uint32_t bit = 1u << (rel & 31u);
                    if (rel & 32u) mine_next |= bit; else mine_cur |= bit;
#if VR_QPREFETCH
                    {
                        const unsigned char* rp = rec_addr(P.tree.wrecs, eidx, RecBytes<KBD>::n);
                        asm volatile("prefetch.global.L2 [%0];" :: "l"(rp));
#if VR_QPREFETCH >= 3
                        asm volatile("prefetch.global.L2 [%0];" :: "l"(rp + 32));
                        asm volatile("prefetch.global.L2 [%0];" :: "l"(rp + 64));
#endif
                    }
#endif
                }
                qcount += (uint32_t)__popc(bal);
#ifdef VR_POOL_DEBUG
                if (qcount >= 32u) {
                    __syncwarp();
                    uint32_t i0, i1, i2, i3;
                    lds128_a(q_warp + (qhead + lane) * kQSlotBytes, i0, i1, i2, i3);
                    const uint32_t fresh = __ballot_sync(0xffffffffu, (i3 & 0x80000000u) != 0u);
                    const uint32_t qh_same = __ballot_sync(0xffffffffu, qhead == __shfl_sync(0xffffffffu, qhead, 0));
                    const uint32_t qc_same = __ballot_sync(0xffffffffu, qcount == __shfl_sync(0xffffffffu, qcount, 0));
                    if (fresh != 0xffffffffu && lane == 0)
                        printf("STALE block %d warp %d from_pool %d iter %u flushes %u: qhead %u qcount %u bal %08x fresh %08x qh_same %08x qc_same %08x slot_iter %u\n",
                               blockIdx.x, warp, (int)from_pool, dbg_iter, dbg_flushes, qhead, qcount, bal, fresh, qh_same, qc_same, i3 & 0x7fffffffu);
                }
#endif
                if (qcount >= 32u) {
                    __syncwarp();
                    drain_window<KBD>(q_warp + qhead * kQSlotBytes, 32u, bs_warp, P.tree.wrecs, P.tree.wide_entries, from_pool ? 11 : 1);
                    uint32_t m = mine_cur;
                    while (m) {  // this lane's terms, in sample order (rt_core.cuh:163)
                        const uint32_t sl = (uint32_t)__ffs((int)m) - 1u;
                        m &= m - 1u;
                        uint32_t cr, cg, cb, pad;
                        lds128_a(q_warp + (qhead + sl) * kQSlotBytes, cr, cg, cb, pad);
                        r = __fadd_rn(r, __uint_as_float(cr)); g = __fadd_rn(g, __uint_as_float(cg)); b = __fadd_rn(b, __uint_as_float(cb));
                    }
                    __syncwarp();   // every owner has read its terms before a later enqueue may reuse the window (racecheck)
                    mine_cur = mine_next;
                    mine_next = 0u;
                    qhead ^= 32u;
                    qcount -= 32u;
                    {   // ray constants back into registers
                        uint32_t a0, a1, a2, a3;
                        lds128_a(rs, a0, a1, a2, a3);
                        R.dx = __uint_as_float(a0); R.dy = __uint_as_float(a1); R.dz = __uint_as_float(a2); R.cx = __uint_as_float(a3);
                        lds128_a(rs + kBlock * 16u, a0, a1, a2, a3);
                        R.cy = __uint_as_float(a0); R.cz = __uint_as_float(a1); R.ix = __uint_as_float(a2); R.iy = __uint_as_float(a3);
                        lds128_a(rs + 2u * kBlock * 16u, a0, a1, a2, a3);
                        R.iz = __uint_as_float(a0); R.tmax = __uint_as_float(a1); R.ds = __uint_as_float(a2);
                        R.ox = fmaxf(R.ix, 0.f); R.oy = fmaxf(R.iy, 0.f); R.oz = fmaxf(R.iz, 0.f);
                    }
                }
            }
            alive = __ballot_sync(0xffffffffu, t < R.tmax);
        } while (POOL ? (can_park ? __popc(alive) > kPoolTheta : alive != 0u) : alive != 0u);
            if (!POOL || !alive) break;
            {
                // ---------------------------------------- park the surviving rays (warp-uniform)
                const bool live = (alive >> lane) & 1u;
                if (qcount) {   // their pending colours first: the accumulators travel with the ray
                    __syncwarp();
                    drain_window<KBD>(q_warp + qhead * kQSlotBytes, qcount, bs_warp, P.tree.wrecs, P.tree.wide_entries, from_pool ? 12 : 2);
                    uint32_t m = mine_cur;
                    while (m) {
                        const uint32_t sl = (uint32_t)__ffs((int)m) - 1u;
                        m &= m - 1u;
                        uint32_t cr, cg, cb, pad;
                        lds128_a(q_warp + (qhead + sl) * kQSlotBytes, cr, cg, cb, pad);
                        r = __fadd_rn(r, __uint_as_float(cr)); g = __fadd_rn(g, __uint_as_float(cg)); b = __fadd_rn(b, __uint_as_float(cb));
                    }
                    __syncwarp();
                    mine_cur = 0u; qcount = 0u; qhead = 0u;
#ifdef VR_POOL_DEBUG
                    ++dbg_flushes;
#endif
                }
                const uint32_t n_live = (uint32_t)__popc(alive);
                pool_lock(ctrl);
                const uint32_t have = lds_uniform(ctrl + 4);
                const bool room = have + n_live <= (uint32_t)kPoolSlots;
                if (room) {
                    if (!dep_done) { pdl_wait_predecessor(); dep_done = true; }   // the pool may still belong to the previous launch
                    if (live) {
                        uint4* dst = pool_base() + have + (uint32_t)__popc(alive & lt_mask);
                        uint32_t a0, a1, a2, a3;
                        stg128_cg(dst, __float_as_uint(t), __float_as_uint(T), __float_as_uint(r), __float_as_uint(g));
                        stg128_cg(dst + kPoolSlots, __float_as_uint(b), W.pux, W.puy, W.puz);
                        if (!kPoolPack) stg128_cg(dst + 2 * kPoolSlots, (uint32_t)W.pdepth, 0u, 0u, 0u);
                        lds128_a(rs, a0, a1, a2, a3);
                        stg128_cg(dst + 3 * kPoolSlots, a0, a1, a2, a3);
                        lds128_a(rs + kBlock * 16u, a0, a1, a2, a3);
                        stg128_cg(dst + 4 * kPoolSlots, a0, a1, a2, a3);
                        lds128_a(rs + 2u * kBlock * 16u, a0, a1, a2, a3);
                        stg128_cg(dst + 5 * kPoolSlots, a0, a1, a2, a3);
                        for (uint32_t j = 0; j < levels; j += 4u) {
                            a1 = a2 = a3 = 0u;
                            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(a0) : "r"(stack_a + j * (kBlock * 4u)) : "memory");
                            if (j + 1u < levels) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(a1) : "r"(stack_a + (j + 1u) * (kBlock * 4u)) : "memory");
                            if (j + 2u < levels) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(a2) : "r"(stack_a + (j + 2u) * (kBlock * 4u)) : "memory");
                            if (j + 3u < levels) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(a3) : "r"(stack_a + (j + 3u) * (kBlock * 4u)) : "memory");
                            stg128_cg(dst + (6u + (j >> 2)) * kPoolSlots, a0, a1, a2, a3);
                        }
#pragma unroll
                        for (int q = 0; q < KQ; ++q) {
                            lds128_a(bs_warp + ((uint32_t)q * 32u + (uint32_t)lane) * 16u, a0, a1, a2, a3);
                            stg128_cg(dst + (6 + kPoolStackQ + q) * kPoolSlots, a0, a1, a2, a3);
                        }
                        t = __int_as_float(0x7fc00001);   // NaN with the "parked" payload: no pixel is written for this lane
                    }
                    __threadfence_block();
                    __syncwarp();
                    if (lane == 0) sts_volatile(ctrl + 4, have + n_live);
                    alive = 0u;
                } else {
                    can_park = false;  // pool full: finish this work item the ordinary way
                }
                pool_unlock(ctrl);
                if (room) break;
                {   // the drain above clobbered the ray constants
                    uint32_t a0, a1, a2, a3;
                    lds128_a(rs, a0, a1, a2, a3);
                    R.dx = __uint_as_float(a0); R.dy = __uint_as_float(a1); R.dz = __uint_as_float(a2); R.cx = __uint_as_float(a3);
                    lds128_a(rs + kBlock * 16u, a0, a1, a2, a3);
                    R.cy = __uint_as_float(a0); R.cz = __uint_as_float(a1); R.ix = __uint_as_float(a2); R.iy = __uint_as_float(a3);
                    lds128_a(rs + 2u * kBlock * 16u, a0, a1, a2, a3);
                    R.iz = __uint_as_float(a0); R.tmax = __uint_as_float(a1); R.ds = __uint_as_float(a2);
                    R.ox = fmaxf(R.ix, 0.f); R.oy = fmaxf(R.iy, 0.f); R.oz = fmaxf(R.iz, 0.f);
                }
            }
        }
        const bool stopped = __float_as_uint(t) == 0x7f800000u;
        if (qcount) {  // tile end: the remaining items (all in the window at qhead)
            __syncwarp();
            drain_window<KBD>(q_warp + qhead * kQSlotBytes, qcount, bs_warp, P.tree.wrecs, P.tree.wide_entries, from_pool ? 13 : 3);
            uint32_t m = mine_cur;
            while (m) {
                const uint32_t sl = (uint32_t)__ffs((int)m) - 1u;
                m &= m - 1u;
                uint32_t cr, cg, cb, pad;
                lds128_a(q_warp + (qhead + sl) * kQSlotBytes, cr, cg, cb, pad);
                r = __fadd_rn(r, __uint_as_float(cr)); g = __fadd_rn(g, __uint_as_float(cg)); b = __fadd_rn(b, __uint_as_float(cb));
            }
        }
        __syncwarp();   // every lane is done with the ring and the basis values before the next tile reuses them

        // this lane's pixel: its own tile, or the tile a parked ray came from
        uint32_t packed;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(packed) : "r"(rs + 2u * kBlock * 16u + 12u) : "memory");
        if constexpr (OUT == kOutRays) {   // this lane's ray: 32 * item + lane slot (offscreen compositing only)
            const uint32_t ray = (packed & 0x3ffffffu) * 32u + (packed >> 26);
            if (packed != 0xffffffffu && ray < (uint32_t)P.n_rays) {
                float out[4] = {0.f, 0.f, 0.f, 0.f};
                if (__float_as_uint(t) != 0x7fc00000u) {   // marched (degenerate rays and misses kept the plain NaN)
                    if (P.opt.render_depth) r = g = b = fminf(r * 0.3f, 1.0f);  // :177-179,189-191
                    if (stopped) {  // :181-184
                        const float sc = __frcp_rn(__fsub_rn(1.f, T));
                        out[0] = __fmul_rn(r, sc); out[1] = __fmul_rn(g, sc); out[2] = __fmul_rn(b, sc); out[3] = 1.f;
                    } else {
                        out[0] = r; out[1] = g; out[2] = b;
                        out[3] = P.opt.render_depth ? 1.f : __fsub_rn(1.f, T);
                    }
                } else if (P.opt.render_depth) {
                    out[3] = 1.f;  // rt_core.cuh:90-91
                }
                const float remain = __fmul_rn(__fsub_rn(1.f, out[3]), P.opt.background_brightness);
                P.rgbaf[ray] = make_float4(__fadd_rn(remain, out[0]), __fadd_rn(remain, out[1]), __fadd_rn(remain, out[2]), out[3]);
            }
            __syncwarp();
            continue;
        }
        int view, tx, ty;
        decode_item<false>(P, packed & 0x3ffffffu, view, tx, ty);
        const int lx = tx * kTW + (int)((packed >> 26) % kTW), ly = ty * kTH + (int)((packed >> 26) / kTW);
        hit = __float_as_uint(t) != 0x7fc00000u;   // lanes without a ray kept the plain NaN
        const bool write_px = packed != 0xffffffffu && lx < P.w && ly < P.h && __float_as_uint(t) != 0x7fc00001u;
        if (write_px) {
            const int px = P.x0 + lx, py = P.y0 + frame_row(P, ly);
            float out[4] = {0.f, 0.f, 0.f, 0.f};
            if (hit) {
                if (P.opt.render_depth) r = g = b = fminf(r * 0.3f, 1.0f);  // :177-179,189-191
                if (stopped) {  // :181-184
                    const float sc = __frcp_rn(__fsub_rn(1.f, T));
                    out[0] = __fmul_rn(r, sc); out[1] = __fmul_rn(g, sc); out[2] = __fmul_rn(b, sc); out[3] = 1.f;
                } else {
                    out[0] = r; out[1] = g; out[2] = b;
                    out[3] = P.opt.render_depth ? 1.f : __fsub_rn(1.f, T);
                }
            } else if (P.tree.N > 0 && P.opt.render_depth) {
                out[3] = 1.f;  // rt_core.cuh:90-91
            }
            const float nalpha = __fsub_rn(1.f, out[3]);
            if (!P.composite) {
                const float remain = __fmul_rn(nalpha, P.opt.background_brightness);
                out[0] = __fadd_rn(remain, out[0]); out[1] = __fadd_rn(remain, out[1]); out[2] = __fadd_rn(remain, out[2]);
            } else {
                out[0] += (float)(init & 0xffu) / 255.f * nalpha;
                out[1] += (float)((init >> 8) & 0xffu) / 255.f * nalpha;
                out[2] += (float)((init >> 16) & 0xffu) / 255.f * nalpha;
            }
            const uint32_t q = quantise(out);
            if (!dep_done) { pdl_wait_predecessor(); dep_done = true; }  // first write of this thread
            const size_t o = ((size_t)view * P.h + ly) * P.w + lx;
            if (OUT == kOutSurface) {
                surf2Dwrite(q, P.surf, px * 4, py, cudaBoundaryModeZero);
            } else {
                if (P.rgba8) reinterpret_cast<uint32_t*>(P.rgba8)[o] = q;
            }
            if (P.rgbaf) P.rgbaf[o] = make_float4(out[0], out[1], out[2], out[3]);
        }
        __syncwarp();
        if (COUNT && P.trace && lane == 0 && !from_pool) {
            unsigned long long t_end;
            unsigned int smid;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            P.trace[4 * (size_t)item + 0] = t_begin;
            P.trace[4 * (size_t)item + 1] = t_end;
            P.trace[4 * (size_t)item + 2] = smid;
            P.trace[4 * (size_t)item + 3] = blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5);
        }
    }
    if (!dep_done) pdl_wait_predecessor();
    if (COUNT) flush_counts(cnt, P.counters);
    rearm_queue<false>(P);
}

}  // namespace vrb
