// Persistent pipeline: the wavefront stages (generate / extend / shade) run inside ONE resident kernel, with the path
// pool in registers + shared memory and warp ballots deciding which stage a warp executes next.
//
// It replaces Renderer::render / render_pixel / trace_internal (src/raytrace.rs:172-198, :79-101).  Every lane owns TWO
// camera paths, both as records in shared memory; registers hold the context of the one being traversed (ray, closest
// hit so far, cursor), the other waits to be shaded or holds a fresh ray.  The warp alternates between
//   extend  : while-while traversal of the paths in flight — the 4-wide tree (128-byte nodes, four 256-bit loads, 4-byte
//             sort / stack keys) or, selectable, the binary tree of 32-byte nodes; lanes vote between the inner-node loop
//             and a leaf step;
//   shade   : when enough lanes hold a finished traversal (or an empty slot), those paths are shaded together —
//             scatter / emit / background, terminated paths deposit beta * radiance with 64-bit fixed-point REDs and are
//             regenerated in place from a global camera-path counter (reserved in chunks, one atomic per 256 paths),
//             the media event of the new ray is pre-sampled — and become "ready" again.
// A lane whose traversal finishes simply starts on its other, ready path and keeps traversing, so the extend
// stage runs with (nearly) full warps and the shade stage with (nearly) full warps, without any queue in global memory:
// HBM only sees the accumulation REDs.  Noise textures are evaluated warp-cooperatively (the 56 gradient terms of
// the 7-octave turbulence are spread over the lanes) instead of by one lane while 31 wait.
//
// The kernel's speed hangs on the SM's 32 KB instruction cache (DESIGN.md section 5b): it is instantiated per scene
// FEATURE SET (FEAT: no code for what a scene cannot contain), and everything that adds code to it is an opt-in instance:
// the in-kernel chain phase (CHAIN, RT_PS_CHAIN=1) and the chain queues with their own kernel (CHAINQ, RT_PS_CHAINQ=1), two
// exact but unprofitable ways to advance paths inside "clear" media without a surface search.  tools/sass_footprint.py
// prints the footprint of an instance by source function.
#include <cuda_runtime.h>

#include <algorithm>
#include <map>
#include <cstdio>
#include <cstdlib>

#include "rt_device.cuh"
#include "scene_internal.h"

namespace rtb {

#define PS_DONE RTB_TRAVERSAL_DONE
#define PS_MIN_DESCEND 8   // lanes that must still be descending inner nodes for the inner loop to keep going
#define PS_LEAVE 12        // lanes that must have finished before the warp leaves the traversal loop (to start them on their other path)
// (8 / 12 instead of round 1's 6 / 8: +0.5 % on C4, +1.8 % on C2, +-0 on C3 with the final kernel; gpurun_out/ab_tune2.txt)
#define PS_WORK 28         // lanes with shading / regeneration work pending that trigger a shade phase ...
#define PS_STALL 14        // ... or lanes that cannot traverse at all (both of their paths wait for the shade phase)
// resident blocks per SM the kernel is compiled for: 6 = 80 registers with 32 B of spills.  Measured on C4:
// 5 blocks (94 registers, no spills) -4 %, 7 blocks (72 registers, 132 B of spills, only 96 KB of L1 left) -6 %
#define PS_MIN_BLOCKS 6
#define PS_CHUNK 256u      // camera paths a warp reserves per atomic

// chain phase (paths that hop from event to event inside a clear medium, rt_device.cuh: wf_chain_step)
#define PS_CHAIN_TRIG 24   // parked chain paths in the warp that start a chain phase ...
#define PS_CHAIN_MIN 12    // ... which goes on while at least this many lanes still hold one

// ST_CHAIN: a finished "traversal" whose hit is the pre-sampled event of a clear medium the ray starts inside — the record
// is what ST_DONE holds, but the chain phase advances it without the shade phase and without a surface search
enum { ST_EMPTY = 0, ST_TRAV = 1, ST_DONE = 2, ST_READY = 3, ST_CHAIN = 4 };

// scheduling thresholds (defaults = the PS_* constants; RT_PS_WORK / RT_PS_STALL / RT_PS_LEAVE / RT_PS_DESCEND / RT_PS_CHAIN_TRIG /
// RT_PS_CHAIN_MIN override them for sweeps; RT_PS_CHAIN_TRIG=0 turns the chain phase off)
struct PsTune {
    int work, stall, leave, descend, chain_trig, chain_min;
};

struct PsCounters {
    unsigned long long next_path, total_paths, rays;
};

// ---- chain queues (CHAINQ instances).  A path whose ray starts inside a CLEAR medium and whose next event lies inside it
// too (wf_chain_eligible) LEAVES the persistent kernel: its record goes to the chain queue in global memory, its slot is
// free.  chain_kernel — a small kernel of its own, so that its code does not share the 32 KB instruction cache with this
// one (DESIGN.md section 5b) — hops such paths from event to event (wf_chain_step) until they leave the medium or end, and
// writes the ones that leave to the exit queue, which the NEXT launch of the persistent kernel consumes before it starts
// new camera paths.  One record = PQ_REC words, SoA over the queue: origin, direction, beta, t, pixel, sample, flags, code
// (the pre-sampled event of the ray: what WfSlot.D.x / D.y hold).
enum { PQ_REC = 14 };
struct ChainCounters {
    unsigned int chain_count, chain_taken;  // records pushed by the persistent kernel / reserved by chain_kernel
    unsigned int exit_count, exit_taken;    // records pushed by chain_kernel / reserved by the next persistent launch
    unsigned int chain_dropped, pad;        // pushes that found the chain queue full (the path then stays in the kernel)
};
struct PsChainIO {
    float* chain;  // [PQ_REC][cap]
    float* exitq;  // [PQ_REC][cap]
    ChainCounters* cc;
    unsigned int cap;
};
__device__ __forceinline__ void queue_store(float* q, unsigned int cap, unsigned int i, const WfSlot& s) {
    q[0 * cap + i] = s.A.x, q[1 * cap + i] = s.A.y, q[2 * cap + i] = s.A.z, q[3 * cap + i] = s.B.x, q[4 * cap + i] = s.B.y, q[5 * cap + i] = s.B.z;
    q[6 * cap + i] = s.C.x, q[7 * cap + i] = s.C.y, q[8 * cap + i] = s.C.z, q[9 * cap + i] = s.D.x;
    q[10 * cap + i] = s.A.w, q[11 * cap + i] = s.C.w, q[12 * cap + i] = s.B.w, q[13 * cap + i] = s.D.y;
}
__device__ __forceinline__ void queue_load(const float* q, unsigned int cap, unsigned int i, WfSlot& s) {
    s.A = f4(q[0 * cap + i], q[1 * cap + i], q[2 * cap + i], q[10 * cap + i]);
    s.B = f4(q[3 * cap + i], q[4 * cap + i], q[5 * cap + i], q[12 * cap + i]);
    s.C = f4(q[6 * cap + i], q[7 * cap + i], q[8 * cap + i], q[11 * cap + i]);
    s.D = f4(q[9 * cap + i], q[13 * cap + i], as_float(0xFFFFFFFFu), 0.f);  // origin primitive: none (the ray starts at a medium event)
}

#define PS_VARIANTS 12
#define PS_DEFAULT_LAYOUT 4    // RT_BVH_LAYOUT / RtParams.bvh_layout override
#define PS_DEFAULT_VARIANT 2   // index into kVariants for the 4-wide layout; RT_PS_VARIANT overrides
#define PS_MAX_SMEM (227u * 1024u)
struct PersistState {
    PsCounters* ctr = nullptr;
    std::map<const void*, int> blocks;  // resident grid of each kernel instance launched so far
    PsChainIO io = {nullptr, nullptr, nullptr, 0u};  // chain / exit queues of the CHAINQ instances (allocated at the first such launch)
};

// One camera path = one record of PS_REC words in shared memory, SoA over the block's threads (conflict-free):
//   origin.xyz, direction.xyz, beta.rgb, t, pixel, sample, flags (depth left | origin face << 16), origin primitive, hit
// hit: -1 miss, prim | face << 24 surface, WF_MEDIUM | m medium (as in WfSlot.D.y).  Every lane owns NS records (2 or 3);
// the slot statuses live in one register (4 bits per slot).  Registers hold only the context of the traversal in
// flight (ray, node-test constants, closest hit so far, cursor), so shading a parked path moves nothing around.
enum { R_OX, R_OY, R_OZ, R_DX, R_DY, R_DZ, R_BR, R_BG, R_BB, R_T, R_PIXEL, R_SAMPLE, R_FLAGS, R_ORIGIN, R_HIT, PS_REC };
#define PS_MAX_SLOTS 4
// field `f` of record `slot` of the calling thread; the pool is [NS][PS_REC][NT] floats at the start of shared memory
#define POOL(slot, f) pool[((slot) * PS_REC + (f)) * NT + threadIdx.x]

// (tried: one 4-bit SET of slots per status, slot_find = a bit-field extract and a find-first-set — FLO is a slow-pipe
// instruction: -0.8 % on C4, -2.4 % on C3; gpurun_out/ab_slots.txt)
__device__ __forceinline__ int slot_status(unsigned int stat, int s) { return (int)((stat >> (4 * s)) & 15u); }
__device__ __forceinline__ unsigned int slot_set(unsigned int stat, int s, int st) { return (stat & ~(15u << (4 * s))) | ((unsigned int)st << (4 * s)); }
template <int NS>
__device__ __forceinline__ int slot_find(unsigned int stat, int want) {  // lowest slot with that status, -1 if none
    int found = -1;
#pragma unroll
    for (int s = NS - 1; s >= 0; --s)
        if (slot_status(stat, s) == want) found = s;
    return found;
}

template <int NT>
__device__ __forceinline__ void rec_load(const float* pool, int slot, WfSlot& s) {
    s.A = f4(POOL(slot, R_OX), POOL(slot, R_OY), POOL(slot, R_OZ), POOL(slot, R_PIXEL));
    s.B = f4(POOL(slot, R_DX), POOL(slot, R_DY), POOL(slot, R_DZ), POOL(slot, R_FLAGS));
    s.C = f4(POOL(slot, R_BR), POOL(slot, R_BG), POOL(slot, R_BB), POOL(slot, R_SAMPLE));
    s.D = f4(POOL(slot, R_T), POOL(slot, R_HIT), POOL(slot, R_ORIGIN), 0.f);
}
template <int NT>
__device__ __forceinline__ void rec_store(float* pool, int slot, const WfSlot& s) {
    POOL(slot, R_OX) = s.A.x, POOL(slot, R_OY) = s.A.y, POOL(slot, R_OZ) = s.A.z, POOL(slot, R_PIXEL) = s.A.w;
    POOL(slot, R_DX) = s.B.x, POOL(slot, R_DY) = s.B.y, POOL(slot, R_DZ) = s.B.z, POOL(slot, R_FLAGS) = s.B.w;
    POOL(slot, R_BR) = s.C.x, POOL(slot, R_BG) = s.C.y, POOL(slot, R_BB) = s.C.z, POOL(slot, R_SAMPLE) = s.C.w;
    POOL(slot, R_T) = s.D.x, POOL(slot, R_HIT) = s.D.y, POOL(slot, R_ORIGIN) = s.D.z;
}

// the same for a record in another lane's column `col` (index of its owner within the block): the chain phase hands the
// parked chain records of the warp to its lowest lanes
#define POOLC(slot, f, col) pool[((slot) * PS_REC + (f)) * NT + (col)]
template <int NT>
__device__ __forceinline__ void rec_load_col(const float* pool, int slot, int col, WfSlot& s) {
    s.A = f4(POOLC(slot, R_OX, col), POOLC(slot, R_OY, col), POOLC(slot, R_OZ, col), POOLC(slot, R_PIXEL, col));
    s.B = f4(POOLC(slot, R_DX, col), POOLC(slot, R_DY, col), POOLC(slot, R_DZ, col), POOLC(slot, R_FLAGS, col));
    s.C = f4(POOLC(slot, R_BR, col), POOLC(slot, R_BG, col), POOLC(slot, R_BB, col), POOLC(slot, R_SAMPLE, col));
    s.D = f4(POOLC(slot, R_T, col), POOLC(slot, R_HIT, col), POOLC(slot, R_ORIGIN, col), 0.f);
}
template <int NT>
__device__ __forceinline__ void rec_store_col(float* pool, int slot, int col, const WfSlot& s) {
    POOLC(slot, R_OX, col) = s.A.x, POOLC(slot, R_OY, col) = s.A.y, POOLC(slot, R_OZ, col) = s.A.z;
    POOLC(slot, R_DX, col) = s.B.x, POOLC(slot, R_DY, col) = s.B.y, POOLC(slot, R_DZ, col) = s.B.z, POOLC(slot, R_FLAGS, col) = s.B.w;
    POOLC(slot, R_BR, col) = s.C.x, POOLC(slot, R_BG, col) = s.C.y, POOLC(slot, R_BB, col) = s.C.z;
    POOLC(slot, R_T, col) = s.D.x, POOLC(slot, R_HIT, col) = s.D.y, POOLC(slot, R_ORIGIN, col) = s.D.z;
}

// 128-bit load from a shared-memory address (the scene copy of the SCENE variants)
__device__ __forceinline__ float4 lds4(uint32_t saddr) {
    float4 v;
    asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}

// Perlin::turbulence (textures.rs:76-88, depth 7) of one point, computed by the whole warp: term = (octave, corner),
// 56 terms over 32 lanes, then a butterfly sum.  `p` must be warp-uniform.  Every lane returns the result.
__device__ __forceinline__ float warp_turbulence(const float* __restrict__ vec, const unsigned short* __restrict__ perm, V3 p) {
    const int lane = (int)(threadIdx.x & 31u);
    float acc = 0.0f;
    // two rounds of 32 terms, NOT unrolled: the kernel's speed hangs on its instruction footprint (32 KB instruction cache)
#pragma unroll 1
    for (int term = lane; term < 56; term += 32) {
        const int oct = term >> 3, di = (term >> 2) & 1, dj = (term >> 1) & 1, dk = term & 1;
        const float scale = (float)(1 << oct);
        const float qx = p.x * scale, qy = p.y * scale, qz = p.z * scale;  // exact: the reference doubles p per octave
        const float fx = floorf(qx), fy = floorf(qy), fz = floorf(qz);
        const float u = qx - fx, v = qy - fy, w = qz - fz;
        const int i = (int)fx, j = (int)fy, k = (int)fz;
        const float uu = u * u * (3.0f - 2.0f * u), vv = v * v * (3.0f - 2.0f * v), ww = w * w * (3.0f - 2.0f * w);
        const int idx = perm[(i + di) & 1023] ^ perm[1024 + ((j + dj) & 1023)] ^ perm[2048 + ((k + dk) & 1023)];
        const float4 g = ld4(vec + 4 * idx);  // (through L1: loads that do not allocate there measured -2.5 %)
        const float wx = u - (float)di, wy = v - (float)dj, wz = w - (float)dk;
        const float bi = di ? uu : 1.0f - uu, bj = dj ? vv : 1.0f - vv, bk = dk ? ww : 1.0f - ww;
        acc += (1.0f / scale) * (bi * bj * bk * (wx * g.x + wy * g.y + wz * g.z));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    return fabsf(acc);
}

__global__ void ps_reset_kernel(PsCounters* c, unsigned long long total, ChainCounters* cc) {
    c->next_path = 0, c->total_paths = total, c->rays = 0;
    if (cc) cc->exit_taken = 0u, cc->chain_count = 0u;  // (exit_count: what the previous chain_kernel left)
}
__global__ void chain_reset_kernel(ChainCounters* cc) { cc->chain_taken = 0u, cc->exit_count = 0u; }

// The chain paths of one launch of the persistent kernel, hopped to their end.  Persistent warps: every lane owns one
// record at a time; lanes whose path left the medium (-> exit queue) or ended take the next records of the queue, 32 lanes'
// worth of reservations per atomic.
#define CHAIN_THREADS 256
__global__ void __launch_bounds__(CHAIN_THREADS) chain_kernel(DSceneView S, DRenderParams P, PsChainIO io, unsigned long long* __restrict__ rays_out) {
    const unsigned int lane = threadIdx.x & 31u;
    const unsigned int lt_mask = (1u << lane) - 1u;
    const unsigned int n = min(io.cc->chain_count, io.cap);
    WfSlot s;
    s.A = s.B = s.C = s.D = f4(0.f, 0.f, 0.f, 0.f);
    bool active = false, drained = false;
    unsigned int n_rays = 0u;
    for (;;) {
        // refill the idle lanes
        const unsigned int m_idle = __ballot_sync(0xffffffffu, !active);
        if (!drained && (__popc(m_idle) >= 8 || m_idle == 0xffffffffu)) {  // (one atomic per 8+ records, not per record)
            const unsigned int want = (unsigned int)__popc(m_idle);
            unsigned int base = 0u;
            if (lane == 0) base = atomicAdd(&io.cc->chain_taken, want);
            base = __shfl_sync(0xffffffffu, base, 0);
            const unsigned int have = base < n ? min(want, n - base) : 0u;
            if (have < want) drained = true;
            const unsigned int rank = (unsigned int)__popc(m_idle & lt_mask);
            if (!active && rank < have) queue_load(io.chain, io.cap, base + rank, s), active = true;
        }
        if (__ballot_sync(0xffffffffu, active) == 0u) break;
        int rc = 1;
        if (active) {
            n_rays += 1u;
            rc = wf_chain_step<MEDIA_FAST>(S, P, s);
            if (rc != 1) active = false;
        }
        const unsigned int m_exit = __ballot_sync(0xffffffffu, rc == 2);
        if (m_exit) {
            const int first = __ffs((int)m_exit) - 1;
            unsigned int base = 0u;
            if ((int)lane == first) base = atomicAdd(&io.cc->exit_count, (unsigned int)__popc(m_exit));
            base = __shfl_sync(0xffffffffu, base, first);
            if (rc == 2) queue_store(io.exitq, io.cap, base + (unsigned int)__popc(m_exit & lt_mask), s);  // (never more exits than chain records: fits)
        }
    }
    for (int off = 16; off > 0; off >>= 1) n_rays += __shfl_down_sync(0xffffffffu, n_rays, off);
    if (lane == 0 && n_rays) atomicAdd(rays_out, (unsigned long long)n_rays);
}

// phase statistics of a debug launch (RT_PS_STATS=1): warp-level step counts and the lanes that were useful in them
enum { PSS_SHADE_PHASES, PSS_SHADE_ACT, PSS_SHADE_DONE, PSS_SHADE_ONPARK, PSS_EXT_PHASES, PSS_INNER_ITERS, PSS_INNER_LANES, PSS_LEAF_STEPS,
       PSS_LEAF_LANES, PSS_LEAF_PRIMS, PSS_EXT_ROUNDS, PSS_EXT_TRAV_LANES, PSS_NOISE, PSS_CHAIN_PHASES, PSS_CHAIN_RECORDS, PSS_CHAIN_ITERS, PSS_CHAIN_LANES,
       PSS_CHAIN_PARKED, PSS_COUNT };

// ---------------------------------------------------------------------------------------------------------------
// Chain phase.  The parked chain records of the warp (ST_CHAIN, wherever they live) go to its lowest lanes, which advance
// them event by event (wf_chain_step: two Philox blocks, one in-ball direction, the media intervals — ~200 instructions
// a step instead of a traversal and a share of a shade phase) while at least `min_lanes` are left.
template <int NT, int NS, int MEDIA, bool STATS, class SV>
__device__ __forceinline__ uint2 chain_phase(float* pool, const SV& S, const DRenderParams& P, int min_lanes, unsigned int stat, unsigned int* st_) {
    const unsigned int lane = threadIdx.x & 31u;
    // lane i takes the i-th parked record, slot 0's first
    int src_slot = -1, src_lane = 0, before = 0, n_chain = 0;
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        const unsigned int mk = __ballot_sync(0xffffffffu, slot_status(stat, k) == ST_CHAIN);
        const int nk = __popc(mk);
        if (src_slot < 0 && (int)lane < before + nk) src_slot = k, src_lane = (int)__fns(mk, 0u, (int)lane - before + 1);
        before += nk;
    }
    n_chain = before;
    const bool mine = src_slot >= 0;
    if (!mine) src_slot = 0;
    const int col = (int)(threadIdx.x & ~31u) + src_lane;
    if (STATS && lane == 0) st_[PSS_CHAIN_PHASES] += 1u, st_[PSS_CHAIN_RECORDS] += (unsigned int)(n_chain < 32 ? n_chain : 32), st_[PSS_CHAIN_PARKED] += (unsigned int)n_chain;
    __syncwarp();
    WfSlot s;
    s.A = s.B = s.C = s.D = f4(0.f, 0.f, 0.f, 0.f);
    if (mine) rec_load_col<NT>(pool, src_slot, col, s);
    int state = mine ? 1 : -1;  // 1: still hopping, 2: left the medium (ready for the extend stage), 0: ended
    unsigned int rays = 0u;
    for (;;) {
        const unsigned int m_act = __ballot_sync(0xffffffffu, state == 1);
        if (__popc(m_act) < min_lanes) break;
        if (STATS && lane == 0) st_[PSS_CHAIN_ITERS] += 1u, st_[PSS_CHAIN_LANES] += (unsigned int)__popc(m_act);
        if (state == 1) {
            rays += 1u;
            const int rc = wf_chain_step<MEDIA>(S, P, s);
            state = rc == 1 ? 1 : (rc == 2 ? 2 : 0);
        }
    }
    if (mine && state != 0) rec_store_col<NT>(pool, src_slot, col, s);
    const unsigned int bit = 1u << src_lane;
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        const unsigned int ready = __reduce_or_sync(0xffffffffu, (mine && state == 2 && src_slot == k) ? bit : 0u);
        const unsigned int ended = __reduce_or_sync(0xffffffffu, (mine && state == 0 && src_slot == k) ? bit : 0u);
        if ((ready >> lane) & 1u) stat = slot_set(stat, k, ST_READY);
        if ((ended >> lane) & 1u) stat = slot_set(stat, k, ST_EMPTY);
    }
    __syncwarp();
    return make_uint2(stat, rays);
}

// WIDE: walk the 4-wide tree (DNode4) with 4-byte stack keys, the first SD stack levels in shared memory (the rest, if a
// ray ever needs them, in local memory); !WIDE: the binary 32-byte-node tree with (link, distance) entries in local memory.
// NT threads per block.  SCENE bit 0: the block keeps a copy of the DNode4 array in shared memory, bit 1: of the
// primitives — ONE large block per SM then shares a single copy, and the L1 that is left holds only what is not copied.
// Dynamic shared memory: [pool NS x PS_REC x NT floats][stack SD x NT keys][nodes4][prims].
#define PS_SCENE_NODES 1
#define PS_SCENE_PRIMS 2
// MOM (the moments family, persist_moments_kernel; IO = PsMomentsIO): every deposit also adds moment2_fixed of its
// fixed-point sample to io.moment2, and path numbers run over the io.n_list pixels of io.plist (ascending pixel ids;
// nullptr: pixel i is i).  The extra inputs ride in the type of `io` rather than in parameters of their own: one more
// parameter, even unused, changes the instruction schedule of existing instances (DESIGN.md section 5d).
struct PsMomentsIO : PsChainIO {
    AccumFx* moment2;
    const uint32_t* plist;
    unsigned int n_list;
};
template <bool STATS, bool WIDE, int SD, int NT, int SCENE, int MEDIA, int NS, bool CHAIN, uint32_t FEAT, bool CHAINQ, bool MOM = false, class IO = PsChainIO>
__device__ __forceinline__ void persist_body(const DSceneView& S_, const DCamera& cam, const DRenderParams& P, PsCounters* __restrict__ ctr,
                                             AccumFx* __restrict__ accum, unsigned long long* __restrict__ rays_out, unsigned int chunk_size,
                                             unsigned long long* __restrict__ stats, const PsTune& tune, const IO& io) {
    const SceneViewF<FEAT>& S = static_cast<const SceneViewF<FEAT>&>(S_);  // same record; SV::feat = what the scene can contain (rt_types.h)
    unsigned int st_[PSS_COUNT];
    if (STATS)
        for (int k = 0; k < PSS_COUNT; ++k) st_[k] = 0u;
#define PS_STAT(k, v)                              \
    if (STATS) {                                   \
        const unsigned int v_ = (unsigned int)(v); \
        if (lane == 0) st_[k] += v_;               \
    }
    extern __shared__ float4 smem_raw[];
    float* const pool = reinterpret_cast<float*>(smem_raw);
    uint32_t* const sstack = reinterpret_cast<uint32_t*>(pool + NS * PS_REC * NT);  // [SD][NT], conflict-free
    uint32_t nodes_saddr = 0u, prims_saddr = 0u;
    if constexpr (SCENE != 0) {
        float4* dst = reinterpret_cast<float4*>(sstack + SD * NT);
        if (SCENE & PS_SCENE_NODES) {
            const float4* src = reinterpret_cast<const float4*>(S.nodes4);
            const int n16 = S.n_nodes4 * (int)(sizeof(DNode4) / 16);
            for (int i = threadIdx.x; i < n16; i += NT) dst[i] = __ldg(src + i);
            nodes_saddr = (uint32_t)__cvta_generic_to_shared(dst);
            dst += n16;
        }
        if (SCENE & PS_SCENE_PRIMS) {
            const float4* src = reinterpret_cast<const float4*>(S.prims);
            const int n16 = S.n_prims * (int)(sizeof(DPrim) / 16);
            for (int i = threadIdx.x; i < n16; i += NT) dst[i] = __ldg(src + i);
            prims_saddr = (uint32_t)__cvta_generic_to_shared(dst);
        }
        __syncthreads();
    }
    const unsigned int lane = threadIdx.x & 31u;
    const unsigned int lt_mask = (1u << lane) - 1u;
    constexpr int DONE = WIDE ? (int)RTB_LINK4_DONE : PS_DONE;
    const int root_link = S.n_prims > 0 ? (WIDE ? 0 : (int)as_uint(ld4(S.nodes).w)) : DONE;
    const unsigned long long total = ctr->total_paths;
    unsigned int npix = (unsigned int)P.width * (unsigned int)P.height;  // pixels the path numbers run over
    if constexpr (MOM) npix = io.n_list;

    unsigned int stat = 0u;  // every slot ST_EMPTY
    // context of the traversal in flight (tslot < 0: none)
    int tslot = -1;
    Ray r;
    r.o = r.d = v3(0.f, 0.f, 0.f);
    NodeRay nr;
    nr.inv = nr.noi = v3(0.f, 0.f, 0.f), nr.pad = 0.f;
    float t_best = 0.f;
    int hit = -1, origin_prim = -1, origin_face = 0, cur = DONE, sp = 0;
    StackEntry stack[WIDE ? 1 : RTB_BVH_STACK];  // binary tree: (node link, entry distance of its box), see stack_pop
    uint32_t lstack[WIDE ? RTB_WIDE_STACK : 1];  // 4-wide tree: the keys above the shared-memory levels
    // (tried: the top of the stack mirrored in a register so that a pop does not wait for its local-memory load — one register
    // more, 12 B more spills, -2 ... -3 % on C2 - C4; gpurun_out/ab_stacktop.txt)
    auto push4 = [&](uint32_t k) {
        if (SD > 0 && sp < SD) sstack[sp * NT + threadIdx.x] = k;
        else lstack[sp - SD] = k;
        sp += 1;
    };
    auto pop4 = [&]() -> int {
        const uint32_t limit = key_limit(t_best, nr.pad);
        while (sp > 0) {
            sp -= 1;
            const uint32_t k = (SD > 0 && sp < SD) ? sstack[sp * NT + threadIdx.x] : lstack[sp - SD];
            if (k <= limit) return (int)(k & 0xFFFFu);
        }
        return DONE;
    };
    // warp-uniform reservation of camera-path numbers
    unsigned long long chunk_next = 0, chunk_end = 0;
    uint32_t chunk_pixel = 0, chunk_sample = 0;  // (pixel, sample) of path chunk_next
    bool exhausted = false;
    bool exits_done = !CHAINQ;  // CHAINQ: the exit queue of the previous launch is served before new camera paths
    unsigned int n_rays = 0;
    // (scenes that need the general media sampler keep to the shade phase: with the out-of-line sampler inside it the chain
    // phase would cost that kernel instance 480 B more spills)
    const bool chain_on = CHAIN && MEDIA != MEDIA_GENERAL && S.clear_media != 0u && tune.chain_trig > 0 && !(MEDIA == MEDIA_ANY && S.media_general);  // warp-uniform

    for (;;) {
        // ---- (1) an idle lane starts traversing one of its ready paths
        if (tslot < 0) {
            const int sl = slot_find<NS>(stat, ST_READY);
            if (sl >= 0) {
                r.o = v3(POOL(sl, R_OX), POOL(sl, R_OY), POOL(sl, R_OZ)), r.d = v3(POOL(sl, R_DX), POOL(sl, R_DY), POOL(sl, R_DZ));
                t_best = POOL(sl, R_T), hit = __float_as_int(POOL(sl, R_HIT)), origin_prim = __float_as_int(POOL(sl, R_ORIGIN));
                origin_face = (int)((__float_as_uint(POOL(sl, R_FLAGS)) >> WF_FACE_SHIFT) & 7u);
                nr = node_ray(r);
                cur = root_link, sp = 0;
                tslot = sl;
                stat = slot_set(stat, sl, ST_TRAV);
            }
        }
        const bool trav = tslot >= 0;
        const int s_done = slot_find<NS>(stat, ST_DONE);
        const int s_work = s_done >= 0 ? s_done : (exhausted ? -1 : slot_find<NS>(stat, ST_EMPTY));
        const unsigned int m_trav = __ballot_sync(0xffffffffu, trav);
        const unsigned int m_work = __ballot_sync(0xffffffffu, s_work >= 0);
        int n_chain = 0;
        if (CHAIN && chain_on) {
#pragma unroll
            for (int k = 0; k < NS; ++k) n_chain += __popc(__ballot_sync(0xffffffffu, slot_status(stat, k) == ST_CHAIN));
        }
        if ((m_trav | m_work) == 0u && n_chain == 0) break;

        if (CHAIN && MEDIA != MEDIA_GENERAL && n_chain > 0 && (n_chain >= tune.chain_trig || (m_trav | m_work) == 0u)) {
            // The registers of the traversal in flight must not stay live across this phase (80 registers: they would be
            // spilled all over the traversal loop).  Ray, origin primitive and face are in the path's record anyway; the
            // closest hit so far goes there too (what the record holds at the end of the traversal, only earlier), and the
            // context is read back — node_ray recomputed — afterwards.  Only the cursor and the stack depth stay in registers.
            const int sl = tslot >= 0 ? tslot : 0;
            if (tslot >= 0) POOL(sl, R_T) = t_best, POOL(sl, R_HIT) = __int_as_float(hit);
            const uint2 res = chain_phase<NT, NS, MEDIA == MEDIA_GENERAL ? MEDIA_FAST : MEDIA, STATS>(pool, S, P, (m_trav | m_work) == 0u ? 1 : tune.chain_min, stat, STATS ? st_ : nullptr);
            stat = res.x, n_rays += res.y;
            r.o = v3(POOL(sl, R_OX), POOL(sl, R_OY), POOL(sl, R_OZ)), r.d = v3(POOL(sl, R_DX), POOL(sl, R_DY), POOL(sl, R_DZ));
            t_best = POOL(sl, R_T), hit = __float_as_int(POOL(sl, R_HIT)), origin_prim = __float_as_int(POOL(sl, R_ORIGIN));
            origin_face = (int)((__float_as_uint(POOL(sl, R_FLAGS)) >> WF_FACE_SHIFT) & 7u);
            nr = node_ray(r);
            continue;
        }

        if (m_work && (m_trav == 0u || __popc(m_work) >= tune.work || __popc(m_work & ~m_trav) >= tune.stall)) {
            // ================================================================ shade / regenerate phase
            const bool act = s_work >= 0;
            const bool shade = s_done >= 0;
            PS_STAT(PSS_SHADE_PHASES, 1)
            PS_STAT(PSS_SHADE_ACT, __popc(m_work))
            PS_STAT(PSS_SHADE_ONPARK, __popc(m_work & m_trav))
            PS_STAT(PSS_SHADE_DONE, __popc(__ballot_sync(0xffffffffu, shade)))
            bool alive = false;
            V3 radiance = v3(0.f, 0.f, 0.f);
            NoiseReq req;
            req.tex = -1, req.p = v3(0.f, 0.f, 0.f);
            int segment_next = 0;
            uint32_t pixel_out = 0u;
            WfSlot s;
            if (shade) {
                n_rays += 1u;
                rec_load<NT>(pool, s_work, s);
                pixel_out = __float_as_uint(s.A.w);
                alive = wf_shade_core(S, P, s, radiance, &req, segment_next);
            }
            // noise textures: one point at a time, all lanes on its 56 gradient terms
            {
                unsigned int m_noise = __ballot_sync(0xffffffffu, req.tex >= 0);
#ifdef RTB_AB_NO_NOISE  // timing A/B only (build flavor "nonoise"): how much of the kernel's time is the FOOTPRINT of this code (instruction cache)
                m_noise = 0u;
#endif
                while (m_noise) {
                    PS_STAT(PSS_NOISE, 1)
                    const int src = __ffs((int)m_noise) - 1;
                    m_noise &= m_noise - 1u;
                    const int tex = __shfl_sync(0xffffffffu, req.tex, src);
                    V3 q;
                    q.x = __shfl_sync(0xffffffffu, req.p.x, src), q.y = __shfl_sync(0xffffffffu, req.p.y, src), q.z = __shfl_sync(0xffffffffu, req.p.z, src);
                    const DTexture& T = S.texs[tex];
                    const float* vec = S.perlin_vec + (size_t)T.a * RTB_PERLIN_POINTS * 4;
                    const unsigned short* perm = S.perlin_perm + (size_t)T.a * RTB_PERLIN_POINTS * 3;
                    const float turb = warp_turbulence(vec, perm, T.scale * q);
                    if ((int)lane == src) {
                        const float g = noise_value(T, q, turb);
                        if (alive) s.C.x *= g, s.C.y *= g, s.C.z *= g;
                        else radiance = g * radiance;
                    }
                }
            }
            if (shade && !alive) {  // the path ended: beta * (emission | background | 0) -> its pixel
                AccumFx* dst = accum + 3 * (size_t)pixel_out;  // 64-bit integer REDs: order-independent sums
#ifdef RTB_AB_FLOAT_RED  // timing A/B only (build flavor "floatred"): round 1's 32-bit float REDs into the same slots; the image is garbage
                if (radiance.x != 0.f) atomicAdd(reinterpret_cast<float*>(dst + 0), radiance.x);
                if (radiance.y != 0.f) atomicAdd(reinterpret_cast<float*>(dst + 1), radiance.y);
                if (radiance.z != 0.f) atomicAdd(reinterpret_cast<float*>(dst + 2), radiance.z);
#else
                if constexpr (MOM) {  // the same sums (a zero sample adds nothing to either) and the squares of the samples
                    AccumFx* dst2 = io.moment2 + 3 * (size_t)pixel_out;
                    const AccumFx q0 = radiance_fixed(radiance.x), q1 = radiance_fixed(radiance.y), q2 = radiance_fixed(radiance.z);
                    if (q0) atomicAdd(dst + 0, q0), atomicAdd(dst2 + 0, moment2_fixed(q0));
                    if (q1) atomicAdd(dst + 1, q1), atomicAdd(dst2 + 1, moment2_fixed(q1));
                    if (q2) atomicAdd(dst + 2, q2), atomicAdd(dst2 + 2, moment2_fixed(q2));
                } else {
                    if (radiance.x != 0.f) atomicAdd(dst + 0, radiance_fixed(radiance.x));
                    if (radiance.y != 0.f) atomicAdd(dst + 1, radiance_fixed(radiance.y));
                    if (radiance.z != 0.f) atomicAdd(dst + 2, radiance_fixed(radiance.z));
                }
#endif
            }
            // regenerate: the next camera paths of the job, handed out in reservation order
            bool need = act && !alive;
            bool from_exit = false;
            unsigned int m_need = __ballot_sync(0xffffffffu, need);
            if (CHAINQ && !exits_done && m_need) {  // paths that chain_kernel took out of a clear medium after the previous launch
                const unsigned int n_exit = min(io.cc->exit_count, io.cap);
                const unsigned int want = (unsigned int)__popc(m_need);
                unsigned int base = 0u;
                if (lane == 0) base = atomicAdd(&io.cc->exit_taken, want);
                base = __shfl_sync(0xffffffffu, base, 0);
                const unsigned int have = base < n_exit ? min(want, n_exit - base) : 0u;
                if (have < want) exits_done = true;
                if (need && (unsigned int)__popc(m_need & lt_mask) < have) {
                    queue_load(io.exitq, io.cap, base + (unsigned int)__popc(m_need & lt_mask), s);  // ray + its pre-sampled event: ready as it is
                    alive = true, need = false, from_exit = true;
                }
                m_need = __ballot_sync(0xffffffffu, need);
            }
            while (m_need) {
                const unsigned int avail = (unsigned int)(chunk_end - chunk_next);
                if (avail == 0u) {
                    if (exhausted) break;
                    unsigned long long base = 0;
                    // (tried: guided self-scheduling, reservations that shrink towards the end of the launch: +2 % on jobs of 2 - 5 ms,
                    // -1.3 % on C4 through the code it adds here; gpurun_out/ab_c1.txt, bench_r2s3.json)
                    const unsigned int cs = chunk_size;
                    if (lane == 0) base = atomicAdd(&ctr->next_path, (unsigned long long)cs);
                    base = __shfl_sync(0xffffffffu, base, 0);
                    chunk_next = base < total ? base : total;
                    chunk_end = base + cs < total ? base + cs : total;
                    if (chunk_next == chunk_end) {
                        exhausted = true;
                        break;
                    }
                    {  // (pixel, sample) of path chunk_next < 2^33: quotient through f64 (exact to +-1, then corrected) instead of the
                       // 64-bit integer division routine — ~90 instructions that the instruction cache would carry for a rare step
                        uint32_t q = (uint32_t)__double2ll_rz((double)(long long)chunk_next * P.inv_npix);
                        long long rem = (long long)chunk_next - (long long)q * (long long)npix;
                        if (rem < 0) q -= 1u, rem += npix;
                        if (rem >= (long long)npix) q += 1u, rem -= npix;
                        chunk_pixel = (uint32_t)rem, chunk_sample = (uint32_t)P.sample_begin + q;
                    }
                    continue;
                }
                const unsigned int want = (unsigned int)__popc(m_need);
                const unsigned int take = want < avail ? want : avail;
                const unsigned int rank = (unsigned int)__popc(m_need & lt_mask);
                if (need && rank < take) {
                    uint32_t pixel = chunk_pixel + rank, sample = chunk_sample;
                    while (pixel >= npix) pixel -= npix, sample += 1u;
                    if constexpr (MOM) {
                        if (io.plist) pixel = __ldg(io.plist + pixel);
                    }
                    wf_init_camera<FEAT>(cam, P, pixel, sample, s);
                    segment_next = 0;
                    alive = true, need = false;
                }
                chunk_next += take;
                chunk_pixel += take;
                while (chunk_pixel >= npix) chunk_pixel -= npix, chunk_sample += 1u;
                m_need = __ballot_sync(0xffffffffu, need);
            }
            // survivors and fresh camera paths alike: media event of the new ray, then "ready"
            if constexpr (!CHAINQ) {
                // survivors and fresh camera paths alike: media event of the new ray, then "ready"
                if (act) {
                    if (alive) {
                        const int code_shaded = __float_as_int(s.D.y);  // the hit this path was shaded at (wf_shade_core leaves it; a fresh camera path: 0)
                        wf_presample_media<MEDIA>(S, P, s, segment_next);
                        rec_store<NT>(pool, s_work, s);
                        // a medium event of a clear medium followed by another one: the path hops on in the chain phase
                        stat = slot_set(stat, s_work, (CHAIN && chain_on && wf_chain_eligible(S, code_shaded, s)) ? ST_CHAIN : ST_READY);
                    } else {
                        stat = slot_set(stat, s_work, ST_EMPTY);
                    }
                }
            } else {
                // the same, except that a path which can hop on without a surface search (a medium event of a clear medium followed
                // by another one) leaves the kernel for chain_kernel: its record goes to the chain queue, its slot is free
                bool eligible = false;
                if (act && alive && !from_exit) {  // (a path from the exit queue brings its pre-sampled event along)
                    const int code_shaded = __float_as_int(s.D.y);
                    wf_presample_media<MEDIA>(S, P, s, segment_next);
                    eligible = wf_chain_eligible(S, code_shaded, s);
                }
                const unsigned int m_el = __ballot_sync(0xffffffffu, eligible);
                if (m_el) {
                    const int first = __ffs((int)m_el) - 1;
                    unsigned int base = 0u;
                    if ((int)lane == first) base = atomicAdd(&io.cc->chain_count, (unsigned int)__popc(m_el));
                    base = __shfl_sync(0xffffffffu, base, first);
                    const unsigned int idx = base + (unsigned int)__popc(m_el & lt_mask);
                    if (eligible) {
                        if (idx < io.cap) queue_store(io.chain, io.cap, idx, s), alive = false;
                        else atomicAdd(&io.cc->chain_dropped, 1u);  // queue full: the path stays here, as any other
                    }
                }
                if (act) {
                    if (alive) {
                        rec_store<NT>(pool, s_work, s);
                        stat = slot_set(stat, s_work, ST_READY);
                    } else {
                        stat = slot_set(stat, s_work, ST_EMPTY);
                    }
                }
            }
            continue;
        }

        // ==================================================================== extend phase
        bool has = trav;
        PS_STAT(PSS_EXT_PHASES, 1)
        for (;;) {
            PS_STAT(PSS_EXT_ROUNDS, 1)
            PS_STAT(PSS_EXT_TRAV_LANES, __popc(__ballot_sync(0xffffffffu, has)))
            // (a) inner nodes: lanes leave the loop when they reach a leaf or run out of nodes
            while (has && (WIDE ? (cur & (int)RTB_LINK4_LEAF) == 0 : cur >= 0)) {
                if (STATS) {
                    const unsigned int am = __activemask();
                    if ((int)lane == __ffs((int)am) - 1) st_[PSS_INNER_ITERS] += 1u, st_[PSS_INNER_LANES] += (unsigned int)__popc(am);
                }
                if constexpr (WIDE) {
                    uint32_t k0, k1, k2, k3;
                    Node4Regs n4;
                    if constexpr ((SCENE & PS_SCENE_NODES) != 0) {
                        const uint32_t a = nodes_saddr + (uint32_t)cur * (uint32_t)sizeof(DNode4);
                        n4.c0 = lds4(a), n4.c1 = lds4(a + 16), n4.c2 = lds4(a + 32), n4.c3 = lds4(a + 48);
                        n4.lz = lds4(a + 64), n4.hz = lds4(a + 80), n4.lk = lds4(a + 96);
                    } else {
                        n4 = node4_fetch(S.nodes4, (uint32_t)cur);
                    }
                    node4_sorted_keys(n4, nr, RTB_T_MIN, t_best, k0, k1, k2, k3);
                    if (k0 == RTB_KEY_MISS) {
                        cur = pop4();
                    } else {
                        if (k3 != RTB_KEY_MISS) push4(k3);
                        if (k2 != RTB_KEY_MISS) push4(k2);
                        if (k1 != RTB_KEY_MISS) push4(k1);
                        cur = (int)(k0 & 0xFFFFu);
                    }
                } else {
                    const char* base = reinterpret_cast<const char*>(S.nodes + cur);
                    const F8 ln = ld8(base), rn = ld8(base + 32);
                    const float4 l0 = ln.lo, l1 = ln.hi, r0 = rn.lo, r1 = rn.hi;
                    float tl, tr;
                    bool hl = slab_node(l0, l1, nr, RTB_T_MIN, t_best, tl);
                    bool hr = slab_node(r0, r1, nr, RTB_T_MIN, t_best, tr);
                    int ll = (int)as_uint(l0.w), lr = (int)as_uint(r0.w);
                    if (hl && hr) {
                        bool left_first = tl <= tr;
                        stack[sp].node = left_first ? lr : ll, stack[sp].tn = left_first ? tr : tl;
                        sp += 1;
                        cur = left_first ? ll : lr;
                    } else if (hl) {
                        cur = ll;
                    } else if (hr) {
                        cur = lr;
                    } else {
                        cur = stack_pop(stack, sp, t_best, nr.pad);
                    }
                }
                if (__popc(__activemask()) < tune.descend) break;
            }
            __syncwarp();
            // (b) one leaf per lane: every primitive of it
            const bool at_leaf = has && cur != DONE && (WIDE ? (cur & (int)RTB_LINK4_LEAF) != 0 : cur < 0);
            if (STATS) {
                const unsigned int lm = __ballot_sync(0xffffffffu, at_leaf);
                PS_STAT(PSS_LEAF_STEPS, lm != 0u)
                PS_STAT(PSS_LEAF_LANES, __popc(lm))
            }
            if (at_leaf) {
                int first, count;
                if (WIDE) {
                    first = cur & 0x7FFF, count = 1;
                } else {
                    const int v = ~cur;
                    first = v & 0xFFFFFF, count = v >> 24;
                }
                if (STATS) st_[PSS_LEAF_PRIMS] += (unsigned int)count;
                for (int i = first; i < first + count; ++i) {
                    PrimRec q;
                    if constexpr ((SCENE & PS_SCENE_PRIMS) != 0) {
                        const uint32_t a = prims_saddr + (uint32_t)i * (uint32_t)sizeof(DPrim);
                        q = prim_from(lds4(a), lds4(a + 16));
                    } else {
                        q = load_prim(S.prims + i);
                    }
                    if ((FEAT & F_MOVING) && (q.meta & PRIM_MOVING)) apply_motion(S, q, time_of_flags(__float_as_uint(POOL(tslot, R_FLAGS))));  // EXTENSION
                    float t;
                    int face;
                    if (hit_prim(S, q, r, RTB_T_MIN, t_best, i == origin_prim, origin_face, t, face))
                        t_best = t, hit = i | (face << 24);  // closer than the pre-sampled medium event, which it replaces
                }
                if constexpr (WIDE) cur = pop4();
                else cur = stack_pop(stack, sp, t_best, nr.pad);
            }
            __syncwarp();
            if (has && cur == DONE) {  // traversal finished: the hit record goes back to the path's slot
                has = false;
                POOL(tslot, R_T) = t_best;
                POOL(tslot, R_HIT) = __int_as_float(hit);
                stat = slot_set(stat, tslot, ST_DONE);
                tslot = -1;
            }
            const unsigned int busy = __ballot_sync(0xffffffffu, has);
            if (busy == 0u) break;
            if (__popc(m_trav & ~busy) >= tune.leave) break;
        }
    }

    for (int off = 16; off > 0; off >>= 1) n_rays += __shfl_down_sync(0xffffffffu, n_rays, off);
    if (lane == 0 && n_rays) atomicAdd(rays_out, (unsigned long long)n_rays);
    if (STATS) {  // per-lane counters (inner iterations are counted by the first active lane, leaf primitives by every lane)
        for (int k = 0; k < PSS_COUNT; ++k) {
            unsigned int v = st_[k];
            for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
            if (lane == 0 && v) atomicAdd(stats + k, (unsigned long long)v);
        }
    }
#undef PS_STAT
}

template <bool STATS, bool WIDE, int SD, int NT, int SCENE, int MEDIA, int NS, bool CHAIN, uint32_t FEAT, bool CHAINQ = false>
__global__ void __launch_bounds__(NT, (STATS || NT > 128) ? 1 : PS_MIN_BLOCKS) persist_kernel(DSceneView S, DCamera cam, DRenderParams P, PsCounters* __restrict__ ctr,
                                                             AccumFx* __restrict__ accum, unsigned long long* __restrict__ rays_out,
                                                             unsigned int chunk_size, unsigned long long* __restrict__ stats, PsTune tune, PsChainIO io) {
    persist_body<STATS, WIDE, SD, NT, SCENE, MEDIA, NS, CHAIN, FEAT, CHAINQ>(S, cam, P, ctr, accum, rays_out, chunk_size, stats, tune, io);
}

// EXTENSION: the moments family (rt_render_moments_fixed_device, rt_render_adaptive) — the product placement (two slots per
// lane, no scene copy, no chain phase / queues / statistics) with second moments and a pixel list.  A kernel of its own, so
// that the instances above stay as they were, instruction for instruction (DESIGN.md section 5b).
template <bool WIDE, int NT, int MEDIA, uint32_t FEAT>
__global__ void __launch_bounds__(NT, NT > 128 ? 1 : PS_MIN_BLOCKS) persist_moments_kernel(DSceneView S, DCamera cam, DRenderParams P, PsCounters* __restrict__ ctr,
                                                                      AccumFx* __restrict__ accum, AccumFx* __restrict__ moment2,
                                                                      const uint32_t* __restrict__ plist, unsigned int n_list,
                                                                      unsigned long long* __restrict__ rays_out, unsigned int chunk_size, PsTune tune) {
    PsMomentsIO io;
    io.chain = io.exitq = nullptr, io.cc = nullptr, io.cap = 0u;
    io.moment2 = moment2, io.plist = plist, io.n_list = n_list;
    persist_body<false, WIDE, 0, NT, 0, MEDIA, 2, false, FEAT, false, true>(S, cam, P, ctr, accum, rays_out, chunk_size, nullptr, tune, io);
}

// ---------------------------------------------------------------------------------------------------------------
void free_persist(RtScene* s) {
    if (!s->ps) return;
    rtb::cache_free(s->ps->ctr, sizeof(PsCounters));
    if (s->ps->io.cc) {
        rtb::cache_free(s->ps->io.chain, (size_t)PQ_REC * s->ps->io.cap * sizeof(float));
        rtb::cache_free(s->ps->io.exitq, (size_t)PQ_REC * s->ps->io.cap * sizeof(float));
        rtb::cache_free(s->ps->io.cc, sizeof(ChainCounters));
    }
    delete s->ps;
    s->ps = nullptr;
}

bool persist_supports(const RtScene* s, const RtParams* p) { return p->max_depth <= WF_DEPTH_MASK && s->flat.prims.size() < (1u << 24); }

namespace {

typedef void (*PersistFn)(DSceneView, DCamera, DRenderParams, PsCounters*, AccumFx*, unsigned long long*, unsigned int, unsigned long long*, PsTune, PsChainIO);
struct Variant {
    int layout, smem_stack, threads, scene, slots;
    PersistFn fn, fn_general, fn_stats;  // fn: scenes with <= 4 single-primitive media; fn_general: any media (rt_device.cuh: sample_media)
    const char* name;
};
// [fast-media instance, general-media instance, stats instance (decides at run time)]
#define PS_INSTANCE(wide, sd, nt, scene, ns, chain) \
    persist_kernel<false, wide, sd, nt, scene, MEDIA_FAST, ns, chain, F_ALL>, persist_kernel<false, wide, sd, nt, scene, MEDIA_GENERAL, ns, false, F_ALL>, \
        persist_kernel<true, wide, sd, nt, scene, MEDIA_ANY, ns, chain, F_ALL>
// The kernel instances the library carries.  Measured on C4 (profiles/r2_ab_variants.txt): [1] is +1.6 % over [0], [2]
// (one 768-thread block per SM instead of six 128-thread blocks: 5 KB more L1, one pool) another +1.8 %.
// RTB_PS_EXPERIMENTS adds the rejected placements (stack levels or scene copies in shared memory: -2 ... -9 %, the L1
// they take away costs more than the shared-memory latency wins) so that the A/B stays reproducible
// (tools/experiments/build_experiments.sh); the product build does not carry them.
const Variant kVariants[] = {
    {2, 0, 128, 0, 2, PS_INSTANCE(false, 0, 128, 0, 2, false), "bvh2, 6 x 128 threads per SM"},  // north_star's 32-byte-node binary tree
    {4, 0, 128, 0, 2, PS_INSTANCE(true, 0, 128, 0, 2, false), "bvh4, 6 x 128 threads per SM"},
    {4, 0, 768, 0, 2, PS_INSTANCE(true, 0, 768, 0, 2, false), "bvh4, 1 x 768 threads per SM"},
#ifdef RTB_PS_EXPERIMENTS
    {4, 0, 640, 0, 2, PS_INSTANCE(true, 0, 640, 0, 2, false), "bvh4, 1 x 640 threads per SM (96 registers)"},
    {4, 0, 896, 0, 2, PS_INSTANCE(true, 0, 896, 0, 2, false), "bvh4, 1 x 896 threads per SM (72 registers)"},
    {4, 0, 1024, 0, 2, PS_INSTANCE(true, 0, 1024, 0, 2, false), "bvh4, 1 x 1024 threads per SM (64 registers)"},
    {4, 8, 128, 0, 2, PS_INSTANCE(true, 8, 128, 0, 2, false), "bvh4, 6 x 128 threads, 8 stack levels in shared memory"},
    {4, 0, 768, 1, 2, PS_INSTANCE(true, 0, 768, 1, 2, false), "bvh4, 1 x 768 threads, nodes in shared memory"},
    {4, 0, 768, 2, 2, PS_INSTANCE(true, 0, 768, 2, 2, false), "bvh4, 1 x 768 threads, primitives in shared memory"},
    {4, 0, 768, 3, 2, PS_INSTANCE(true, 0, 768, 3, 2, false), "bvh4, 1 x 768 threads, nodes + primitives in shared memory"},
    {4, 0, 640, 3, 2, PS_INSTANCE(true, 0, 640, 3, 2, false), "bvh4, 1 x 640 threads, nodes + primitives in shared memory"},
#endif
    // The chain phase (wf_chain_step) as an opt-in instance, RT_PS_CHAIN=1: it removes 7 % of C4's warp instructions and
    // still loses 10 %, because the instructions the kernel then executes per frame (39 KB) no longer fit the SM's 32 KB
    // instruction cache (profiles/r2_chain_phase.txt) — carrying its code in the default instance cost 13 % even switched off.
    {4, 0, 768, 0, 2, PS_INSTANCE(true, 0, 768, 0, 2, true), "bvh4, 1 x 768 threads per SM, chain phase for clear media"},
};
const int kNumVariants = (int)(sizeof(kVariants) / sizeof(kVariants[0]));

// Feature-specialised instances of the product variant (bvh4, 1 x 768 threads, fast media): the first whose mask covers the
// scene's features is launched, so that the kernel holds no code the scene cannot reach.  Not a dispatch on speed of the
// tests themselves: what counts is that the ~31 KB of instructions final_scene executes per frame lie contiguous and
// below the 32 KB of the SM's instruction cache (DESIGN.md section 5; RT_PS_FEAT=0 launches the generic instance).
// (Registers: 24 warps = 6 per SM sub-partition leave 80 registers a thread and 24 - 52 B of spills; 23 or 22 warps do not
// help, a sub-partition still holds 6 of them; 20 warps at 96 registers measured -2.6 %, profiles/r2_ab_variants.txt run i.)
struct FeatInstance {
    uint32_t mask;
    int threads;
    PersistFn fn;
    PersistFn fn_q;  // the same with the chain queues (CHAINQ), for scenes with clear media; nullptr: none built
    const char* name;
};
#define PS_FEAT_INSTANCE(mask, nt) mask, nt, persist_kernel<false, true, 0, nt, 0, MEDIA_FAST, 2, false, mask>
#define PS_FEAT_INSTANCE_Q(mask, nt) persist_kernel<false, true, 0, nt, 0, MEDIA_FAST, 2, false, mask, true>
constexpr uint32_t kFeatSpheres = F_SPHERE | F_BIG;                                                           // random (C1, C2), simple
constexpr uint32_t kFeatBoxes = F_BOX | F_INSTBOX | F_INSTANCE | F_MEDIA | F_BOXMEDIA;                        // cornell_box, cornell_smoke (C3)
constexpr uint32_t kFeatFinal = F_SPHERE | F_BOX | F_INSTANCE | F_BIG | F_MEDIA | F_NOISE | F_IMAGE;          // final_scene (C4, C5)
const FeatInstance kFeatInstances[] = {
    {PS_FEAT_INSTANCE(kFeatSpheres, 768), nullptr, "spheres"},
    {PS_FEAT_INSTANCE(kFeatBoxes, 768), PS_FEAT_INSTANCE_Q(kFeatBoxes, 768), "boxes, instances, box media"},
    {PS_FEAT_INSTANCE(kFeatFinal, 768), PS_FEAT_INSTANCE_Q(kFeatFinal, 768), "spheres, world-space boxes, sphere media, noise and image textures"},
    {PS_FEAT_INSTANCE(F_ALL, 768), PS_FEAT_INSTANCE_Q(F_ALL, 768), "everything"},
};
// Chain queues: OPT-IN (RT_PS_CHAINQ=1), for scenes with clear media (FlatScene.clear_media) and the fast media sampler.
// Exact (identical images and ray counts, also with queues far too small) and measured (profiles/r2_chain_phase.txt,
// section 6): on C4 the main launch of the persistent kernel gets 37 % shorter, but what it saves in total is 8 % — the chain
// segments had been cheap riders of its phases — and chain_kernel costs 10 %: 2318 against 2313 Mpaths/s; C3 loses 19 %.
bool want_chain_queues(const RtScene* s) {
    if (s->flat.clear_media == 0u || s->view.media_general) return false;
    if (const char* e = getenv("RT_PS_CHAINQ")) return atoi(e) != 0;
    return false;
}
PersistFn pick_feature_instance(const RtScene* s, int vi, PersistFn generic, int* threads, bool* queues) {
    *queues = false;
    if (vi != PS_DEFAULT_VARIANT || s->view.media_general) return generic;
    bool specialise = true;
    if (const char* e = getenv("RT_PS_FEAT")) specialise = atoi(e) != 0;
    const bool q = want_chain_queues(s);
    for (const FeatInstance& f : kFeatInstances)
        if ((s->flat.features & ~f.mask) == 0u && (specialise || f.mask == F_ALL) && (!q || f.fn_q)) {
            *threads = f.threads, *queues = q;
            return q ? f.fn_q : f.fn;
        }
    return generic;
}

size_t variant_smem(const Variant& V, const RtScene* s) {
    size_t bytes = (size_t)V.slots * PS_REC * V.threads * sizeof(float) + (size_t)V.smem_stack * V.threads * sizeof(uint32_t);
    if (V.scene & PS_SCENE_NODES) bytes += s->flat.nodes4.size() * sizeof(DNode4);
    if (V.scene & PS_SCENE_PRIMS) bytes += s->flat.prims.size() * sizeof(DPrim);
    return bytes;
}

int pick_variant(const RtScene* s, const RtParams* p) {
    int layout = p->bvh_layout;
    if (layout == 0)
        if (const char* e = getenv("RT_BVH_LAYOUT")) layout = atoi(e);
    if (layout == 0) layout = PS_DEFAULT_LAYOUT;
    if (layout != 2 && s->flat.nodes4.empty()) layout = 2;  // the scene does not fit the 16-bit links of the wide tree
    if (layout == 2) return 0;
    int vi = PS_DEFAULT_VARIANT;
    if (const char* e = getenv("RT_PS_VARIANT")) vi = std::max(1, std::min(kNumVariants - 1, atoi(e)));
    if (const char* e = getenv("RT_PS_CHAIN"))
        if (atoi(e) != 0 && s->flat.clear_media != 0u) vi = kNumVariants - 1;
    if (variant_smem(kVariants[vi], s) > PS_MAX_SMEM) vi = 1;  // the scene copy does not fit beside the path pool
    return vi;
}

// the resident grid of a kernel instance (cached per instance in w->blocks under `key`), and the shared-memory carve-out
int size_grid(RtScene* s, PersistState* w, const void* key, const void* kernel, int NT, size_t smem, const char* name) {
    if (w->blocks.find(key) != w->blocks.end()) return RT_OK;
    int per_sm = 0, sms = 0;
    CU_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, NT, smem));
    if (per_sm < 1) return set_error(RT_ERR_CUDA, "persistent pipeline: kernel instance '%s' does not fit an SM", name);
    if (const char* e = getenv("RT_PS_BLOCKS_PER_SM")) per_sm = std::min(per_sm, std::max(1, atoi(e)));
    // Ask for exactly the shared memory the resident blocks need (+1 KB per block the runtime reserves); whatever is left
    // of the SM's 228 KB is L1, which holds the BVH, the primitives and the traversal stacks.  The driver's
    // default carve-out was larger than needed and cost 5 % (L1 hit rate 92 %).
    int need_kb = (int)((per_sm * (smem + 1024) + 1023) / 1024);
    int percent = std::min(100, (need_kb * 100 + 227) / 228);
    if (const char* e = getenv("RT_PS_CARVEOUT")) percent = atoi(e);
    CU_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, percent));
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    w->blocks[key] = per_sm * std::max(1, sms);  // persistent: exactly what is co-resident
    return RT_OK;
}

// one launch of `total` camera paths over `npix` pixels: the grid (at most the resident one) and the reservation size
void launch_shape(int resident, unsigned long long total, int NT, unsigned long long npix, int* blocks, unsigned int* chunk) {
    *blocks = (int)std::min<unsigned long long>((unsigned long long)resident, (total + 2 * NT - 1) / (2 * NT));
    // small jobs: smaller reservations so that every warp gets work
    unsigned long long per_warp = total / ((unsigned long long)*blocks * (NT / 32) * 4ull);
    *chunk = (unsigned int)std::min<unsigned long long>(PS_CHUNK, std::max<unsigned long long>(32ull, per_warp));
    *chunk = (unsigned int)std::min<unsigned long long>(*chunk, std::max<unsigned long long>(1ull, npix));
}

PsTune read_tune() {
    PsTune tune = {PS_WORK, PS_STALL, PS_LEAVE, PS_MIN_DESCEND, PS_CHAIN_TRIG, PS_CHAIN_MIN};
    if (const char* e = getenv("RT_PS_CHAIN_TRIG")) tune.chain_trig = atoi(e);
    if (const char* e = getenv("RT_PS_CHAIN_MIN")) tune.chain_min = std::max(1, atoi(e));
    if (const char* e = getenv("RT_PS_WORK")) tune.work = atoi(e);
    if (const char* e = getenv("RT_PS_STALL")) tune.stall = atoi(e);
    if (const char* e = getenv("RT_PS_LEAVE")) tune.leave = atoi(e);
    if (const char* e = getenv("RT_PS_DESCEND")) tune.descend = atoi(e);
    return tune;
}

// ---- the moments family: the feature masks and media forms the default path picks (pick_feature_instance, the general
// media sampler) on the 4-wide product placement, and the binary tree's variant for scenes beyond the 16-bit links of the
// 4-wide tree.  RT_PS_VARIANT, RT_PS_CHAIN, RT_PS_CHAINQ and RT_PS_STATS do not apply to it.
typedef void (*MomentsFn)(DSceneView, DCamera, DRenderParams, PsCounters*, AccumFx*, AccumFx*, const uint32_t*, unsigned int, unsigned long long*,
                          unsigned int, PsTune);
struct MomentsInstance {
    uint32_t mask;
    MomentsFn fn;
};
const MomentsInstance kMomentsFeat[] = {
    {kFeatSpheres, persist_moments_kernel<true, 768, MEDIA_FAST, kFeatSpheres>},
    {kFeatBoxes, persist_moments_kernel<true, 768, MEDIA_FAST, kFeatBoxes>},
    {kFeatFinal, persist_moments_kernel<true, 768, MEDIA_FAST, kFeatFinal>},
    {F_ALL, persist_moments_kernel<true, 768, MEDIA_FAST, F_ALL>},
};
const MomentsFn kMomentsWideGeneral = persist_moments_kernel<true, 768, MEDIA_GENERAL, F_ALL>;
const MomentsFn kMomentsBinary = persist_moments_kernel<false, 128, MEDIA_FAST, F_ALL>;
const MomentsFn kMomentsBinaryGeneral = persist_moments_kernel<false, 128, MEDIA_GENERAL, F_ALL>;

MomentsFn pick_moments_instance(const RtScene* s, const RtParams* p, int* vi) {
    *vi = pick_variant(s, p) == 0 ? 0 : PS_DEFAULT_VARIANT;
    if (*vi == 0) return s->view.media_general ? kMomentsBinaryGeneral : kMomentsBinary;
    if (s->view.media_general) return kMomentsWideGeneral;
    bool specialise = true;
    if (const char* e = getenv("RT_PS_FEAT")) specialise = atoi(e) != 0;
    for (const MomentsInstance& f : kMomentsFeat)
        if ((s->flat.features & ~f.mask) == 0u && (specialise || f.mask == F_ALL)) return f.fn;
    return kMomentsFeat[3].fn;
}

}  // namespace

int persist_layout_used(const RtScene* s, const RtParams* p) { return kVariants[pick_variant(s, p)].layout; }

// Scene creation asks the driver for the kernel a default render of this scene will launch: CUDA loads kernel images
// lazily, and for a job of a few milliseconds (C1 is 2 ms of work) that load would otherwise sit inside the first render.
void persist_preload(const RtScene* s) {
    RtParams p{};
    p.max_depth = 1;
    const Variant& V = kVariants[pick_variant(s, &p)];
    cudaFuncAttributes fa;
    const int vi = pick_variant(s, &p);
    int nt = V.threads;
    bool queues = false;
    if (cudaFuncGetAttributes(&fa, s->view.media_general ? V.fn_general : pick_feature_instance(s, vi, V.fn, &nt, &queues)) != cudaSuccess) cudaGetLastError();
    if (queues && cudaFuncGetAttributes(&fa, chain_kernel) != cudaSuccess) cudaGetLastError();
}

int launch_persist(RtScene* s, const DCamera& cam, const RtParams* p, int begin, int count, AccumFx* d_accum, cudaStream_t stream, RtProgressFn cb,
                   void* user, int* launches) {
    if (!persist_supports(s, p)) return set_error(RT_ERR_UNSUPPORTED, "persistent pipeline: max_depth above %d or more than 2^24 primitives", WF_DEPTH_MASK);
    if (p->bvh_layout != 0 && p->bvh_layout != 2 && p->bvh_layout != 4) return set_error(RT_ERR_INVALID, "render: bvh_layout must be 0 (auto), 2 or 4");
    if (p->max_depth <= 0) return RT_OK;  // every path returns Color::ZERO at once (raytrace.rs:87-89)
    if (!s->ps) {
        s->ps = new PersistState();
        CU_TRY(rtb::cache_malloc((void**)&s->ps->ctr, sizeof(PsCounters)));
    }
    PersistState* w = s->ps;
    const int vi = pick_variant(s, p);
    const Variant& V = kVariants[vi];
    int NT = V.threads;
    bool queues = false;
    const PersistFn kernel = s->view.media_general ? V.fn_general : pick_feature_instance(s, vi, V.fn, &NT, &queues);
    if (getenv("RT_PS_STATS")) queues = false;  // (the statistics instance has no queues)
    const size_t smem = variant_smem(V, s) / V.threads * NT;  // (every term of it is per thread for the variant feature instances exist for)
    const void* const key = getenv("RT_PS_STATS") ? (const void*)V.fn_stats : (const void*)kernel;
    if (w->blocks.find(key) == w->blocks.end()) {
        // (the statistics instance only when it will be launched: touching a kernel makes the driver load it, which a 3 ms job notices)
        if (getenv("RT_PS_STATS")) CU_TRY(cudaFuncSetAttribute(V.fn_stats, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int rc = size_grid(s, w, key, (const void*)kernel, NT, smem, V.name);
        if (rc != RT_OK) return rc;
    }
    const unsigned long long npix = (unsigned long long)p->width * p->height;
    // one launch = up to 2^29 camera paths when progress is reported (a quarter of a second on C4), 2^33 otherwise: every
    // launch ends with a tail in which the longest paths run on a mostly idle machine
    int samples_per_launch = (int)std::min<unsigned long long>(1u << 30, std::max<unsigned long long>(1, (1ull << (cb ? 29 : 33)) / npix));
    // Chain queues: one launch = 2^27 camera paths (RT_PS_CHAINQ_LOG2_PATHS), and queues of 2^24 records (RT_PS_CHAINQ_LOG2_CAP; 2 x
    // 896 MB) — final_scene pushes ~0.1 records per path; a push that finds the queue full leaves the path in the kernel.
    PsChainIO io = {nullptr, nullptr, nullptr, 0u};
    int chain_blocks = 0;
    if (queues) {
        int log2_paths = 27, log2_cap = 24;
        if (const char* e = getenv("RT_PS_CHAINQ_LOG2_PATHS")) log2_paths = std::max(10, std::min(33, atoi(e)));
        if (const char* e = getenv("RT_PS_CHAINQ_LOG2_CAP")) log2_cap = std::max(8, std::min(28, atoi(e)));
        samples_per_launch = (int)std::min<unsigned long long>((unsigned long long)samples_per_launch, std::max<unsigned long long>(1, (1ull << log2_paths) / npix));
        const unsigned int cap = 1u << log2_cap;
        if (w->io.cc && w->io.cap != cap) {  // another capacity asked for: start over
            rtb::cache_free(w->io.chain, (size_t)PQ_REC * w->io.cap * sizeof(float)), rtb::cache_free(w->io.exitq, (size_t)PQ_REC * w->io.cap * sizeof(float));
            rtb::cache_free(w->io.cc, sizeof(ChainCounters));
            w->io = PsChainIO{nullptr, nullptr, nullptr, 0u};
        }
        if (!w->io.cc) {
            CU_TRY(rtb::cache_malloc((void**)&w->io.chain, (size_t)PQ_REC * cap * sizeof(float)));
            CU_TRY(rtb::cache_malloc((void**)&w->io.exitq, (size_t)PQ_REC * cap * sizeof(float)));
            CU_TRY(rtb::cache_malloc((void**)&w->io.cc, sizeof(ChainCounters)));
            w->io.cap = cap;
        }
        io = w->io;
        CU_TRY(cudaMemsetAsync(io.cc, 0, sizeof(ChainCounters), stream));
        int per_sm = 0, sms = 0;
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, chain_kernel, CHAIN_THREADS, 0));
        CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
        chain_blocks = std::max(1, per_sm) * std::max(1, sms);
    }
    const PsTune tune = read_tune();
    int done = 0;
    while (done < count) {
        int samples = std::min(count - done, samples_per_launch);
        unsigned long long total = npix * (unsigned long long)samples;
        DRenderParams P = device_params(p, begin + done, 1, 1);
        int blocks = 0;
        unsigned int chunk = 0u;
        launch_shape(w->blocks[key], total, NT, npix, &blocks, &chunk);
        ps_reset_kernel<<<1, 1, 0, stream>>>(w->ctr, total, io.cc);
        if (getenv("RT_PS_STATS")) {  // debug: phase statistics on stderr (slower kernel; never used by the bench)
            unsigned long long* d_stats = nullptr;
            CU_TRY(cudaMalloc(&d_stats, PSS_COUNT * sizeof(unsigned long long)));
            CU_TRY(cudaMemsetAsync(d_stats, 0, PSS_COUNT * sizeof(unsigned long long), stream));
            V.fn_stats<<<blocks, NT, smem, stream>>>(s->view, cam, P, w->ctr, d_accum, s->d_rays, chunk, d_stats, tune, io);
            unsigned long long h[PSS_COUNT];
            CU_TRY(cudaMemcpyAsync(h, d_stats, sizeof h, cudaMemcpyDeviceToHost, stream));
            CU_TRY(cudaStreamSynchronize(stream));
            cudaFree(d_stats);
            static const char* names[PSS_COUNT] = {"shade_phases", "shade_act_lanes", "shade_done_lanes", "shade_onpark_lanes", "ext_phases", "inner_iters",
                                                   "inner_lanes", "leaf_steps", "leaf_lanes", "leaf_prims", "ext_rounds", "ext_trav_lanes", "noise_evals",
                                                   "chain_phases", "chain_records", "chain_iters", "chain_lanes", "chain_parked"};
            fprintf(stderr, "persist stats [%s] (%llu paths):", V.name, total);
            for (int k = 0; k < PSS_COUNT; ++k) fprintf(stderr, " %s=%llu", names[k], h[k]);
            fprintf(stderr, "\n");
        } else {
            kernel<<<blocks, NT, smem, stream>>>(s->view, cam, P, w->ctr, d_accum, s->d_rays, chunk, nullptr, tune, io);
        }
        CU_TRY(cudaGetLastError());
        *launches += 2;
        done += samples;
        if (queues) {  // the chain paths of this launch, hopped to their end; those that leave their medium wait for the next launch
            chain_reset_kernel<<<1, 1, 0, stream>>>(io.cc);
            chain_kernel<<<chain_blocks, CHAIN_THREADS, 0, stream>>>(s->view, P, io, s->d_rays);
            CU_TRY(cudaGetLastError());
            *launches += 2;
        }
        if (cb) {
            CU_TRY(cudaStreamSynchronize(stream));
            cb(done, count, user);
        }
    }
    // drain: launches without new camera paths until no path is left in either queue (each takes a tenth of the previous one's)
    for (int round = 0; queues && round < 1024; ++round) {
        ChainCounters h;
        CU_TRY(cudaMemcpyAsync(&h, io.cc, sizeof h, cudaMemcpyDeviceToHost, stream));
        CU_TRY(cudaStreamSynchronize(stream));
        const unsigned int n_exit = std::min(h.exit_count, io.cap);
        if (getenv("RT_PS_CHAINQ_VERBOSE")) fprintf(stderr, "chain queues: drain round %d, %u exits, %u pushes dropped so far\n", round, n_exit, h.chain_dropped);
        if (n_exit == 0u) break;
        DRenderParams P = device_params(p, begin + count, 1, 1);
        const int blocks = (int)std::min<unsigned long long>((unsigned long long)w->blocks[key], ((unsigned long long)n_exit + 2 * NT - 1) / (2 * NT));
        ps_reset_kernel<<<1, 1, 0, stream>>>(w->ctr, 0ull, io.cc);
        kernel<<<blocks, NT, smem, stream>>>(s->view, cam, P, w->ctr, d_accum, s->d_rays, 32u, nullptr, tune, io);
        chain_reset_kernel<<<1, 1, 0, stream>>>(io.cc);
        chain_kernel<<<chain_blocks, CHAIN_THREADS, 0, stream>>>(s->view, P, io, s->d_rays);
        CU_TRY(cudaGetLastError());
        *launches += 4;
    }
    return RT_OK;
}

int launch_persist_moments(RtScene* s, const DCamera& cam, const RtParams* p, int begin, int count, AccumFx* d_accum, AccumFx* d_moment2,
                           const uint32_t* d_list, unsigned int n_list, cudaStream_t stream, int* launches) {
    if (!persist_supports(s, p)) return set_error(RT_ERR_UNSUPPORTED, "persistent pipeline: max_depth above %d or more than 2^24 primitives", WF_DEPTH_MASK);
    if (p->bvh_layout != 0 && p->bvh_layout != 2 && p->bvh_layout != 4) return set_error(RT_ERR_INVALID, "render: bvh_layout must be 0 (auto), 2 or 4");
    if (p->max_depth <= 0 || n_list == 0u) return RT_OK;
    if (!s->ps) {
        s->ps = new PersistState();
        CU_TRY(rtb::cache_malloc((void**)&s->ps->ctr, sizeof(PsCounters)));
    }
    PersistState* w = s->ps;
    int vi = 0;
    const MomentsFn kernel = pick_moments_instance(s, p, &vi);
    const Variant& V = kVariants[vi];
    const int NT = V.threads;
    const size_t smem = variant_smem(V, s);
    int rc = size_grid(s, w, (const void*)kernel, (const void*)kernel, NT, smem, "moments");
    if (rc != RT_OK) return rc;
    const PsTune tune = read_tune();
    const int samples_per_launch = (int)std::min<unsigned long long>(1u << 30, std::max<unsigned long long>(1, (1ull << 33) / n_list));
    for (int done = 0; done < count;) {
        const int samples = std::min(count - done, samples_per_launch);
        const unsigned long long total = (unsigned long long)n_list * (unsigned long long)samples;
        DRenderParams P = device_params(p, begin + done, 1, 1);
        P.inv_npix = 1.0 / (double)n_list;
        int blocks = 0;
        unsigned int chunk = 0u;
        launch_shape(w->blocks[(const void*)kernel], total, NT, n_list, &blocks, &chunk);
        ps_reset_kernel<<<1, 1, 0, stream>>>(w->ctr, total, nullptr);
        kernel<<<blocks, NT, smem, stream>>>(s->view, cam, P, w->ctr, d_accum, d_moment2, d_list, n_list, s->d_rays, chunk, tune);
        CU_TRY(cudaGetLastError());
        *launches += 2;
        done += samples;
    }
    return RT_OK;
}

}  // namespace rtb
