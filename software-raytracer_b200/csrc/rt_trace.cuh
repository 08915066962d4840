// rt_trace.cuh - closest-hit back ends shared by the render kernels (rt_kernels.cu, rt_wavefront.cu):
// shared-memory staging of the scene per CTA, the MODE dispatch, and the host-side choice of variant.
#pragma once
#include "rt_device.cuh"
#include "rt_kernels.h"
#include "rt_bvh_lane.cuh"

namespace rtb {

constexpr int kTileW = 16, kTileH = 8;          // CTA tile: 4 warps, each an 8x4 pixel block
constexpr int kThreads = 128;
static_assert(kThreads == kLaneThreads, "rt_bvh_lane.cuh lays the traversal stacks out for CTAs of kThreads threads");
#ifndef RTB_BVH_POP_CULL
#define RTB_BVH_POP_CULL 1             // big (global-memory) BVHs: keep the far child's entry distance on the stack, skip stale pops
#endif
#ifndef RTB_REGEN_MIN_BLOCKS
#define RTB_REGEN_MIN_BLOCKS 6      // register budget of the render kernel: 65536 / (128 * 6) -> 80 registers
#endif
#ifndef RTB_REGEN_STASH_BLOCKS
#define RTB_REGEN_STASH_BLOCKS 7    // k_render_regen<.., STASH>: 72 registers
#endif

// ---- closest-hit back ends -------------------------------------------------------------------
// MODE 0: brute force, geometry staged in shared memory      MODE 1: brute force from global (L1)
// MODE 2: BVH, nodes + refs + geometry staged in shared mem  MODE 3: BVH from global (L1/L2); when the 8-wide quantised
//                                                                    form exists (bvh_wide.h) MODE 3 traverses that one
// MODE 4: flat two-level accelerator (flat_build.h), everything staged in shared memory
// Shared memory layout: [BVH stack: stack_entries x blockDim ints][spheres][cubes][nodes][refs]
//                       MODE 4: [cluster boxes per octant: 16 x n_clusters float4][candidate queues: kFlatQueue x blockDim bytes][spheres][cubes][level-1 boxes][cull records, packed pairs][prim ids][cull slots]
struct TraceCtx {
    const float4* sph; const float4* box; const float4* nodes; const int* refs;
    int* stack; float* stack_t; int stride;
    FlatView fl;
    unsigned char* q;          // MODE 4/5: this thread's candidate queue, entries `stride` bytes apart
    unsigned char* coop;       // MODE 5: this WARP's scratch for the cooperative levels 2/3
    const uint4* wnodes; const int* wrefs; int wentries; uint32_t k47;   // MODE 3 with the wide BVH: stack = [3 * wentries][thread] words
};

// MODE 5 = MODE 4 with warp-cooperative levels 2 and 3 (closest_hit_flat_coop below); per-warp scratch layout:
// [ray: 6 x 32 floats (o, d)][pairs: kCoopPairs x u16][sphere candidates: kCoopCands x u16][best key: 32 x u64]
constexpr int kCoopPairs = 64;                  // (owner lane, cluster) pairs per call; more -> per-lane fallback
#ifndef RTB_COOP_CANDS
#define RTB_COOP_CANDS 768
#endif
constexpr int kCoopCands = RTB_COOP_CANDS;      // sphere candidates per call (every pair full + every lane's level-1 queue full would be 64 * 8 + 32 * 56 = 2304:
                                                // 4.6 KB per warp, which held the kernel at 6 CTAs per SM); a call whose upper bound is larger takes the per-lane fallback
constexpr int kCoopBytesPerWarp = 6 * 32 * 4 + kCoopPairs * 2 + kCoopCands * 2 + 32 * 8;

// Float4 i of the staged cull records (cull_pair): records j, j + 1 of a cluster (j = 0, 2, 4, 6) or of the singles become
// [x_j x_j+1 y_j y_j+1][z_j z_j+1 R'_j R'_j+1] in place; a cluster's pad stays as it is. With an odd number of singles the last
// pair's second half is zeros and one float4 more is staged than the host holds: it fits the slack of flat_staged_bytes(),
// which counts one cull-slot byte per record, pads included, plus 16 bytes.
__device__ __forceinline__ float4 flat_stage_cull(const float4* __restrict__ cull, int n_clusters, int n_singles, int i) {
    const int nclu = kClusterStride * n_clusters;
    int j, last;                                   // the pair's first record, the last record of its group
    if (i < nclu) {
        const int w = i % kClusterStride;
        if (w == 8) return __ldg(cull + i);
        j = i - w + (w & ~1); last = i - w + 7;
    } else {
        j = nclu + ((i - nclu) & ~1); last = nclu + n_singles - 1;
    }
    const float4 a = __ldg(cull + j), b = j + 1 <= last ? __ldg(cull + j + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
    return ((i - j) & 1) ? make_float4(a.z, b.z, a.w, b.w) : make_float4(a.x, b.x, a.y, b.y);
}

template <int MODE>
__device__ __forceinline__ TraceCtx setup_trace(const SceneView& sc, const BvhView& bv, const FlatView& fl, float4* smem) {
    TraceCtx t;
    t.sph = sc.sph; t.box = sc.box; t.nodes = bv.nodes; t.refs = bv.refs; t.stack = nullptr; t.stack_t = nullptr; t.stride = blockDim.x;
    t.fl = fl; t.q = nullptr;
    t.wnodes = bv.wnodes; t.wrefs = bv.wrefs; t.wentries = bv.wstack_entries; t.k47 = bv.q2f_hi;
    float4* p = smem;
    t.coop = nullptr;
    if (MODE == 4 || MODE == 5) {
#ifndef RTB_FLAT_NO_OCT
        // the per-octant cluster boxes FIRST: every query addresses them per lane (base + octant), and at offset 0 of the dynamic
        // shared memory that address is one add instead of the whole layout computation re-done in vector registers
        for (int i = threadIdx.x; i < 8 * fl.n_clusters; i += blockDim.x) flat_fill_oct(fl.boxes, i >> 3, i & 7, p);
        t.fl.oct = p; p += 16 * fl.n_clusters;
#endif
        t.q = reinterpret_cast<unsigned char*>(p) + threadIdx.x;
        p += (kFlatQueue * blockDim.x + 15) / 16;
        if (MODE == 5) {
            t.coop = reinterpret_cast<unsigned char*>(p) + (threadIdx.x >> 5) * kCoopBytesPerWarp;
            p += ((blockDim.x >> 5) * kCoopBytesPerWarp + 15) / 16;
        }
        const int ng = sc.n_sph + 2 * sc.n_box, nb = 2 * (fl.n_clusters + fl.n_cubes), ncull = kClusterStride * fl.n_clusters + fl.n_singles;
        const int nslot = 8 * fl.n_clusters + fl.n_singles;
        const int np = sc.n_sph + sc.n_box;
        for (int i = threadIdx.x; i < ng; i += blockDim.x) p[i] = i < sc.n_sph ? __ldg(sc.sph + i) : __ldg(sc.box + (i - sc.n_sph));
        t.sph = p; t.box = p + sc.n_sph; p += ng;
        for (int i = threadIdx.x; i < nb; i += blockDim.x) p[i] = __ldg(fl.boxes + i);
        t.fl.boxes = p; p += nb;
        const int nstaged = ncull + (fl.n_singles & 1);
        for (int i = threadIdx.x; i < nstaged; i += blockDim.x) p[i] = flat_stage_cull(fl.cull, fl.n_clusters, fl.n_singles, i);
        t.fl.cull = p; p += nstaged;
        int* ids = reinterpret_cast<int*>(p);
        for (int i = threadIdx.x; i < np; i += blockDim.x) ids[i] = __ldg(fl.prim_id + i);
        t.fl.prim_id = ids;
        unsigned char* slots = reinterpret_cast<unsigned char*>(ids + np);
        for (int i = threadIdx.x; i < nslot; i += blockDim.x) slots[i] = __ldg(fl.cull_slot + i);
        t.fl.cull_slot = slots;
        __syncthreads();
        return t;
    }
    if (MODE >= 2) {
        t.stack = reinterpret_cast<int*>(p) + threadIdx.x;
        t.stack_t = reinterpret_cast<float*>(t.stack + bv.stack_entries * blockDim.x);
        p += (2 * bv.stack_entries * blockDim.x + 3) / 4;      // links + entry distances
    }
    if (MODE == 0 || MODE == 2) {
        const int ng = sc.n_sph + 2 * sc.n_box;
        for (int i = threadIdx.x; i < ng; i += blockDim.x)
            p[i] = i < sc.n_sph ? __ldg(sc.sph + i) : __ldg(sc.box + (i - sc.n_sph));
        t.sph = p; t.box = p + sc.n_sph;
        p += ng;
        if (MODE == 2) {
            for (int i = threadIdx.x; i < 4 * bv.n_nodes; i += blockDim.x) p[i] = __ldg(bv.nodes + i);
            t.nodes = p;
            p += 4 * bv.n_nodes;
            int* r = reinterpret_cast<int*>(p);
            for (int i = threadIdx.x; i < bv.n_refs; i += blockDim.x) r[i] = __ldg(bv.refs + i);
            t.refs = r;
        }
        __syncthreads();
    }
    return t;
}

// COUNT (BVH modes 2 and 3 over the binary tree only): the lane's traversal work is added to *tcnt.
template <int MODE, bool COUNT = false>
__device__ __forceinline__ Hit trace(const SceneView& sc, const TraceCtx& t, float3 o, float3 d, TravCount* tcnt = nullptr) {
    if (MODE == 4 || MODE == 5) return closest_hit_flat(sc, t.fl, t.sph, t.box, t.q, t.stride, o, d);
    if (MODE == 3 && t.wnodes) return closest_hit_bvh8(sc, t.sph, t.box, t.wnodes, t.wrefs, t.stack, t.stride, t.wentries, t.k47, o, d);
    if (MODE >= 2) return closest_hit_bvh<COUNT, MODE == 3>(sc, t.sph, t.box, t.nodes, t.refs, t.stack, t.stride, o, d, (RTB_BVH_POP_CULL && MODE == 3) ? t.stack_t : nullptr, tcnt);
    return closest_hit(sc, t.sph, t.box, o, d);
}

// Adds a lane's traversal counts to the context's counters [8..12] (queries, node visits, sphere / cube / triangle tests):
// warp reduce, one atomic per warp and counter. Must be reached by all 32 lanes.
__device__ __forceinline__ void flush_trav_count(const TravCount& tc, unsigned int queries, unsigned long long* __restrict__ counters) {
    unsigned int v[5] = {queries, tc.nodes, tc.sph, tc.box, tc.tri};
#pragma unroll
    for (int k = 0; k < 5; ++k) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], off);
        if ((threadIdx.x & 31) == 0 && v[k]) atomicAdd(counters + 8 + k, (unsigned long long)v[k]);
    }
}


// ---- warp-cooperative flat traversal ------------------------------------------------------------------------------
// Levels 2 and 3 of the flat accelerator per lane leave most of the warp idle: a lane has 0.9 hit clusters and 0.9
// candidates on average but the warp loops for the lane with the most (2.5 and 3.9 iterations on Scene1, 9 and 7 lanes
// active; profiles/r1q_summary_flat_reuse_1024spp.txt). Here the warp pools the work: every lane publishes its ray,
// the (lane, cluster) pairs of all lanes are enumerated with a prefix sum into one list and each lane culls ONE pair
// (whoever's it is); the surviving (lane, primitive) candidates are appended to a second list the same way and each
// lane runs ONE strict test per pass, returning the result to the owning lane as the minimum of
// (order-preserving bits of t, object id) in shared memory - exactly the reference's "closest, lowest id on ties". Lanes without work
// of their own (sky pixels, finished pixels) serve the others. Must be called by all 32 lanes; `active` = has a ray.
__device__ __forceinline__ unsigned int warp_incl_scan(unsigned int v, int lane) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned int n = __shfl_up_sync(0xffffffffu, v, off);
        if (lane >= off) v += n;
    }
    return v;
}

// the rare per-lane fallback, kept out of line so it does not dilute the instruction cache of the hot loop. It culls one record at a
// time: with the packed culls' register pairs in this callee, the 72-register form of the caller spills its path state across the
// whole query (172 B of spill stores instead of none); the fallback's speed does not matter.
static __device__ __noinline__ Hit flat_levels23_outlined(const SceneView& sc, const FlatView& fv, const float4* __restrict__ sph,
                                                   const float4* __restrict__ box, unsigned char* __restrict__ q, int qstride,
                                                   float3 o, float3 d, unsigned int cm, int nq) {
    return flat_levels23<false>(sc, fv, sph, box, q, qstride, o, d, cm, nq);
}

__device__ __forceinline__ Hit closest_hit_flat_coop(const SceneView& sc, const FlatView& fv, const float4* __restrict__ sph,
                                                     const float4* __restrict__ box, unsigned char* __restrict__ q, int qstride,
                                                     unsigned char* __restrict__ coop, float3 o, float3 d, bool active) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    float* const ray_s = reinterpret_cast<float*>(coop);
    unsigned short* const pairs = reinterpret_cast<unsigned short*>(coop + 6 * 32 * 4);
    unsigned short* const cand = pairs + kCoopPairs;
    unsigned long long* const key = reinterpret_cast<unsigned long long*>(cand + kCoopCands);

    int nq = 0, nq_cubes = 0;
    unsigned int cm = 0u;
    if (active) cm = flat_level1(sc, fv, q, qstride, o, d, nq, nq_cubes);
    // ---- level 2: (lane, cluster) pairs, one per lane per pass ----
    const unsigned int cnt = (unsigned int)__popc(cm);
    const unsigned int incl = warp_incl_scan(cnt, lane);
    const unsigned int n_pairs = __shfl_sync(FULL, incl, 31);
    const unsigned int own_all = __reduce_add_sync(FULL, (unsigned int)(nq - nq_cubes));
    if (n_pairs > (unsigned int)kCoopPairs || own_all + 8u * n_pairs > (unsigned int)kCoopCands) {   // rare: every lane works for itself
        Hit h;
        h.id = -1; h.t = 0.f; h.n = f3(0.f, 0.f, 0.f); h.p = f3(0.f, 0.f, 0.f);
        if (active) h = flat_levels23_outlined(sc, fv, sph, box, q, qstride, o, d, cm, nq);
        return h;
    }
    ray_s[lane] = o.x; ray_s[32 + lane] = o.y; ray_s[64 + lane] = o.z;
    ray_s[96 + lane] = d.x; ray_s[128 + lane] = d.y; ray_s[160 + lane] = d.z;
    reinterpret_cast<unsigned int*>(key)[lane] = 0xffffffffu; reinterpret_cast<unsigned int*>(key)[32 + lane] = 0xffffffffu;
    {
        unsigned int m = cm, j = incl - cnt;
        while (m) { const int k = __ffs((int)m) - 1; m &= m - 1u; pairs[j++] = (unsigned short)((lane << 8) | k); }
    }
    __syncwarp();
    // sphere candidates: every lane's level-1 singles (pass 0, as owner) + the survivors of the pair it culls (as worker)
    unsigned int n_cand = 0u;                                 // warp-uniform
    unsigned int base = 0u;
    do {
        unsigned int m8 = 0u, pr = 0u;
        if (base + (unsigned int)lane < n_pairs) {
            pr = pairs[base + lane];
            const int ow = (int)(pr >> 8);
            m8 = flat_cull8(fv, (int)(pr & 255u), f3(ray_s[ow], ray_s[32 + ow], ray_s[64 + ow]), f3(ray_s[96 + ow], ray_s[128 + ow], ray_s[160 + ow]));
        }
        const unsigned int own = base == 0u ? (unsigned int)(nq - nq_cubes) : 0u;
        const unsigned int contrib = own + (unsigned int)__popc(m8);
        const unsigned int incl2 = warp_incl_scan(contrib, lane);
        unsigned int j = n_cand + incl2 - contrib;
        for (unsigned int i = 0; i < own; ++i) cand[j++] = (unsigned short)((lane << 8) | q[(nq_cubes + (int)i) * qstride]);
        while (m8) { const int b = __clz((int)m8) - 24; m8 &= ~(0x80u >> b); cand[j++] = (unsigned short)((pr & 0xff00u) | fv.cull_slot[8 * (pr & 255u) + b]); }
        n_cand += __shfl_sync(FULL, incl2, 31);
        base += 32u;
    } while (base < n_pairs);
    // cubes stay with their own lane: in rooms of cubes every ray has a similar number of them, so there is nothing to pool,
    // and the ray-only half of the cube test is computed once
    float cube_t = __int_as_float(0x7f800000);
    int cube_id = 0x7fffffff, cube_code = -1;
    float3 bn = f3(0.f, 0.f, 0.f);
    if (nq_cubes > 0) {
        const BoxRay br = box_ray(d);
        for (int i = 0; i < nq_cubes; ++i) {
            const int code = (int)q[i * qstride], j = code - sc.n_sph;
            float dist; float3 nrm;
            if (box_hit_pre(box[2 * j], box[2 * j + 1], o, br, dist, nrm)) {
                const int oid = fv.prim_id[code];
                if (dist < cube_t || (dist == cube_t && oid < cube_id)) { cube_t = dist; cube_id = oid; cube_code = code; bn = nrm; }
            }
        }
    }
    __syncwarp();
    // ---- level 3, spheres: one strict test per lane per pass; the owner gets the minimum of (t, object id) ----
    // Two native 32-bit shared-memory minima per pass - first the distance, then, among the candidates that have the owner's smallest
    // distance so far, the object id - instead of one 64-bit atomicMin on (distance, id), which is a compare-and-swap loop in shared
    // memory (4 % of the kernel's instructions at 10-12 active threads; C2 110.2 -> 108.9 ms, C1 2.05 -> 1.96 ms, same bits:
    // profiles/r4q_ab_key32.txt). Passes are ordered by __syncwarp; a pass that lowers the distance resets the id word before it
    // competes for it. Lexicographic minimum of (t, id): the reference's "closest, lowest index on ties" (Raytracer.cpp:127-137).
    unsigned int* const key_t = reinterpret_cast<unsigned int*>(key);      // [0..31] order-preserving bits of t, [32..63] (object id << 8) | code
    for (base = 0u; base < n_cand; base += 32u) {
        const unsigned int i = base + (unsigned int)lane;
        unsigned int ob = 0xffffffffu, idc = 0xffffffffu;
        int ow = 0;
        if (i < n_cand) {
            const unsigned int e = cand[i];
            ow = (int)(e >> 8);
            const int code = (int)(e & 255u);
            float t = 0.f;
            if (sphere_t(sph[code], f3(ray_s[ow], ray_s[32 + ow], ray_s[64 + ow]), f3(ray_s[96 + ow], ray_s[128 + ow], ray_s[160 + ow]), t) && t == t) {
                ob = __float_as_uint(t);
                ob ^= (unsigned int)((int)ob >> 31) | 0x80000000u;
                idc = ((unsigned int)fv.prim_id[code] << 8) | (unsigned int)code;
            }
        }
        const unsigned int before = idc != 0xffffffffu ? key_t[ow] : 0u;
        if (idc != 0xffffffffu && ob < before) atomicMin(key_t + ow, ob);
        __syncwarp();
        const unsigned int now = idc != 0xffffffffu ? key_t[ow] : 0u;
        if (idc != 0xffffffffu && now < before && ob == now) key_t[32 + ow] = 0xffffffffu;     // a new smallest distance: its ids start afresh (same value from every writer)
        __syncwarp();
        if (idc != 0xffffffffu && ob == now) atomicMin(key_t + 32 + ow, idc);
        __syncwarp();
    }
    const unsigned int kid = key_t[32 + lane];               // 0xffffffff: no sphere was hit
    float best_t = cube_t; int best_id = cube_id, best_code = cube_code;
    if (active && kid != 0xffffffffu) {
        unsigned int ob = key_t[lane];
        ob ^= (unsigned int)((int)~ob >> 31) | 0x80000000u;
        const float st = __uint_as_float(ob);
        const int sid = (int)(kid >> 8);
        if (st < best_t || (st == best_t && sid < best_id)) { best_t = st; best_id = sid; best_code = (int)(kid & 255u); }
    }
    __syncwarp();                                             // everyone is done with the scratch before the next call
    return flat_finish(sc, sph, o, d, best_t, best_id, best_code, bn);
}

// Per-lane trace for all lanes of a warp (inactive lanes get a miss); MODE 5 pools levels 2/3 across the warp.
template <int MODE, bool COUNT = false>
__device__ __forceinline__ Hit trace_all(const SceneView& sc, const TraceCtx& t, float3 o, float3 d, bool active, TravCount* tcnt = nullptr) {
    if (MODE == 5) return closest_hit_flat_coop(sc, t.fl, t.sph, t.box, t.q, t.stride, t.coop, o, d, active);
    Hit h;
    h.id = -1; h.t = 0.f; h.n = f3(0.f, 0.f, 0.f); h.p = f3(0.f, 0.f, 0.f);
    if (active) h = trace<MODE, COUNT>(sc, t, o, d, tcnt);
    return h;
}

// ---- host: variant + dynamic shared memory size for a back end -----------------------------------
inline size_t staged_bytes(const SceneView& sc) { return (size_t)(sc.n_sph + 2 * sc.n_box) * sizeof(float4); }
inline size_t flat_staged_bytes(const SceneView& sc, const FlatView& fl, int threads) {
    const size_t ncull = (size_t)kClusterStride * fl.n_clusters + fl.n_singles;
    return (size_t)kFlatQueue * threads + staged_bytes(sc) + (size_t)2 * (fl.n_clusters + fl.n_cubes) * 16 + (size_t)16 * fl.n_clusters * 16 + ncull * 16 + (size_t)(sc.n_sph + sc.n_box) * 4 + ncull + 16;
}
inline int pick_mode(const SceneView& sc, const AccelSel& ac, size_t& smem, int threads = kThreads, bool coop = false) {
    const size_t geo = staged_bytes(sc);
    if (ac.kind == kAccelFlat) {
        smem = flat_staged_bytes(sc, ac.flat, threads);
        if (coop) { smem += (size_t)(threads / 32) * kCoopBytesPerWarp + 16; return 5; }
        return 4;
    }
    if (ac.kind == kAccelBrute) {
        if (geo <= kMaxStagedBytes) { smem = geo; return 0; }
        smem = 0; return 1;
    }
    const BvhView& bv = ac.bvh;
    if (bv.wnodes) { smem = ((size_t)3 * bv.wstack_entries * threads * sizeof(int) + 15) / 16 * 16; return 3; }
    const size_t stack = ((size_t)2 * bv.stack_entries * threads * sizeof(int) + 15) / 16 * 16;
    const size_t all = stack + geo + (size_t)bv.n_nodes * 64 + (size_t)bv.n_refs * 4 + 16;
    if (all <= kMaxBvhStagedBytes) { smem = all; return 2; }
    smem = stack; return 3;
}

}  // namespace rtb
