// rt_wavefront.cu - the WAVEFRONT pipeline (RT_PIPELINE_WAVEFRONT): the same path tracer as the regeneration
// megakernel (rt_kernels.cu k_render_regen), split into stream-ordered stages over device-resident queues:
//
//   k_wf_generate   raygen: one path per (pixel, sample) of the wave; with REUSE it shades the pixel's cached primary hit
//                   (the context's per-pixel cache, rt_kernels.cu k_primary_cache)
//                   and emits the first SECONDARY ray; live paths get consecutive slots of state set 0
//   k_wf_intersect  persistent threads: every warp pulls batches of 32 queue entries through an atomic cursor
//                   and runs the closest-hit back end (brute / BVH / flat, scene staged per CTA once)
//   k_wf_shade      path_ends / scatter_segment per entry; surviving paths are COMPACTED into consecutive slots of
//                   the other state set: warp ballot + prefix popcount, one atomicAdd per CTA pass (block_slot)
//   k_wf_accumulate per pixel, the wave's samples are added in sample order; k_wf_commit adds the launch's sum
//                   into the accumulation buffer
//
// A wave is all pixels x S samples (S <= 64, up to 128 M paths). No host synchronisation anywhere: queue lengths stay
// in device memory (one counter and one cursor per bounce round, zeroed per wave) and the persistent kernels
// read them there. Path state lives in two DENSE ping-pong sets of SoA float4 arrays: slot i of a round's set is its
// i-th surviving path (plus its path id = wave-local sample x tile-major pixel), so every kernel reads and writes
// consecutive records. Every path's arithmetic is the megakernel's (same device
// functions, same Philox counters) and samples are summed in the same order: the result is BIT-IDENTICAL to
// k_render_regen (asserted by tests/test_gpu_parity.py), whichever order the queues end up in.
#include "rt_kernels.h"

#include <cstdio>
#include <mutex>

#include "rt_devbuf.h"
#include "rt_device.cuh"
#include "rt_trace.cuh"

namespace rtb {

struct WavefrontBuffers {
    // Path state lives in DENSE ping-pong sets: slot i of round r's set is the i-th surviving path, so every kernel reads and
    // writes consecutive records (with one fixed slot per path and a queue of path ids the survivors of the later rounds are
    // scattered and a 32-byte sector carries one useful record: the shade kernel moved 3.8x its useful bytes).
    DeviceArray<float4> ray_o[2], ray_d[2];           // per slot: o, (d, depth)
    DeviceArray<float4> thr[2], rad[2];               // per slot: T, L
    DeviceArray<uint32_t> q[2];                       // per slot: path id (tile-major pixel + npad * sample)
    DeviceArray<float4> hit_nt; DeviceArray<int> hit_id;   // per slot of the current round: (normal, t), object id
    DeviceArray<float4> wave_rad;                     // per PATH id: radiance of the finished path
    DeviceArray<unsigned int> counters;               // [0..63] queue lengths per round, [64..127] cursors
    DeviceArray<float4> launch_acc;                   // per pixel: this launch's sum
    size_t paths() const { return q[1].capacity(); }  // paths the per-path arrays hold (alloc_paths: all of them or none)
};

namespace {

constexpr int kMaxRounds = 64;
constexpr size_t kBytesPerPath = 2 * (4 * 16 + 4) + 16 + 4 + 16;   // two state sets + path id each, hit record, finished radiance: 172 B

struct WaveGeom { int tiles_x, tiles_y, npad; };
__host__ __device__ inline WaveGeom wave_geom(int w, int h) {
    WaveGeom g; g.tiles_x = (w + 7) / 8; g.tiles_y = (h + 3) / 4; g.npad = g.tiles_x * g.tiles_y * 32;
    return g;
}
// tile-major pixel index -> pixel: 8x4 tiles, so the 32 lanes of a warp cover a compact block like the megakernel's
__device__ __forceinline__ bool tile_to_pixel(const FrameView& fr, int tiles_x, int ti, int& px, int& py) {
    const int tile = ti >> 5, lane = ti & 31;
    px = (tile % tiles_x) * 8 + (lane & 7);
    py = (tile / tiles_x) * 4 + (lane >> 3);
    return px < fr.width && py < fr.height;
}

// append `pid` to a queue for the lanes with want == true: one atomicAdd per warp
__device__ __forceinline__ void warp_push(bool want, uint32_t pid, uint32_t* __restrict__ q, unsigned int* __restrict__ count) {
    const unsigned mask = __ballot_sync(0xffffffffu, want);
    if (mask == 0u) return;
    const int lane = threadIdx.x & 31;
    unsigned int base = 0;
    if (lane == (__ffs((int)mask) - 1)) base = atomicAdd(count, (unsigned int)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, __ffs((int)mask) - 1);
    if (want) q[base + __popc(mask & ((1u << lane) - 1u))] = pid;
}

// Slot allocation for a whole CTA of NW warps: ONE atomicAdd on the counter per CTA pass instead of one per warp (a wave of
// 133 M paths is 4 M warps, all adding to the same word), and the segment counters ride along: `delivered` is summed over the
// CTA and added to seg_counter[0 .. n_seg) by the same thread. Must be reached by every thread of the CTA.
template <int NW>
__device__ __forceinline__ unsigned int block_slot(bool want, unsigned int* __restrict__ count,
                                                   unsigned int delivered, unsigned long long* __restrict__ seg_counter, int n_seg) {
    __shared__ unsigned int s_cnt[NW], s_del[NW], s_base;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned mask = __ballot_sync(0xffffffffu, want);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) delivered += __shfl_down_sync(0xffffffffu, delivered, off);
    __syncthreads();                                         // the previous pass has read s_base / s_cnt
    if (lane == 0) { s_cnt[w] = (unsigned int)__popc(mask); s_del[w] = delivered; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int c = 0, dl = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) { const unsigned int t = s_cnt[i]; s_cnt[i] = c; c += t; dl += s_del[i]; }
        s_base = c ? atomicAdd(count, c) : 0u;
        if (dl) for (int k = 0; k < n_seg; ++k) atomicAdd(seg_counter + k, (unsigned long long)dl);
    }
    __syncthreads();
    return s_base + s_cnt[w] + (unsigned int)__popc(mask & ((1u << lane) - 1u));      // this thread's slot in the next set, if it wants one
}

template <bool REUSE>
__global__ void __launch_bounds__(256) k_wf_generate(SceneView sc, FrameView fr, int tiles_x, int npad, uint32_t s_first, int s_wave,
                                                      const float4* __restrict__ prim_nt, const int* __restrict__ prim_id,
                                                      float4* __restrict__ ray_o, float4* __restrict__ ray_d, float4* __restrict__ thr,
                                                      float4* __restrict__ rad, float4* __restrict__ wave_rad,
                                                      uint32_t* __restrict__ q0, unsigned int* __restrict__ counters,
                                                      unsigned long long* __restrict__ seg_counter) {
    const uint32_t np = (uint32_t)npad * (uint32_t)s_wave;
    const uint32_t pid = blockIdx.x * blockDim.x + threadIdx.x;             // the grid covers np rounded up to warps
    bool live = false;
    unsigned int delivered = 0;
    float4 so = make_float4(0.f, 0.f, 0.f, 0.f), sd = so, sT = so, sL = so;
    if (pid < np) {
        const int ti = (int)(pid % (uint32_t)npad);
        const uint32_t s = s_first + pid / (uint32_t)npad;
        int px, py;
        if (tile_to_pixel(fr, tiles_x, ti, px, py)) {
            const uint32_t pixel = (uint32_t)px + (uint32_t)py * (uint32_t)fr.width;
            float3 o = fr.cam_pos, d = ray_dir(fr, px, py);
            float3 T = f3(0.f, 0.f, 0.f), L = f3(0.f, 0.f, 0.f);
            int depth = 0;
            live = true;
            if (REUSE) {
                const float4 nt = __ldg(prim_nt + pixel);
                Hit h0;
                h0.id = __ldg(prim_id + pixel); h0.t = nt.w; h0.n = f3(nt.x, nt.y, nt.z);
                h0.p = f3(o.x + d.x * nt.w, o.y + d.y * nt.w, o.z + d.z * nt.w);
                delivered = 1;                                               // the reused primary segment
                float3 c;
                if (primary_ends(sc, fr, h0, c)) { wave_rad[pid] = make_float4(c.x, c.y, c.z, 0.f); live = false; }
                else scatter_segment(sc, fr, h0, pixel, s, o, d, T, L, depth);
            }
            if (live) { so = make_float4(o.x, o.y, o.z, 0.f); sd = make_float4(d.x, d.y, d.z, __int_as_float(depth)); sT = make_float4(T.x, T.y, T.z, 0.f); sL = make_float4(L.x, L.y, L.z, 0.f); }
        }
    }
    const unsigned int slot = block_slot<8>(live, counters, delivered, seg_counter, REUSE ? 2 : 0);      // segments + reused (not traced) segments
    if (live) { ray_o[slot] = so; ray_d[slot] = sd; thr[slot] = sT; rad[slot] = sL; q0[slot] = pid; }
}

// Persistent threads: the grid is sized to the machine, not to the queue. Each warp claims 32 consecutive entries.
template <int MODE>
__global__ void __launch_bounds__(kThreads, 6) k_wf_intersect(SceneView sc, BvhView bv, FlatView fl, const uint32_t* __restrict__ q,
                                                               const unsigned int* __restrict__ count_ptr, unsigned int* __restrict__ cursor,
                                                               const float4* __restrict__ ray_o, const float4* __restrict__ ray_d,
                                                               float4* __restrict__ hit_nt, int* __restrict__ hit_id) {
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);
    const unsigned int count = *count_ptr;
    const int lane = threadIdx.x & 31;
    for (;;) {
        unsigned int base = 0;
        if (lane == 0) base = atomicAdd(cursor, 32u);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= count) break;
        const unsigned int i = base + (unsigned int)lane;
        if (i < count) {
            const uint32_t pid = i;                          // dense state: slot = queue position
            const float4 o4 = ray_o[pid], d4 = ray_d[pid];
            const Hit h = trace<MODE>(sc, tc, f3(o4.x, o4.y, o4.z), f3(d4.x, d4.y, d4.z));
            hit_nt[pid] = make_float4(h.n.x, h.n.y, h.n.z, h.t);
            hit_id[pid] = h.id;
        }
    }
}


// BVH scenes: persistent threads with PER-LANE ray replacement and POSTPONED leaves ("speculative while-while").
// With one ray per lane per batch (k_wf_intersect above) a warp runs until its longest traversal ends: on the
// 10 000-sphere scene 5 of 32 lanes are active on average (profiles/r1l_summary_c3_bvh.txt). Here every lane is
// a small state machine - IDLE (needs a ray), ACTIVE, DONE (hit pending):
//   node phase  lanes holding an inner node step through it together; a lane that reaches a leaf stashes it
//               (one pending leaf) and keeps traversing - culling against a best distance that is merely not
//               yet as tight as it could be, so the candidate set stays conservative; the phase ends when
//               fewer than kNodeMin lanes still hold an inner node;
//   leaf phase  the stashed leaves are tested together with the strict reference arithmetic (with ~70 node
//               visits and ~5 leaves per ray, testing a leaf the moment one lane reaches it would drag the whole
//               warp through the leaf code at almost every step);
//   refill      as soon as kRefill lanes are free, the DONE lanes write their hits together and every free lane
//               claims the next queue entry (one atomicAdd per warp).
// Same candidate semantics, strict tests and tie rule as closest_hit_bvh(): bit-identical results (tested).
// k_refill: free lanes that trigger a refill pass; k_node_min: lanes with inner-node work below which the warp turns
// to its pending leaves (RT_OPT_WF_REFILL / RT_OPT_WF_NODE_MIN; defaults measured on the 10k-sphere scene)

#ifndef RTB_WF_BVH_MIN_BLOCKS
#define RTB_WF_BVH_MIN_BLOCKS 8      // 63 registers, no spills: the kernel waits on node fetches (issue slots 52 % busy at 6), +8 % at 8
#endif
#ifndef RTB_WF_NODE_UNROLL
#define RTB_WF_NODE_UNROLL 2           // node steps per warp vote in the node phase: the vote, its count and the branch are ~10 of a step's ~90
                                       // instructions. Measured (profiles/r2ad_ab_node_unroll.txt): C3 92.9 / 88.3 / 89.3 / 88.4 ms and C4 23.2 / 22.1 /
                                       // 22.2 / 22.1 ms per step with 1 / 2 / 3 / 4 (streaming kernel: 2 best, 3 and 4 lose)
#endif
template <int MODE, bool COUNT = false, bool QUANT = false>
__global__ void __launch_bounds__(kThreads, RTB_WF_BVH_MIN_BLOCKS) k_wf_intersect_bvh(SceneView sc, BvhView bv, FlatView fl, const uint32_t* __restrict__ q,
                                                                   const unsigned int* __restrict__ count_ptr, unsigned int* __restrict__ cursor,
                                                                   const float4* __restrict__ ray_o, const float4* __restrict__ ray_d,
                                                                   float4* __restrict__ hit_nt, int* __restrict__ hit_id, int kRefill, int kNodeMin,
                                                                   unsigned long long* __restrict__ counters) {
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);
    const float4* __restrict__ nodes = tc.nodes;
    const int* __restrict__ refs = tc.refs;
    const uint4* __restrict__ qnodes = (MODE == 3 && QUANT) ? bv.qnodes : nullptr;     // 32-byte quantised nodes (the host built them: QUANT)
    const unsigned int count = *count_ptr;
    const int lane = threadIdx.x & 31;
    constexpr unsigned FULL = 0xffffffffu;

    BvhLane L;                                               // rt_bvh_lane.cuh: traversal state + shared-memory stack
    L.init(tc.stack);
    uint32_t pid = 0;
    float3 o = f3(0.f, 0.f, 0.f), d = f3(0.f, 0.f, 1.f);
    bool exhausted = false;
    TravCount cnt = {0u, 0u, 0u, 0u};                          // COUNT only
    unsigned int n_queries = 0;

    for (;;) {
        // ---- refill ---------------------------------------------------------------------------------------
        const unsigned m_free = __ballot_sync(FULL, L.state != BvhLane::ACTIVE);
        if (__popc(m_free) >= kRefill || m_free == FULL) {
            if (L.state == BvhLane::DONE) {                  // write the pending hits together
                const Hit h = L.finish(tc.sph, o, d);
                hit_nt[pid] = make_float4(h.n.x, h.n.y, h.n.z, h.t);
                hit_id[pid] = h.id;
                L.state = BvhLane::IDLE;
            }
            if (!exhausted) {
                const unsigned m_idle = __ballot_sync(FULL, L.state == BvhLane::IDLE);
                unsigned int base = 0;
                const int leader = __ffs((int)m_idle) - 1;
                if (lane == leader) base = atomicAdd(cursor, (unsigned int)__popc(m_idle));
                base = __shfl_sync(FULL, base, leader);
                if (L.state == BvhLane::IDLE) {
                    const unsigned int i = base + (unsigned int)__popc(m_idle & ((1u << lane) - 1u));
                    if (i < count) {
                        pid = i;                             // dense state: slot = queue position
                        const float4 o4 = ray_o[pid], d4 = ray_d[pid];
                        o = f3(o4.x, o4.y, o4.z); d = f3(d4.x, d4.y, d4.z);
                        L.begin(o, d, QUANT, bv.q_org, bv.q_step);
                        if (COUNT) ++n_queries;
                    }
                }
                if (base + (unsigned int)__popc(m_idle) >= count) exhausted = true;       // warp-uniform
            }
            if (!__any_sync(FULL, L.state == BvhLane::ACTIVE)) break;    // nothing left to traverse (DONE lanes were flushed above)
        }
        // ---- node phase: at least one step, then for as long as enough lanes hold an inner node ----------------
        for (;;) {
#pragma unroll
            for (int u = 0; u < RTB_WF_NODE_UNROLL; ++u)
                if (L.in_node()) L.node_step<COUNT, MODE == 3, QUANT ? 1 : 0>(nodes, cnt, qnodes, bv.q2f16);
            if (__popc(__ballot_sync(FULL, L.in_node())) < kNodeMin) break;
        }
        // ---- leaf phase: the stashed leaves (and a second one waiting in `cur`), strict tests ---------------------
        if (L.state == BvhLane::ACTIVE) L.leaf_step<COUNT>(sc, tc.sph, tc.box, refs, MODE == 3 ? bv.slots : nullptr, o, d, cnt);
    }
    if (COUNT) flush_trav_count(cnt, n_queries, counters);
}

// ---- STREAMING variant: the whole path in the persistent kernel (RT_PIPELINE_STREAM) ----------------------------------
// The bounce-round pipeline above moves every path's state through HBM once per bounce (~170 B per segment), needs two more
// kernels per round and runs its late rounds - a few per cent of the paths - on an almost empty machine, which is why it wants
// waves of 128 M paths (22 GB of state). Here the lane that finishes a traversal SHADES its hit on the spot and goes on with
// the scattered ray; a lane whose path ended stores the path's radiance (16 B) and claims the next path id from one global
// cursor (ids are sample-major over tile-major pixels, like the wavefront's). The traversal is the state machine of
// k_wf_intersect_bvh (speculative while-while, postponed leaves, refill at kRefill free lanes); the shading block runs for the
// DONE lanes of a warp together under the same refill condition. Path state that is only needed at a hit (throughput, radiance
// so far, depth, pixel, sample) lives in shared memory, 9 words per thread, so the traversal keeps its 64 registers.
// No queues, no per-bounce state, no rounds: HBM sees the primary-hit cache (20 B per path) and the finished radiance (16 B per
// path); samples are added per pixel in sample order by k_wf_accumulate afterwards, so the sum is BIT-IDENTICAL to the
// megakernel's and to the wavefront pipeline's (tests/test_gpu_round2.py).
constexpr int kStreamStateWords = 9;       // T.xyz, L.xyz, depth, pixel, sample - per thread, [word][thread] in shared memory
#ifndef RTB_WF_STREAM_MIN_BLOCKS
#define RTB_WF_STREAM_MIN_BLOCKS 8
#endif
#ifndef RTB_STREAM_SHADE_NOINLINE
#define RTB_STREAM_SHADE_NOINLINE 0    // measured (profiles/r2t_ab.txt): as a call the kernel is 6 % SLOWER on both BVH scenes
#endif
#if RTB_STREAM_SHADE_NOINLINE
#define RTB_STREAM_SHADE_ATTR __noinline__
#else
#define RTB_STREAM_SHADE_ATTR __forceinline__
#endif
// The shading of one finished traversal of the streaming kernel. Inlined, its ~40 live values (Philox block, normalisations, the sky's
// powers) set the register count of the whole kernel and the traversal loop spills a little at 64 registers; as a CALL
// (RTB_STREAM_SHADE_NOINLINE=1) the loop keeps its registers, but the call's argument traffic and the parameter structs read through
// generic pointers cost more than the spills: C3 101.0 -> 107.3 ms, C4 28.9 -> 30.7 ms per step. Returns true when the path goes on
// with the scattered ray (o, d); false when it ended (radiance stored).
static __device__ RTB_STREAM_SHADE_ATTR bool stream_shade(const SceneView& sc, const FrameView& fr, const Hit& h, float* __restrict__ ps, float3& o, float3& d,
                                                          float4* __restrict__ wave_rad, uint32_t pid) {
    float3 T = f3(ps[0], ps[kThreads], ps[2 * kThreads]), Lr = f3(ps[3 * kThreads], ps[4 * kThreads], ps[5 * kThreads]);
    int depth = __float_as_int(ps[6 * kThreads]);
    float3 c;
    if (path_ends(sc, fr, h, d, T, Lr, depth, c)) {
        wave_rad[pid] = make_float4(c.x, c.y, c.z, 0.f);
        return false;
    }
    scatter_segment(sc, fr, h, __float_as_uint(ps[7 * kThreads]), __float_as_uint(ps[8 * kThreads]), o, d, T, Lr, depth);
    ps[0] = T.x; ps[kThreads] = T.y; ps[2 * kThreads] = T.z; ps[3 * kThreads] = Lr.x; ps[4 * kThreads] = Lr.y; ps[5 * kThreads] = Lr.z;
    ps[6 * kThreads] = __int_as_float(depth);
    return true;
}

template <int MODE, bool REUSE, bool COUNT, bool QUANT = false>
__global__ void __launch_bounds__(kThreads, RTB_WF_STREAM_MIN_BLOCKS) k_wf_stream(const __grid_constant__ SceneView sc, const __grid_constant__ BvhView bv, const __grid_constant__ FlatView fl,
                                                                                const __grid_constant__ FrameView fr, int tiles_x, int npad,
                                                                                uint32_t s_first, unsigned int n_paths, const float4* __restrict__ prim_nt,
                                                                                const int* __restrict__ prim_id, float4* __restrict__ wave_rad,
                                                                                unsigned int* __restrict__ cursor, int kRefill, int kNodeMin,
                                                                                unsigned long long* __restrict__ seg_counter) {
    extern __shared__ float4 smem[];
    float* const ps = reinterpret_cast<float*>(smem) + threadIdx.x;           // this thread's path state, words kThreads apart
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem + (kStreamStateWords * kThreads + 3) / 4);
    const float4* __restrict__ nodes = tc.nodes;
    const int* __restrict__ refs = tc.refs;
    const uint4* __restrict__ qnodes = (MODE == 3 && QUANT) ? bv.qnodes : nullptr;     // 32-byte quantised nodes (the host built them: QUANT)
    const int lane = threadIdx.x & 31;
    constexpr unsigned FULL = 0xffffffffu;

    BvhLane L;                                               // rt_bvh_lane.cuh: traversal state + shared-memory stack
    L.init(tc.stack);
    uint32_t pid = 0;
    float3 o = f3(0.f, 0.f, 0.f), d = f3(0.f, 0.f, 1.f);
    bool exhausted = false;
    TravCount cnt = {0u, 0u, 0u, 0u};
    unsigned int segs = 0, traced = 0;

    for (;;) {
        // ---- shade + refill ---------------------------------------------------------------------------------
        const unsigned m_free = __ballot_sync(FULL, L.state != BvhLane::ACTIVE);
        if (__popc(m_free) >= kRefill || m_free == FULL) {
            if (L.state == BvhLane::DONE) {                  // the finished traversals of the warp are shaded together
                const Hit h = L.finish(tc.sph, o, d);
                ++segs; ++traced;
                if (stream_shade(sc, fr, h, ps, o, d, wave_rad, pid)) L.begin(o, d, QUANT, bv.q_org, bv.q_step);
                else L.state = BvhLane::IDLE;
            }
            if (!exhausted) {                                // every idle lane claims the next path id: one atomicAdd per warp
                const unsigned m_idle = __ballot_sync(FULL, L.state == BvhLane::IDLE);
                if (m_idle) {
                    unsigned int base = 0;
                    const int leader = __ffs((int)m_idle) - 1;
                    if (lane == leader) base = atomicAdd(cursor, (unsigned int)__popc(m_idle));
                    base = __shfl_sync(FULL, base, leader);
                    if (L.state == BvhLane::IDLE) {
                        const unsigned int i = base + (unsigned int)__popc(m_idle & ((1u << lane) - 1u));
                        int px, py;
                        if (i < n_paths && tile_to_pixel(fr, tiles_x, (int)(i % (unsigned int)npad), px, py)) {
                            pid = i;
                            const uint32_t pixel = (uint32_t)px + (uint32_t)py * (uint32_t)fr.width;
                            const uint32_t sample = s_first + i / (unsigned int)npad;
                            o = fr.cam_pos; d = ray_dir(fr, px, py);
                            float3 T = f3(0.f, 0.f, 0.f), Lr = f3(0.f, 0.f, 0.f);
                            int depth = 0;
                            bool live = true;
                            if (REUSE) {                     // start from the pixel's cached primary hit (k_primary_cache)
                                const float4 nt = __ldg(prim_nt + pixel);
                                Hit h0;
                                h0.id = __ldg(prim_id + pixel); h0.t = nt.w; h0.n = f3(nt.x, nt.y, nt.z);
                                h0.p = f3(o.x + d.x * nt.w, o.y + d.y * nt.w, o.z + d.z * nt.w);
                                ++segs;                      // the reused primary segment: delivered, not traced
                                float3 c;
                                if (primary_ends(sc, fr, h0, c)) { wave_rad[pid] = make_float4(c.x, c.y, c.z, 0.f); live = false; }
                                else scatter_segment(sc, fr, h0, pixel, sample, o, d, T, Lr, depth);
                            }
                            if (live) {
                                ps[0] = T.x; ps[kThreads] = T.y; ps[2 * kThreads] = T.z; ps[3 * kThreads] = Lr.x; ps[4 * kThreads] = Lr.y; ps[5 * kThreads] = Lr.z;
                                ps[6 * kThreads] = __int_as_float(depth); ps[7 * kThreads] = __uint_as_float(pixel); ps[8 * kThreads] = __uint_as_float(sample);
                                L.begin(o, d, QUANT, bv.q_org, bv.q_step);
                            }
                        }
                    }
                    if (base + (unsigned int)__popc(m_idle) >= n_paths) exhausted = true;       // warp-uniform
                }
            }
            if (!__any_sync(FULL, L.state == BvhLane::ACTIVE)) {
                if (exhausted) break;                        // no traversal in flight, nothing left to claim (DONE lanes were shaded above)
                continue;                                    // this pass's paths all ended at once (sky pixels): claim more
            }
        }
        // ---- node phase: at least one step, then for as long as enough lanes hold an inner node ----------------
        for (;;) {
#pragma unroll
            for (int u = 0; u < RTB_WF_NODE_UNROLL; ++u)
                if (L.in_node()) L.node_step<COUNT, MODE == 3, QUANT ? 1 : 0>(nodes, cnt, qnodes, bv.q2f16);
            if (__popc(__ballot_sync(FULL, L.in_node())) < kNodeMin) break;
        }
        // ---- leaf phase: the stashed leaves (and a second one waiting in `cur`), strict tests ---------------------
        if (L.state == BvhLane::ACTIVE) L.leaf_step<COUNT>(sc, tc.sph, tc.box, refs, MODE == 3 ? bv.slots : nullptr, o, d, cnt);
    }
    // segment counters: delivered [0..1], executed [2..3]; one atomic per warp and counter
    unsigned int tot = segs, tot_tr = traced;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) { tot += __shfl_down_sync(FULL, tot, off); tot_tr += __shfl_down_sync(FULL, tot_tr, off); }
    if (lane == 0 && tot) {
        atomicAdd(seg_counter, (unsigned long long)tot); atomicAdd(seg_counter + 1, (unsigned long long)tot);
        atomicAdd(seg_counter + 2, (unsigned long long)tot_tr); atomicAdd(seg_counter + 3, (unsigned long long)tot_tr);
    }
    if (COUNT) flush_trav_count(cnt, traced, seg_counter);
}

// The same state machine over the 8-WIDE quantised BVH (bvh_wide.h): a node step tests eight children at once, the
// line's nearest inner child becomes the lane's next node and the other hit children wait on the stack as one group
// with the smallest of their entry parameters (groups that start behind the best hit are dropped at the pop); the node's
// leaf candidates (up to 24 refs, one bit each) are kept in one of two pending slots and tested in the leaf phase.
// A ray makes about 2.2 times fewer node steps than in the binary tree and each step is five 16-byte loads from ONE
// 80-byte record instead of four from a 64-byte one.
#ifndef RTB_WF_BVH8_MIN_BLOCKS
#define RTB_WF_BVH8_MIN_BLOCKS 5
#endif
__global__ void __launch_bounds__(kThreads, RTB_WF_BVH8_MIN_BLOCKS) k_wf_intersect_bvh8(SceneView sc, BvhView bv, const uint32_t* __restrict__ q,
                                                                     const unsigned int* __restrict__ count_ptr, unsigned int* __restrict__ cursor,
                                                                     const float4* __restrict__ ray_o, const float4* __restrict__ ray_d,
                                                                     float4* __restrict__ hit_nt, int* __restrict__ hit_id, int kRefill, int kNodeMin) {
    extern __shared__ float4 smem[];
    const int stride = blockDim.x, E = bv.wstack_entries;
    int* const stk = reinterpret_cast<int*>(smem) + threadIdx.x;            // [group base: E][group bits: E][bound: E] x [thread]
    float* const stk_t = reinterpret_cast<float*>(stk + 2 * E * stride);
    const uint4* __restrict__ wn = bv.wnodes;
    const int* __restrict__ refs = bv.wrefs;
    const unsigned int count = *count_ptr;
    const int lane = threadIdx.x & 31;
    constexpr unsigned FULL = 0xffffffffu;
    constexpr uint32_t NONE = 0xffffffffu;
    enum { IDLE = 0, ACTIVE = 1, DONE = 2 };

    int state = IDLE, sp = 0;
    uint32_t pid = 0, node = NONE, t0x = 0, t0b = 0, t1x = 0, t1b = 0;
    float node_t = 0.f;
    float3 o = f3(0.f, 0.f, 0.f), d = f3(0.f, 0.f, 1.f);
    WideRay wr = wide_ray(d, bv.q2f_hi);
    BestHit b;
    b.t = 0.f; b.id = 0; b.ref = 0; b.have = false; b.n = f3(0.f, 0.f, 0.f);
    bool exhausted = false;

    // next node from the waiting groups (octant order inside a group); NONE when nothing is left in front of the best hit
    auto pop_node = [&]() {
        node = NONE;
        while (sp > 0) {
            const float bound = stk_t[(sp - 1) * stride];
            if (bound > b.t) { --sp; continue; }
            const uint32_t gx = (uint32_t)stk[(sp - 1) * stride];
            uint32_t gy = (uint32_t)stk[(E + sp - 1) * stride];
            const int p = 31 - __clz((int)gy);
            gy &= ~(1u << p);
            if (gy & 0xff000000u) stk[(E + sp - 1) * stride] = (int)gy; else --sp;
            const uint32_t slot = (uint32_t)(p - 24) ^ (wr.octinv4 & 7u);
            node = gx + (uint32_t)__popc(gy & 0xffu & ((1u << slot) - 1u));
            node_t = bound;
            return;
        }
    };

    for (;;) {
        // ---- refill ---------------------------------------------------------------------------------------
        const unsigned m_free = __ballot_sync(FULL, state != ACTIVE);
        if (__popc(m_free) >= kRefill || m_free == FULL) {
            if (state == DONE) {                             // write the pending hits together
                Hit h;
                h.id = -1; h.t = 0.f; h.n = f3(0.f, 0.f, 0.f);
                if (b.have) {
                    h.id = b.id; h.t = b.t;
                    if (b.ref >= 0 && b.ref < kTriRef) {
                        const float4 s4 = sc.sph[b.ref];
                        const float3 p = f3(o.x + d.x * b.t, o.y + d.y * b.t, o.z + d.z * b.t);             // Object.hpp:136
                        h.n = normalized3(f3(p.x - s4.x, p.y - s4.y, p.z - s4.z));                         // Object.hpp:137
                    } else h.n = b.n;
                }
                hit_nt[pid] = make_float4(h.n.x, h.n.y, h.n.z, h.t);
                hit_id[pid] = h.id;
                state = IDLE;
            }
            if (!exhausted) {
                const unsigned m_idle = __ballot_sync(FULL, state == IDLE);
                unsigned int base = 0;
                const int leader = __ffs((int)m_idle) - 1;
                if (lane == leader) base = atomicAdd(cursor, (unsigned int)__popc(m_idle));
                base = __shfl_sync(FULL, base, leader);
                if (state == IDLE) {
                    const unsigned int i = base + (unsigned int)__popc(m_idle & ((1u << lane) - 1u));
                    if (i < count) {
                        pid = i;                             // dense state: slot = queue position
                        const float4 o4 = ray_o[pid], d4 = ray_d[pid];
                        o = f3(o4.x, o4.y, o4.z); d = f3(d4.x, d4.y, d4.z);
                        wr = wide_ray(d, bv.q2f_hi);
                        b.t = __int_as_float(0x7f800000); b.id = 0x7fffffff; b.ref = 0; b.have = false;
                        node = 0u; node_t = -b.t; t0b = t1b = 0u; sp = 0; state = ACTIVE;
                    }
                }
                if (base + (unsigned int)__popc(m_idle) >= count) exhausted = true;       // warp-uniform
            }
            if (!__any_sync(FULL, state == ACTIVE)) break;    // nothing left to traverse (DONE lanes were flushed above)
        }
        // ---- node phase: at least one step, then for as long as enough lanes have a node and room for its leaf candidates ----
        for (;;) {
            if (state == ACTIVE && node != NONE && !t1b) {
                const uint4* __restrict__ np = wn + 5u * node;
                const uint4 w0 = np[0], w1 = np[1], w2 = np[2], w3 = np[3], w4 = np[4];
                uint32_t near_bit; float e1, e2;
                const uint32_t hm = wide_node_hits(w0, w1, w2, w3, w4, o, wr, b.t, near_bit, e1, e2);
                const uint32_t tb = hm & 0x00ffffffu;
                if (tb) { if (!t0b) { t0x = w1.y; t0b = tb; } else { t1x = w1.y; t1b = tb; } }
                uint32_t gy = (hm & 0xff000000u) | (w0.w >> 24);
                if (gy & 0xff000000u) {
                    gy &= ~(1u << near_bit);
                    if (gy & 0xff000000u) { stk[sp * stride] = (int)w1.x; stk[(E + sp) * stride] = (int)gy; stk_t[sp * stride] = e2; ++sp; }
                    const uint32_t slot = (near_bit - 24u) ^ (wr.octinv4 & 7u);
                    node = w1.x + (uint32_t)__popc(gy & 0xffu & ((1u << slot) - 1u));
                    node_t = e1;
                } else {
                    pop_node();
                    if (node == NONE && !t0b) state = DONE;
                }
            }
            if (__popc(__ballot_sync(FULL, state == ACTIVE && node != NONE && !t1b)) < kNodeMin) break;
        }
        // ---- leaf phase: the pending candidates, strict tests; then drop a next node that now starts behind the best hit ----
        if (state == ACTIVE) {
            for (;;) {
                uint32_t base; int bit;
                if (t0b) { bit = __ffs((int)t0b) - 1; t0b &= t0b - 1u; base = t0x; }
                else if (t1b) { bit = __ffs((int)t1b) - 1; t1b &= t1b - 1u; base = t1x; }
                else break;
                test_ref(sc, sc.sph, sc.box, refs[base + (uint32_t)bit], o, d, b);
            }
            if (node != NONE && node_t > b.t) node = NONE;
            if (node == NONE) pop_node();
            if (node == NONE) state = DONE;
        }
    }
}

__global__ void __launch_bounds__(256) k_wf_shade(SceneView sc, FrameView fr, int tiles_x, int npad, uint32_t s_first,
                                                   const uint32_t* __restrict__ q_in, const unsigned int* __restrict__ count_ptr,
                                                   uint32_t* __restrict__ q_out, unsigned int* __restrict__ count_out,
                                                   const float4* __restrict__ ray_o, const float4* __restrict__ ray_d, const float4* __restrict__ thr,
                                                   const float4* __restrict__ rad, float4* __restrict__ ray_o2, float4* __restrict__ ray_d2,
                                                   float4* __restrict__ thr2, float4* __restrict__ rad2,
                                                   const float4* __restrict__ hit_nt, const int* __restrict__ hit_id,
                                                   float4* __restrict__ wave_rad, unsigned long long* __restrict__ seg_counter) {
    const unsigned int count = *count_ptr;
    const unsigned int stride = gridDim.x * blockDim.x;
    // whole CTAs stay in the loop together: the compaction needs every thread
    for (unsigned int base = blockIdx.x * blockDim.x; base < count; base += stride) {
        const unsigned int i = base + threadIdx.x;
        bool live = false;
        unsigned int done = 0;
        uint32_t pid = 0;
        float4 so = make_float4(0.f, 0.f, 0.f, 0.f), sd = so, sT = so, sL = so;
        if (i < count) {
            pid = q_in[i];
            const int ti = (int)(pid % (uint32_t)npad);
            const uint32_t s = s_first + pid / (uint32_t)npad;
            int px, py;
            tile_to_pixel(fr, tiles_x, ti, px, py);
            const uint32_t pixel = (uint32_t)px + (uint32_t)py * (uint32_t)fr.width;
            const float4 o4 = ray_o[i], d4 = ray_d[i], T4 = thr[i], L4 = rad[i], nt = hit_nt[i];
            float3 o = f3(o4.x, o4.y, o4.z), d = f3(d4.x, d4.y, d4.z), T = f3(T4.x, T4.y, T4.z), L = f3(L4.x, L4.y, L4.z);
            int depth = __float_as_int(d4.w);
            Hit h;
            h.id = hit_id[i]; h.t = nt.w; h.n = f3(nt.x, nt.y, nt.z);
            h.p = f3(o.x + d.x * nt.w, o.y + d.y * nt.w, o.z + d.z * nt.w);            // as in closest_hit*()
            ++done;
            float3 c;
            if (path_ends(sc, fr, h, d, T, L, depth, c)) wave_rad[pid] = make_float4(c.x, c.y, c.z, 0.f);
            else {
                scatter_segment(sc, fr, h, pixel, s, o, d, T, L, depth);
                so = make_float4(o.x, o.y, o.z, 0.f); sd = make_float4(d.x, d.y, d.z, __int_as_float(depth));
                sT = make_float4(T.x, T.y, T.z, 0.f); sL = make_float4(L.x, L.y, L.z, 0.f);
                live = true;
            }
        }
        const unsigned int slot = block_slot<8>(live, count_out, done, seg_counter, 4);  // ray compaction + the four segment counters
        if (live) { ray_o2[slot] = so; ray_d2[slot] = sd; thr2[slot] = sT; rad2[slot] = sL; q_out[slot] = pid; }
    }
}

__global__ void k_wf_accumulate(FrameView fr, int tiles_x, int npad, int s_wave, const float4* __restrict__ wave_rad,
                                float4* __restrict__ launch_acc) {
    const int ti = blockIdx.x * blockDim.x + threadIdx.x;
    if (ti >= npad) return;
    int px, py;
    if (!tile_to_pixel(fr, tiles_x, ti, px, py)) return;
    const size_t pixel = (size_t)px + (size_t)py * fr.width;
    float4 a = launch_acc[pixel];
    for (int s = 0; s < s_wave; ++s) {                       // sample order: the megakernel's summation order
        const float4 c = wave_rad[(size_t)s * npad + ti];
        a.x += c.x; a.y += c.y; a.z += c.z;
    }
    launch_acc[pixel] = a;
}

__global__ void k_wf_commit(int n, const float4* __restrict__ launch_acc, float4* __restrict__ accum) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    float4 a = accum[p];
    const float4 c = launch_acc[p];
    a.x += c.x; a.y += c.y; a.z += c.z;
    accum[p] = a;
}

template <typename K>
cudaError_t optin(K kernel) { return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxStagedBytes); }

cudaError_t ensure_optin() {
    // the attribute is per DEVICE: a process may hold contexts on several GPUs (rt_create_multi), used from several host threads
    static bool done_on[64] = {false};
    static std::mutex mu;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    bool& done = done_on[dev & 63];
    if (done) return cudaSuccess;
#define RTB_WF_OPTIN(K) \
    if ((e = optin(K<0>)) != cudaSuccess) return e; if ((e = optin(K<1>)) != cudaSuccess) return e; \
    if ((e = optin(K<2>)) != cudaSuccess) return e; if ((e = optin(K<3>)) != cudaSuccess) return e; \
    if ((e = optin(K<4>)) != cudaSuccess) return e;
    RTB_WF_OPTIN(k_wf_intersect)
    if ((e = optin(k_wf_intersect_bvh<2>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_intersect_bvh<3>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_intersect_bvh<2, true>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_intersect_bvh<3, true>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_intersect_bvh<3, false, true>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_intersect_bvh<3, true, true>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_stream<3, true, false, true>)) != cudaSuccess) return e; if ((e = optin(k_wf_stream<3, false, false, true>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_stream<3, true, true, true>)) != cudaSuccess) return e; if ((e = optin(k_wf_stream<3, false, true, true>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_intersect_bvh8)) != cudaSuccess) return e;
    if ((e = optin(k_wf_stream<2, true, false>)) != cudaSuccess) return e; if ((e = optin(k_wf_stream<2, false, false>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_stream<3, true, false>)) != cudaSuccess) return e; if ((e = optin(k_wf_stream<3, false, false>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_stream<2, true, true>)) != cudaSuccess) return e; if ((e = optin(k_wf_stream<2, false, true>)) != cudaSuccess) return e;
    if ((e = optin(k_wf_stream<3, true, true>)) != cudaSuccess) return e; if ((e = optin(k_wf_stream<3, false, true>)) != cudaSuccess) return e;
#undef RTB_WF_OPTIN
    done = true;
    return cudaSuccess;
}

}  // namespace

WavefrontBuffers* wavefront_create() { return new WavefrontBuffers(); }

// frees the path state (everything that scales with the wave); the small counter block stays
void wavefront_release(WavefrontBuffers* wb) {
    if (!wb) return;
    DeviceArray<unsigned int> counters = std::move(wb->counters);
    *wb = WavefrontBuffers();
    wb->counters = std::move(counters);
}

void wavefront_destroy(WavefrontBuffers* wb) { delete wb; }

namespace {
// every per-path array for `n` paths, or none of them on failure (launch_acc, the per-pixel sum, stays)
cudaError_t alloc_paths(WavefrontBuffers* wb, size_t n) {
    return reserve_all(n, wb->ray_o[0], wb->ray_d[0], wb->thr[0], wb->rad[0], wb->ray_o[1], wb->ray_d[1], wb->thr[1], wb->rad[1],
                       wb->hit_nt, wb->hit_id, wb->wave_rad, wb->q[0], wb->q[1]);
}
}  // namespace

cudaError_t launch_render_wavefront(WavefrontBuffers* wb, const SceneView& sc, const AccelSel& ac, const FrameView& fr,
                                    float4* accum, uint32_t s_begin, int n_samples, const PrimCache* prim_cache, unsigned long long* seg_counter,
                                    cudaStream_t st, bool bvh_refill, int k_refill, int k_node_min, int wave_mpaths, bool count_traversal, bool streaming) {
    if (k_refill < 1) k_refill = 1; if (k_refill > 32) k_refill = 32;
    if (k_node_min < 1) k_node_min = 1; if (k_node_min > 32) k_node_min = 32;
    if (n_samples <= 0) return cudaSuccess;
    const bool reuse = prim_cache != nullptr;
    const float4* prim_nt = reuse ? prim_cache->nt : nullptr;
    const int* prim_id = reuse ? prim_cache->id : nullptr;
    cudaError_t e = ensure_optin();
    if (e != cudaSuccess) return e;
    const WaveGeom g = wave_geom(fr.width, fr.height);
    const size_t npix = (size_t)fr.width * fr.height;
    // Samples per wave. The late bounce rounds of a wave hold a few per cent of its paths, and a persistent intersect kernel
    // needs ~150 k rays just to fill the machine once, so small waves spend most of their rounds in the tail: on the
    // 1 M-triangle mesh at 1080p 8 M / 34 M / 136 M paths per wave give 3.1 / 4.7 / 5.4 G segments/s (profiles/r1A_wave_sweep.log).
    // Default 128 M paths (172 B each, ~22 GB), at most 64 samples per pixel, never more than a third of the free memory; if
    // the allocation fails all the same (another context or process took the memory) the wave is halved until it fits.
    size_t wave_paths = (size_t)(wave_mpaths >= 1 && wave_mpaths <= 1024 ? wave_mpaths : 128) << 20;
    if (const char* wp = getenv("RTB200_WAVE_MPATHS")) { const long v = atol(wp); if (v >= 1 && v <= 1024) wave_paths = (size_t)v << 20; }
    size_t sb; const int mode = pick_mode(sc, ac, sb);
    // the streaming kernel walks the binary BVH; other back ends fall back to the bounce-round kernels (identical results)
    streaming = streaming && (mode == 2 || mode == 3) && !ac.bvh.wnodes;
    const size_t bytes_per_path = streaming ? sizeof(float4) : kBytesPerPath;
    {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
            const size_t have = streaming ? wb->wave_rad.capacity() * sizeof(float4) : wb->paths() * kBytesPerPath;
            const size_t budget = (free_b + have) / 3 / bytes_per_path;
            if (wave_paths > budget) wave_paths = budget;
        }
    }
    int s_cap = (int)(wave_paths / (size_t)g.npad);
    if (s_cap < 1) s_cap = 1;
    if (s_cap > 64) s_cap = 64;
    if (s_cap > n_samples) s_cap = n_samples;
    // equal waves: 16 samples with room for 15 are two waves of 8, not 15 + a single-sample wave that runs mostly in its tail
    { const int n_waves = (n_samples + s_cap - 1) / s_cap; s_cap = (n_samples + n_waves - 1) / n_waves; }
    if ((size_t)g.npad * s_cap >= (size_t)1 << 32) return cudaErrorInvalidValue;
    if (wb->launch_acc.capacity() < npix) {
        cudaStreamSynchronize(st);
        if ((e = wb->launch_acc.reserve(npix)) != cudaSuccess) return e;
    }
    if ((streaming ? wb->wave_rad.capacity() : wb->paths()) < (size_t)g.npad * s_cap) {
        cudaStreamSynchronize(st);
        for (;;) {
            // the streaming kernel needs only the finished radiance per path
            e = streaming ? wb->wave_rad.reserve((size_t)g.npad * s_cap) : alloc_paths(wb, (size_t)g.npad * s_cap);
            if (e == cudaSuccess) break;
            if (e != cudaErrorMemoryAllocation || s_cap == 1) return e;      // s_cap == 1: not even one sample per pixel fits
            s_cap = (s_cap + 1) / 2;
        }
    }
    if (getenv("RTB200_DEBUG")) {
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        fprintf(stderr, "[rtb200] wavefront launch: %d samples, %d per wave (%zu M paths, %s), free %.1f of %.1f GB\n", n_samples, s_cap, ((size_t)g.npad * s_cap) >> 20,
                streaming ? "streaming" : "bounce rounds", free_b / 1e9, total_b / 1e9);
    }
    if ((e = wb->counters.reserve(2 * kMaxRounds)) != cudaSuccess) return e;
    const int rounds = reuse ? fr.max_bounces : fr.max_bounces + 1;
    if (!streaming && rounds > kMaxRounds - 1) return cudaErrorInvalidValue;      // one queue counter per bounce round; the streaming kernel has no rounds

    int device = 0, sms = 0;
    cudaGetDevice(&device);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const int persistent_blocks = sms * 8;
    const bool count = count_traversal && (mode == 2 || mode == 3) && bvh_refill && !ac.bvh.wnodes;

    if ((e = cudaMemsetAsync(wb->launch_acc.get(), 0, npix * sizeof(float4), st)) != cudaSuccess) return e;
    for (int s0 = 0; s0 < n_samples; s0 += s_cap) {
        const int sw = n_samples - s0 < s_cap ? n_samples - s0 : s_cap;
        const uint32_t s_first = s_begin + (uint32_t)s0;
        const size_t np = (size_t)g.npad * sw;
        if ((e = cudaMemsetAsync(wb->counters.get(), 0, 2 * kMaxRounds * sizeof(unsigned int), st)) != cudaSuccess) return e;
        if (streaming) {
            // one persistent launch per wave: paths are claimed from counters[0], traced and shaded to the end in the kernel
            const size_t ssb = sb + (size_t)((kStreamStateWords * kThreads + 3) / 4) * sizeof(float4);
            const int blocks = sms * RTB_WF_STREAM_MIN_BLOCKS;
#define RTB_STREAM_ARGS sc, ac.bvh, ac.flat, fr, g.tiles_x, g.npad, s_first, (unsigned int)np, prim_nt, prim_id, wb->wave_rad.get(), wb->counters.get(), k_refill, k_node_min, seg_counter
#define RTB_STREAM_LAUNCH(M, Q)                                                                                                     \
            if (reuse) { if (count) k_wf_stream<M, true, true, Q><<<blocks, kThreads, ssb, st>>>(RTB_STREAM_ARGS);                  \
                         else k_wf_stream<M, true, false, Q><<<blocks, kThreads, ssb, st>>>(RTB_STREAM_ARGS); }                    \
            else { if (count) k_wf_stream<M, false, true, Q><<<blocks, kThreads, ssb, st>>>(RTB_STREAM_ARGS);                       \
                   else k_wf_stream<M, false, false, Q><<<blocks, kThreads, ssb, st>>>(RTB_STREAM_ARGS); }
            if (mode == 2) { RTB_STREAM_LAUNCH(2, false) } else if (ac.bvh.qnodes) { RTB_STREAM_LAUNCH(3, true) } else { RTB_STREAM_LAUNCH(3, false) }
#undef RTB_STREAM_LAUNCH
#undef RTB_STREAM_ARGS
            k_wf_accumulate<<<(g.npad + 255) / 256, 256, 0, st>>>(fr, g.tiles_x, g.npad, sw, wb->wave_rad.get(), wb->launch_acc.get());
            continue;
        }
        const int gen_blocks = (int)((np + 255) / 256);
        if (reuse) k_wf_generate<true><<<gen_blocks, 256, 0, st>>>(sc, fr, g.tiles_x, g.npad, s_first, sw, prim_nt, prim_id, wb->ray_o[0].get(), wb->ray_d[0].get(),
                                                                    wb->thr[0].get(), wb->rad[0].get(), wb->wave_rad.get(), wb->q[0].get(), wb->counters.get(), seg_counter);
        else k_wf_generate<false><<<gen_blocks, 256, 0, st>>>(sc, fr, g.tiles_x, g.npad, s_first, sw, prim_nt, prim_id, wb->ray_o[0].get(), wb->ray_d[0].get(),
                                                               wb->thr[0].get(), wb->rad[0].get(), wb->wave_rad.get(), wb->q[0].get(), wb->counters.get(), seg_counter);
        for (int r = 0; r < rounds; ++r) {
            const int a = r & 1, b = a ^ 1;                  // this round's dense state set, the next round's
            const uint32_t* qin = wb->q[a].get();
            uint32_t* qout = wb->q[b].get();
            unsigned int* cnt = wb->counters.get() + r;
            unsigned int* cur = wb->counters.get() + kMaxRounds + r;
#define RTB_WF_ARGS sc, ac.bvh, ac.flat, qin, cnt, cur, wb->ray_o[a].get(), wb->ray_d[a].get(), wb->hit_nt.get(), wb->hit_id.get()
            switch (mode) {
                case 0: k_wf_intersect<0><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS); break;
                case 1: k_wf_intersect<1><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS); break;
                case 2: if (count) k_wf_intersect_bvh<2, true><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS, k_refill, k_node_min, seg_counter);
                        else if (bvh_refill) k_wf_intersect_bvh<2><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS, k_refill, k_node_min, seg_counter);
                        else k_wf_intersect<2><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS);
                        break;
                case 3: if (bvh_refill && ac.bvh.wnodes) k_wf_intersect_bvh8<<<sms * RTB_WF_BVH8_MIN_BLOCKS, kThreads, sb, st>>>(sc, ac.bvh, qin, cnt, cur, wb->ray_o[a].get(), wb->ray_d[a].get(), wb->hit_nt.get(), wb->hit_id.get(), k_refill, k_node_min);
                        else if (count && ac.bvh.qnodes) k_wf_intersect_bvh<3, true, true><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS, k_refill, k_node_min, seg_counter);
                        else if (count) k_wf_intersect_bvh<3, true><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS, k_refill, k_node_min, seg_counter);
                        else if (bvh_refill && ac.bvh.qnodes) k_wf_intersect_bvh<3, false, true><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS, k_refill, k_node_min, seg_counter);
                        else if (bvh_refill) k_wf_intersect_bvh<3><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS, k_refill, k_node_min, seg_counter);
                        else k_wf_intersect<3><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS);
                        break;
                default: k_wf_intersect<4><<<persistent_blocks, kThreads, sb, st>>>(RTB_WF_ARGS); break;
            }
#undef RTB_WF_ARGS
            k_wf_shade<<<sms * 8, 256, 0, st>>>(sc, fr, g.tiles_x, g.npad, s_first, qin, cnt, qout, cnt + 1, wb->ray_o[a].get(), wb->ray_d[a].get(), wb->thr[a].get(), wb->rad[a].get(), wb->ray_o[b].get(), wb->ray_d[b].get(), wb->thr[b].get(), wb->rad[b].get(),
                                                 wb->hit_nt.get(), wb->hit_id.get(), wb->wave_rad.get(), seg_counter);
        }
        k_wf_accumulate<<<(g.npad + 255) / 256, 256, 0, st>>>(fr, g.tiles_x, g.npad, sw, wb->wave_rad.get(), wb->launch_acc.get());
    }
    k_wf_commit<<<(int)((npix + 255) / 256), 256, 0, st>>>((int)npix, wb->launch_acc.get(), accum);
    return cudaGetLastError();
}

}  // namespace rtb
