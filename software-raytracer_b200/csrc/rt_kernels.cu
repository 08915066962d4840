// rt_kernels.cu - hand-written CUDA kernels for sm_100a: primary visibility, the path-tracing
// render kernel (persistent-lane megakernel with in-register sample regeneration), preview
// shading, resolve, and the small test-hook kernels.
//
// Compiled with -fmad=false (see rt_device.cuh for the parity rules).
#include "rt_kernels.h"

#include <cstdlib>
#include <atomic>
#include <mutex>

#include "rt_device.cuh"
#include "rt_filter.cuh"
#include "rt_resolve.cuh"
#include "rt_trace.cuh"

namespace rtb {

namespace {

__device__ __forceinline__ bool tile_pixel(const FrameView& fr, int& px, int& py) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    px = blockIdx.x * kTileW + (warp & 1) * 8 + (lane & 7);
    py = blockIdx.y * kTileH + (warp >> 1) * 4 + (lane >> 3);
    return px < fr.width && py < fr.height;
}

// ---- primary visibility AOVs ----------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(kThreads) k_primary_aov(SceneView sc, BvhView bv, FlatView fl, FrameView fr, int* __restrict__ out_id,
                                                           float* __restrict__ out_t, float* __restrict__ out_n,
                                                           float* __restrict__ out_p) {
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);
    int px, py;
    if (!tile_pixel(fr, px, py)) return;
    const size_t p = (size_t)px + (size_t)py * fr.width;
    Hit h = trace<MODE>(sc, tc, fr.cam_pos, ray_dir(fr, px, py));
    if (out_id) out_id[p] = h.id;
    if (out_t) out_t[p] = h.t;
    if (out_n) { out_n[3 * p] = h.n.x; out_n[3 * p + 1] = h.n.y; out_n[3 * p + 2] = h.n.z; }
    if (out_p) { out_p[3 * p] = h.p.x; out_p[3 * p + 1] = h.p.y; out_p[3 * p + 2] = h.p.z; }
}

__global__ void k_ray_dirs(FrameView fr, float* __restrict__ out) {
    int px = blockIdx.x * blockDim.x + threadIdx.x, py = blockIdx.y;
    if (px >= fr.width) return;
    float3 d = ray_dir(fr, px, py);
    size_t p = (size_t)px + (size_t)py * fr.width;
    out[3 * p] = d.x; out[3 * p + 1] = d.y; out[3 * p + 2] = d.z;
}

// rt_read_sample_dirs: the primary direction of global sample `sample` of every pixel, as the jittered render kernels draw it
__global__ void k_sample_dirs(FrameView fr, PixelFilter pf, uint32_t sample, float* __restrict__ out) {
    int px = blockIdx.x * blockDim.x + threadIdx.x, py = blockIdx.y;
    if (px >= fr.width) return;
    const uint32_t pixel = (uint32_t)px + (uint32_t)py * (uint32_t)fr.width;
    float3 d = filtered_ray_dir(fr, pf, px, py, pixel, sample);
    out[3 * (size_t)pixel] = d.x; out[3 * (size_t)pixel + 1] = d.y; out[3 * (size_t)pixel + 2] = d.z;
}

template <int MODE, bool COUNT = false>
__global__ void __launch_bounds__(kThreads) k_trace_rays(SceneView sc, BvhView bv, FlatView fl, const float* __restrict__ org,
                                                          const float* __restrict__ dir, int n,
                                                          int* __restrict__ out_id, float* __restrict__ out_t,
                                                          float* __restrict__ out_n, float* __restrict__ out_p,
                                                          unsigned long long* __restrict__ counters) {
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    TravCount cnt = {0u, 0u, 0u, 0u};
    if (i < n) {
        Hit h = trace<MODE, COUNT>(sc, tc, f3(org[3 * i], org[3 * i + 1], org[3 * i + 2]),
                                   f3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]), &cnt);
        out_id[i] = h.id; out_t[i] = h.t;
        out_n[3 * i] = h.n.x; out_n[3 * i + 1] = h.n.y; out_n[3 * i + 2] = h.n.z;
        out_p[3 * i] = h.p.x; out_p[3 * i + 1] = h.p.y; out_p[3 * i + 2] = h.p.z;
    }
    if (COUNT) flush_trav_count(cnt, i < n ? 1u : 0u, counters);
}

// ---- the per-pixel primary-hit cache (RT_OPT_PRIMARY_REUSE) ------------------------------------------------------
// GetRayDirection shoots every sample of a pixel through the pixel CORNER (no jitter, Raytracer.cpp:106-122), so the primary
// closest-hit query of a pixel has the same inputs - and the same result - for every sample of every frame until the camera,
// the scene, the resolution or the environment colours change. It is traced ONCE, here, into (normal, t) + object id per pixel
// (20 B, y-up row-major like the accumulation buffer; a miss keeps GetEnvironmentColor(d) instead of the normal); the render
// kernels start every sample from it. counters[2..3] (queries executed) += pixels.
template <int MODE>
__global__ void __launch_bounds__(kThreads) k_primary_cache(SceneView sc, BvhView bv, FlatView fl, FrameView fr, float4* __restrict__ prim_nt,
                                                             int* __restrict__ prim_id, unsigned long long* __restrict__ counters) {
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);
    int px, py;
    if (tile_pixel(fr, px, py)) {
        const size_t p = (size_t)px + (size_t)py * fr.width;
        const float3 d = ray_dir(fr, px, py);
        const Hit h = trace<MODE>(sc, tc, fr.cam_pos, d);
        // a pixel whose primary ray misses has ONE radiance for every sample of every frame: the environment colour of its ray is
        // kept in place of the normal (rt_device.cuh primary_ends), so that a sky pixel costs a load, not two SFU powers, per call
        const float3 v = h.id >= 0 ? h.n : env_color(fr, d);
        prim_nt[p] = make_float4(v.x, v.y, v.z, h.t);
        prim_id[p] = h.id;
    }
    if (threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) {
        atomicAdd(counters + 2, (unsigned long long)fr.width * fr.height); atomicAdd(counters + 3, (unsigned long long)fr.width * fr.height);
    }
}
// the cached primary hit of a pixel as the closest-hit functions return it (hit point = o + d * t, Object.hpp:136 / :229)
__device__ __forceinline__ Hit cached_primary(const PrimCache& pc, uint32_t pixel, float3 o, float3 d) {
    const float4 nt = __ldg(pc.nt + pixel);
    Hit h;
    h.id = __ldg(pc.id + pixel); h.t = nt.w; h.n = f3(nt.x, nt.y, nt.z);
    h.p = h.id >= 0 ? f3(o.x + d.x * nt.w, o.y + d.y * nt.w, o.z + d.z * nt.w) : f3(0.f, 0.f, 0.f);
    return h;
}

__global__ void k_env_color(FrameView fr, const float* __restrict__ dir, int n, float* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float3 c = env_color(fr, f3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]));
    out[3 * i] = c.x; out[3 * i + 1] = c.y; out[3 * i + 2] = c.z;
}

template <int MODE>
__global__ void __launch_bounds__(kThreads) k_pick(SceneView sc, BvhView bv, FlatView fl, FrameView fr, int px, int py, int* out_id) {
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);       // all threads stage; thread 0 traces the one ray
    if (threadIdx.x == 0) *out_id = trace<MODE>(sc, tc, fr.cam_pos, ray_dir(fr, px, py)).id;
}

__global__ void k_selftest_uniform(int* failures) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;       // 32768 threads
    const uint32_t w = k << 17;
    if (__float_as_uint(unit_from_word(w)) != __float_as_uint(unit_from_word_div(w))) atomicAdd(failures, 1);
}

// normalized3() (shared reciprocal) against normalized3_div() (three IEEE divisions) on 64 vectors per thread: components uniform in
// [-1, 1] like the sampler's, products of those with random powers of two across and beyond the fast path's range (2^-56 .. 2^56),
// mantissas of all ones / all zeros / one bit, exact zeros. Bits must be equal, NaN patterns included.
__global__ void k_selftest_normalize(int* failures, uint32_t seed) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    int bad = 0;
    for (uint32_t it = 0; it < 64u; ++it) {
        const uint4 w = philox4x32_10(tid, it, 0u, 0u, seed, 0x5e1f7e57u);
        float v[3];
        const uint32_t ws[3] = {w.x, w.y, w.z};
        const uint32_t kind = w.w & 7u;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const uint32_t u = ws[k];
            float f = (unit_from_word(u) - 0.5f) * 2.f;                              // the sampler's own values
            if (kind >= 2u) f = __uint_as_float((u & 0x807fffffu) | ((127u - 56u + ((u >> 23) % 113u)) << 23));   // random sign, mantissa, exponent
            if (kind == 5u) f = __uint_as_float((__float_as_uint(f) & 0xff800000u) | ((u & 0x00800000u) ? 0x007fffffu : 0u));
            if (kind == 6u) f = __uint_as_float((__float_as_uint(f) & 0xff800000u) | (1u << (u % 23u)));
            if (kind == 7u && (w.w >> 3) % 3u == (uint32_t)k) f = (u & 1u) ? 0.f : -0.f;
            v[k] = f;
        }
        if (kind == 3u) { v[1] = v[0] * 0x1p-20f; v[2] = v[0] * 0x1p-38f; }          // very different magnitudes
        if (kind == 4u) { const float sc = __uint_as_float((127u - 30u + (w.w >> 8) % 61u) << 23); v[0] *= sc; v[1] *= sc; v[2] *= sc; }
        const float3 a = normalized3(f3(v[0], v[1], v[2])), b = normalized3_div(f3(v[0], v[1], v[2]));
        if (__float_as_uint(a.x) != __float_as_uint(b.x) || __float_as_uint(a.y) != __float_as_uint(b.y) || __float_as_uint(a.z) != __float_as_uint(b.z)) ++bad;
    }
    if (bad) atomicAdd(failures, bad);
}

// The packed pair ops (add2 / sub2 / mul2 / fma2: add / sub / mul / fma.rn.f32x2) against the scalar .rn ops, half by half, on 2^26
// operand sets per call. Each operand draws its own kind - any bit pattern (NaN and infinities included), subnormals, +-0 / +-inf /
// +-FLT_MAX / +-smallest normal, exponents near overflow and near underflow, ordinary magnitudes, the sampler's values, edge mantissas -
// so mixed exponents come from mixing kinds; one set in eight makes c cancel a * b exactly. Bits must be equal; two NaNs count as equal.
__device__ __forceinline__ float selftest_operand(uint32_t u, uint32_t kind) {
    const uint32_t sign = u & 0x80000000u;
    switch (kind & 7u) {
    case 0u: return __uint_as_float(u);
    case 1u: return __uint_as_float(u & 0x807fffffu);                                              // subnormal or zero
    case 2u: {
        const uint32_t special[8] = {0u, 0x7f800000u, 0x7f7fffffu, 0x00800000u, 0x00000001u, 0x3f800000u, 0x7f000000u, 0x00ffffffu};
        return __uint_as_float(sign | special[(u >> 8) & 7u]);
    }
    case 3u: return __uint_as_float(sign | ((250u + (u >> 23) % 5u) << 23) | (u & 0x007fffffu));      // near overflow
    case 4u: return __uint_as_float(sign | ((1u + (u >> 23) % 24u) << 23) | (u & 0x007fffffu));       // just above the subnormals
    case 5u: return __uint_as_float(sign | ((97u + (u >> 23) % 61u) << 23) | (u & 0x007fffffu));      // 2^-30 .. 2^30
    case 6u: return (unit_from_word(u) - 0.5f) * 2.f;                                                 // the sampler's own values
    default: return __uint_as_float(sign | ((u >> 8) & 0x7f800000u) | ((u & 1u) ? 0x007fffffu : (1u << (u % 23u))));
    }
}
__device__ __forceinline__ bool same_bits(float a, float b) { return __float_as_uint(a) == __float_as_uint(b) || (a != a && b != b); }
__global__ void k_selftest_packed(int* failures, uint32_t seed) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    int bad = 0;
    for (uint32_t it = 0; it < 64u; ++it) {
        const uint4 w0 = philox4x32_10(tid, it, 0u, 0u, seed, 0x9ac4ed2fu), w1 = philox4x32_10(tid, it, 1u, 0u, seed, 0x9ac4ed2fu);
        const uint32_t k = w1.w;
        const fpair a = fp(selftest_operand(w0.x, k), selftest_operand(w0.y, k >> 3));
        const fpair b = fp(selftest_operand(w0.z, k >> 6), selftest_operand(w0.w, k >> 9));
        fpair c = fp(selftest_operand(w1.x, k >> 12), selftest_operand(w1.y, k >> 15));
        if (((k >> 18) & 7u) == 0u) c = fp(-__fmul_rn(a.x, b.x), -__fmul_rn(a.y, b.y));           // exact cancellation in the fma
        const fpair s = add2(a, b), d = sub2(a, b), m = mul2(a, b), f = fma2(a, b, c);
        bad += !same_bits(s.x, __fadd_rn(a.x, b.x)) + !same_bits(s.y, __fadd_rn(a.y, b.y));
        bad += !same_bits(d.x, __fsub_rn(a.x, b.x)) + !same_bits(d.y, __fsub_rn(a.y, b.y));
        bad += !same_bits(m.x, __fmul_rn(a.x, b.x)) + !same_bits(m.y, __fmul_rn(a.y, b.y));
        bad += !same_bits(f.x, __fmaf_rn(a.x, b.x, c.x)) + !same_bits(f.y, __fmaf_rn(a.y, b.y, c.y));
    }
    if (bad) atomicAdd(failures, bad);
}

__global__ void k_philox(uint4 ctr, uint2 key, uint4* out) { *out = philox4x32_10(ctr.x, ctr.y, ctr.z, ctr.w, key.x, key.y); }

// ---- the render kernel -----------------------------------------------------------------------
// One lane owns one pixel for the whole launch and walks its samples [s_begin, s_begin+n) in
// order. The loop is flat over path SEGMENTS: every iteration does one closest-hit query (the
// ~90 % part) and a short divergent shading tail. A lane whose path ends starts its next sample
// in the same iteration slot ("regeneration"), so the warp stays full until a lane runs out of
// samples; with many samples per launch the per-lane totals converge (law of large numbers) and
// neighbouring pixels finish together. Per-pixel sums are kept in registers in sample order and
// added to the float4 accumulation buffer once - no atomics, bit-reproducible for a given
// (seed, sample range), independent of the launch shape.
//
// REUSE (primary-hit reuse): the primary closest-hit query of a pixel has the same inputs - and the same
// result - for every sample (k_primary_cache above). With REUSE every sample starts from the cached hit:
// it still draws its own Philox block there and scatters its own secondary ray, so every sample's radiance
// is bit-identical to the non-reuse loop (asserted by the tests). A pixel whose primary ray misses (or
// max_bounces == 0) has the same value for every sample: the value is added n times, in order.
// seg_counter[0..1] count path segments DELIVERED (what the reference traces), seg_counter[2..3] the
// closest-hit queries actually EXECUTED (with REUSE: the secondary and later segments; the cache pass adds its own).
// STASH (REUSE only): the pixel's cached primary hit and direction wait in shared memory for the next sample instead of in ten registers
// across the closest-hit query, which brings the kernel to 72 registers = 7 CTAs per SM. The stash costs 1.5 % at equal occupancy and
// the seventh CTA gives 4 %: Scene1 1080p 1024 spp 108.2 -> 105.5 ms; a 640x480 launch (2400 CTAs: 2.3 instead of 2.7 waves, the last
// as long and emptier) loses 4 %, so the launcher takes this form for large grids only (profiles/r4u_ab_stash.txt). Same bits.
//
// JITTER (a pixel filter, rt_filter.cuh; never with REUSE): every sample starts from its own primary direction, filtered_ray_dir() of its
// global sample index, instead of the pixel's corner ray d0 - the non-reuse loop with a different d0. k_render_regen_aa below.
template <int MODE, bool REUSE, bool COUNT, bool STASH, bool JITTER>
__device__ __forceinline__ void render_regen(const SceneView& sc, const BvhView& bv, const FlatView& fl, const FrameView& fr, float4* __restrict__ accum,
                                             uint32_t s_begin, int n_samples, const PrimCache& prim, unsigned long long* __restrict__ seg_counter,
                                             const PixelFilter& pf) {
    static_assert(!(JITTER && REUSE), "a jittered primary ray is not the cached one");
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);
    int px, py;
    const bool inside = tile_pixel(fr, px, py);              // no early return: the warp reduce below needs every lane
    const uint32_t pixel = inside ? (uint32_t)px + (uint32_t)py * (uint32_t)fr.width : 0u;
    if (!inside) n_samples = 0;

    const float3 d0 = JITTER ? f3(0.f, 0.f, 0.f) : ray_dir(fr, px, py);
    float3 acc = f3(0.f, 0.f, 0.f);
    float3 o = fr.cam_pos, d = JITTER ? filtered_ray_dir(fr, pf, px, py, pixel, s_begin) : d0;
    float3 T = f3(0.f, 0.f, 0.f), L = f3(0.f, 0.f, 0.f);
    int s = 0, depth = 0;
    unsigned int segs = 0, traced = 0;

    // REUSE prologue: the pixel's cached primary hit. A miss (or max_bounces == 0) consumes no random number, so
    // every sample of the pixel has the same value: add it n times, in order, and the lane is done.
    Hit h0;
    h0.id = -1; h0.t = 0.f; h0.n = f3(0.f, 0.f, 0.f); h0.p = f3(0.f, 0.f, 0.f);
    TravCount cnt = {0u, 0u, 0u, 0u};
    static_assert(!STASH || REUSE, "the stash holds the cached primary hit");
    __shared__ float stash[STASH ? 10 * kThreads : 1];
    float* const st = stash + (STASH ? threadIdx.x : 0);
    if (REUSE) {
        if (n_samples > 0) {
            h0 = cached_primary(prim, pixel, o, d);
            if (STASH) {
                st[0] = h0.p.x; st[kThreads] = h0.p.y; st[2 * kThreads] = h0.p.z; st[3 * kThreads] = h0.n.x; st[4 * kThreads] = h0.n.y; st[5 * kThreads] = h0.n.z;
                st[6 * kThreads] = __int_as_float(h0.id); st[7 * kThreads] = d0.x; st[8 * kThreads] = d0.y; st[9 * kThreads] = d0.z;
            }
            float3 c;
            if (primary_ends(sc, fr, h0, c)) {
                for (; s < n_samples; ++s) { acc.x += c.x; acc.y += c.y; acc.z += c.z; }
                segs = (unsigned int)n_samples;
            } else {
                scatter_segment(sc, fr, h0, pixel, s_begin, o, d, T, L, depth);
                segs = 1;
            }
        }
    }
    // Main loop: one closest-hit query per lane per iteration, then ONE pass through each shading block - the
    // flag (instead of continue/break) lets the warp reconverge before the scatter block.
    while (__any_sync(0xffffffffu, s < n_samples)) {
        const bool live = s < n_samples;                     // lanes that are done keep serving the others in MODE 5
        Hit h = trace_all<MODE, COUNT>(sc, tc, o, d, live, &cnt);
        if (live) {
            ++segs; ++traced;
            bool scatter = true;
            float3 c;
            if (path_ends(sc, fr, h, d, T, L, depth, c)) {
                acc.x += c.x; acc.y += c.y; acc.z += c.z;
                ++s; depth = 0; o = fr.cam_pos;
                scatter = false;                             // no reuse: trace the primary ray again
                if (STASH) {
                    d = f3(st[7 * kThreads], st[8 * kThreads], st[9 * kThreads]);
                    if (s < n_samples) {                     // next sample starts from the cached primary hit (scatter_segment reads id, n, p)
                        h.p = f3(st[0], st[kThreads], st[2 * kThreads]); h.n = f3(st[3 * kThreads], st[4 * kThreads], st[5 * kThreads]);
                        h.id = __float_as_int(st[6 * kThreads]); h.t = 0.f;
                        ++segs; scatter = true;
                    }
                } else {
                    d = JITTER ? filtered_ray_dir(fr, pf, px, py, pixel, s_begin + (uint32_t)s) : d0;
                    if (REUSE && s < n_samples) { h = h0; ++segs; scatter = true; }   // next sample starts from the cached primary hit
                }
            }
            if (scatter) scatter_segment(sc, fr, h, pixel, s_begin + (uint32_t)s, o, d, T, L, depth);
        }
    }

    if (inside) {
        float4 a = accum[pixel];
        a.x += acc.x; a.y += acc.y; a.z += acc.z;
        accum[pixel] = a;
    }

    // segment counts: warp reduce, one atomic per warp and counter
    unsigned int total = segs, total_tr = traced;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        total += __shfl_down_sync(0xffffffffu, total, off);
        total_tr += __shfl_down_sync(0xffffffffu, total_tr, off);
    }
    if ((threadIdx.x & 31) == 0 && total) {
        atomicAdd(seg_counter, (unsigned long long)total); atomicAdd(seg_counter + 1, (unsigned long long)total);
        atomicAdd(seg_counter + 2, (unsigned long long)total_tr); atomicAdd(seg_counter + 3, (unsigned long long)total_tr);
    }
    if (COUNT) flush_trav_count(cnt, traced, seg_counter);
}
template <int MODE, bool REUSE, bool COUNT = false, bool STASH = false>
__global__ void __launch_bounds__(kThreads, STASH ? RTB_REGEN_STASH_BLOCKS : RTB_REGEN_MIN_BLOCKS) k_render_regen(SceneView sc, BvhView bv, FlatView fl, FrameView fr, float4* __restrict__ accum,
                                                            uint32_t s_begin, int n_samples, PrimCache prim,
                                                            unsigned long long* __restrict__ seg_counter) {
    render_regen<MODE, REUSE, COUNT, STASH, false>(sc, bv, fl, fr, accum, s_begin, n_samples, prim, seg_counter, PixelFilter{kFilterNone, 0.f});
}
// the same loop with a pixel filter: one jittered primary ray per sample (no primary-hit reuse)
template <int MODE, bool COUNT = false>
__global__ void __launch_bounds__(kThreads, RTB_REGEN_MIN_BLOCKS) k_render_regen_aa(SceneView sc, BvhView bv, FlatView fl, FrameView fr, float4* __restrict__ accum,
                                                                                    uint32_t s_begin, int n_samples,
                                                                                    unsigned long long* __restrict__ seg_counter, PixelFilter pf) {
    render_regen<MODE, false, COUNT, false, true>(sc, bv, fl, fr, accum, s_begin, n_samples, PrimCache{nullptr, nullptr}, seg_counter, pf);
}

// ---- resolve: sum/count -> Reinhard -> truncating ARGB8 pack (Raytracer.cpp:73-75): resolve_pixel() in rt_resolve.cuh ----------
// ---- frame fused into the render (rt_render_frame) --------------------------------------------------------------------
// An interactive frame is rt_render_spp(1) + rt_resolve_rgba8: render kernel, resolve kernel, 3.7 MB (720p) over PCIe, one after the
// other - the copy alone is a third of the frame. The reference resolves every pixel the moment it is traced (SetScreenPixel inside
// renderArea, Raytracer.cpp:63-76,250). With a FrameOut the pixel-pool kernel does the same at the granularity of a warp's CHUNK (two
// tiles of 32 pixels, all traced by that warp): when the chunk's last pixel is done the warp resolves the chunk and stores its rows
// to the device surface and to the caller's page-locked surface (whole 128-byte lines over PCIe, spread over the whole render). Chunk
// bookkeeping is warp-uniform: pixels left per in-flight chunk as the eight bytes of one 64-bit register, the chunks' first tiles in
// shared memory (8 words per warp behind the trace layout).
struct FrameOut {
    uint32_t* out;         // device surface (whole image), nullptr: not fused
    uint32_t* out2;        // mapped page-locked host surface or nullptr
    float count;           // samples in the accumulation buffer after this launch
    int flip_y;
    int smem_off;          // byte offset of the kPoolSlots x (threads / 32) chunk words in dynamic shared memory
};

// ---- few samples per pixel: warp-level pixel pool -------------------------------------------------------------
// With one lane per pixel a launch of n samples keeps a warp busy for the LONGEST of its 32 pixels' work; for large
// n that averages out (29.8 of 32 lanes alive at 1024 spp), but an interactive 1-spp frame runs ~4.5 warp iterations
// for 2.1 segments per path. Here the grid is PERSISTENT (one wave of CTAs): a warp claims chunks of `pool_tiles` consecutive
// 8x4 pixel tiles from one cursor per launch (one atomicAdd per chunk, requested ahead of time) and its lanes pull PIXELS
// from the current chunk (one ballot + popcount): a lane that finishes a pixel's n samples starts the next
// pixel at once. One pixel is still traced by one lane, samples in order, one write: the same bits as k_render_regen.
// Tile shape of the pixel pool: 32 pixels, kPoolTW wide. A chunk is two tiles side by side, and its rows are what chunk_done() sends
// over PCIe in one piece: 8x4 tiles give 64-byte rows, 16x2 tiles 128-byte rows (one full line per store instruction and row).
#ifndef RTB_POOL_TILE_W
#define RTB_POOL_TILE_W 32             // measured (profiles/r2y_ab_pool_tile_shape.txt, 720p 1 spp): render alone 0.145 (8x4) / 0.142 (16x2) / 0.138 ms (32x1)
#endif
constexpr int kPoolTW = RTB_POOL_TILE_W, kPoolTH = 32 / kPoolTW;
constexpr int kPoolSlots = 8;          // chunks of one warp that may be in flight with frame output (one byte of a 64-bit register each)
static_assert(kPoolTW == 8 || kPoolTW == 16 || kPoolTW == 32, "pool tiles are 8x4, 16x2 or 32x1");
// A chunk whose last pixel finished: the warp resolves its 64 sums (L2 loads: they were written by lanes of this warp) and stores the
// rows to the device surface and to the host surface - 32 lanes at once, once per chunk. OUT of line: inlined at both retire points
// its four copies of the resolve (six IEEE divisions with their slow paths each) made the render loop 1000 instructions longer.
// (Resolving each pixel where its sum is written - for the one or two lanes that finish in a pass, in almost every pass - was worse still.)
static __device__ __noinline__ void pool_chunk_out(const float4* accum, uint32_t* out, uint32_t* out2, float count, int flip_y, int width, int height,
                                                   int tiles_x, unsigned int n_tiles, int pool_tiles, unsigned int t0, int lane) {
#pragma unroll 1
    for (int p = 0; p < 2; ++p) {                            // the chunk row-major, 2 * kPoolTW pixels per row: 32 consecutive positions per pass
        const int q = 32 * p + lane, row = q / (2 * kPoolTW), xx = q % (2 * kPoolTW);
        const unsigned int tile = t0 + (unsigned int)(xx / kPoolTW);
        if ((xx / kPoolTW) < pool_tiles && tile < n_tiles) {
            const int x = (int)(tile % (unsigned int)tiles_x) * kPoolTW + (xx % kPoolTW), y = (int)(tile / (unsigned int)tiles_x) * kPoolTH + row;
            if (x < width && y < height) {
                const uint32_t v = resolve_pixel(__ldcg(accum + ((size_t)x + (size_t)y * width)), count);
                const size_t dst = (size_t)x + (size_t)(flip_y ? height - 1 - y : y) * width;
                out[dst] = v;
                if (out2) out2[dst] = v;
            }
        }
    }
}
// The pixel-pool loop as the body of k_render_pool (JITTER false) and k_render_pool_aa (JITTER true: every sample of a pixel starts from
// its own filtered_ray_dir(), rt_filter.cuh, instead of the pixel's d0; no primary-hit reuse). A macro rather than a device function: inlined
// from a device function, the loop of the existing kernels came out with a different register allocation (the same result, other SASS).
// Expects the kernel parameters below and `pf` in scope.
#define RTB_RENDER_POOL_BODY(JITTER)                                                                                                                                                                                \
    extern __shared__ float4 smem[];                                                                                                                                                                                \
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);                                                                                                                                                        \
    constexpr unsigned FULL = 0xffffffffu;                                                                                                                                                                          \
    const int lane = threadIdx.x & 31;                                                                                                                                                                              \
    const int tiles_x = (fr.width + kPoolTW - 1) / kPoolTW, tiles_y = (fr.height + kPoolTH - 1) / kPoolTH;                                                                                                          \
    const unsigned int n_tiles = (unsigned int)tiles_x * (unsigned int)tiles_y;                                                                                                                                     \
    /* frame output (FRAME: its own instantiation, the bookkeeping costs registers; requires pool_tiles <= 2): see FrameOut */                                                                                      \
    constexpr bool fuse = FRAME;                                                                                                                                                                                    \
    unsigned int* const chunk_tile = reinterpret_cast<unsigned int*>(reinterpret_cast<unsigned char*>(smem) + fo.smem_off) + (threadIdx.x >> 5) * kPoolSlots;                                                       \
    unsigned long long left8 = 0ull;                          /* pixels not yet finished of the chunks in flight, byte (seq % kPoolSlots) */                                                                        \
    int seq_cur = -1, my_seq = 0;                             /* chunks are numbered per warp in claim order */                                                                                                     \
    /* a lane can finish two pixels in one pass: the one it was tracing, and a fresh one whose primary ray misses (or a chunk slot */                                                                               \
    /* outside the image): the chunk numbers of both, -1 = none */                                                                                                                                                  \
    int fin_a = -1, fin_b = -1;                                                                                                                                                                                     \
    uint32_t pixel = 0;                                       /* the lane's current pixel */                                                                                                                        \
    /* end of a pass: the finished pixels leave their chunks' counts; a chunk that reaches zero is resolved and sent (ONE call site) */                                                                             \
    auto retire = [&]() {                                                                                                                                                                                           \
_Pragma("unroll 1")                                                                                                                                                                                                    \
        for (int e = 0; e < 2; ++e) {                                                                                                                                                                               \
            const int mine = e ? fin_b : fin_a;                                                                                                                                                                     \
            unsigned m_fin = __ballot_sync(FULL, mine >= 0);                                                                                                                                                        \
            while (m_fin) {                                                                                                                                                                                         \
                const int sq = __shfl_sync(FULL, mine, __ffs((int)m_fin) - 1);                                                                                                                                      \
                const unsigned same = __ballot_sync(FULL, mine == sq);                                                                                                                                              \
                m_fin &= ~same;                                                                                                                                                                                     \
                const int sh = 8 * (sq & (kPoolSlots - 1));                                                                                                                                                         \
                left8 -= (unsigned long long)__popc(same) << sh;                                                                                                                                                    \
                if (((left8 >> sh) & 0xffull) == 0ull) {                                                                                                                                                            \
                    __syncwarp();                            /* the chunk's sums were written by lanes of this warp */                                                                                              \
                    pool_chunk_out(accum, fo.out, fo.out2, fo.count, fo.flip_y, fr.width, fr.height, tiles_x, n_tiles, pool_tiles, chunk_tile[sq & (kPoolSlots - 1)], lane);                                        \
                }                                                                                                                                                                                                   \
            }                                                                                                                                                                                                       \
        }                                                                                                                                                                                                           \
        fin_a = -1; fin_b = -1;                                                                                                                                                                                     \
    };                                                                                                                                                                                                              \
    /* the warp's current chunk of `pool_tiles` tiles, claimed from the launch's cursor; the NEXT chunk is requested as soon as */                                                                                  \
    /* the current one is half handed out, so the atomic's round trip overlaps the tracing (its result is first read when needed) */                                                                                \
    unsigned int tile0 = 0, claimed = 0;                                                    /* warp-uniform */                                                                                                      \
    int next = 0, total = 0;                                                                                                                                                                                        \
    bool have_claim = false, drained = false;                                                                                                                                                                       \
    bool busy = false;                                                                                                                                                                                              \
    float3 d0 = f3(0.f, 0.f, 1.f), acc = f3(0.f, 0.f, 0.f), o = fr.cam_pos, d = d0;                                                                                                                                 \
    float3 T = f3(0.f, 0.f, 0.f), L = f3(0.f, 0.f, 0.f);                                                                                                                                                            \
    int s = 0, depth = 0;                                                                                                                                                                                           \
    unsigned int segs = 0, traced = 0;                                                                                                                                                                              \
    Hit h0;                                                                                                                                                                                                         \
    h0.id = -1; h0.t = 0.f; h0.n = f3(0.f, 0.f, 0.f); h0.p = f3(0.f, 0.f, 0.f);                                                                                                                                     \
                                                                                                                                                                                                                    \
    /* One iteration: closest hit for the lanes that hold a ray -> end-of-path handling -> idle lanes (also those that finished a pixel */                                                                          \
    /* just now) take the next pixels of the chunk -> ONE scatter block for continuing paths, restarted samples and fresh pixels. */                                                                                \
    /* (The first version scattered fresh pixels inside the pick-up: a second copy of the scatter code that ran in almost every */                                                                                  \
    /* iteration for the handful of lanes that had just taken a pixel.) */                                                                                                                                          \
    for (;;) {                                                                                                                                                                                                      \
        Hit h = trace_all<MODE>(sc, tc, o, d, busy);                                                                                                                                                                \
        bool scat = false;                                                                                                                                                                                          \
        if (busy) {                                                                                                                                                                                                 \
            ++segs; ++traced;                                                                                                                                                                                       \
            float3 c;                                                                                                                                                                                               \
            if (path_ends(sc, fr, h, d, T, L, depth, c)) {                                                                                                                                                          \
                acc.x += c.x; acc.y += c.y; acc.z += c.z;                                                                                                                                                           \
                ++s; depth = 0; o = fr.cam_pos; d = d0;     /* no reuse: the next iteration traces the primary ray again */                                                                                         \
                if (JITTER && s < n_samples) d = filtered_ray_dir(fr, pf, (int)(pixel % (uint32_t)fr.width), (int)(pixel / (uint32_t)fr.width), pixel, s_begin + (uint32_t)s);                                      \
                if (s >= n_samples) {                                                                                                                                                                               \
                    float4 a = accum[pixel];                                                                                                                                                                        \
                    a.x += acc.x; a.y += acc.y; a.z += acc.z;                                                                                                                                                       \
                    accum[pixel] = a;                                                                                                                                                                               \
                    if (fuse) fin_a = my_seq;                                                                                                                                                                       \
                    busy = false;                                                                                                                                                                                   \
                } else if (REUSE) { h = h0; ++segs; scat = true; }     /* next sample from the cached primary hit */                                                                                                \
            } else scat = true;                                                                                                                                                                                     \
        }                                                                                                                                                                                                           \
        const unsigned m_need = __ballot_sync(FULL, !busy);                                                                                                                                                         \
        if (!have_claim && !drained && 2 * next >= total) {  /* ask for the next chunk early */                                                                                                                     \
            if (lane == 0) claimed = atomicAdd(tile_cursor, (unsigned int)pool_tiles);                                                                                                                              \
            have_claim = true;                                                                                                                                                                                      \
        }                                                                                                                                                                                                           \
        /* (frame output: the chunk kPoolSlots claims back must be complete before its bookkeeping slot is used again - else wait a pass. */                                                                        \
        /* With 4 slots that happened often enough - one deep path under 31 lanes racing through sky chunks - to cost 15 % of the kernel.) */                                                                       \
        if (m_need != 0u && next >= total && have_claim && !(fuse && ((left8 >> (8 * ((seq_cur + 1) & (kPoolSlots - 1)))) & 0xffull) != 0ull)) {   /* the current chunk is handed out: switch to the claimed one */ \
            tile0 = __shfl_sync(FULL, claimed, 0);                                                                                                                                                                  \
            have_claim = false;                                                                                                                                                                                     \
            if (tile0 >= n_tiles) { drained = true; total = 0; }                                                                                                                                                    \
            else { const unsigned int rem = n_tiles - tile0; total = (int)(rem < (unsigned int)pool_tiles ? rem : (unsigned int)pool_tiles) * 32; }                                                                 \
            next = 0;                                                                                                                                                                                               \
            if (fuse && total > 0) {                                                                                                                                                                                \
                ++seq_cur;                                                                                                                                                                                          \
                left8 += (unsigned long long)total << (8 * (seq_cur & (kPoolSlots - 1)));                                                                                                                           \
                if (lane == 0) chunk_tile[seq_cur & (kPoolSlots - 1)] = tile0;                                                                                                                                      \
            }                                                                                                                                                                                                       \
        }                                                                                                                                                                                                           \
        if (m_need != 0u && next < total) {                                                                                                                                                                         \
            const int idx = next + __popc(m_need & ((1u << lane) - 1u));                                                                                                                                            \
            next += __popc(m_need);                                                                                                                                                                                 \
            if (!busy && idx < total) {                                                                                                                                                                             \
                const unsigned int tile = tile0 + (unsigned int)(idx >> 5);                                                                                                                                         \
                const int px = (int)(tile % (unsigned int)tiles_x) * kPoolTW + (idx % kPoolTW), py = (int)(tile / (unsigned int)tiles_x) * kPoolTH + ((idx & 31) / kPoolTW);                                        \
                if (fuse) { my_seq = seq_cur; if (!(px < fr.width && py < fr.height)) fin_b = my_seq; }   /* nothing to trace for this slot of the chunk */                                                         \
                if (px < fr.width && py < fr.height) {                                                                                                                                                              \
                    pixel = (uint32_t)px + (uint32_t)py * (uint32_t)fr.width;                                                                                                                                       \
                    d0 = JITTER ? filtered_ray_dir(fr, pf, px, py, pixel, s_begin) : ray_dir(fr, px, py);                                                                                                           \
                    acc = f3(0.f, 0.f, 0.f); o = fr.cam_pos; d = d0; s = 0; depth = 0;                                                                                                                              \
                    busy = true;                                                                                                                                                                                    \
                    if (REUSE) {                                                                                                                                                                                    \
                        h0 = cached_primary(prim, pixel, o, d);                                                                                                                                                     \
                        float3 c;                                                                                                                                                                                   \
                        if (primary_ends(sc, fr, h0, c)) {                                                                                                                                                          \
                            /* the primary ray misses (or max_bounces == 0): every sample of the pixel has the value c */                                                                                           \
                            for (; s < n_samples; ++s) { acc.x += c.x; acc.y += c.y; acc.z += c.z; }                                                                                                                \
                            segs += (unsigned int)n_samples;                                                                                                                                                        \
                            float4 a = accum[pixel];                                                                                                                                                                \
                            a.x += acc.x; a.y += acc.y; a.z += acc.z;                                                                                                                                               \
                            accum[pixel] = a;                                                                                                                                                                       \
                            if (fuse) fin_b = my_seq;                                                                                                                                                               \
                            busy = false;                    /* takes another pixel in the next pass */                                                                                                             \
                        } else { h = h0; ++segs; scat = true; }                                                                                                                                                     \
                    }                                                                                                                                                                                               \
                }                                                                                                                                                                                                   \
            }                                                                                                                                                                                                       \
        }                                                                                                                                                                                                           \
        if (fuse) retire();                                                                                                                                                                                         \
        if (scat) scatter_segment(sc, fr, h, pixel, s_begin + (uint32_t)s, o, d, T, L, depth);                                                                                                                      \
        if (!__any_sync(FULL, busy) && drained) break;      /* not drained: the next pass switches to the claimed chunk */                                                                                          \
    }                                                                                                                                                                                                               \
                                                                                                                                                                                                                    \
    unsigned int total_s = segs, total_tr = traced;                                                                                                                                                                 \
_Pragma("unroll")                                                                                                                                                                                                   \
    for (int off = 16; off > 0; off >>= 1) {                                                                                                                                                                        \
        total_s += __shfl_down_sync(FULL, total_s, off);                                                                                                                                                            \
        total_tr += __shfl_down_sync(FULL, total_tr, off);                                                                                                                                                          \
    }                                                                                                                                                                                                               \
    if (lane == 0 && total_s) {                                                                                                                                                                                     \
        atomicAdd(seg_counter, (unsigned long long)total_s); atomicAdd(seg_counter + 1, (unsigned long long)total_s);                                                                                               \
        atomicAdd(seg_counter + 2, (unsigned long long)total_tr); atomicAdd(seg_counter + 3, (unsigned long long)total_tr);                                                                                         \
    }                                                                                                                                                                                                               \

template <int MODE, bool REUSE, bool FRAME>
__global__ void __launch_bounds__(kThreads, RTB_REGEN_MIN_BLOCKS) k_render_pool(SceneView sc, BvhView bv, FlatView fl, FrameView fr, float4* __restrict__ accum,
                                                           uint32_t s_begin, int n_samples, int pool_tiles, PrimCache prim,
                                                           unsigned int* __restrict__ tile_cursor, unsigned long long* __restrict__ seg_counter, FrameOut fo) {
    const PixelFilter pf = {kFilterNone, 0.f};
    RTB_RENDER_POOL_BODY(false)
}
// the same with a pixel filter: one jittered primary ray per sample (no primary-hit reuse)
template <int MODE, bool FRAME>
__global__ void __launch_bounds__(kThreads, RTB_REGEN_MIN_BLOCKS) k_render_pool_aa(SceneView sc, BvhView bv, FlatView fl, FrameView fr, float4* __restrict__ accum,
                                                              uint32_t s_begin, int n_samples, int pool_tiles,
                                                              unsigned int* __restrict__ tile_cursor, unsigned long long* __restrict__ seg_counter, FrameOut fo,
                                                              PixelFilter pf) {
    constexpr bool REUSE = false;
    const PrimCache prim = {nullptr, nullptr};
    RTB_RENDER_POOL_BODY(true)
}
#undef RTB_RENDER_POOL_BODY

// ---- BVH render kernel with warp-level phase scheduling ---------------------------------------
// Same lane-owns-a-pixel / regeneration scheme as k_render_regen, but the BVH traversal is an
// explicit per-lane state machine and the WARP decides what runs next, so no lane waits for the
// slowest ray of its warp:
//   NODE  one inner-node visit (two slab tests, push far child with its entry distance)
//   LEAF  one primitive test with the strict reference arithmetic
//   WAIT  traversal finished: the hit is pending shading
//   DEAD  the lane's pixel has all its samples
// Each warp iteration ballots the states and runs exactly ONE of: the shading block (when nothing is
// traversing any more, or at least `wait_k` lanes are waiting), the NODE block or the LEAF block
// (whichever has more lanes). Shaded lanes immediately get their next ray (scatter or next sample), so
// traversal runs with most lanes busy instead of the mean/max trip-count ratio of a per-ray loop.
// Results are bit-identical to the other back ends (same candidate semantics, same strict tests).
#ifndef RTB_BVH_MIN_BLOCKS
#define RTB_BVH_MIN_BLOCKS 5
#endif
template <int MODE>
__global__ void __launch_bounds__(kThreads, RTB_BVH_MIN_BLOCKS) k_render_bvh(SceneView sc, BvhView bv, FlatView fl, FrameView fr,
                                                                           float4* __restrict__ accum, uint32_t s_begin,
                                                                           int n_samples, unsigned long long* __restrict__ seg_counter,
                                                                           int wait_k) {
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);
    const float4* __restrict__ nodes = tc.nodes;
    const int* __restrict__ refs = tc.refs;
    int* const stk = tc.stack;                                   // [entry][thread] links
    float* const stk_t = tc.stack_t;                             // entry distances
    const int stride = tc.stride;
    constexpr unsigned FULL = 0xffffffffu;
    enum { NODE = 0, LEAF = 1, WAIT = 2, DEAD = 3 };

    int px, py;
    const bool inside = tile_pixel(fr, px, py);
    const uint32_t pixel = inside ? (uint32_t)px + (uint32_t)py * (uint32_t)fr.width : 0u;
    const float3 d0 = ray_dir(fr, px, py);
    float3 acc = f3(0.f, 0.f, 0.f);
    float3 o = fr.cam_pos, d = d0;
    float3 T = f3(0.f, 0.f, 0.f), L = f3(0.f, 0.f, 0.f);
    int s = 0, depth = 0;
    unsigned int segs = 0;

    // traversal state
    float ix, iy, iz, ox, oy, oz;
    float best_t; int best_id, best_ref;
    int cur = 0, li = 0, lend = 0, sp = 0;
    int st = (inside && n_samples > 0) ? NODE : DEAD;

    auto begin_ray = [&]() {
        const float big = 1e30f;
        ix = fabsf(d.x) > 1e-30f ? 1.f / d.x : copysignf(big, d.x);
        iy = fabsf(d.y) > 1e-30f ? 1.f / d.y : copysignf(big, d.y);
        iz = fabsf(d.z) > 1e-30f ? 1.f / d.z : copysignf(big, d.z);
        ox = -o.x * ix; oy = -o.y * iy; oz = -o.z * iz;
        best_t = __int_as_float(0x7f800000); best_id = 0x7fffffff; best_ref = 0;
        cur = 0; sp = 0; st = NODE;
    };
    auto enter = [&](int link) -> bool {                     // false: empty leaf, keep popping
        if (link >= 0) { cur = link; st = NODE; return true; }
        const unsigned v = (unsigned)(~link);
        const int cnt = (int)(v >> 24);
        if (cnt == 0) return false;
        li = (int)(v & 0xffffffu); lend = li + cnt; st = LEAF;
        return true;
    };
    auto pop = [&]() {
        for (;;) {
            if (sp == 0) { st = WAIT; return; }
            --sp;
            const int link = stk[sp * stride];
            const float tn = stk_t[sp * stride];
            if (tn > best_t) continue;                           // entered after the best hit found since the push
            if (enter(link)) return;
        }
    };
    if (st == NODE) begin_ray();

    int alive_cnt = __popc(__ballot_sync(FULL, st != DEAD));
    int k_eff = max(1, min(wait_k, (alive_cnt * 3) >> 2));
    for (;;) {
        const unsigned m_node = __ballot_sync(FULL, st == NODE);
        const unsigned m_leaf = __ballot_sync(FULL, st == LEAF);
        const unsigned m_wait = __ballot_sync(FULL, st == WAIT);
        if ((m_node | m_leaf) == 0u || __popc(m_wait) >= k_eff) {
            if (m_wait == 0u) break;                             // nothing traversing, nothing pending: all lanes done
            if (st == WAIT) {
                Hit h;
                h.id = -1; h.t = 0.f; h.n = f3(0.f, 0.f, 0.f); h.p = f3(0.f, 0.f, 0.f);
                if (best_id != 0x7fffffff) {
                    h.id = best_id; h.t = best_t;
                    h.p = f3(o.x + d.x * best_t, o.y + d.y * best_t, o.z + d.z * best_t);
                    if (best_ref >= 0) {
                        const float4 sp4 = tc.sph[best_ref];
                        h.n = normalized3(f3(h.p.x - sp4.x, h.p.y - sp4.y, h.p.z - sp4.z));
                    } else {                                     // cube: the normal comes out of the same test again
                        float dist; float3 nrm = f3(0.f, 0.f, 0.f);
                        box_hit(tc.box[2 * (~best_ref)], tc.box[2 * (~best_ref) + 1], o, d, dist, nrm);
                        h.n = nrm;
                    }
                }
                ++segs;
                float3 c;
                if (shade_segment(sc, fr, h, pixel, s_begin + (uint32_t)s, o, d, T, L, depth, c)) {
                    acc.x += c.x; acc.y += c.y; acc.z += c.z;
                    ++s; depth = 0; o = fr.cam_pos; d = d0;
                }
                if (s < n_samples) begin_ray(); else st = DEAD;
            }
            alive_cnt = __popc(__ballot_sync(FULL, st != DEAD));
            k_eff = max(1, min(wait_k, (alive_cnt * 3) >> 2));
            continue;
        }
        if (__popc(m_node) >= __popc(m_leaf)) {
            if (st == NODE) {
                const float4 n0 = nodes[4 * cur], n1 = nodes[4 * cur + 1], n2 = nodes[4 * cur + 2];
                const int2 ch = *reinterpret_cast<const int2*>(nodes + 4 * cur + 3);
                float a, b;
                a = fmaf(n0.x, ix, ox); b = fmaf(n0.y, ix, ox);
                float lo0 = fminf(a, b), hi0 = fmaxf(a, b);
                a = fmaf(n0.z, iy, oy); b = fmaf(n0.w, iy, oy);
                lo0 = fmaxf(lo0, fminf(a, b)); hi0 = fminf(hi0, fmaxf(a, b));
                a = fmaf(n1.x, iz, oz); b = fmaf(n1.y, iz, oz);
                lo0 = fmaxf(lo0, fminf(a, b)); hi0 = fminf(hi0, fmaxf(a, b));
                a = fmaf(n1.z, ix, ox); b = fmaf(n1.w, ix, ox);
                float lo1 = fminf(a, b), hi1 = fmaxf(a, b);
                a = fmaf(n2.x, iy, oy); b = fmaf(n2.y, iy, oy);
                lo1 = fmaxf(lo1, fminf(a, b)); hi1 = fminf(hi1, fmaxf(a, b));
                a = fmaf(n2.z, iz, oz); b = fmaf(n2.w, iz, oz);
                lo1 = fmaxf(lo1, fminf(a, b)); hi1 = fminf(hi1, fmaxf(a, b));
                const bool h0 = lo0 <= hi0 && hi0 >= 0.f && lo0 <= best_t;
                const bool h1 = lo1 <= hi1 && hi1 >= 0.f && lo1 <= best_t;
                if (h0 && h1) {
                    const bool swap = lo1 < lo0;
                    stk[sp * stride] = swap ? ch.x : ch.y;
                    stk_t[sp * stride] = swap ? lo0 : lo1;
                    ++sp;
                    if (!enter(swap ? ch.y : ch.x)) pop();
                } else if (h0) { if (!enter(ch.x)) pop(); }
                else if (h1) { if (!enter(ch.y)) pop(); }
                else pop();
            }
        } else {
            if (st == LEAF) {
                const int r = refs[li];
                ++li;
                if (r >= 0) {
                    float t;
                    if (sphere_t(tc.sph[r], o, d, t)) {
                        const int oid = sc.sph_id[r];
                        if (t < best_t || (t == best_t && oid < best_id)) { best_t = t; best_id = oid; best_ref = r; }
                    }
                } else {
                    const int j = ~r;
                    float dist; float3 nrm;
                    if (box_hit(tc.box[2 * j], tc.box[2 * j + 1], o, d, dist, nrm)) {
                        const int oid = sc.box_id[j];
                        if (dist < best_t || (dist == best_t && oid < best_id)) { best_t = dist; best_id = oid; best_ref = r; }
                    }
                }
                if (li == lend) pop();
            }
        }
    }

    if (inside) {
        float4 a4 = accum[pixel];
        a4.x += acc.x; a4.y += acc.y; a4.z += acc.z;
        accum[pixel] = a4;
    }
    unsigned int total = segs;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) total += __shfl_down_sync(FULL, total, off);
    if ((threadIdx.x & 31) == 0 && total) {
        atomicAdd(seg_counter, (unsigned long long)total); atomicAdd(seg_counter + 1, (unsigned long long)total);
        atomicAdd(seg_counter + 2, (unsigned long long)total); atomicAdd(seg_counter + 3, (unsigned long long)total);
    }
}

// ---- preview mode (SIMPLEDRAW, Raytracer.cpp:147-160): one primary ray, overwrite ----------
__device__ __forceinline__ float3 preview_color(const SceneView& sc, const FrameView& fr, const Hit& h, float3 d) {
    if (h.id < 0) return env_color(fr, d);
    const float4 m0 = __ldg(sc.mat + 3 * h.id), m1 = __ldg(sc.mat + 3 * h.id + 1);
    const float3 base = f3(m0.x, m0.y, m0.z), emis = f3(m1.x, m1.y, m1.z);
    const float k = m1.w, sm = m0.w;
    const float3 refl = env_color(fr, reflect3(d, h.n));                       // :148
    float fres = 0.f;
    if (h.id == fr.selected_id) {                                              // :153-157
        fres = 1.f - dot3(scale3(h.n, -1.f), d);
        fres = maxsel(fres, 0.f);
        fres = smoothstep1(0.f, 0.5f, fres);
    }
    const float3 a = cadd(cadd(cscale(base, 1.f - k), cscale(cscale(refl, k), sm)), emis);
    return clerp(a, col(3.f, 3.f, 0.f), fres);                                 // :159
}

template <int MODE>
__global__ void __launch_bounds__(kThreads) k_render_preview(SceneView sc, BvhView bv, FlatView fl, FrameView fr, float4* __restrict__ accum,
                                                              unsigned long long* __restrict__ seg_counter) {
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);
    int px, py;
    if (!tile_pixel(fr, px, py)) return;
    const size_t pixel = (size_t)px + (size_t)py * fr.width;
    const float3 d = ray_dir(fr, px, py);
    const float3 c = preview_color(sc, fr, trace<MODE>(sc, tc, fr.cam_pos, d), d);
    accum[pixel] = make_float4(c.x, c.y, c.z, 0.f);
    if (threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) {
        for (int k = 0; k < 4; ++k) atomicAdd(seg_counter + k, (unsigned long long)fr.width * fr.height);
    }
}

// ---- block-filled frames: SCREEN_SCALE / progressive resolution (Raytracer.cpp:233-248, 330-341) -------------
// `steps` = ceil(1 / (SCREEN_SCALE * progressiveResolutionScaler)): one path per steps x steps block, traced
// through the block's first pixel and written to every pixel of the block. Blocks start at each column strip's
// first column (the reference's 16 worker strips) and are clipped to the strip and the image. One thread per
// block; path mode adds the block's sample sum to all its pixels, preview mode overwrites them.
template <int MODE>
__global__ void __launch_bounds__(kThreads) k_render_blocks(SceneView sc, BvhView bv, FlatView fl, FrameView fr, float4* __restrict__ accum,
                                                             uint32_t s_begin, int n_samples, int steps, int strip_w, int bps, int n_strips,
                                                             unsigned long long* __restrict__ seg_counter) {
    extern __shared__ float4 smem[];
    const TraceCtx tc = setup_trace<MODE>(sc, bv, fl, smem);
    const int cols = n_strips * bps, rows = (fr.height + steps - 1) / steps;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int col_i = t % cols, row = t / cols;
    const int strip = col_i / bps, x0 = strip * strip_w, x1 = min(x0 + strip_w, fr.width);
    const int px = x0 + (col_i % bps) * steps, py = row * steps;
    const bool valid = row < rows && px < x1 && py < fr.height;
    unsigned int segs = 0;
    if (valid) {
        const uint32_t pixel = (uint32_t)px + (uint32_t)py * (uint32_t)fr.width;
        const float3 d0 = ray_dir(fr, px, py);
        float3 acc = f3(0.f, 0.f, 0.f);
        if (fr.mode == 1) {
            acc = preview_color(sc, fr, trace<MODE>(sc, tc, fr.cam_pos, d0), d0);
            segs = 1;
        } else {
            float3 o = fr.cam_pos, d = d0, T = f3(0.f, 0.f, 0.f), L = f3(0.f, 0.f, 0.f);
            int s = 0, depth = 0;
            while (s < n_samples) {
                const Hit h = trace<MODE>(sc, tc, o, d);
                ++segs;
                float3 c;
                if (shade_segment(sc, fr, h, pixel, s_begin + (uint32_t)s, o, d, T, L, depth, c)) {
                    acc.x += c.x; acc.y += c.y; acc.z += c.z;
                    ++s; depth = 0; o = fr.cam_pos; d = d0;
                }
            }
        }
        for (int j = py; j < py + steps && j < fr.height; ++j)
            for (int i = px; i < px + steps && i < x1; ++i) {
                const size_t p = (size_t)i + (size_t)j * fr.width;
                if (fr.mode == 1) accum[p] = make_float4(acc.x, acc.y, acc.z, 0.f);
                else { float4 a = accum[p]; a.x += acc.x; a.y += acc.y; a.z += acc.z; accum[p] = a; }
            }
    }
    if (segs) for (int k = 0; k < 4; ++k) atomicAdd(seg_counter + k, (unsigned long long)segs);
}

// ---- resolve kernels (resolve_pixel(): above k_render_pool, which resolves finished pixels itself) -----------
// Generic slice resolve: pixels [first, first+n) of a width x height image; `accum` points at
// the slice. Output row = flip ? (H-1-y) : y (Raytracer.cpp:64), tightly packed width*4 pitch,
// `out` points at the start of the WHOLE image when whole_image_out, else at the slice.
// out2 (optional): a second whole-image destination - the caller's page-locked HOST surface, written straight over PCIe
// by the kernel's coalesced stores (zero-copy), so that an interactive frame needs no separate device-to-host copy.
__global__ void k_resolve(const float4* __restrict__ accum, float count, int width, int height, int first, int n,
                          int flip_y, uint32_t* __restrict__ out, int out_is_slice, uint32_t* __restrict__ out2) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int p = first + i;
    const int x = p % width, y = p / width;
    const uint32_t v = resolve_pixel(accum[i], count);
    const size_t dst = (size_t)x + (size_t)(flip_y ? height - 1 - y : y) * width;
    out[out_is_slice ? (size_t)i : dst] = v;
    if (out2) out2[dst] = v;
}

// ---- fused multi-GPU reduce + resolve over peer memory -----------------------------------------
// One thread per pixel of this rank's slice: float4 loads from every rank's accumulation buffer (the
// peers' are NVLink P2P mappings: plain ld.global on peer addresses), summed in rank order, then the
// same resolve as k_resolve, stored into the destination surface (a peer store when it is rank 0's).
__global__ void k_resolve_fused(PeerPtrs peers, int world, float count, int width, int height, int first, int n, int flip_y,
                                uint32_t* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int p = first + i;
    float4 sum = peers.p[0][p];
    for (int r = 1; r < world; ++r) {
        const float4 v = peers.p[r][p];
        sum.x += v.x; sum.y += v.y; sum.z += v.z;
    }
    const int x = p % width, y = p / width;
    out[(size_t)x + (size_t)(flip_y ? height - 1 - y : y) * width] = resolve_pixel(sum, count);
}

// ---- fused multi-GPU reduce into one device's buffer (rt_group_denoise_rgba8 / rt_group_temporal_rgba8) ---------------------
// k_resolve_fused without the resolve: the float4 sum, formed by the same rank-order loop (so resolve_pixel(out[p], total) gives
// k_resolve_fused's bits), stored at pixel p of `out` (a peer store when it is another device's). 16 B read per rank, 16 B written.
__global__ void k_reduce_fused(PeerPtrs peers, int world, int first, int n, float4* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int p = first + i;
    float4 sum = peers.p[0][p];
    for (int r = 1; r < world; ++r) {
        const float4 v = peers.p[r][p];
        sum.x += v.x; sum.y += v.y; sum.z += v.z;
    }
    out[p] = sum;
}

// ---- the same with the inter-rank ordering on the device (rt_exchange_resolve; one process per GPU) -------------------------
// No collective library and no host synchronisation: ranks signal each other through flag words in device memory that the
// peers have mapped (CUDA IPC over NVLink). Epochs only grow, so nothing is ever reset and a late reader cannot see a stale
// "ready". Every wait is bounded (kExchTimeoutNs): a peer that died makes the exchange fail instead of hanging the GPU.
// NOTE: the ranks must run on DIFFERENT devices (kernels of two ranks on one GPU are not guaranteed to run concurrently).
constexpr unsigned long long kExchTimeoutNs = 4000000000ull;
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// One warp: lane r < world polls flags[r] until it reaches `epoch` (wrap-safe compare). false: timed out, *error is set.
__device__ __forceinline__ bool warp_wait_flags(const uint32_t* flags, int world, uint32_t epoch, uint32_t* error) {
    const int lane = threadIdx.x & 31;
    bool ok = lane >= world;
    const unsigned long long t0 = global_ns();
    while (!__all_sync(0xffffffffu, ok)) {
        if (!ok) ok = (int)(ld_acquire_sys(flags + lane) - epoch) >= 0;
        if (global_ns() - t0 > kExchTimeoutNs) {
            if (lane == 0) atomicExch(error, 1u);
            return false;
        }
    }
    return true;
}
__global__ void __launch_bounds__(256) k_resolve_fused_sync(PeerPtrs peers, ExchPeers fl, int rank, int world, uint32_t epoch, float count,
                                                             int width, int height, int first, int n, int flip_y, uint32_t* __restrict__ out) {
    ExchFlags* const mine = fl.f[rank];
    if (threadIdx.x < 32) {
        if (blockIdx.x == 0 && threadIdx.x < world) {
            // this rank's render finished before this kernel started (stream order): publish it to every rank
            __threadfence_system();
            st_release_sys(&fl.f[threadIdx.x]->arrive[rank], epoch);
        }
        warp_wait_flags(mine->arrive, world, epoch, &mine->error);
    }
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const int p = first + i;
        float4 sum = peers.p[0][p];
        for (int r = 1; r < world; ++r) {
            const float4 v = peers.p[r][p];
            sum.x += v.x; sum.y += v.y; sum.z += v.z;
        }
        const int x = p % width, y = p / width;
        out[(size_t)x + (size_t)(flip_y ? height - 1 - y : y) * width] = resolve_pixel(sum, count);
    }
    // the last CTA tells every rank: my slice is in the surface, and I am done reading your buffers
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(&mine->blocks_done, 1u);
        if (prev == gridDim.x - 1) {
            mine->blocks_done = 0u;
            __threadfence_system();
            for (int r = 0; r < world; ++r) st_release_sys(&fl.f[r]->done[rank], epoch);
        }
    }
}
__global__ void k_exchange_wait(ExchFlags* mine, int world, uint32_t epoch) { warp_wait_flags(mine->done, world, epoch, &mine->error); }

}  // namespace

// ---- launchers --------------------------------------------------------------------------------
static inline dim3 tile_grid(int w, int h) { return dim3((w + kTileW - 1) / kTileW, (h + kTileH - 1) / kTileH); }

template <typename K>
static cudaError_t optin(K kernel) { return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxStagedBytes); }

static cudaError_t ensure_smem_optin() {
    // the attribute is per DEVICE: a process may hold contexts on several GPUs (rt_create_multi), used from several host threads
    static bool done_on[64] = {false};
    static std::mutex mu;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    bool& done = done_on[dev & 63];
    if (done) return cudaSuccess;
#define RTB_OPTIN(K) \
    if ((e = optin(K<0>)) != cudaSuccess) return e; \
    if ((e = optin(K<1>)) != cudaSuccess) return e; \
    if ((e = optin(K<2>)) != cudaSuccess) return e; \
    if ((e = optin(K<3>)) != cudaSuccess) return e; \
    if ((e = optin(K<4>)) != cudaSuccess) return e;
#define RTB_OPTIN2(K) \
    if ((e = optin(K<0, false>)) != cudaSuccess) return e; if ((e = optin(K<0, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<1, false>)) != cudaSuccess) return e; if ((e = optin(K<1, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<2, false>)) != cudaSuccess) return e; if ((e = optin(K<2, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<3, false>)) != cudaSuccess) return e; if ((e = optin(K<3, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<4, false>)) != cudaSuccess) return e; if ((e = optin(K<4, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<5, false>)) != cudaSuccess) return e; if ((e = optin(K<5, true>)) != cudaSuccess) return e;
#define RTB_OPTIN3(K) \
    if ((e = optin(K<0, false, false>)) != cudaSuccess) return e; if ((e = optin(K<0, true, false>)) != cudaSuccess) return e; if ((e = optin(K<0, false, true>)) != cudaSuccess) return e; if ((e = optin(K<0, true, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<1, false, false>)) != cudaSuccess) return e; if ((e = optin(K<1, true, false>)) != cudaSuccess) return e; if ((e = optin(K<1, false, true>)) != cudaSuccess) return e; if ((e = optin(K<1, true, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<2, false, false>)) != cudaSuccess) return e; if ((e = optin(K<2, true, false>)) != cudaSuccess) return e; if ((e = optin(K<2, false, true>)) != cudaSuccess) return e; if ((e = optin(K<2, true, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<3, false, false>)) != cudaSuccess) return e; if ((e = optin(K<3, true, false>)) != cudaSuccess) return e; if ((e = optin(K<3, false, true>)) != cudaSuccess) return e; if ((e = optin(K<3, true, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<4, false, false>)) != cudaSuccess) return e; if ((e = optin(K<4, true, false>)) != cudaSuccess) return e; if ((e = optin(K<4, false, true>)) != cudaSuccess) return e; if ((e = optin(K<4, true, true>)) != cudaSuccess) return e; \
    if ((e = optin(K<5, false, false>)) != cudaSuccess) return e; if ((e = optin(K<5, true, false>)) != cudaSuccess) return e; if ((e = optin(K<5, false, true>)) != cudaSuccess) return e; if ((e = optin(K<5, true, true>)) != cudaSuccess) return e;
    RTB_OPTIN2(k_render_regen) RTB_OPTIN3(k_render_pool) RTB_OPTIN(k_render_preview) RTB_OPTIN(k_primary_aov) RTB_OPTIN(k_trace_rays) RTB_OPTIN(k_pick) RTB_OPTIN(k_render_blocks)
    RTB_OPTIN(k_primary_cache)
    if ((e = optin(k_render_bvh<2>)) != cudaSuccess) return e;
    if ((e = optin(k_render_bvh<3>)) != cudaSuccess) return e;
    // the counting instantiations (RT_OPT_TRAVERSAL_STATS): binary BVH only
    if ((e = optin(k_trace_rays<2, true>)) != cudaSuccess) return e;
    if ((e = optin(k_trace_rays<3, true>)) != cudaSuccess) return e;
    if ((e = optin(k_render_regen<2, true, true>)) != cudaSuccess) return e;
    if ((e = optin(k_render_regen<3, true, true>)) != cudaSuccess) return e;
    if ((e = optin(k_render_regen<2, false, true>)) != cudaSuccess) return e;
    if ((e = optin(k_render_regen<3, false, true>)) != cudaSuccess) return e;
    if ((e = optin(k_render_regen<5, true, false, true>)) != cudaSuccess) return e;      // the 7-CTA form (STASH)
    // the pixel filter's forms
    RTB_OPTIN2(k_render_pool_aa)
    if ((e = optin(k_render_regen_aa<0>)) != cudaSuccess) return e; if ((e = optin(k_render_regen_aa<1>)) != cudaSuccess) return e;
    if ((e = optin(k_render_regen_aa<2>)) != cudaSuccess) return e; if ((e = optin(k_render_regen_aa<3>)) != cudaSuccess) return e;
    if ((e = optin(k_render_regen_aa<4>)) != cudaSuccess) return e; if ((e = optin(k_render_regen_aa<5>)) != cudaSuccess) return e;
    if ((e = optin(k_render_regen_aa<2, true>)) != cudaSuccess) return e; if ((e = optin(k_render_regen_aa<3, true>)) != cudaSuccess) return e;
#undef RTB_OPTIN
#undef RTB_OPTIN2
#undef RTB_OPTIN3
    done = true;
    return cudaSuccess;
}

#define RTB_DISPATCH(MODE, K, GRID, SMEM, ST, ...)                                     \
    switch (MODE) {                                                                    \
        case 0: K<0><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break;                \
        case 1: K<1><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break;                \
        case 2: K<2><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break;                \
        case 3: K<3><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break;                \
        default: K<4><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break;               \
    }
#define RTB_DISPATCH2(MODE, FLAG, K, GRID, SMEM, ST, ...)                                                  \
    switch (MODE) {                                                                                        \
        case 0: if (FLAG) K<0, true><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); else K<0, false><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break; \
        case 1: if (FLAG) K<1, true><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); else K<1, false><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break; \
        case 2: if (FLAG) K<2, true><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); else K<2, false><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break; \
        case 3: if (FLAG) K<3, true><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); else K<3, false><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break; \
        case 4: if (FLAG) K<4, true><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); else K<4, false><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break; \
        default: if (FLAG) K<5, true><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); else K<5, false><<<GRID, kThreads, SMEM, ST>>>(__VA_ARGS__); break; \
    }

cudaError_t launch_primary_aov(const SceneView& sc, const AccelSel& ac, const FrameView& fr, int* id, float* t,
                               float* n, float* p, cudaStream_t st) {
    cudaError_t e = ensure_smem_optin();
    if (e != cudaSuccess) return e;
    size_t sb; const int mode = pick_mode(sc, ac, sb);
    RTB_DISPATCH(mode, k_primary_aov, tile_grid(fr.width, fr.height), sb, st, sc, ac.bvh, ac.flat, fr, id, t, n, p)
    return cudaGetLastError();
}

cudaError_t launch_ray_dirs(const FrameView& fr, float* out, cudaStream_t st) {
    k_ray_dirs<<<dim3((fr.width + 127) / 128, fr.height), 128, 0, st>>>(fr, out);
    return cudaGetLastError();
}

cudaError_t launch_sample_dirs(const FrameView& fr, PixelFilter pf, uint32_t sample, float* out, cudaStream_t st) {
    k_sample_dirs<<<dim3((fr.width + 127) / 128, fr.height), 128, 0, st>>>(fr, pf, sample, out);
    return cudaGetLastError();
}

cudaError_t launch_trace_rays(const SceneView& sc, const AccelSel& ac, const float* org, const float* dir, int n,
                              int* id, float* t, float* nrm, float* pt, cudaStream_t st, unsigned long long* counters) {
    if (n <= 0) return cudaSuccess;
    cudaError_t e = ensure_smem_optin();
    if (e != cudaSuccess) return e;
    size_t sb; const int mode = pick_mode(sc, ac, sb);
    const dim3 grid((n + kThreads - 1) / kThreads);
    if (counters && (mode == 2 || mode == 3) && !ac.bvh.wnodes) {
        if (mode == 2) k_trace_rays<2, true><<<grid, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, org, dir, n, id, t, nrm, pt, counters);
        else k_trace_rays<3, true><<<grid, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, org, dir, n, id, t, nrm, pt, counters);
        return cudaGetLastError();
    }
    RTB_DISPATCH(mode, k_trace_rays, grid, sb, st, sc, ac.bvh, ac.flat, org, dir, n, id, t, nrm, pt, nullptr)
    return cudaGetLastError();
}

cudaError_t launch_primary_cache(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* prim_nt, int* prim_id,
                                 unsigned long long* counters, cudaStream_t st) {
    cudaError_t e = ensure_smem_optin();
    if (e != cudaSuccess) return e;
    size_t sb; const int mode = pick_mode(sc, ac, sb);
    RTB_DISPATCH(mode, k_primary_cache, tile_grid(fr.width, fr.height), sb, st, sc, ac.bvh, ac.flat, fr, prim_nt, prim_id, counters)
    return cudaGetLastError();
}

cudaError_t launch_env_color(const FrameView& fr, const float* dir, int n, float* out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    k_env_color<<<(n + 127) / 128, 128, 0, st>>>(fr, dir, n, out);
    return cudaGetLastError();
}

cudaError_t launch_philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t* dev_out4, cudaStream_t st) {
    k_philox<<<1, 1, 0, st>>>(make_uint4(ctr[0], ctr[1], ctr[2], ctr[3]), make_uint2(key[0], key[1]), (uint4*)dev_out4);
    return cudaGetLastError();
}

cudaError_t launch_selftest_uniform(int* dev_failures, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(dev_failures, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    k_selftest_uniform<<<32768 / 256, 256, 0, st>>>(dev_failures);
    return cudaGetLastError();
}

cudaError_t launch_selftest_normalize(int* dev_failures, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(dev_failures, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    k_selftest_normalize<<<16384, 256, 0, st>>>(dev_failures, 0x2b200u);            // 2^28 vectors
    return cudaGetLastError();
}

cudaError_t launch_selftest_packed(int* dev_failures, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(dev_failures, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    k_selftest_packed<<<4096, 256, 0, st>>>(dev_failures, 0xf32c2u);                 // 2^26 operand sets
    return cudaGetLastError();
}

cudaError_t launch_pick(const SceneView& sc, const AccelSel& ac, const FrameView& fr, int px, int py, int* dev_id, cudaStream_t st) {
    cudaError_t e = ensure_smem_optin();
    if (e != cudaSuccess) return e;
    size_t sb; const int mode = pick_mode(sc, ac, sb);
    RTB_DISPATCH(mode, k_pick, 1, sb, st, sc, ac.bvh, ac.flat, fr, px, py, dev_id)
    return cudaGetLastError();
}

// 32-pixel tiles = 10 000 CTAs: about ten waves of 148 x 7 (1080p has 64 800 tiles, 720p 28 800, 640x480 9600). Below it the two forms are
// within the run-to-run noise of each other (profiles/r4z_ab_stash_threshold.txt: 720p 64 spp 3.71 vs 3.77 ms, 960x540 and 640x480 equal;
// 2560x1440 12.68 vs 13.07 ms), so small grids stay on the form they were tuned and profiled with.
constexpr long long kStashMinWarpTiles = 40000;

cudaError_t launch_render_regen(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* accum,
                                uint32_t s_begin, int n_samples, const PrimCache* prim_cache, unsigned long long* seg_counter, cudaStream_t st, int pool_override, bool flat_coop,
                                bool count_traversal, FrameTarget* frame, const PixelFilter* filter) {
    if (n_samples <= 0) return cudaSuccess;
    if (filter) prim_cache = nullptr;                         // every sample traces its own jittered primary ray
    const bool reuse_primary = prim_cache != nullptr;
    PrimCache prim;
    prim.nt = prim_cache ? prim_cache->nt : nullptr; prim.id = prim_cache ? prim_cache->id : nullptr;
    cudaError_t e = ensure_smem_optin();
    if (e != cudaSuccess) return e;
    // few samples per launch: lanes pull pixels from chunks of tiles claimed by their warp (k_render_pool); many: one pixel per lane.
    // Measured on B200 (scratch/pool_sweep.py, Scene1, persistent grid + primary-hit cache): 1 spp 720p 0.174 (one pixel per lane) ->
    // 0.158 ms with chunks of 2 tiles, 1080p 0.364 -> 0.257 ms; 2 spp pays at 1080p only (0.549 -> 0.514 ms); from 4 spp on one pixel
    // per lane wins, and larger chunks lose to the imbalance between warps at the end of the launch (8 tiles: 0.295 ms at 720p).
    const long long n_tiles_all = (long long)((fr.width + kPoolTW - 1) / kPoolTW) * ((fr.height + kPoolTH - 1) / kPoolTH);
    int pool_tiles = 1;
    if (count_traversal) pool_override = 1;                   // the counting instantiations exist for the one-pixel-per-lane kernel only
    if (pool_override > 0) pool_tiles = pool_override > 32 ? 32 : pool_override;
    else if (n_samples == 1 || (n_samples == 2 && n_tiles_all >= 50000)) pool_tiles = 2;
    // the pooled flat traversal pays from ~16 spp per launch on; short launches (the pixel pool's) run the per-lane form
    static const bool pool_coop = [] { const char* v = getenv("RTB200_POOL_COOP"); return v && v[0] == '1'; }();   // A/B: pooled levels 2/3 in the pixel-pool kernel too
    size_t sb; const int mode = pick_mode(sc, ac, sb, kThreads, flat_coop && (pool_tiles < 2 ? n_samples >= 16 : pool_coop));
    if (pool_tiles >= 2) {
        // persistent grid: at most one resident wave of CTAs; the warps claim tiles until the image is handed out
        int dev = 0;
        cudaGetDevice(&dev);
        static std::atomic<int> sms_of[64];                  // per device; the attribute query costs microseconds of every frame
        int sms = sms_of[dev & 63].load(std::memory_order_relaxed);
        if (sms == 0) { cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); sms_of[dev & 63].store(sms, std::memory_order_relaxed); }
        const long long n_tiles = n_tiles_all;
        const long long chunks = (n_tiles + pool_tiles - 1) / pool_tiles;
        long long blocks = (chunks + kThreads / 32 - 1) / (kThreads / 32);
        if (blocks > (long long)sms * RTB_REGEN_MIN_BLOCKS) blocks = (long long)sms * RTB_REGEN_MIN_BLOCKS;
        unsigned int* cursor = reinterpret_cast<unsigned int*>(seg_counter + kTileCursorSlot);
        // (the kernel's last warp putting the cursor back itself instead of this memset node: measured, no gain - 0.187 vs 0.185 ms per 720p frame)
        if ((e = cudaMemsetAsync(cursor, 0, sizeof(unsigned int), st)) != cudaSuccess) return e;
        FrameOut fo;
        fo.out = nullptr; fo.out2 = nullptr; fo.count = 0.f; fo.flip_y = 0; fo.smem_off = 0;
        if (frame && frame->surface && pool_tiles == 2) {     // resolve + host copy inside the render (FrameOut)
            fo.out = frame->surface; fo.out2 = frame->mapped_host; fo.count = (float)frame->samples_after; fo.flip_y = frame->flip_y;
            fo.smem_off = (int)((sb + 15) / 16 * 16);
            sb = (size_t)fo.smem_off + (size_t)(kThreads / 32) * kPoolSlots * sizeof(unsigned int);
            frame->fused = true;
        }
#define RTB_POOL_CASE(M) case M: \
            if (filter) { if (fo.out) k_render_pool_aa<M, true><<<(unsigned int)blocks, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, pool_tiles, cursor, seg_counter, fo, *filter); \
                          else k_render_pool_aa<M, false><<<(unsigned int)blocks, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, pool_tiles, cursor, seg_counter, fo, *filter); } \
            else if (fo.out) { if (reuse_primary) k_render_pool<M, true, true><<<(unsigned int)blocks, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, pool_tiles, prim, cursor, seg_counter, fo); \
                          else k_render_pool<M, false, true><<<(unsigned int)blocks, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, pool_tiles, prim, cursor, seg_counter, fo); } \
            else { if (reuse_primary) k_render_pool<M, true, false><<<(unsigned int)blocks, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, pool_tiles, prim, cursor, seg_counter, fo); \
                   else k_render_pool<M, false, false><<<(unsigned int)blocks, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, pool_tiles, prim, cursor, seg_counter, fo); } \
            break;
        switch (mode) { RTB_POOL_CASE(0) RTB_POOL_CASE(1) RTB_POOL_CASE(2) RTB_POOL_CASE(3) RTB_POOL_CASE(4) default: RTB_POOL_CASE(5) }
#undef RTB_POOL_CASE
        return cudaGetLastError();
    }
    if (count_traversal && (mode == 2 || mode == 3) && !ac.bvh.wnodes) {
        const dim3 grid = tile_grid(fr.width, fr.height);
        if (filter && mode == 2) k_render_regen_aa<2, true><<<grid, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, seg_counter, *filter);
        else if (filter) k_render_regen_aa<3, true><<<grid, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, seg_counter, *filter);
        else if (mode == 2 && reuse_primary) k_render_regen<2, true, true><<<grid, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, prim, seg_counter);
        else if (mode == 2) k_render_regen<2, false, true><<<grid, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, prim, seg_counter);
        else if (reuse_primary) k_render_regen<3, true, true><<<grid, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, prim, seg_counter);
        else k_render_regen<3, false, true><<<grid, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, prim, seg_counter);
        return cudaGetLastError();
    }
    // large grids of the pooled flat traversal with the primary-hit cache (the headline configuration): the 7-CTA form (k_render_regen STASH)
    static const bool no_stash = [] { const char* v = getenv("RTB200_REGEN_STASH"); return v && v[0] == '0'; }();    // A/B
    static const long long stash_min = [] { const char* v = getenv("RTB200_STASH_MIN_TILES"); return v ? atoll(v) : kStashMinWarpTiles; }();   // A/B
    if (filter) {
        const dim3 grid = tile_grid(fr.width, fr.height);
#define RTB_AA_CASE(M) case M: k_render_regen_aa<M><<<grid, kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, seg_counter, *filter); break;
        switch (mode) { RTB_AA_CASE(0) RTB_AA_CASE(1) RTB_AA_CASE(2) RTB_AA_CASE(3) RTB_AA_CASE(4) default: RTB_AA_CASE(5) }
#undef RTB_AA_CASE
        return cudaGetLastError();
    }
    if (mode == 5 && reuse_primary && !no_stash && n_tiles_all >= stash_min) {
        k_render_regen<5, true, false, true><<<tile_grid(fr.width, fr.height), kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, prim, seg_counter);
        return cudaGetLastError();
    }
    RTB_DISPATCH2(mode, reuse_primary, k_render_regen, tile_grid(fr.width, fr.height), sb, st, sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, prim, seg_counter)
    return cudaGetLastError();
}

cudaError_t launch_render_bvh(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* accum, uint32_t s_begin,
                              int n_samples, unsigned long long* seg_counter, int wait_k, cudaStream_t st) {
    if (n_samples <= 0) return cudaSuccess;
    cudaError_t e = ensure_smem_optin();
    if (e != cudaSuccess) return e;
    if (ac.bvh.wnodes) return launch_render_regen(sc, ac, fr, accum, s_begin, n_samples, nullptr, seg_counter, st);   // the scheduled kernel walks binary nodes only (and, like it, re-traces every primary ray)
    size_t sb; const int mode = pick_mode(sc, ac, sb);
    if (mode == 2) k_render_bvh<2><<<tile_grid(fr.width, fr.height), kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, seg_counter, wait_k);
    else if (mode == 3) k_render_bvh<3><<<tile_grid(fr.width, fr.height), kThreads, sb, st>>>(sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples, seg_counter, wait_k);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

cudaError_t launch_render_preview(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* accum,
                                  unsigned long long* seg_counter, cudaStream_t st) {
    cudaError_t e = ensure_smem_optin();
    if (e != cudaSuccess) return e;
    size_t sb; const int mode = pick_mode(sc, ac, sb);
    RTB_DISPATCH(mode, k_render_preview, tile_grid(fr.width, fr.height), sb, st, sc, ac.bvh, ac.flat, fr, accum, seg_counter)
    return cudaGetLastError();
}

cudaError_t launch_render_blocks(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* accum, uint32_t s_begin,
                                 int n_samples, int steps, int strip_w, unsigned long long* seg_counter, cudaStream_t st) {
    cudaError_t e = ensure_smem_optin();
    if (e != cudaSuccess) return e;
    if (steps < 1) steps = 1;
    if (strip_w <= 0 || strip_w > fr.width) strip_w = fr.width;
    const int n_strips = (fr.width + strip_w - 1) / strip_w, bps = (strip_w + steps - 1) / steps;
    const int rows = (fr.height + steps - 1) / steps;
    const long long threads = (long long)n_strips * bps * rows;
    size_t sb; const int mode = pick_mode(sc, ac, sb);
    RTB_DISPATCH(mode, k_render_blocks, (unsigned int)((threads + kThreads - 1) / kThreads), sb, st, sc, ac.bvh, ac.flat, fr, accum, s_begin, n_samples,
                 steps, strip_w, bps, n_strips, seg_counter)
    return cudaGetLastError();
}

cudaError_t launch_resolve(const float4* accum, uint32_t samples, int width, int height, int first, int n, int flip_y,
                           uint32_t* out, int out_is_slice, cudaStream_t st, uint32_t* mapped_host_out) {
    if (n <= 0) return cudaSuccess;
    k_resolve<<<(n + 255) / 256, 256, 0, st>>>(accum, (float)samples, width, height, first, n, flip_y, out, out_is_slice, mapped_host_out);
    return cudaGetLastError();
}

cudaError_t launch_resolve_fused(const PeerPtrs& peers, int world, uint32_t samples, int width, int height, int first, int n,
                                 int flip_y, uint32_t* out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    k_resolve_fused<<<(n + 255) / 256, 256, 0, st>>>(peers, world, (float)samples, width, height, first, n, flip_y, out);
    return cudaGetLastError();
}

cudaError_t launch_reduce_fused(const PeerPtrs& peers, int world, int first, int n, float4* out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    k_reduce_fused<<<(n + 255) / 256, 256, 0, st>>>(peers, world, first, n, out);
    return cudaGetLastError();
}

cudaError_t launch_resolve_fused_sync(const PeerPtrs& peers, const ExchPeers& flags, int rank, int world, uint32_t epoch, uint32_t samples,
                                      int width, int height, int first, int n, int flip_y, uint32_t* out, cudaStream_t st) {
    // n == 0 still signals: the other ranks wait for this one
    k_resolve_fused_sync<<<n > 0 ? (n + 255) / 256 : 1, 256, 0, st>>>(peers, flags, rank, world, epoch, (float)samples, width, height, first, n, flip_y, out);
    k_exchange_wait<<<1, 32, 0, st>>>(flags.f[rank], world, epoch);
    return cudaGetLastError();
}

}  // namespace rtb
