// rt_filter.cuh - the pixel filter (rt_set_pixel_filter): one sub-pixel offset of the primary ray per sample, drawn from the
// sample's own Philox block, so that accumulating samples integrates the radiance over the filter's footprint (anti-aliased edges).
// Shared by the jittered render kernels and rt_read_sample_dirs (rt_kernels.cu), and compiled for the host by the tests
// (tests/host_emu/filter_emu.cpp). The definition (DESIGN.md 5):
//   words   (w.x, w.y) of Philox4x32-10 with counter (pixel, global sample index, 0, 1) and the context's key. Every other stream
//           of the renderer has counter word 3 = 0, so this block is disjoint from the path's blocks (pixel, sample, depth, 0);
//           it does not depend on the shard, the world size or the launch shape.
//   unit    u = (float)(w >> 8) * 2^-24, exact, in [0, 1)
//   box     j = (2u - 1) * r: uniform on [-r, r)
//   tent    v = 2u; j = (v < 1 ? sqrt(v) - 1 : 1 - sqrt(2 - v)) * r: density (r - |j|) / r^2 on (-r, r)
//   ray     ray_dir with (float)px replaced by (float)px + jx (and py by py + jy), the remaining operations in ray_dir's order; a zero
//           offset gives ray_dir's bits. The footprint is centred on the reference's own ray, the pixel CORNER, so the image does not
//           shift against the unfiltered one and the primary-hit cache (corner rays) stays the guide of the denoiser and the
//           temporal reprojection.
#pragma once
#include "rt_device.cuh"

namespace rtb {

enum { kFilterNone = 0, kFilterBox = 1, kFilterTent = 2 };   // RT_FILTER_* (include/rt_b200.h)
struct PixelFilter { int type; float radius; };

__host__ __device__ __forceinline__ float filter_unit(uint32_t w) { return (float)(w >> 8) * 0x1p-24f; }
__host__ __device__ __forceinline__ float filter_offset(int type, float radius, uint32_t w) {
    if (type == kFilterNone) return 0.f;
    const float u = filter_unit(w);
    if (type == kFilterBox) return (u * 2.f - 1.f) * radius;
    const float v = u * 2.f;
    return (v < 1.f ? sqrtf(v) - 1.f : 1.f - sqrtf(2.f - v)) * radius;
}

// the primary direction of global sample `sample` of pixel (px, py), pixel = px + py * width
__device__ __forceinline__ float3 filtered_ray_dir(const FrameView& f, PixelFilter pf, int px, int py, uint32_t pixel, uint32_t sample) {
#ifdef RTB_PHILOX_PLAIN_KEYS
    const uint4 w = philox4x32_10(pixel, sample, 0u, 1u, f.seed_lo, f.seed_hi);
#else
    const uint4 w = philox4x32_10_ks(pixel, sample, 0u, 1u, f.key_sched);
#endif
    const float jx = filter_offset(pf.type, pf.radius, w.x), jy = filter_offset(pf.type, pf.radius, w.y);
    float nX = (((float)px + jx) / (float)f.width) * 2.f - 1.f;
    float nY = (((float)py + jy) / (float)f.height) * 2.f - 1.f;
    float3 u = scale3(f.u_axis, nX);
    float3 v = scale3(f.v_axis, nY);
    return normalized3(add3(add3(u, v), f.fwd));
}

}  // namespace rtb
