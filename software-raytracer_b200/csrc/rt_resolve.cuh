// rt_resolve.cuh - sum/count -> Reinhard -> truncating ARGB8 pack of one pixel (Raytracer.cpp:73-75), shared by the resolve kernels
// (rt_kernels.cu) and the denoiser's last pass (rt_denoise.cu).
#pragma once
#include "rt_device.cuh"

namespace rtb {

__device__ __forceinline__ uint32_t pack_lane(float v) {
    const float s = v * 255.f;                              // Common.hpp:190-193 (int)(c*255)
    int i;
    // out-of-range and NaN conversions give INT_MIN on the reference's x86 targets (cvttss2si)
    if (!(s > -2147483904.0f && s < 2147483648.0f)) i = (int)0x80000000;
    else i = __float2int_rz(s);
    if (i > 255) i = 255;                                   // :195-198
    return (uint32_t)(i & 0xff);                            // (Uint8) :200-203
}
__device__ __forceinline__ uint32_t resolve_pixel(float4 a, float count) {
    float r = a.x, g = a.y, b = a.z;
    if (count > 0.f) { r = r / count; g = g / count; b = b / count; }      // sum -> mean; count 0: already a mean
    const float R = c0(r / c0(1.f + r)), G = c0(g / c0(1.f + g)), B = c0(b / c0(1.f + b));   // :74
    return (pack_lane(R) << 16) | (pack_lane(G) << 8) | pack_lane(B);                        // alpha byte 0
}

}  // namespace rtb
