// rt_denoise.cuh - the per-tap weight and the per-pixel combine of the edge-avoiding a-trous filter (rt_denoise_rgba8,
// rt_read_denoised; kernels in rt_denoise.cu). __host__ __device__ and free of CUDA-only calls, so that
// tests/host_emu/cuda_shim.h can compile them for the CPU and tests/denoise_reference.py can pin them.
//
// Pass i (0-based, step s = 2^i) replaces the mean radiance c of every pixel p whose primary ray hits something by
//     sum_q w_pq c_q / sum_q w_pq,   q = p + s (dx, dy), dx, dy in -2..2 (dy outer, dx inner), taps outside the image skipped,
//     w_pq = h[dx] h[dy] [id_q == id_p] max(0, n_p . n_q)^P exp(-(|t_p - t_q| / dz_p + (l_p - l_q)^2 kc))
// with h = (1, 4, 6, 4, 1) / 16, dz_p = (sigma_z s) max(|t_p|, 1e-3), kc = 4^i N / sigma_c^2 (N = samples, at least 1) and
// l = Y / (1 + Y) the Reinhard-mapped luminance of the pass input. Pixels whose primary ray misses are copied. Every operation is
// float32, evaluated in the order written here; the reference (tests/denoise_reference.py) uses the same order.
#pragma once

namespace rtb {

constexpr int kDenoiseMaxPasses = 8;

// Reinhard-mapped luminance of a mean radiance (Rec. 709 weights)
__host__ __device__ __forceinline__ float dn_luma(float r, float g, float b) {
    const float Y = 0.2126f * r + 0.7152f * g + 0.0722f * b;
    return Y / (1.f + Y);
}

// B3-spline tap weight h[d] for d in -2..2
__host__ __device__ __forceinline__ float dn_h(int d) { return d == 0 ? 0.375f : (d == 1 || d == -1) ? 0.25f : 0.0625f; }

// The constants of one pass, computed once on the host.
struct DenoisePass {
    int step;          // s = 2^i
    int pow_log2;      // log2(P): max(0, n_p . n_q) is squared this many times
    float sz;          // sigma_z * s
    float kc;          // 4^i * N / sigma_c^2, as ((float)4^i * (float)N) / (sigma_c * sigma_c)
};
__host__ __device__ __forceinline__ DenoisePass dn_pass(int i, int pow_log2, float sigma_c, float sigma_z, unsigned int samples) {
    DenoisePass p;
    p.step = 1 << i;
    p.pow_log2 = pow_log2;
    p.sz = sigma_z * (float)p.step;
    p.kc = ((float)(1u << (2 * i)) * (float)(samples > 0u ? samples : 1u)) / (sigma_c * sigma_c);
    return p;
}

// Depth scale of the centre pixel: (sigma_z s) max(|t_p|, 1e-3). |t| because a sphere's primary t can be negative.
__host__ __device__ __forceinline__ float dn_depth_scale(const DenoisePass& ps, float tp) { return ps.sz * fmaxf(fabsf(tp), 1e-3f); }

// Weight of one tap whose object id equals the centre's: h[dx] h[dy] max(0, n_p . n_q)^P exp(-(|t_p - t_q| / dz + (l_p - l_q)^2 kc)).
__host__ __device__ __forceinline__ float dn_weight(float hw, float4 np, float dz, float lp, float4 nq, float lq, const DenoisePass& ps) {
    float d = np.x * nq.x + np.y * nq.y + np.z * nq.z;
    d = d > 0.f ? d : 0.f;
    for (int k = 0; k < ps.pow_log2; ++k) d = d * d;
    const float dl = lp - lq;
    const float e = fabsf(np.w - nq.w) / dz + dl * dl * ps.kc;
    return hw * d * expf(-e);
}

// Running sums of one pixel's taps.
struct DenoiseAcc { float r, g, b, w; };
__host__ __device__ __forceinline__ void dn_add(DenoiseAcc& a, float w, float4 c) {
    a.r += w * c.x; a.g += w * c.y; a.b += w * c.z; a.w += w;
}
// The filtered pixel as the next pass reads it: (r, g, b, l).
__host__ __device__ __forceinline__ float4 dn_finish(const DenoiseAcc& a) {
    const float r = a.r / a.w, g = a.g / a.w, b = a.b / a.w;
    float4 o;
    o.x = r; o.y = g; o.z = b; o.w = dn_luma(r, g, b);
    return o;
}

// Pass input of a pixel from the accumulation buffer: mean = sum / count (count 0: already a mean, like the plain resolve) and l.
__host__ __device__ __forceinline__ float4 dn_mean(float4 a, float count) {
    float r = a.x, g = a.y, b = a.z;
    if (count > 0.f) { r = r / count; g = g / count; b = b / count; }
    float4 o;
    o.x = r; o.y = g; o.z = b; o.w = dn_luma(r, g, b);
    return o;
}

}  // namespace rtb
