// rt_temporal.cuh - the per-pixel math of the temporal resolve (rt_temporal_rgba8, rt_read_temporal; kernel in rt_temporal.cu):
// projection of the current primary hit into the previous pose, tap validity, bilinear accumulation of the history, the blend,
// and the per-pixel colour tolerance of the filter behind it. __host__ __device__ and free of CUDA-only calls, so that
// tests/host_emu/cuda_shim.h can compile them for the CPU and tests/temporal_reference.py can pin them.
//
// A pose is the origin o and the axes (u, v, f) of FrameView: ray_dir(F, x, y) = normalize(u nX + v nY + f) with
// nX = (x / W) 2 - 1, nY = (y / H) 2 - 1 (pixel corners). Pixel p = (x, y) of the current pose F' with a primary hit
// (id_p >= 0, normal n_p, t_p) reprojects as
//     X = o' + ray_dir(F', p) t_p;  (a, b, c) = M^-1 (X - o), M = [u v f] of the previous pose F (columns)
//     no history if !(c > 0); xq = ((a / c + 1) 0.5) W, yq = ((b / c + 1) 0.5) H   (pixel-corner space, the inverse of ray_dir)
// and gathers the 2 x 2 taps q = (floor(xq) + i, floor(yq) + j), bilinear weights b_q, of the history H (colour, weight W_H) and
// the previous guides G (id, normal, t). Tap q counts when it lies in the image, id_q == id_p,
// |X_q - X| <= tau_z |X - o| with X_q = o + ray_dir(F, q) t_q, and n_p . n_q >= tau_n. With A = sum b_q W_H(q) over the taps
// that count (order (0,0), (1,0), (0,1), (1,1)), the prior is P = sum b_q W_H(q) H(q) / A with weight w_P = min(cap, A)
// (w_P = 0 if A == 0). The output is O = (S + w_P P) / (N + w_P) for a pixel with w_P > 0, id_p >= 0 and N > 0 (S the
// sample sum, N the sample count), else the plain mean; its weight N_eff is N + w_P, resp. N.
//
// M^-1 is computed on the host in double (tp_inverse) and rounded to float. Every other operation is float32 in the order
// written in the code; dot products and lengths are (xx + yy) + zz. The reference (tests/temporal_reference.py) uses the same order.
#pragma once

namespace rtb {

enum { kTpKeep = 0, kTpZero = 1, kTpCopy = 2, kTpReproject = 3 };   // how a call obtains the prior (rt_capi.cu present())

// The part of a FrameView that places rays: origin and axes (a camera pose at a resolution).
struct TemporalPose { float3 o, u, v, f; };

// The previous call's history H (r, g, b, W_H) and guides G ((normal, t), id) per pixel.
struct TemporalHist { const float4* h; const float4* nt; const int* id; };

// Inverse of the column matrix [u v f] in double, rounded to float, row-major: rows (v x f, f x u, u x v) / det,
// det = u . (v x f), a x b = (a.y b.z - a.z b.y, a.z b.x - a.x b.z, a.x b.y - a.y b.x). A singular basis gives inf / NaN
// entries, whose projections fail the c > 0 test or the image bounds.
__host__ __device__ inline void tp_inverse(const TemporalPose& p, float m[9]) {
    const double u[3] = {p.u.x, p.u.y, p.u.z}, v[3] = {p.v.x, p.v.y, p.v.z}, f[3] = {p.f.x, p.f.y, p.f.z};
    const double* pairs[3][2] = {{v, f}, {f, u}, {u, v}};
    double r[3][3];
    for (int i = 0; i < 3; ++i) {
        const double* a = pairs[i][0];
        const double* b = pairs[i][1];
        r[i][0] = a[1] * b[2] - a[2] * b[1];
        r[i][1] = a[2] * b[0] - a[0] * b[2];
        r[i][2] = a[0] * b[1] - a[1] * b[0];
    }
    const double det = (u[0] * r[0][0] + u[1] * r[0][1]) + u[2] * r[0][2];
    for (int i = 0; i < 3; ++i)
        for (int k = 0; k < 3; ++k) m[3 * i + k] = (float)(r[i][k] / det);
}

// ray_dir (rt_device.cuh) with plain IEEE divisions; the device's normalized3 gives the same bits (rt_selftest(1)).
__host__ __device__ __forceinline__ float3 tp_ray_dir(const TemporalPose& f, int W, int H, int px, int py) {
    const float nX = ((float)px / (float)W) * 2.f - 1.f;
    const float nY = ((float)py / (float)H) * 2.f - 1.f;
    const float x = (f.u.x * nX + f.v.x * nY) + f.f.x;
    const float y = (f.u.y * nX + f.v.y * nY) + f.f.y;
    const float z = (f.u.z * nX + f.v.z * nY) + f.f.z;
    const float len = sqrtf((x * x + y * y) + z * z);
    return make_float3(x / len, y / len, z / len);
}

// The prior of pixel (x, y) with a primary hit (id idp, guide np = (normal, t)) reprojected from the previous pose:
// (P.rgb, w_P), all zero when no tap counts. m: tp_inverse(prev).
__host__ __device__ inline float4 tp_reproject(const TemporalPose& cur, const TemporalPose& prev, const float* m, int W, int H, int x, int y,
                                               int idp, float4 np, const TemporalHist& hist, float cap, float tau_z, float tau_n) {
    const float4 none = make_float4(0.f, 0.f, 0.f, 0.f);
    const float3 dp = tp_ray_dir(cur, W, H, x, y);
    const float X0 = cur.o.x + dp.x * np.w, X1 = cur.o.y + dp.y * np.w, X2 = cur.o.z + dp.z * np.w;
    const float d0 = X0 - prev.o.x, d1 = X1 - prev.o.y, d2 = X2 - prev.o.z;
    const float a = (m[0] * d0 + m[1] * d1) + m[2] * d2;
    const float b = (m[3] * d0 + m[4] * d1) + m[5] * d2;
    const float c = (m[6] * d0 + m[7] * d1) + m[8] * d2;
    if (!(c > 0.f)) return none;                               // behind the previous camera (or NaN)
    const float xq = ((a / c + 1.f) * 0.5f) * (float)W;
    const float yq = ((b / c + 1.f) * 0.5f) * (float)H;
    if (!(xq > -1.f && xq < (float)W && yq > -1.f && yq < (float)H)) return none;   // every tap outside the image (or NaN)
    const float fx0 = floorf(xq), fy0 = floorf(yq);
    const int x0 = (int)fx0, y0 = (int)fy0;
    const float fx = xq - fx0, fy = yq - fy0, gx = 1.f - fx, gy = 1.f - fy;
    const float lim = tau_z * sqrtf((d0 * d0 + d1 * d1) + d2 * d2);
    float A = 0.f, R = 0.f, G = 0.f, B = 0.f;
    for (int k = 0; k < 4; ++k) {
        const int qx = x0 + (k & 1), qy = y0 + (k >> 1);
        if (qx < 0 || qx >= W || qy < 0 || qy >= H) continue;
        const size_t q = (size_t)qx + (size_t)qy * (size_t)W;
        if (hist.id[q] != idp) continue;
        const float4 nq = hist.nt[q];
        const float3 dq = tp_ray_dir(prev, W, H, qx, qy);
        const float e0 = (prev.o.x + dq.x * nq.w) - X0, e1 = (prev.o.y + dq.y * nq.w) - X1, e2 = (prev.o.z + dq.z * nq.w) - X2;
        if (!(sqrtf((e0 * e0 + e1 * e1) + e2 * e2) <= lim)) continue;
        if (!((np.x * nq.x + np.y * nq.y) + np.z * nq.z >= tau_n)) continue;
        const float4 hq = hist.h[q];
        const float wq = ((k & 1) ? fx : gx) * ((k >> 1) ? fy : gy) * hq.w;
        A = A + wq;
        R = R + wq * hq.x; G = G + wq * hq.y; B = B + wq * hq.z;
    }
    if (!(A > 0.f)) return none;
    return make_float4(R / A, G / A, B / A, A < cap ? A : cap);
}

// The prior of an identical pose: the history itself, its weight capped.
__host__ __device__ __forceinline__ float4 tp_copy(float4 hp, float cap) { return make_float4(hp.x, hp.y, hp.z, hp.w < cap ? hp.w : cap); }

// The output of one pixel as (O.rgb, N_eff): the blend where there is a prior, a hit and samples, else the plain mean
// (sum / N; N == 0: the buffer already holds a mean), bit for bit the value the plain resolve packs.
__host__ __device__ __forceinline__ float4 tp_output(float4 S, float N, int idp, float4 P) {
    if (P.w > 0.f && idp >= 0 && N > 0.f) {
        const float d = N + P.w;
        return make_float4((S.x + P.w * P.x) / d, (S.y + P.w * P.y) / d, (S.z + P.w * P.z) / d, d);
    }
    if (N > 0.f) return make_float4(S.x / N, S.y / N, S.z / N, N);
    return make_float4(S.x, S.y, S.z, N);
}

// Colour tolerance of a-trous pass i (step s = 2^i) at a pixel of weight N_eff: (4^i max(N_eff, 1)) / sigma_c^2, with
// sc2 = sigma_c * sigma_c. For N_eff = N it is the kc of dn_pass (rt_denoise.cuh), bit for bit.
__host__ __device__ __forceinline__ float tp_kc(int step, float neff, float sc2) {
    return ((float)(step * step) * (neff > 0.f ? neff : 1.f)) / sc2;
}

}  // namespace rtb
