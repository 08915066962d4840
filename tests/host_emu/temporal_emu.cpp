// Host build of the temporal resolve's per-pixel math (csrc/rt_temporal.cuh) and of the filter's per-pixel count form
// (rt_denoise.cuh weights with rt_temporal.cuh tp_kc) through cuda_shim.h: rt_temporal.cu's and rt_denoise.cu's kernels as plain
// loops (test infrastructure only - the product runs the CUDA kernels).
#include "cuda_shim.h"

#include <vector>

#include "../../software-raytracer_b200/csrc/rt_denoise.cuh"
#include "../../software-raytracer_b200/csrc/rt_temporal.cuh"

using namespace rtb;

static TemporalPose pose_of(const float* p) {
    TemporalPose r;
    r.o = make_float3(p[0], p[1], p[2]); r.u = make_float3(p[3], p[4], p[5]);
    r.v = make_float3(p[6], p[7], p[8]); r.f = make_float3(p[9], p[10], p[11]);
    return r;
}

extern "C" {

// pose: 12 floats (o, u, v, f); m: 9 floats, row-major
void emu_tp_inverse(const float* pose, float* m) { tp_inverse(pose_of(pose), m); }

// The prior of every pixel (mode kTpReproject; pixels without a hit: zeros). w*h arrays: id int32, nt / hist_h / hist_nt / out float4.
void emu_tp_reproject(const float* cur, const float* prev, int w, int h, const int* id, const float* nt_f, const float* hist_h,
                      const float* hist_nt, const int* hist_id, float cap, float tau_z, float tau_n, float* out_f) {
    const TemporalPose pc = pose_of(cur), pp = pose_of(prev);
    float m[9];
    tp_inverse(pp, m);
    const float4* nt = reinterpret_cast<const float4*>(nt_f);
    TemporalHist hist;
    hist.h = reinterpret_cast<const float4*>(hist_h); hist.nt = reinterpret_cast<const float4*>(hist_nt); hist.id = hist_id;
    float4* out = reinterpret_cast<float4*>(out_f);
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            const size_t p = (size_t)x + (size_t)y * w;
            out[p] = id[p] >= 0 ? tp_reproject(pc, pp, m, w, h, x, y, id[p], nt[p], hist, cap, tau_z, tau_n) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
}

// tp_copy / tp_output per pixel over n pixels
void emu_tp_copy(const float* hist_h, int n, float cap, float* out_f) {
    for (int p = 0; p < n; ++p) reinterpret_cast<float4*>(out_f)[p] = tp_copy(reinterpret_cast<const float4*>(hist_h)[p], cap);
}
void emu_tp_output(const float* S, float N, const int* id, const float* P, int n, float* out_f) {
    for (int p = 0; p < n; ++p)
        reinterpret_cast<float4*>(out_f)[p] = tp_output(reinterpret_cast<const float4*>(S)[p], N, id[p], reinterpret_cast<const float4*>(P)[p]);
}

// The filter's per-pixel count form over (O, N_eff) images; out: (r, g, b, l) of the last pass.
void emu_tp_filter(const float* o4, const float* nt_f, const int* id, int w, int h, int passes, int pow_log2, float sigma_color,
                   float sigma_depth, float* out_f) {
    const float4* src = reinterpret_cast<const float4*>(o4);
    const float4* nt = reinterpret_cast<const float4*>(nt_f);
    const size_t n = (size_t)w * h;
    const float sc2 = sigma_color * sigma_color;
    std::vector<float4> cur(n), next(n);
    for (size_t p = 0; p < n; ++p) cur[p] = make_float4(src[p].x, src[p].y, src[p].z, dn_luma(src[p].x, src[p].y, src[p].z));
    for (int i = 0; i < passes; ++i) {
        DenoisePass ps = dn_pass(i, pow_log2, sigma_color, sigma_depth, 1u);
        const int s = ps.step;
        for (int y = 0; y < h; ++y)
            for (int x = 0; x < w; ++x) {
                const size_t p = (size_t)x + (size_t)y * w;
                const int idp = id[p];
                if (idp < 0) { next[p] = cur[p]; continue; }
                ps.kc = tp_kc(s, src[p].w, sc2);
                const float4 np = nt[p], cp = cur[p];
                const float dz = dn_depth_scale(ps, np.w);
                DenoiseAcc a = {0.f, 0.f, 0.f, 0.f};
                for (int dy = -2; dy <= 2; ++dy) {
                    const int qy = y + dy * s;
                    if (qy < 0 || qy >= h) continue;
                    for (int dx = -2; dx <= 2; ++dx) {
                        const int qx = x + dx * s;
                        if (qx < 0 || qx >= w) continue;
                        const size_t q = (size_t)qx + (size_t)qy * w;
                        if (id[q] != idp) continue;
                        dn_add(a, dn_weight(dn_h(dx) * dn_h(dy), np, dz, cp.w, nt[q], cur[q].w, ps), cur[q]);
                    }
                }
                next[p] = dn_finish(a);
            }
        cur.swap(next);
    }
    float4* out = reinterpret_cast<float4*>(out_f);
    for (size_t p = 0; p < n; ++p) out[p] = cur[p];
}

}  // extern "C"
