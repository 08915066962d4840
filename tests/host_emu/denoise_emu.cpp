// Host build of the denoiser's tap weight and combine (csrc/rt_denoise.cuh) through cuda_shim.h: the passes of rt_denoise.cu's
// kernels as plain loops (test infrastructure only - the product runs the CUDA kernels).
#include "cuda_shim.h"

#include <vector>

#include "../../software-raytracer_b200/csrc/rt_denoise.cuh"

using namespace rtb;

extern "C" {

// accum: w*h float4 sums, nt: w*h float4 (normal, t), id: w*h int32; out: w*h float4 (r, g, b, l) of the last pass.
int emu_denoise(const float* accum, unsigned int samples, const float* nt_f, const int* id, int w, int h, int passes, int pow_log2,
                float sigma_color, float sigma_depth, float* out_f) {
    const float4* acc = reinterpret_cast<const float4*>(accum);
    const float4* nt = reinterpret_cast<const float4*>(nt_f);
    const size_t n = (size_t)w * h;
    std::vector<float4> cur(n), next(n);
    for (size_t p = 0; p < n; ++p) cur[p] = dn_mean(acc[p], (float)samples);
    for (int i = 0; i < passes; ++i) {
        const DenoisePass ps = dn_pass(i, pow_log2, sigma_color, sigma_depth, samples);
        const int s = ps.step;
        for (int y = 0; y < h; ++y)
            for (int x = 0; x < w; ++x) {
                const size_t p = (size_t)x + (size_t)y * w;
                const int idp = id[p];
                if (idp < 0) { next[p] = cur[p]; continue; }
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
    return 0;
}

}  // extern "C"
