// Host build of the pixel filter (csrc/rt_filter.cuh) through cuda_shim.h: filter_offset() on given Philox words and
// filtered_ray_dir() of every pixel of a frame (test infrastructure only - the product runs the CUDA kernels).
#include "cuda_shim.h"
#define RTB_HOST_EMULATION 1
#include "../../software-raytracer_b200/csrc/rt_filter.cuh"
#include "../../software-raytracer_b200/csrc/rt_host_pack.h"

using namespace rtb;

extern "C" {

void emu_filter_offsets(int type, float radius, const uint32_t* words, int n, float* out) {
    for (int i = 0; i < n; ++i) out[i] = filter_offset(type, radius, words[i]);
}

// width * height * 3 floats, y-up: the primary direction of global sample `sample` of every pixel (the seed of `par` is the key)
void emu_sample_dirs(const rt_camera* cam, const rt_params* par, int type, float radius, uint32_t sample, float* out) {
    FrameView fr;
    fill_frame_view(*cam, *par, fr);
    const PixelFilter pf = {type, radius};
    for (int py = 0; py < fr.height; ++py)
        for (int px = 0; px < fr.width; ++px) {
            const uint32_t pixel = (uint32_t)px + (uint32_t)py * (uint32_t)fr.width;
            const float3 d = filtered_ray_dir(fr, pf, px, py, pixel, sample);
            out[3 * (size_t)pixel] = d.x; out[3 * (size_t)pixel + 1] = d.y; out[3 * (size_t)pixel + 2] = d.z;
        }
}

}  // extern "C"
