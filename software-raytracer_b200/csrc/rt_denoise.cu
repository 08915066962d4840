// rt_denoise.cu - the edge-avoiding a-trous filter behind rt_denoise_rgba8 / rt_read_denoised: one launch per pass, guided by the
// context's primary-hit cache (object id, normal, t per pixel; rt_kernels.cu k_primary_cache). Tap weight and combine: rt_denoise.cuh.
//
// Pass 0 reads the accumulation buffer (sum / count) and computes the Reinhard luminance l itself; every pass stores (r, g, b, l) so
// that the next one does not recompute l per tap; the last pass stores the Reinhard + ARGB8 pack of the plain resolve (device surface
// and, optionally, the caller's page-locked surface) or the filtered mean as (r, g, b, 0).
//
// Small steps stage the CTA's 32 x 8 tile plus its 2s apron of colour, guide and id in shared memory (36 B per staged pixel); larger
// steps, whose apron exceeds the tile, read the taps through L1 (__ldg). Compiled with -fmad=false like every file.
//
// The per-pixel count form (NEFF, behind the temporal resolve of rt_temporal.cu) filters a blend of samples and reprojected
// history: every pass reads (r, g, b, l) images, and the colour tolerance of pixel p uses its own weight N_eff(p) instead of the
// sample count (rt_temporal.cuh tp_kc).
#include "rt_kernels.h"

#include <cstdlib>

#include "rt_denoise.cuh"
#include "rt_resolve.cuh"
#include "rt_temporal.cuh"

namespace rtb {

namespace {

constexpr int kDnTileW = 32, kDnTileH = 8;
constexpr int kDnMaxStagedStep = 4;   // (32 + 16) x (8 + 16) x 36 B = 41.5 KB: the largest step whose staged tile fits 48 KB

enum { kDnOutNext = 0, kDnOutMean = 1, kDnOutArgb = 2 };

struct DenoiseIO {
    const float4* accum;       // pass 0 input: the accumulation buffer; NEFF: (r, g, b, N_eff) per pixel (rt_temporal.cu)
    float count;               // its sample count (0: it already holds a mean); NEFF: sigma_c * sigma_c
    const float4* cin;         // later passes: (r, g, b, l) of the previous pass
    const float4* nt;          // guides: (normal, t) and object id per pixel (-1: the primary ray missed)
    const int* id;
    int width, height;
    int copy_only;             // 1: every pixel is copied (no filtering; passes == 0 or preview)
    float4* out;               // kDnOutNext / kDnOutMean
    uint32_t* argb;            // kDnOutArgb: device surface (whole image) ...
    uint32_t* argb_host;       // ... and the device alias of a page-locked host surface, or nullptr
    int flip_y;
};

template <bool FIRST>
__device__ __forceinline__ float4 dn_load(const DenoiseIO& io, size_t q) {
    if (FIRST) return dn_mean(__ldg(io.accum + q), io.count);
    return __ldg(io.cin + q);
}

template <int OUT, bool NEFF>
__device__ __forceinline__ void dn_store(const DenoiseIO& io, int x, int y, float4 o) {
    const size_t p = (size_t)x + (size_t)y * io.width;
    if (OUT == kDnOutNext) io.out[p] = o;
    else if (OUT == kDnOutMean) io.out[p] = make_float4(o.x, o.y, o.z, NEFF ? __ldg(io.accum + p).w : 0.f);
    else {
        const uint32_t v = resolve_pixel(o, 0.f);               // a mean already: count 0
        const size_t dst = (size_t)x + (size_t)(io.flip_y ? io.height - 1 - y : y) * io.width;
        io.argb[dst] = v;
        if (io.argb_host) io.argb_host[dst] = v;
    }
}

template <bool FIRST, bool STAGED, int OUT, bool NEFF>
__global__ void __launch_bounds__(kDnTileW * kDnTileH) k_denoise_pass(DenoiseIO io, DenoisePass ps) {
    extern __shared__ float4 dn_smem[];
    const int W = io.width, H = io.height, s = ps.step;
    const int x = blockIdx.x * kDnTileW + threadIdx.x, y = blockIdx.y * kDnTileH + threadIdx.y;
    // staged layout: colour[n], (normal, t)[n], id[n] over the (32 + 4s) x (8 + 4s) window; ids outside the image are -1
    const int apron = 2 * s, sw = kDnTileW + 2 * apron, n = sw * (kDnTileH + 2 * apron);
    float4* s_c = dn_smem;
    float4* s_nt = dn_smem + n;
    int* s_id = reinterpret_cast<int*>(dn_smem + 2 * n);
    if (STAGED) {
        const int x0 = blockIdx.x * kDnTileW - apron, y0 = blockIdx.y * kDnTileH - apron;
        for (int k = threadIdx.y * kDnTileW + threadIdx.x; k < n; k += kDnTileW * kDnTileH) {
            const int gx = x0 + k % sw, gy = y0 + k / sw;
            int idq = -1;
            if (gx >= 0 && gx < W && gy >= 0 && gy < H) {
                const size_t q = (size_t)gx + (size_t)gy * W;
                idq = __ldg(io.id + q);
                if (idq >= 0) { s_nt[k] = __ldg(io.nt + q); s_c[k] = dn_load<FIRST>(io, q); }
            }
            s_id[k] = idq;
        }
        __syncthreads();
    }
    if (x >= W || y >= H) return;
    const size_t p = (size_t)x + (size_t)y * W;
    const int kc = (threadIdx.y + apron) * sw + threadIdx.x + apron;   // centre in the staged window
    const int idp = io.copy_only ? -1 : STAGED ? s_id[kc] : __ldg(io.id + p);
    if (idp < 0) {                                             // sky (or no filtering): copied unchanged
        dn_store<OUT, NEFF>(io, x, y, dn_load<FIRST>(io, p));
        return;
    }
    const float4 np = STAGED ? s_nt[kc] : __ldg(io.nt + p);
    const float4 cp = STAGED ? s_c[kc] : dn_load<FIRST>(io, p);
    const float dz = dn_depth_scale(ps, np.w);
    DenoisePass pp = ps;
    if (NEFF) pp.kc = tp_kc(s, __ldg(io.accum + p).w, io.count);
    DenoiseAcc acc = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
    for (int dy = -2; dy <= 2; ++dy) {
        const float hy = dn_h(dy);
        const int qy = y + dy * s;
        if (!STAGED && (qy < 0 || qy >= H)) continue;
#pragma unroll 1
        for (int dx = -2; dx <= 2; ++dx) {
            const int qx = x + dx * s;
            float4 nq, cq;
            if (STAGED) {
                const int k = kc + dy * s * sw + dx * s;
                if (s_id[k] != idp) continue;
                nq = s_nt[k]; cq = s_c[k];
            } else {
                if (qx < 0 || qx >= W) continue;
                const size_t q = (size_t)qx + (size_t)qy * W;
                if (__ldg(io.id + q) != idp) continue;
                nq = __ldg(io.nt + q); cq = dn_load<FIRST>(io, q);
            }
            const float w = dn_weight(dn_h(dx) * hy, np, dz, cp.w, nq, cq.w, pp);
            dn_add(acc, w, cq);
        }
    }
    dn_store<OUT, NEFF>(io, x, y, dn_finish(acc));
}

template <bool FIRST, bool STAGED, bool NEFF = false>
cudaError_t dn_launch(int out, dim3 grid, size_t smem, cudaStream_t st, const DenoiseIO& io, const DenoisePass& ps) {
    const dim3 block(kDnTileW, kDnTileH);
    if (out == kDnOutNext) k_denoise_pass<FIRST, STAGED, kDnOutNext, NEFF><<<grid, block, smem, st>>>(io, ps);
    else if (out == kDnOutMean) k_denoise_pass<FIRST, STAGED, kDnOutMean, NEFF><<<grid, block, smem, st>>>(io, ps);
    else k_denoise_pass<FIRST, STAGED, kDnOutArgb, NEFF><<<grid, block, smem, st>>>(io, ps);
    return cudaGetLastError();
}

// Largest step staged in shared memory (measured: DESIGN.md 8). RTB200_DENOISE_STAGE=<0|1|2|4> overrides it for A/B runs.
int stage_max_step() {
    static const int v = [] {
        const char* e = getenv("RTB200_DENOISE_STAGE");
        const int k = e ? atoi(e) : kDenoiseStageDefault;
        return k < 0 ? 0 : k > kDnMaxStagedStep ? kDnMaxStagedStep : k;
    }();
    return v;
}

}  // namespace

cudaError_t launch_denoise(const DenoiseLaunch& d, cudaStream_t st) {
    const int W = d.width, H = d.height;
    if (W <= 0 || H <= 0) return cudaSuccess;
    const dim3 grid((W + kDnTileW - 1) / kDnTileW, (H + kDnTileH - 1) / kDnTileH);
    DenoiseIO io;
    io.accum = d.accum; io.count = (float)d.samples; io.cin = nullptr;
    io.nt = d.nt; io.id = d.id; io.width = W; io.height = H; io.copy_only = d.passes == 0 ? 1 : 0;
    io.out = nullptr; io.argb = d.argb; io.argb_host = d.argb_host; io.flip_y = d.flip_y;
    const int last_out = d.argb ? kDnOutArgb : kDnOutMean;
    if (d.passes == 0) {                                       // the plain mean / resolve, through the same store
        io.out = d.buf[0];
        return dn_launch<true, false>(last_out, grid, 0, st, io, dn_pass(0, d.pow_log2, d.sigma_color, d.sigma_depth, d.samples));
    }
    const int stage_max = stage_max_step();
    const bool neff = d.neff != nullptr;
    if (neff) { io.accum = d.neff; io.count = d.sigma_color * d.sigma_color; }
    for (int i = 0; i < d.passes; ++i) {
        const DenoisePass ps = dn_pass(i, d.pow_log2, d.sigma_color, d.sigma_depth, d.samples);
        const bool staged = ps.step <= stage_max;
        const int a = 2 * ps.step;
        const size_t smem = staged ? (size_t)(kDnTileW + 2 * a) * (kDnTileH + 2 * a) * (2 * sizeof(float4) + sizeof(int)) : 0;
        const int out = i == d.passes - 1 ? last_out : kDnOutNext;
        io.cin = i > 0 || neff ? d.buf[(i - 1) & 1] : nullptr;   // NEFF pass 0: buf[1]
        io.out = d.buf[i & 1];
        cudaError_t e;
        if (neff) e = staged ? dn_launch<false, true, true>(out, grid, smem, st, io, ps) : dn_launch<false, false, true>(out, grid, smem, st, io, ps);
        else if (i == 0) e = staged ? dn_launch<true, true>(out, grid, smem, st, io, ps) : dn_launch<true, false>(out, grid, smem, st, io, ps);
        else e = staged ? dn_launch<false, true>(out, grid, smem, st, io, ps) : dn_launch<false, false>(out, grid, smem, st, io, ps);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace rtb
