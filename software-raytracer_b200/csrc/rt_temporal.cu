// rt_temporal.cu - the temporal resolve behind rt_temporal_rgba8 / rt_read_temporal: one launch per call, one thread per pixel.
// Per-pixel math (projection, tap validity, bilinear gather, blend): rt_temporal.cuh. Prior bookkeeping: rt_capi.cu present().
//
// Each thread reads its sample sum S, its primary-hit cache entry and - when the prior is rebuilt - up to four taps of the
// previous history H and guides G; it writes the prior (when rebuilt), the new H and G into the other half of their ping-pong
// pairs (the taps of other threads still read the old ones), and one output: the (r, g, b, l) input of the filter's first pass
// (rt_denoise.cu, per-pixel count form), nothing (the caller reads H), or the ARGB8 pack of the plain resolve (device surface and,
// optionally, the caller's page-locked surface). Compiled with -fmad=false like every file.
#include "rt_kernels.h"

#include "rt_denoise.cuh"
#include "rt_resolve.cuh"
#include "rt_temporal.cuh"

namespace rtb {

namespace {

constexpr int kTpTileW = 32, kTpTileH = 8;

__global__ void __launch_bounds__(kTpTileW * kTpTileH) k_temporal(TemporalLaunch t) {
    const int W = t.width, H = t.height;
    const int x = blockIdx.x * kTpTileW + threadIdx.x, y = blockIdx.y * kTpTileH + threadIdx.y;
    if (x >= W || y >= H) return;
    const size_t p = (size_t)x + (size_t)y * W;
    const float4 S = __ldg(t.accum + p);
    const int idp = t.id ? __ldg(t.id + p) : -1;
    const float4 np = idp >= 0 ? __ldg(t.nt + p) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 P;
    if (t.mode == kTpKeep) P = t.prior[p];
    else {
        P = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t.mode == kTpCopy) P = tp_copy(__ldg(t.hist.h + p), t.cap);
        else if (t.mode == kTpReproject && idp >= 0) P = tp_reproject(t.cur, t.prev, t.m, W, H, x, y, idp, np, t.hist, t.cap, t.tau_z, t.tau_n);
        t.prior[p] = P;
    }
    const float4 O = tp_output(S, t.count, idp, P);
    t.h_out[p] = O;
    t.nt_out[p] = np;
    t.id_out[p] = idp;
    if (t.next) t.next[p] = make_float4(O.x, O.y, O.z, dn_luma(O.x, O.y, O.z));
    else if (t.argb) {
        const uint32_t v = resolve_pixel(O, 0.f);                   // a mean already: count 0
        const size_t dst = (size_t)x + (size_t)(t.flip_y ? H - 1 - y : y) * W;
        t.argb[dst] = v;
        if (t.argb_host) t.argb_host[dst] = v;
    }
}

}  // namespace

cudaError_t launch_temporal(const TemporalLaunch& t, cudaStream_t st) {
    if (t.width <= 0 || t.height <= 0) return cudaSuccess;
    const dim3 grid((t.width + kTpTileW - 1) / kTpTileW, (t.height + kTpTileH - 1) / kTpTileH), block(kTpTileW, kTpTileH);
    k_temporal<<<grid, block, 0, st>>>(t);
    return cudaGetLastError();
}

}  // namespace rtb
