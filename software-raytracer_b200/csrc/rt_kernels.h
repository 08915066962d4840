// rt_kernels.h - host-visible launchers of the CUDA kernels in rt_kernels.cu, rt_wavefront.cu, rt_denoise.cu and rt_temporal.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "rt_device.cuh"
#include "rt_filter.cuh"
#include "rt_temporal.cuh"

namespace rtb {

// Which closest-hit back end a launch uses, with the device views it needs.
enum { kAccelBrute = 0, kAccelBvh = 1, kAccelFlat = 2 };
struct AccelSel {
    int kind;
    BvhView bvh;
    FlatView flat;
};

// Geometry lists up to this size are staged into shared memory by every CTA
// (8192 spheres); larger scenes go through the BVH or read global memory.
constexpr size_t kMaxStagedBytes = 128 * 1024;
// A BVH (stack + geometry + nodes + refs) up to this size is staged whole; smaller keeps more CTAs per SM.
constexpr size_t kMaxBvhStagedBytes = 48 * 1024;


// Layout of the counter block the render launchers get (rt_ctx::d_counters, or an offset into it for the autotuner's scratch):
// [0..3] segment counters, [8..12] traversal statistics, [kTileCursorSlot] the tile cursor of the pixel-pool kernel.
constexpr int kTileCursorSlot = 13;

struct PeerPtrs { const float4* p[16]; };      // every rank's accumulation buffer, rank order (RT_MAX_PEERS)

// Per-pixel primary-hit cache of a context (RT_OPT_PRIMARY_REUSE): (normal, t) and object id (-1 = miss) per pixel, y-up row-major.
struct PrimCache { const float4* nt; const int* id; };

cudaError_t launch_primary_aov(const SceneView& sc, const AccelSel& ac, const FrameView& fr, int* id, float* t,
                               float* n, float* p, cudaStream_t st);
cudaError_t launch_ray_dirs(const FrameView& fr, float* out, cudaStream_t st);
// filtered_ray_dir() (rt_filter.cuh) of global sample `sample` for every pixel: width * height * 3 floats
cudaError_t launch_sample_dirs(const FrameView& fr, PixelFilter pf, uint32_t sample, float* out, cudaStream_t st);
cudaError_t launch_trace_rays(const SceneView& sc, const AccelSel& ac, const float* org, const float* dir, int n,
                              int* id, float* t, float* nrm, float* pt, cudaStream_t st,
                              unsigned long long* counters = nullptr);   // non-NULL + binary BVH: the counting instantiation (counters[8..12])
// One primary closest-hit query per pixel into the context's cache; counters[2..3] += width * height.
cudaError_t launch_primary_cache(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* prim_nt, int* prim_id,
                                 unsigned long long* counters, cudaStream_t st);
cudaError_t launch_env_color(const FrameView& fr, const float* dir, int n, float* out, cudaStream_t st);
cudaError_t launch_philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t* dev_out4, cudaStream_t st);
cudaError_t launch_selftest_uniform(int* dev_failures, cudaStream_t st);
cudaError_t launch_selftest_normalize(int* dev_failures, cudaStream_t st);
cudaError_t launch_selftest_packed(int* dev_failures, cudaStream_t st);
cudaError_t launch_pick(const SceneView& sc, const AccelSel& ac, const FrameView& fr, int px, int py, int* dev_id, cudaStream_t st);
// A frame rendered INTO a surface (rt_render_frame): when the launch is the pixel-pool kernel's (1-2 samples), finished pixels are
// resolved into `surface` by the render kernel itself and - with `mapped_host` - copied to the caller's page-locked surface chunk by
// chunk while the render goes on; `fused` tells the caller whether that happened (else it resolves as usual).
struct FrameTarget {
    uint32_t* surface = nullptr;       // device surface, whole image
    uint32_t* mapped_host = nullptr;   // device pointer of the page-locked host surface, or nullptr
    uint32_t samples_after = 0;        // samples in the accumulation buffer once this launch is done
    int flip_y = 1;
    bool fused = false;                // out
};
// prim_cache != NULL: primary-hit reuse (every sample starts from the cached primary hit); NULL: every sample re-traces it.
cudaError_t launch_render_regen(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* accum,
                                uint32_t s_begin, int n_samples, const PrimCache* prim_cache, unsigned long long* seg_counter, cudaStream_t st,
                                int pool_override = 0,    // 0: automatic; 1: always one pixel per lane; n >= 2: pool of n tiles per warp
                                bool flat_coop = true,    // flat accelerator: warp-cooperative levels 2/3 (rt_trace.cuh)
                                bool count_traversal = false,    // binary-BVH back ends: count node visits / primitive tests into seg_counter[8..12]
                                FrameTarget* frame = nullptr,
                                const PixelFilter* filter = nullptr);   // non-NULL: the jittered forms, one primary ray per sample (prim_cache ignored)
cudaError_t launch_render_bvh(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* accum, uint32_t s_begin,
                              int n_samples, unsigned long long* seg_counter, int wait_k, cudaStream_t st);
cudaError_t launch_render_preview(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* accum,
                                  unsigned long long* seg_counter, cudaStream_t st);
cudaError_t launch_render_blocks(const SceneView& sc, const AccelSel& ac, const FrameView& fr, float4* accum, uint32_t s_begin,
                                 int n_samples, int steps, int strip_w, unsigned long long* seg_counter, cudaStream_t st);
cudaError_t launch_resolve(const float4* accum, uint32_t samples, int width, int height, int first, int n, int flip_y,
                           uint32_t* out, int out_is_slice, cudaStream_t st,
                           uint32_t* mapped_host_out = nullptr);   // device alias of a page-locked host surface (whole image, tight pitch): also written, zero-copy

cudaError_t launch_resolve_fused(const PeerPtrs& peers, int world, uint32_t samples, int width, int height, int first, int n,
                                 int flip_y, uint32_t* out, cudaStream_t st);
// The sum of launch_resolve_fused, unresolved: pixels [first, first+n) of every rank's buffer added in rank order into out[first ..]
// (whole-image buffer, y-up like the accumulation buffers).
cudaError_t launch_reduce_fused(const PeerPtrs& peers, int world, int first, int n, float4* out, cudaStream_t st);

// ---- denoised resolve (rt_denoise.cu; filter in rt_denoise.cuh) ----------------------------------------------------
// Largest a-trous step whose pass stages its tile + apron in shared memory; larger steps read through L1 (measured: DESIGN.md 8).
constexpr int kDenoiseStageDefault = 4;
struct DenoiseLaunch {
    const float4* accum; uint32_t samples;     // the accumulation buffer (samples 0: it holds a mean)
    const float4* nt; const int* id;           // guides: the primary-hit cache (unused when passes == 0)
    int width, height;
    int passes;                                // 0: no filtering (the plain mean / resolve)
    int pow_log2;                              // log2 of the normal power P
    float sigma_color, sigma_depth;
    float4* buf[2];                            // ping-pong (r, g, b, l) images; the result of a mean output is in buf[(passes - 1) & 1]
                                               // (buf[0] for passes == 0) as (r, g, b, 0)
    uint32_t* argb;                            // non-NULL: the last pass packs ARGB8 into this device surface instead (whole image) ...
    uint32_t* argb_host;                       // ... and into this device alias of a page-locked host surface, if non-NULL
    int flip_y;
    const float4* neff;                        // non-NULL: the per-pixel count form behind the temporal resolve: pass 0 reads its (r, g, b, l)
                                               // input from buf[1] (accum and samples are unused), each pixel's colour tolerance uses N_eff
                                               // = neff[p].w instead of samples (rt_temporal.cuh tp_kc), and a mean output stores (r, g, b, N_eff)
};
cudaError_t launch_denoise(const DenoiseLaunch& d, cudaStream_t st);

// ---- temporal resolve (rt_temporal.cu; per-pixel math in rt_temporal.cuh) -------------------------------------------
struct TemporalLaunch {
    const float4* accum; float count;          // S and N (count 0: the buffer holds a mean)
    const float4* nt; const int* id;           // the current primary-hit cache; id NULL: no guides (preview), every pixel the plain mean
    int width, height;
    int mode;                                  // kTpKeep / kTpZero / kTpCopy / kTpReproject
    float cap, tau_z, tau_n;
    TemporalPose cur, prev;                    // the current pose and the history's
    float m[9];                                // tp_inverse(prev)
    TemporalHist hist;                         // the history the taps read
    float4* prior;                             // (P.rgb, w_P) per pixel: read (kTpKeep) or rewritten
    float4* h_out; float4* nt_out; int* id_out;   // the new history and guides
    float4* next;                              // non-NULL: (O, l) for the filter's first pass ...
    uint32_t* argb;                            // ... else, non-NULL: the ARGB8 pack of O into this device surface (whole image) ...
    uint32_t* argb_host;                       // ... and into this device alias of a page-locked host surface, if non-NULL
    int flip_y;
};
cudaError_t launch_temporal(const TemporalLaunch& t, cudaStream_t st);

// Exchange flags of one rank (rt_exchange_*): arrive[r] / done[r] are written by rank r (over NVLink when r is a peer) with
// the epoch of the exchange; epochs only grow. 256 bytes, zeroed once when the context is created.
struct ExchFlags {
    uint32_t arrive[16];           // rank r: "my samples of epoch e are in my accumulation buffer"
    uint32_t done[16];             // rank r: "my slice of epoch e is in the destination surface and I have read your buffer"
    uint32_t error;                // set when a wait timed out (a peer never signalled)
    uint32_t blocks_done;          // CTAs of the running fused kernel that have finished (local)
    uint32_t pad[30];
};
struct ExchPeers { ExchFlags* f[16]; };
// The fused reduce + resolve with the ordering done on the device: signal arrive -> wait for every rank's -> reduce + resolve
// this rank's slice -> signal done; then a one-warp kernel waits for every rank's done.
cudaError_t launch_resolve_fused_sync(const PeerPtrs& peers, const ExchPeers& flags, int rank, int world, uint32_t epoch, uint32_t samples,
                                      int width, int height, int first, int n, int flip_y, uint32_t* out, cudaStream_t st);

}  // namespace rtb

namespace rtb {
// ---- wavefront pipeline (rt_wavefront.cu) ----------------------------------------------------------
struct WavefrontBuffers;                        // device buffers of one context, owned by the C-ABI layer
WavefrontBuffers* wavefront_create();
void wavefront_destroy(WavefrontBuffers* wb);
// Adds samples [s_begin, s_begin + n_samples) of every pixel into accum, bit-identical to launch_render_regen.
// cudaErrorMemoryAllocation: not even the smallest wave fits in device memory - the caller renders with the megakernel instead.
cudaError_t launch_render_wavefront(WavefrontBuffers* wb, const SceneView& sc, const AccelSel& ac, const FrameView& fr,
                                    float4* accum, uint32_t s_begin, int n_samples, const PrimCache* prim_cache,
                                    unsigned long long* seg_counter, cudaStream_t st, bool bvh_refill = true,
                                    int k_refill = 8, int k_node_min = 8,
                                    int wave_mpaths = 0,    // paths per wave in units of 2^20 (0: default 128, capped by free memory)
                                    bool count_traversal = false,
                                    bool streaming = false);   // RT_PIPELINE_STREAM: one persistent kernel traces AND shades whole paths (binary-BVH back ends)
void wavefront_release(WavefrontBuffers* wb);   // frees the device buffers (scene / resolution change); they are reallocated on the next use
}  // namespace rtb
