// rt_ctx.h - the context behind the C-ABI handle (include/rt_b200.h), shared by rt_capi.cu (single-device entry points)
// and rt_group.cu (library-owned multi-GPU). Internal: nothing here is part of the ABI.
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "../../include/rt_b200.h"
#include "rt_devbuf.h"
#include "rt_device.cuh"
#include "rt_kernels.h"
#include "bvh_build.h"
#include "bvh_wide.h"
#include "flat_build.h"
#include "mesh.h"
#include "scene_json.h"

using namespace rtb;       // internal header: only rt_capi.cu and rt_group.cu include it

// One-process-per-GPU exchange (rt_exchange_*): what a context knows about its peers.
struct ExchangeState {
    bool ready = false;
    int rank = 0, world = 1;
    const float4* accum[RT_MAX_PEERS] = {};
    ExchFlags* flags[RT_MAX_PEERS] = {};
    uint32_t* dst = nullptr;
    uint32_t epoch = 0;
};

struct rt_ctx {
    int device = 0;
    int sm_count = 0;
    std::string err;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;         // around the last render
    cudaEvent_t ev2 = nullptr, ev3 = nullptr;         // around the last resolve
    cudaEvent_t ev_tune[5] = {};                      // autotuners

    HostScene scene;
    rt_camera cam;
    rt_params par;
    FrameView frame;
    SceneView view;
    bool frame_dirty = true;

    // device scene
    DeviceArray<float4> d_sph; DeviceArray<int> d_sph_id;
    DeviceArray<float4> d_box; DeviceArray<int> d_box_id;
    DeviceArray<float4> d_mat;
    // mesh extension: triangle records (mesh.h)
    TriRecords tris;
    DeviceArray<float4> d_tri; DeviceArray<int> d_tri_obj;

    // BVH (built lazily; see bvh_build.h)
    HostBvh bvh;
    BvhView bview;
    DeviceArray<float4> d_bvh_nodes; DeviceArray<int> d_bvh_refs;
    DeviceArray<float4> d_bvh_slots;   // leaf-ordered primitive slots (BVHs too large to stage in shared memory)
    DeviceArray<uint4> d_bvh_qnodes;   // 32-byte quantised nodes of the same tree (bvh_build.h HostQNodes)
    int opt_bvh_quant = 1;             // RT_OPT_BVH_QUANT
    HostWideBvh wide;                  // 8-wide quantised form for BVHs read from global memory (bvh_wide.h)
    DeviceArray<uint4> d_wide_nodes; DeviceArray<int> d_wide_refs;
    bool bvh_valid = false;

    // flat two-level accelerator for small scenes (built lazily; see flat_build.h)
    HostFlat flat;
    FlatView fview;
    DeviceArray<float4> d_flat_boxes, d_flat_cull; DeviceArray<unsigned char> d_flat_slots; DeviceArray<int> d_flat_ids;
    bool flat_valid = false;

    WavefrontBuffers* wf = nullptr;    // RT_PIPELINE_WAVEFRONT state (rt_wavefront.cu), allocated on first use

    // frame buffers, width x height each
    DeviceArray<float4> d_accum;
    DeviceArray<uint32_t> d_argb;
    DeviceArray<unsigned long long> d_counters;   // kCounters words, see rt_reset_accumulation
    // per-pixel primary-hit cache (RT_OPT_PRIMARY_REUSE; rt_kernels.cu k_primary_cache): valid until the camera, the scene or
    // the resolution changes
    DeviceArray<float4> d_prim_nt; DeviceArray<int> d_prim_id;
    bool prim_valid = false;
    DeviceArray<float4> d_denoise[2];             // ping-pong images of the denoiser (rt_denoise.cu), allocated on first use
    DeviceArray<float4> d_gather;                 // member 0 of a group: the rank-order sum of every member's buffer (rt_group.cu),
                                                  // allocated on first use
    // temporal resolve (rt_temporal.cu), allocated on first use, 88 B per pixel: history H and guides G as ping-pong pairs (half
    // tp_cur holds the last call's), the prior P
    DeviceArray<float4> d_tp_h[2], d_tp_nt[2]; DeviceArray<int> d_tp_id[2];
    DeviceArray<float4> d_tp_prior;
    int tp_cur = 0;
    bool tp_valid = false;                        // a history exists; it belongs to tp_pose, tp_epoch and tp_key
    TemporalPose tp_pose = {};
    uint64_t tp_epoch = 0, tp_key = 0;
    uint64_t accum_epoch = 0;                     // bumped whenever the accumulation restarts or is replaced (rt_reset_accumulation,
                                                  // rt_write_accum, rt_set_sample_count, a resize)
    uint64_t radiance_key = 0;                    // bumped whenever the expected radiance changes (scene, mesh, radiance parameters)
    DeviceArray<ExchFlags> d_flags;               // this context's exchange flags (rt_exchange_*), zeroed at creation
    ExchangeState exch;
    DeviceArray<uint32_t> d_scratch;              // small device scratch (philox / pick)

    // accumulation state
    uint32_t samples = 0;          // samples per pixel in the buffer (global, after any external reduce)
    uint32_t next_sample = 0;      // next global sample index
    uint64_t paths = 0, total_paths = 0, total_segments_base = 0;
    int rank = 0, world = 1;
    int pixel_step = 1, strip_columns = 0;   // block-filled frames (rt_set_pixel_step)
    int opt_pipeline = RT_PIPELINE_AUTO, opt_accel = RT_ACCEL_AUTO, opt_bvh_threshold = 512;
    int opt_bvh_sched = 0, opt_bvh_wait_k = 20, opt_bvh_leaf = 4, opt_primary_reuse = 1;
    int opt_trav_stats = 0;            // RT_OPT_TRAVERSAL_STATS
    int opt_bvh_wide = 0;              // 0 (default) binary nodes, 1 wide nodes for BVHs of kWideMinPrims+ primitives, 2 always (tests)
    int opt_wf_refill = 8, opt_wf_node_min = 8, opt_wf_wave_mpaths = 0, opt_pool_tiles = 0, opt_flat_coop = 2;   // flat_coop: 0 off, 1 on, 2 measured per scene
    int tuned_flat_coop = 1;
    int tuned_accel = -1;          // RT_ACCEL_AUTO decision for the current scene/camera/params (-1: not measured yet)
    int tuned_pipeline = -1;       // RT_PIPELINE_AUTO decision for large BVH scenes (-1: not measured yet)
    float tune_pipe_ms[3] = {0.f, 0.f, 0.f};
    DeviceArray<float4> d_tune;
    float tune_ms[4] = {0.f, 0.f, 0.f, 0.f};
    int used_pipeline = RT_PIPELINE_REGEN, used_accel = RT_ACCEL_BRUTE;
    float last_render_ms = 0.f, last_resolve_ms = 0.f;
    bool render_timed = false, resolve_timed = false;
};
constexpr int kCounters = 32;      // the autotuners use d_counters + 4 as a scratch block of the same layout (rt_kernels.h kTileCursorSlot)


// helpers of rt_capi.cu that rt_group.cu uses
namespace rtb_capi {
int fail(rt_ctx* c, int code, const std::string& msg);
int prepare(rt_ctx* c);
int enable_peer_access_to(rt_ctx* c, const void* ptr, const char* what);   // no-op for the context's own device
int resolve_fused_unchecked(rt_ctx* c, const void* const* accum_ptrs, int world, uint32_t total_samples, int first_pixel, int n_pixels,
                            void* dst, int flip_y);

// Where a presented image goes: an ARGB8 host surface, or (argb NULL) the float (r, g, b, .) image of the filter or the temporal blend.
struct PresentOut {
    uint32_t* argb; int pitch_bytes; int flip_y;
    float* rgba;
};
// What present() resolves: a sum image (width * height float4 on the context's device) holding `samples` samples per pixel; `full`:
// it holds every sample of the image (not a shard's part), which the temporal history needs.
struct PresentSrc {
    const float4* sum; uint32_t samples; bool full;
};
// present()'s argument checks (output, temporal and filter parameters), with the messages of the single-context calls; *pow_log2:
// log2 of the filter's normal power
int check_present(rt_ctx* c, const char* fn, const PresentOut& out, bool full, const rt_temporal_params* tp, const rt_denoise_params* dn,
                  int* pow_log2 = nullptr);
// src NULL: the context's own accumulation buffer, {d_accum, samples, world == 1} after prepare() and the optional render
int present(rt_ctx* c, const char* fn, const PresentOut& out, const rt_temporal_params* tp, const rt_denoise_params* dn,
            const PresentSrc* src, const int* spp = nullptr);
}
