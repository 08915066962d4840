// rt_group.cu - library-owned multi-GPU (include/rt_b200.h rt_create_multi / rt_group_*): one host process, one context per
// device, samples sharded over the devices, ONE exchange per resolve - the fused reduce + resolve kernel reading every
// member's accumulation buffer over NVLink peer mappings and writing device 0's surface. Replaces what the reference does
// with 16 worker threads and a spin gate (Raytracer.cpp:331-342, 374-384, 598-607): "spawn" = rt_create_multi, "frame" =
// rt_group_render_spp (asynchronous launches on every device's stream), "join" = the event waits of rt_group_resolve_rgba8.
// The denoised and temporal resolves run the same exchange with the reduce kernel instead, which gathers the unresolved sum on
// device 0, and then present it there like a single context.
// No torch, no NCCL, no IPC: in one process the peers' buffers are ordinary device pointers once peer access is enabled, and
// the ordering between the devices' streams is expressed with CUDA events.
#include <cuda_runtime.h>

#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "rt_ctx.h"

struct rt_group {
    std::vector<rt_ctx*> ctx;
    std::vector<cudaEvent_t> ev_rendered, ev_read;    // per member, on its device (exchange())
    std::string err;
};

static thread_local std::string g_group_create_error;

namespace {

int gfail(rt_group* g, int code, const std::string& msg) {
    if (g) g->err = msg; else g_group_create_error = msg;
    return code;
}
int member_fail(rt_group* g, int i, int rc) {
    char buf[48];
    snprintf(buf, sizeof buf, "member %d (device %d): ", i, g->ctx[(size_t)i]->device);
    g->err = std::string(buf) + rt_last_error(g->ctx[(size_t)i]);
    return rc;
}
#define RTG_CUDA(g, call)                                                                       \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) return gfail(g, RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
    } while (0)

// fn(member index) on every member; with `threads` each member gets a host thread (calls that block: uploads, BVH builds,
// autotuning), otherwise they are issued one after the other (asynchronous launches). Returns the first failure.
template <typename F>
int for_members(rt_group* g, bool threads, F fn) {
    const int n = (int)g->ctx.size();
    std::vector<int> rc((size_t)n, RT_OK);
    if (threads && n > 1) {
        std::vector<std::thread> th;
        for (int i = 0; i < n; ++i) th.emplace_back([&, i] { rc[(size_t)i] = fn(i); });
        for (std::thread& t : th) t.join();
    } else {
        for (int i = 0; i < n; ++i) rc[(size_t)i] = fn(i);
    }
    for (int i = 0; i < n; ++i) if (rc[(size_t)i] < 0) return member_fail(g, i, rc[(size_t)i]);
    return rc.empty() ? RT_OK : rc[0];
}

// Every member's accumulation buffer (rank order) and the sum of their sample counts; the members must agree on the resolution.
int collect(rt_group* g, const char* fn, const void** accum, uint32_t& total) {
    const int w = g->ctx[0]->par.width, h = g->ctx[0]->par.height;
    total = 0;
    for (size_t i = 0; i < g->ctx.size(); ++i) {
        rt_ctx* c = g->ctx[i];
        const int rc = rtb_capi::prepare(c);
        if (rc != RT_OK) return member_fail(g, (int)i, rc);
        if (c->par.width != w || c->par.height != h) return gfail(g, RT_ERR_INVALID, std::string(fn) + ": members differ in resolution");
        total += c->samples;
        accum[i] = c->d_accum.get();
    }
    return RT_OK;
}

// The ordering between the members' streams around one exchange (the fused resolve, the reduce):
//   1. every member records "rendered": its samples are in its buffer;
//   2. each member waits for every other member's "rendered" and runs launch(i, first, count) over its slice of the pixels,
//      [n_px * i / n, n_px * (i + 1) / n);
//   3. it records "read": its slice is written and it has read every buffer;
//   4. every member waits for every "read": nobody touches its buffer again (next reset / render) before all have read it, and
//      whatever member 0 enqueues next sees the whole result.
// launch returns RT_OK or the group's error code (it sets g->err).
template <typename F>
int exchange(rt_group* g, F launch) {
    const int n = (int)g->ctx.size();
    for (int i = 0; i < n; ++i) {
        RTG_CUDA(g, cudaSetDevice(g->ctx[(size_t)i]->device));
        RTG_CUDA(g, cudaEventRecord(g->ev_rendered[(size_t)i], g->ctx[(size_t)i]->stream));
    }
    const long long n_px = (long long)g->ctx[0]->par.width * g->ctx[0]->par.height;
    for (int i = 0; i < n; ++i) {
        rt_ctx* c = g->ctx[(size_t)i];
        RTG_CUDA(g, cudaSetDevice(c->device));
        for (int j = 0; j < n; ++j) if (j != i) RTG_CUDA(g, cudaStreamWaitEvent(c->stream, g->ev_rendered[(size_t)j], 0));
        const int first = (int)(n_px * i / n), count = (int)(n_px * (i + 1) / n) - first;
        const int rc = launch(i, first, count);
        if (rc != RT_OK) return rc;
        RTG_CUDA(g, cudaSetDevice(c->device));
        RTG_CUDA(g, cudaEventRecord(g->ev_read[(size_t)i], c->stream));
    }
    for (int i = 0; i < n; ++i) {
        rt_ctx* c = g->ctx[(size_t)i];
        RTG_CUDA(g, cudaSetDevice(c->device));
        for (int j = 0; j < n; ++j) if (j != i) RTG_CUDA(g, cudaStreamWaitEvent(c->stream, g->ev_read[(size_t)j], 0));
    }
    return RT_OK;
}

// The group's denoised and temporal resolves: the rank-order sum of every member's buffer is gathered into member 0's d_gather
// (k_reduce_fused, each member storing its slice over NVLink), and member 0 presents it as the whole image's samples through the
// single-context path, with its own primary-hit guides, history, pose, accumulation epoch and radiance key (every setter is broadcast,
// so they are the group's). Checks everything before the first launch.
int group_present(rt_group* g, const char* fn, const rtb_capi::PresentOut& out, const rt_temporal_params* tp, const rt_denoise_params* dn) {
    if (!g) return RT_ERR_INVALID;
    const int n = (int)g->ctx.size();
    rt_ctx* c0 = g->ctx[0];
    int rc = rtb_capi::check_present(c0, fn, out, true, tp, dn);
    if (rc != RT_OK) return member_fail(g, 0, rc);
    const void* accum[RT_MAX_PEERS] = {};
    uint32_t total = 0;
    if ((rc = collect(g, fn, accum, total)) != RT_OK) return rc;
    const size_t px = (size_t)c0->par.width * c0->par.height;
    RTG_CUDA(g, cudaSetDevice(c0->device));
    if (c0->d_gather.capacity() < px) {
        RTG_CUDA(g, cudaStreamSynchronize(c0->stream));
        RTG_CUDA(g, c0->d_gather.reserve(px));
    }
    float4* sum = c0->d_gather.get();
    PeerPtrs pp;
    memset(&pp, 0, sizeof pp);
    for (int r = 0; r < n; ++r) pp.p[r] = (const float4*)accum[r];
    rc = exchange(g, [&](int i, int first, int count) -> int {
        RTG_CUDA(g, launch_reduce_fused(pp, n, first, count, sum, g->ctx[(size_t)i]->stream));   // peer access was enabled at creation
        return RT_OK;
    });
    if (rc != RT_OK) return rc;
    const rtb_capi::PresentSrc src = {sum, total, true};
    rc = rtb_capi::present(c0, fn, out, tp, dn, &src);
    return rc < 0 ? member_fail(g, 0, rc) : rc;
}

}  // namespace

extern "C" {

const char* rt_group_last_error(const rt_group* g) { return g ? g->err.c_str() : g_group_create_error.c_str(); }

int rt_create_multi(int n_devices, const int* cuda_devices, rt_group** out) {
    if (!out) return gfail(nullptr, RT_ERR_INVALID, "rt_create_multi: out is NULL");
    *out = nullptr;
    if (n_devices < 1 || n_devices > RT_MAX_PEERS) return gfail(nullptr, RT_ERR_INVALID, "rt_create_multi: 1 .. 16 devices");
    std::vector<int> dev((size_t)n_devices);
    for (int i = 0; i < n_devices; ++i) {
        dev[(size_t)i] = cuda_devices ? cuda_devices[i] : i;
        for (int j = 0; j < i; ++j)
            if (dev[(size_t)j] == dev[(size_t)i]) return gfail(nullptr, RT_ERR_INVALID, "rt_create_multi: a device is listed twice");
    }
    rt_group* g = new (std::nothrow) rt_group();
    if (!g) return gfail(nullptr, RT_ERR_NOMEM, "rt_create_multi: out of host memory");
    auto bail = [&](int rc, const std::string& msg) { rt_group_destroy(g); return gfail(nullptr, rc, msg); };
    for (int i = 0; i < n_devices; ++i) {
        rt_ctx* c = nullptr;
        const int rc = rt_create(dev[(size_t)i], &c);
        if (rc != RT_OK) return bail(rc, std::string("rt_create_multi: ") + rt_last_error(nullptr));
        g->ctx.push_back(c);
        rt_set_shard(c, i, n_devices);
    }
    // every member reads every other member's accumulation buffer and writes member 0's surface
    for (int i = 0; i < n_devices; ++i) {
        cudaError_t e = cudaSetDevice(dev[(size_t)i]);
        for (int j = 0; j < n_devices && e == cudaSuccess; ++j) {
            if (i == j) continue;
            int can = 0;
            e = cudaDeviceCanAccessPeer(&can, dev[(size_t)i], dev[(size_t)j]);
            if (e == cudaSuccess && !can) {
                char buf[128];
                snprintf(buf, sizeof buf, "rt_create_multi: device %d cannot access device %d (no peer path)", dev[(size_t)i], dev[(size_t)j]);
                return bail(RT_ERR_CUDA, buf);
            }
            if (e == cudaSuccess) e = cudaDeviceEnablePeerAccess(dev[(size_t)j], 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
        }
        cudaEvent_t a = nullptr, b = nullptr;
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&a, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b, cudaEventDisableTiming);
        g->ev_rendered.push_back(a); g->ev_read.push_back(b);
        if (e != cudaSuccess) return bail(RT_ERR_CUDA, std::string("rt_create_multi: ") + cudaGetErrorString(e));
    }
    *out = g;
    return RT_OK;
}

int rt_group_destroy(rt_group* g) {
    if (!g) return RT_ERR_INVALID;
    for (size_t i = 0; i < g->ctx.size(); ++i) {
        cudaSetDevice(g->ctx[i]->device);
        if (g->ctx[i]->stream) cudaStreamSynchronize(g->ctx[i]->stream);      // nobody still reads a buffer that is about to go
    }
    for (size_t i = 0; i < g->ctx.size(); ++i) {
        cudaSetDevice(g->ctx[i]->device);
        if (i < g->ev_rendered.size() && g->ev_rendered[i]) cudaEventDestroy(g->ev_rendered[i]);
        if (i < g->ev_read.size() && g->ev_read[i]) cudaEventDestroy(g->ev_read[i]);
        rt_destroy(g->ctx[i]);
    }
    delete g;
    return RT_OK;
}

int rt_group_size(const rt_group* g) { return g ? (int)g->ctx.size() : RT_ERR_INVALID; }

rt_ctx* rt_group_ctx(rt_group* g, int index) { return g && index >= 0 && (size_t)index < g->ctx.size() ? g->ctx[(size_t)index] : nullptr; }

int rt_group_set_scene(rt_group* g, const rt_object* objects, int n) {
    if (!g) return RT_ERR_INVALID;
    return for_members(g, true, [&](int i) { return rt_set_scene(g->ctx[(size_t)i], objects, n); });
}

int rt_group_load_scene(rt_group* g, const char* json_path) {
    if (!g) return RT_ERR_INVALID;
    return for_members(g, true, [&](int i) { return rt_load_scene(g->ctx[(size_t)i], json_path); });
}

int rt_group_set_mesh(rt_group* g, int object_index, const float* vertices_xyz, int n_vertices, const int32_t* indices, int n_triangles) {
    if (!g) return RT_ERR_INVALID;
    return for_members(g, true, [&](int i) { return rt_set_mesh(g->ctx[(size_t)i], object_index, vertices_xyz, n_vertices, indices, n_triangles); });
}

int rt_group_set_camera(rt_group* g, const rt_camera* cam) {
    if (!g) return RT_ERR_INVALID;
    return for_members(g, false, [&](int i) { return rt_set_camera(g->ctx[(size_t)i], cam); });
}

int rt_group_set_params(rt_group* g, const rt_params* p) {
    if (!g) return RT_ERR_INVALID;
    return for_members(g, false, [&](int i) { return rt_set_params(g->ctx[(size_t)i], p); });
}

int rt_group_set_option(rt_group* g, int option, int value) {
    if (!g) return RT_ERR_INVALID;
    return for_members(g, false, [&](int i) { return rt_set_option(g->ctx[(size_t)i], option, value); });
}

int rt_group_reset_accumulation(rt_group* g) {
    if (!g) return RT_ERR_INVALID;
    return for_members(g, false, [&](int i) { return rt_reset_accumulation(g->ctx[(size_t)i]); });
}

int rt_group_render_spp(rt_group* g, int spp) {
    if (!g) return RT_ERR_INVALID;
    // A member that still has to build its BVH or measure its back ends blocks inside rt_render_spp: give every member a
    // host thread then, so the devices prepare side by side. Afterwards a render is one asynchronous launch per device.
    bool cold = false;
    for (rt_ctx* c : g->ctx)
        if ((c->opt_accel == RT_ACCEL_AUTO && c->tuned_accel < 0) || (!c->bvh_valid && !c->flat_valid) || (c->opt_pipeline == RT_PIPELINE_AUTO && c->tuned_pipeline < 0)) cold = true;
    return for_members(g, cold, [&](int i) { return rt_render_spp(g->ctx[(size_t)i], spp); });
}

int rt_group_resolve_rgba8(rt_group* g, uint32_t* host_out, int pitch_bytes, int flip_y) {
    if (!g) return RT_ERR_INVALID;
    const int n = (int)g->ctx.size();
    rt_ctx* c0 = g->ctx[0];
    const int w = c0->par.width;
    if (!host_out || pitch_bytes < w * 4) return gfail(g, RT_ERR_INVALID, "rt_group_resolve_rgba8: bad output buffer");
    if (n == 1) {
        const int rc = rt_resolve_rgba8(c0, host_out, pitch_bytes, flip_y);
        return rc < 0 ? member_fail(g, 0, rc) : rc;
    }
    const void* accum[RT_MAX_PEERS] = {};
    uint32_t total = 0;
    int rc = collect(g, "rt_group_resolve_rgba8", accum, total);
    if (rc != RT_OK) return rc;
    rc = exchange(g, [&](int i, int first, int count) {
        const int r = rtb_capi::resolve_fused_unchecked(g->ctx[(size_t)i], accum, n, total, first, count, c0->d_argb.get(), flip_y);   // peer access was enabled at creation
        return r < 0 ? member_fail(g, i, r) : r;
    });
    if (rc != RT_OK) return rc;
    rc = rt_read_surface(c0, host_out, pitch_bytes);
    return rc < 0 ? member_fail(g, 0, rc) : rc;
}

int rt_group_denoise_rgba8(rt_group* g, const rt_denoise_params* p, uint32_t* host_out, int pitch_bytes, int flip_y) {
    rt_denoise_params d;
    if (!p) rt_default_denoise_params(&d);
    return group_present(g, "rt_group_denoise_rgba8", {host_out, pitch_bytes, flip_y, nullptr}, nullptr, p ? p : &d);
}

int rt_group_read_denoised(rt_group* g, const rt_denoise_params* p, float* host_rgba) {
    rt_denoise_params d;
    if (!p) rt_default_denoise_params(&d);
    return group_present(g, "rt_group_read_denoised", {nullptr, 0, 0, host_rgba}, nullptr, p ? p : &d);
}

// dn NULL: no filter
int rt_group_temporal_rgba8(rt_group* g, const rt_temporal_params* tp, const rt_denoise_params* dn, uint32_t* host_out, int pitch_bytes, int flip_y) {
    rt_temporal_params d;
    if (!tp) rt_default_temporal_params(&d);
    return group_present(g, "rt_group_temporal_rgba8", {host_out, pitch_bytes, flip_y, nullptr}, tp ? tp : &d, dn);
}

int rt_group_read_temporal(rt_group* g, const rt_temporal_params* tp, const rt_denoise_params* dn, float* host_rgba) {
    rt_temporal_params d;
    if (!tp) rt_default_temporal_params(&d);
    return group_present(g, "rt_group_read_temporal", {nullptr, 0, 0, host_rgba}, tp ? tp : &d, dn);
}

int rt_group_reset_temporal(rt_group* g) {
    if (!g) return RT_ERR_INVALID;
    return rt_reset_temporal(g->ctx[0]);                       // the history lives on member 0
}

int rt_group_get_stats(rt_group* g, rt_stats* out) {
    if (!g || !out) return RT_ERR_INVALID;
    memset(out, 0, sizeof *out);
    for (size_t i = 0; i < g->ctx.size(); ++i) {
        rt_stats s;
        const int rc = rt_get_stats(g->ctx[i], &s);
        if (rc != RT_OK) return member_fail(g, (int)i, rc);
        out->paths += s.paths; out->segments += s.segments; out->samples += s.samples;
        out->total_paths += s.total_paths; out->total_segments += s.total_segments;
        out->traced_segments += s.traced_segments; out->total_traced_segments += s.total_traced_segments;
        if (s.last_render_ms > out->last_render_ms) out->last_render_ms = s.last_render_ms;
        if (i == 0) { out->n_objects = s.n_objects; out->pipeline = s.pipeline; out->accel = s.accel; out->sm_count = s.sm_count; out->last_resolve_ms = s.last_resolve_ms; }
    }
    return RT_OK;
}

}  // extern "C"
