// rt_capi.cu - the C-ABI (include/rt_b200.h) over the CUDA kernels: context, scene upload as
// SoA, camera/parameter state, launch orchestration, accumulation bookkeeping.
//
// No CPU fallback lives here: every compute entry point launches kernels or fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "rt_ctx.h"
#include "rt_denoise.cuh"
#include "rt_host_pack.h"

using namespace rtb;

static thread_local std::string g_create_error;

namespace rtb_capi {
int fail(rt_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}
}  // namespace rtb_capi
using rtb_capi::fail;

namespace {

int cuda_fail(rt_ctx* c, cudaError_t e, const char* what) {
    return fail(c, RT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define RT_CUDA(ctx, call)                                              \
    do {                                                                \
        cudaError_t e__ = (call);                                       \
        if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call);      \
    } while (0)

// scene and accelerator arrays: at least 16 elements, also for an empty scene
template <typename T>
cudaError_t ensure_capacity(DeviceArray<T>& a, size_t need) { return a.reserve(need < 16 ? 16 : need); }

void build_frame(rt_ctx* c) {
    fill_frame_view(c->cam, c->par, c->frame);
    c->frame_dirty = false;
}

int ensure_buffers(rt_ctx* c) {
    size_t px = (size_t)c->par.width * c->par.height;
    if (c->d_accum.capacity() < px) {
        c->exch.ready = false;                                 // peers hold mappings of the old buffers
        const cudaError_t e = reserve_all(px, c->d_accum, c->d_argb);
        if (e != cudaSuccess) return cuda_fail(c, e, "frame buffers");
        RT_CUDA(c, cudaMemsetAsync(c->d_accum.get(), 0, px * sizeof(float4), c->stream));
        c->samples = 0; c->next_sample = 0; c->paths = 0;
    }
    return RT_OK;
}

int upload_scene(rt_ctx* c) {
    const std::vector<rt_object>& objs = c->scene.objects;
    std::vector<float4> sph, box, mat;
    std::vector<int> sph_id, box_id;
    pack_scene(objs, sph, sph_id, box, box_id, mat);
    RT_CUDA(c, cudaStreamSynchronize(c->stream));             // nothing in flight may still read the old arrays
    RT_CUDA(c, ensure_capacity(c->d_sph, sph.size()));
    RT_CUDA(c, ensure_capacity(c->d_sph_id, sph_id.size()));
    RT_CUDA(c, ensure_capacity(c->d_box, box.size()));
    RT_CUDA(c, ensure_capacity(c->d_box_id, box_id.size()));
    RT_CUDA(c, ensure_capacity(c->d_mat, mat.size()));
    if (!sph.empty()) {
        RT_CUDA(c, cudaMemcpyAsync(c->d_sph.get(), sph.data(), sph.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
        RT_CUDA(c, cudaMemcpyAsync(c->d_sph_id.get(), sph_id.data(), sph_id.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    if (!box.empty()) {
        RT_CUDA(c, cudaMemcpyAsync(c->d_box.get(), box.data(), box.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
        RT_CUDA(c, cudaMemcpyAsync(c->d_box_id.get(), box_id.data(), box_id.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    if (!mat.empty())
        RT_CUDA(c, cudaMemcpyAsync(c->d_mat.get(), mat.data(), mat.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
    c->scene.meshes.resize(objs.size());
    build_tri_records(objs, c->scene.meshes, c->tris);
    const size_t nt = (size_t)c->tris.count();
    RT_CUDA(c, ensure_capacity(c->d_tri, nt * 3));
    RT_CUDA(c, ensure_capacity(c->d_tri_obj, nt));
    if (nt) {
        RT_CUDA(c, cudaMemcpyAsync(c->d_tri.get(), c->tris.rec.data(), nt * 48, cudaMemcpyHostToDevice, c->stream));
        RT_CUDA(c, cudaMemcpyAsync(c->d_tri_obj.get(), c->tris.obj.data(), nt * 4, cudaMemcpyHostToDevice, c->stream));
    }
    RT_CUDA(c, cudaStreamSynchronize(c->stream));             // host vectors die at return
    c->view.sph = c->d_sph.get(); c->view.sph_id = c->d_sph_id.get();
    c->view.box = c->d_box.get(); c->view.box_id = c->d_box_id.get();
    c->view.mat = c->d_mat.get();
    c->view.n_sph = (int)sph_id.size(); c->view.n_box = (int)box_id.size(); c->view.n_obj = (int)objs.size();
    c->view.tri = c->d_tri.get(); c->view.tri_obj = c->d_tri_obj.get(); c->view.n_tri = (int)nt;
    c->bvh_valid = false; c->flat_valid = false; c->tuned_accel = c->tuned_pipeline = -1;
    c->prim_valid = false;
    return RT_OK;
}

// (Re)builds and uploads the BVH when the scene changed or a ray origin lies outside the extent its
// box inflation was derived from.
constexpr int kWideMinPrims = 1024;    // below this the whole BVH2 is staged in shared memory anyway (kMaxBvhStagedBytes)
int ensure_bvh(rt_ctx* c, float origin_extent) {
    if (c->bvh_valid && origin_extent <= c->bvh.extent) return RT_OK;
    const size_t prims = (size_t)c->view.n_sph + c->view.n_box + c->view.n_tri;
    if (prims >= ((size_t)1 << 24)) return fail(c, RT_ERR_INVALID, "scene has 2^24 or more primitives: not supported by the BVH's 24-bit leaf links");
    const bool want_wide = c->opt_bvh_wide == 2 || (c->opt_bvh_wide == 1 && prims >= (size_t)kWideMinPrims);
    build_bvh(c->scene.objects, origin_extent, c->bvh, want_wide ? std::min(c->opt_bvh_leaf, kWideMaxLeaf) : c->opt_bvh_leaf, &c->tris, c->par.eps);
    if (c->bvh.max_depth + 2 > 62) return fail(c, RT_ERR_INVALID, "BVH too deep for the traversal stack");
    // leaf links carry the first ref index in 24 bits (bvh_build.h BvhNode): more refs would alias
    if (c->bvh.refs.size() >= ((size_t)1 << 24)) return fail(c, RT_ERR_INVALID, "scene has 2^24 or more BVH leaf references: not supported by the 24-bit leaf links");
    c->wide = HostWideBvh();
    if (want_wide) build_wide_bvh(c->bvh, c->wide);           // not usable (huge extents, oversized leaves): the BVH2 is traversed
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    RT_CUDA(c, ensure_capacity(c->d_bvh_nodes, c->bvh.nodes.size() * 4));
    RT_CUDA(c, ensure_capacity(c->d_bvh_refs, c->bvh.refs.size()));
    RT_CUDA(c, cudaMemcpyAsync(c->d_bvh_nodes.get(), c->bvh.nodes.data(), c->bvh.nodes.size() * sizeof(BvhNode), cudaMemcpyHostToDevice, c->stream));
    if (!c->bvh.refs.empty())
        RT_CUDA(c, cudaMemcpyAsync(c->d_bvh_refs.get(), c->bvh.refs.data(), c->bvh.refs.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    if (c->wide.usable) {
        RT_CUDA(c, ensure_capacity(c->d_wide_nodes, c->wide.nodes.size() * 5));
        RT_CUDA(c, ensure_capacity(c->d_wide_refs, c->wide.refs.size()));
        RT_CUDA(c, cudaMemcpyAsync(c->d_wide_nodes.get(), c->wide.nodes.data(), c->wide.nodes.size() * sizeof(WideNode), cudaMemcpyHostToDevice, c->stream));
        if (!c->wide.refs.empty())
            RT_CUDA(c, cudaMemcpyAsync(c->d_wide_refs.get(), c->wide.refs.data(), c->wide.refs.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    // leaf-ordered primitive slots for BVHs that are traversed from global memory (rt_trace.cuh pick_mode: MODE 3)
    c->bview.slots = nullptr;
    {
        std::vector<float4> sph, box, mat; std::vector<int> sph_id, box_id;
        pack_scene(c->scene.objects, sph, sph_id, box, box_id, mat);
        const size_t staged = ((size_t)2 * (c->bvh.max_depth + 2) * 128 * sizeof(int)) + (sph.size() + box.size()) * sizeof(float4) +
                              c->bvh.nodes.size() * 64 + c->bvh.refs.size() * 4 + 16;
        if (staged > kMaxBvhStagedBytes && !c->wide.usable && !c->bvh.refs.empty()) {
            std::vector<float> slots;
            build_leaf_slots(c->bvh, reinterpret_cast<const float*>(sph.data()), sph_id.data(), reinterpret_cast<const float*>(box.data()), box_id.data(), &c->tris, slots);
            RT_CUDA(c, ensure_capacity(c->d_bvh_slots, slots.size() / 4));
            RT_CUDA(c, cudaMemcpyAsync(c->d_bvh_slots.get(), slots.data(), slots.size() * sizeof(float), cudaMemcpyHostToDevice, c->stream));
            RT_CUDA(c, cudaStreamSynchronize(c->stream));     // the host vector dies here
            c->bview.slots = c->d_bvh_slots.get();
        }
    }
    // ... and the 32-byte quantised form of the nodes for the persistent kernels (one 256-bit load per node visit)
    c->bview.qnodes = nullptr; c->bview.q2f16 = 0x4B00u;
    if (c->bview.slots && c->opt_bvh_quant) {
        HostQNodes qn;
        build_qnodes(c->bvh, qn);
        if (qn.usable) {
            RT_CUDA(c, ensure_capacity(c->d_bvh_qnodes, qn.words.size() / 4));
            RT_CUDA(c, cudaMemcpyAsync(c->d_bvh_qnodes.get(), qn.words.data(), qn.words.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
            RT_CUDA(c, cudaStreamSynchronize(c->stream));
            c->bview.qnodes = c->d_bvh_qnodes.get();
            c->bview.q_org = make_float3(qn.org[0], qn.org[1], qn.org[2]);
            c->bview.q_step = make_float3(qn.step[0], qn.step[1], qn.step[2]);
        }
    }
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    c->bview.nodes = c->d_bvh_nodes.get(); c->bview.refs = c->d_bvh_refs.get();
    c->bview.n_nodes = (int)c->bvh.nodes.size(); c->bview.n_refs = (int)c->bvh.refs.size();
    c->bview.stack_entries = c->bvh.max_depth + 2;
    c->bview.wnodes = c->wide.usable ? c->d_wide_nodes.get() : nullptr; c->bview.wrefs = c->wide.usable ? c->d_wide_refs.get() : nullptr;
    c->bview.n_wnodes = c->wide.usable ? (int)c->wide.nodes.size() : 0; c->bview.n_wrefs = c->wide.usable ? (int)c->wide.refs.size() : 0;
    c->bview.wstack_entries = c->wide.depth + 2;
    c->bview.q2f_hi = 0x47u;
    c->bvh_valid = true;
    return RT_OK;
}

// (Re)builds and uploads the flat accelerator; c->flat.usable tells whether the scene qualifies.
int ensure_flat(rt_ctx* c, float origin_extent) {
    if (c->flat_valid && origin_extent <= c->flat.extent) return RT_OK;
    build_flat(c->scene.objects, origin_extent, c->flat, c->par.eps);
    c->flat_valid = true;
    memset(&c->fview, 0, sizeof c->fview);
    if (!c->flat.usable) return RT_OK;
    const HostFlat& f = c->flat;
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    RT_CUDA(c, ensure_capacity(c->d_flat_boxes, f.boxes.size() / 4));
    RT_CUDA(c, ensure_capacity(c->d_flat_cull, f.cull.size() / 4));
    RT_CUDA(c, ensure_capacity(c->d_flat_slots, f.cull_slot.size()));
    RT_CUDA(c, ensure_capacity(c->d_flat_ids, f.prim_id.size()));
    if (!f.boxes.empty()) RT_CUDA(c, cudaMemcpyAsync(c->d_flat_boxes.get(), f.boxes.data(), f.boxes.size() * 4, cudaMemcpyHostToDevice, c->stream));
    if (!f.cull.empty()) RT_CUDA(c, cudaMemcpyAsync(c->d_flat_cull.get(), f.cull.data(), f.cull.size() * 4, cudaMemcpyHostToDevice, c->stream));
    if (!f.cull_slot.empty()) RT_CUDA(c, cudaMemcpyAsync(c->d_flat_slots.get(), f.cull_slot.data(), f.cull_slot.size(), cudaMemcpyHostToDevice, c->stream));
    if (!f.prim_id.empty()) RT_CUDA(c, cudaMemcpyAsync(c->d_flat_ids.get(), f.prim_id.data(), f.prim_id.size() * 4, cudaMemcpyHostToDevice, c->stream));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    c->fview.boxes = c->d_flat_boxes.get(); c->fview.cull = c->d_flat_cull.get(); c->fview.cull_slot = c->d_flat_slots.get(); c->fview.prim_id = c->d_flat_ids.get();
    c->fview.n_clusters = f.n_clusters; c->fview.n_cubes = f.n_cubes; c->fview.n_singles = f.n_singles; c->fview.kappa = f.kappa;
    return RT_OK;
}

float camera_extent(const rt_ctx* c) {
    float e = 0.f;
    for (int k = 0; k < 3; ++k) e = fmaxf(e, fabsf(c->cam.pos[k]));
    return e;
}

// Makes the requested back end ready for rays whose origins lie within origin_extent of the axes and fills
// the launch selector. A flat request on a scene that does not qualify degrades to the BVH.
int make_accel(rt_ctx* c, int rt_accel, float origin_extent, AccelSel& ac) {
    memset(&ac, 0, sizeof ac);
    int rc;
    if (rt_accel == RT_ACCEL_FLAT) {
        if ((rc = ensure_flat(c, origin_extent)) != RT_OK) return rc;
        if (c->flat.usable && c->view.n_tri == 0) { ac.kind = kAccelFlat; ac.flat = c->fview; return RT_OK; }
        rt_accel = RT_ACCEL_BVH;
    }
    if (rt_accel == RT_ACCEL_BVH) {
        if ((rc = ensure_bvh(c, origin_extent)) != RT_OK) return rc;
        ac.kind = kAccelBvh; ac.bvh = c->bview;
        return RT_OK;
    }
    ac.kind = kAccelBrute;
    return RT_OK;
}
int accel_of(const AccelSel& ac) { return ac.kind == kAccelFlat ? RT_ACCEL_FLAT : ac.kind == kAccelBvh ? RT_ACCEL_BVH : RT_ACCEL_BRUTE; }

// The back end a launch should use. Explicit options win; RT_ACCEL_AUTO uses the measured choice when there
// is one (autotune_accel), else: flat for scenes that qualify, BVH from `bvh_threshold` primitives, brute force
// below 8.
int want_accel(rt_ctx* c) {
    if (c->opt_accel != RT_ACCEL_AUTO) return c->opt_accel;
    if (c->tuned_accel >= 0) return c->tuned_accel;
    const int n = c->view.n_sph + c->view.n_box + c->view.n_tri;
    if (n >= c->opt_bvh_threshold || c->view.n_tri > 0) return RT_ACCEL_BVH;
    if (n >= 8 && n <= kFlatMaxPrims) return RT_ACCEL_FLAT;
    return RT_ACCEL_BRUTE;
}

// The per-pixel primary-hit cache (RT_OPT_PRIMARY_REUSE): traced once with the back end of the moment (all back ends give
// identical hits) and kept until the camera, the scene or the resolution changes.
int ensure_prim_cache(rt_ctx* c, const AccelSel& ac) {
    const size_t px = (size_t)c->par.width * c->par.height;
    if (c->prim_valid && c->d_prim_nt.capacity() >= px) return RT_OK;
    if (c->d_prim_nt.capacity() < px) {
        RT_CUDA(c, cudaStreamSynchronize(c->stream));
        const cudaError_t e = reserve_all(px, c->d_prim_nt, c->d_prim_id);
        if (e != cudaSuccess) return cuda_fail(c, e, "primary-hit cache");
    }
    RT_CUDA(c, launch_primary_cache(c->view, ac, c->frame, c->d_prim_nt.get(), c->d_prim_id.get(), c->d_counters.get(), c->stream));
    c->prim_valid = true;
    return RT_OK;
}

// what the render launchers take: the cache when reuse is on, NULL when every sample re-traces its primary ray
const PrimCache* prim_cache_arg(rt_ctx* c, PrimCache& pc) {
    if (!c->opt_primary_reuse) return nullptr;
    pc.nt = c->d_prim_nt.get(); pc.id = c->d_prim_id.get();
    return &pc;
}

// RT_ACCEL_AUTO between 8 and `bvh_threshold` primitives: all back ends give identical results and which
// one is fastest depends on the scene, so the first path-mode render after a scene/camera/parameter change
// of at least 64 spp times 16 spp of each into a scratch buffer and keeps the fastest. Below 8 primitives brute force,
// above the threshold the BVH.
int autotune_accel(rt_ctx* c, int spp) {
    if (c->opt_accel != RT_ACCEL_AUTO || c->tuned_accel >= 0) return RT_OK;
    // Measuring costs about 100 samples per pixel of work: only when the call itself is long enough to amortise it
    // (an interactive 1-spp frame loop keeps the heuristic choice of want_accel()); camera moves do not re-trigger it.
    if (spp < 64) { c->tuned_flat_coop = c->view.n_box == 0; return RT_OK; }
    const int n = c->view.n_sph + c->view.n_box + c->view.n_tri;
    if (n < 8) { c->tuned_accel = RT_ACCEL_BRUTE; return RT_OK; }
    if (n >= c->opt_bvh_threshold || c->view.n_tri > 0) { c->tuned_accel = RT_ACCEL_BVH; return RT_OK; }
    // candidates: brute force, BVH, flat. Whether the flat back end pools levels 2/3 across the warp is NOT measured here:
    // the two variants differ by less than the noise of a 16-spp run (2.618 vs 2.614 ms on Scene1) although the pooled one
    // is 8 % faster over 256+ spp; RT_OPT_FLAT_COOP 2 uses it for scenes without cubes (cube rooms lose ~10 % with it).
    const int kinds[4] = {RT_ACCEL_BRUTE, RT_ACCEL_BVH, RT_ACCEL_FLAT, RT_ACCEL_FLAT};
    const bool flat_coop = c->opt_flat_coop == 2 ? c->view.n_box == 0 : c->opt_flat_coop != 0;
    const bool coop[4] = {false, false, flat_coop, false};
    const int n_cand = 3;
    AccelSel sel[4];
    int rc;
    for (int k = 0; k < n_cand; ++k) if ((rc = make_accel(c, kinds[k], camera_extent(c), sel[k])) != RT_OK) return rc;
    const size_t px = (size_t)c->par.width * c->par.height;
    RT_CUDA(c, ensure_capacity(c->d_tune, px));
    cudaEvent_t* e = c->ev_tune;
    unsigned long long* dummy = c->d_counters.get() + 4;      // not part of the reported statistics
    cudaError_t err = cudaSuccess;
    PrimCache pc;
    if (c->opt_primary_reuse && (rc = ensure_prim_cache(c, sel[n_cand - 1])) != RT_OK) return rc;
    const PrimCache* prim = prim_cache_arg(c, pc);
    for (int pass = 0; pass < 2 && err == cudaSuccess; ++pass) {   // pass 0 warms the instruction cache
        cudaEventRecord(e[0], c->stream);
        for (int k = 0; k < n_cand && err == cudaSuccess; ++k) {
            err = launch_render_regen(c->view, sel[k], c->frame, c->d_tune.get(), 0u, 16, prim, dummy, c->stream, 1, coop[k]);
            cudaEventRecord(e[k + 1], c->stream);
        }
    }
    if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);
    if (err == cudaSuccess) for (int k = 0; k < n_cand; ++k) cudaEventElapsedTime(&c->tune_ms[k], e[k], e[k + 1]);
    if (err != cudaSuccess) return cuda_fail(c, err, "autotune_accel");
    int best = 0;
    for (int k = 1; k < n_cand; ++k) {
        if (kinds[k] == RT_ACCEL_FLAT && sel[k].kind != kAccelFlat) continue;   // scene does not qualify
        if (c->tune_ms[k] < c->tune_ms[best]) best = k;
    }
    c->tuned_flat_coop = flat_coop ? 1 : 0;
    if (getenv("RTB200_DEBUG"))
        fprintf(stderr, "[rtb200] autotune: brute %.3f ms, bvh %.3f ms, flat %.3f ms -> candidate %d\n", c->tune_ms[0], c->tune_ms[1], c->tune_ms[2], best);
    c->tuned_accel = kinds[best];
    return RT_OK;
}

// RT_PIPELINE_AUTO: the regeneration megakernel, except for BVH scenes too large to stage in shared memory
// (thousands of primitives), where the first path-mode render of 8+ samples times the megakernel, the bounce-round wavefront
// pipeline and the streaming kernel with up to 16 samples per pixel and keeps the fastest (identical results).
constexpr int kWavefrontMinSpp = 8;    // RT_PIPELINE_AUTO: calls shorter than this cannot fill a wave and stay on the megakernel
int autotune_pipeline(rt_ctx* c, const AccelSel& ac, int spp) {
    if (c->opt_pipeline != RT_PIPELINE_AUTO) return RT_OK;
    if (c->tuned_pipeline >= 0 || spp < kWavefrontMinSpp) return RT_OK;   // short calls always use the megakernel (rt_render_spp)
    const size_t prims = (size_t)c->view.n_sph + c->view.n_box + c->view.n_tri;
    // (the wavefront pipeline keeps one queue counter per bounce round: 60 rounds at most)
    if (ac.kind != kAccelBvh || prims < 2048 || c->pixel_step > 1 || c->par.max_bounces > 60) { c->tuned_pipeline = RT_PIPELINE_REGEN; return RT_OK; }
    const size_t px = (size_t)c->par.width * c->par.height;
    RT_CUDA(c, ensure_capacity(c->d_tune, px));
    if (!c->wf) c->wf = wavefront_create();
    cudaEvent_t* e = c->ev_tune;
    unsigned long long* dummy = c->d_counters.get() + 4;
    PrimCache pc;
    int rc;
    if (c->opt_primary_reuse && (rc = ensure_prim_cache(c, ac)) != RT_OK) return rc;
    const PrimCache* prim = prim_cache_arg(c, pc);
    cudaError_t err = cudaSuccess;
    // The wavefront pipelines' rate depends on how many samples share a wave (launch_render_wavefront: up to 64 per wave), so they
    // are measured with what a call of this length will really run, up to 64 samples per pixel - with 16 a 64-sample call on the
    // 1 M-triangle scene was given to the streaming kernel (26.7 ms) although the bounce rounds take 22-23 ms at that length. The
    // megakernel's time is linear in the sample count: it is timed with up to 16 and scaled. Candidates: 0 megakernel, 1 bounce-round
    // wavefront, 2 streaming kernel.
    const int n_tune = spp < 64 ? spp : 64;
    const int n_regen = n_tune < 16 ? n_tune : 16;
    bool usable[3] = {true, true, true};
    for (int pass = 0; pass < 2 && err == cudaSuccess; ++pass) {   // pass 0 allocates the wavefront buffers and warms up
        cudaEventRecord(e[0], c->stream);
        err = launch_render_regen(c->view, ac, c->frame, c->d_tune.get(), 0u, pass ? n_regen : 1, prim, dummy, c->stream);
        cudaEventRecord(e[1], c->stream);
        for (int k = 1; k <= 2 && err == cudaSuccess; ++k) {
            if (usable[k]) {
                const cudaError_t we = launch_render_wavefront(c->wf, c->view, ac, c->frame, c->d_tune.get(), 0u, n_tune, prim, dummy, c->stream, c->opt_bvh_sched == 0,
                                                               c->opt_wf_refill, c->opt_wf_node_min, c->opt_wf_wave_mpaths, false, k == 2);
                if (we == cudaErrorMemoryAllocation) usable[k] = false;      // no room for even the smallest wave: not a candidate
                else err = we;
            }
            cudaEventRecord(e[k + 1], c->stream);
        }
    }
    if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);
    float ms[3] = {0.f, 0.f, 0.f};
    if (err == cudaSuccess) for (int k = 0; k < 3; ++k) cudaEventElapsedTime(&ms[k], e[k], e[k + 1]);
    if (err != cudaSuccess) return cuda_fail(c, err, "autotune_pipeline");
    ms[0] *= (float)n_tune / (float)n_regen;
    c->tune_pipe_ms[0] = ms[0]; c->tune_pipe_ms[1] = ms[1]; c->tune_pipe_ms[2] = ms[2];
    const int kinds[3] = {RT_PIPELINE_REGEN, RT_PIPELINE_WAVEFRONT, RT_PIPELINE_STREAM};
    int best = 0;
    for (int k = 1; k < 3; ++k) if (usable[k] && ms[k] < ms[best]) best = k;
    if (getenv("RTB200_DEBUG"))
        fprintf(stderr, "[rtb200] pipeline autotune (%d spp): megakernel %.3f ms, wavefront %.3f ms%s, stream %.3f ms%s -> %d\n", n_tune, ms[0], ms[1],
                usable[1] ? "" : " (no memory)", ms[2], usable[2] ? "" : " (no memory)", kinds[best]);
    c->tuned_pipeline = kinds[best];
    // the bounce-round pipeline's path state (up to tens of GB) is not kept when it lost
    if (kinds[best] != RT_PIPELINE_WAVEFRONT && c->opt_pipeline == RT_PIPELINE_AUTO) { cudaStreamSynchronize(c->stream); wavefront_release(c->wf); }
    return RT_OK;
}

}  // namespace

namespace rtb_capi {
int prepare(rt_ctx* c) {
    if (!c) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    if (c->frame_dirty) build_frame(c);
    return ensure_buffers(c);
}

// Makes `ptr` (device memory of any context, or a CUDA-IPC mapping) loadable from kernels on this context's device.
int enable_peer_access_to(rt_ctx* c, const void* ptr, const char* what) {
    cudaPointerAttributes at;
    cudaError_t e = cudaPointerGetAttributes(&at, ptr);
    if (e != cudaSuccess || (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)) {
        cudaGetLastError();
        return fail(c, RT_ERR_INVALID, std::string(what) + ": not a device pointer");
    }
    if (at.device == c->device) return RT_OK;
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, c->device, at.device) != cudaSuccess || !can) {
        cudaGetLastError();
        char buf[160];
        snprintf(buf, sizeof buf, "%s: device %d cannot access memory of device %d (no peer path)", what, c->device, at.device);
        return fail(c, RT_ERR_CUDA, buf);
    }
    e = cudaDeviceEnablePeerAccess(at.device, 0);              // for the current device = c->device (prepare() set it)
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
    if (e != cudaSuccess) return cuda_fail(c, e, "cudaDeviceEnablePeerAccess");
    return RT_OK;
}
// rt_resolve_fused without the per-pointer look-ups: for callers that have established peer access themselves (rt_group.cu)
int resolve_fused_unchecked(rt_ctx* c, const void* const* accum_ptrs, int world, uint32_t total_samples, int first_pixel, int n_pixels,
                            void* dst, int flip_y) {
    RT_CUDA(c, cudaSetDevice(c->device));
    PeerPtrs pp;
    memset(&pp, 0, sizeof pp);
    for (int r = 0; r < world; ++r) pp.p[r] = (const float4*)accum_ptrs[r];
    RT_CUDA(c, launch_resolve_fused(pp, world, total_samples, c->par.width, c->par.height, first_pixel, n_pixels, flip_y,
                                    (uint32_t*)dst, c->stream));
    return RT_OK;
}
}  // namespace rtb_capi
using rtb_capi::prepare;
using rtb_capi::enable_peer_access_to;

extern "C" {

int rt_abi_version(void) { return RT_B200_ABI_VERSION; }

const char* rt_last_error(const rt_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

void rt_default_params(rt_params* p) {
    if (!p) return;
    memset(p, 0, sizeof *p);
    p->width = 1280; p->height = 720;                          // Raytracer.cpp:26-27
    p->max_bounces = 2;                                        // :32
    p->mode = RT_MODE_PREVIEW;                                 // SIMPLEDRAW = true :35
    p->selected_id = -1;                                       // selectedObject = NULL :53
    // SunDirection = float3(1,-1,-1).Normalized() (:55,:264): three divisions by sqrtf(3)
    float len = sqrtf(1.f * 1.f + -1.f * -1.f + -1.f * -1.f);
    p->sun_dir[0] = 1.f / len; p->sun_dir[1] = -1.f / len; p->sun_dir[2] = -1.f / len;
    const float sky[3] = {(float).2, (float).35, 1.0f}, hor[3] = {(float)1.0, 0.9f, 0.5f};
    for (int i = 0; i < 3; ++i) { p->sky[i] = sky[i] * 10.0f; p->horizon[i] = hor[i] * 5.0f; }   // :56-57
    p->ground[0] = .08f; p->ground[1] = .06f; p->ground[2] = .03f;                                // :58
    p->sun[0] = p->sun[1] = p->sun[2] = 500.f;                                                    // :59
    p->dissipation = 0.8f;                                     // :166
    p->eps = .00001f;                                          // :177
    p->seed_lo = 0; p->seed_hi = 0;
}

void rt_default_camera(rt_camera* c) {
    if (!c) return;
    memset(c, 0, sizeof *c);
    c->right[0] = 1.f; c->up[1] = 1.f; c->forward[2] = 1.f;    // Transform defaults Common.hpp:282-285
    c->fov_deg = 55;                                           // Raytracer.cpp:31
}

// Transform::RotateAboutAxis (Common.hpp:287-291): Rodrigues per basis vector, in the
// reference's expression order (host libm cosf/sinf, like the reference).
void rt_rotate_camera(rt_camera* c, float angle, const float axis[3]) {
    if (!c || !axis) return;
    auto rot = [&](float* b) {
        float ax = axis[0], ay = axis[1], az = axis[2];
        float cx = ay * b[2] - b[1] * az, cy = b[0] * az - ax * b[2], cz = ax * b[1] - b[0] * ay;   // Cross(axis, b) Common.hpp:94-96
        float dt = ax * b[0] + ay * b[1] + az * b[2];
        float co = cosf(angle), si = sinf(angle);
        float r0 = (b[0] * co + cx * si) + (ax * dt) * (1 - co);
        float r1 = (b[1] * co + cy * si) + (ay * dt) * (1 - co);
        float r2 = (b[2] * co + cz * si) + (az * dt) * (1 - co);
        b[0] = r0; b[1] = r1; b[2] = r2;
    };
    rot(c->forward); rot(c->up); rot(c->right);
}

int rt_create(int cuda_device, rt_ctx** out) {
    if (!out) return fail(nullptr, RT_ERR_INVALID, "rt_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, RT_ERR_CUDA, std::string("rt_create: no CUDA device (") + cudaGetErrorString(e) + "); this library has no CPU fallback");
    if (cuda_device < 0 || cuda_device >= count) return fail(nullptr, RT_ERR_INVALID, "rt_create: device index out of range");
    if ((e = cudaSetDevice(cuda_device)) != cudaSuccess) return cuda_fail(nullptr, e, "cudaSetDevice");
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, cuda_device)) != cudaSuccess) return cuda_fail(nullptr, e, "cudaGetDeviceProperties");
    if (prop.major != 10) {
        char buf[160];
        snprintf(buf, sizeof buf, "rt_create: device %d is sm_%d%d; this library carries sm_100a code only", cuda_device, prop.major, prop.minor);
        return fail(nullptr, RT_ERR_CUDA, buf);
    }
    rt_ctx* c = new (std::nothrow) rt_ctx();
    if (!c) return fail(nullptr, RT_ERR_NOMEM, "rt_create: out of host memory");
    c->device = cuda_device;
    c->sm_count = prop.multiProcessorCount;
    if (const char* q = getenv("RTB200_BVH_QUANT")) c->opt_bvh_quant = q[0] != '0';      // A/B runs of the quantised nodes (RT_OPT_BVH_QUANT)
    rt_default_params(&c->par);
    rt_default_camera(&c->cam);
    memset(&c->view, 0, sizeof c->view);
    memset(&c->bview, 0, sizeof c->bview);
    if ((e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreate(&c->ev0)) != cudaSuccess || (e = cudaEventCreate(&c->ev1)) != cudaSuccess ||
        (e = cudaEventCreate(&c->ev2)) != cudaSuccess || (e = cudaEventCreate(&c->ev3)) != cudaSuccess ||
        (e = cudaEventCreate(&c->ev_tune[0])) != cudaSuccess || (e = cudaEventCreate(&c->ev_tune[1])) != cudaSuccess ||
        (e = cudaEventCreate(&c->ev_tune[2])) != cudaSuccess || (e = cudaEventCreate(&c->ev_tune[3])) != cudaSuccess ||
        (e = cudaEventCreate(&c->ev_tune[4])) != cudaSuccess ||
        (e = c->d_counters.reserve(kCounters)) != cudaSuccess ||
        (e = c->d_scratch.reserve(4096 / sizeof(uint32_t))) != cudaSuccess ||
        (e = c->d_flags.reserve(1)) != cudaSuccess ||
        (e = cudaMemset(c->d_flags.get(), 0, sizeof(ExchFlags))) != cudaSuccess ||
        (e = cudaMemset(c->d_counters.get(), 0, kCounters * sizeof(unsigned long long))) != cudaSuccess) {
        int rc = cuda_fail(nullptr, e, "rt_create");
        rt_destroy(c);
        return rc;
    }
    c->stream = c->own_stream;
    // an empty scene is valid (everything is sky), like a failed Scene::Load in the reference
    int rc = upload_scene(c);
    if (rc != RT_OK) { g_create_error = c->err; rt_destroy(c); return rc; }
    *out = c;
    return RT_OK;
}

int rt_destroy(rt_ctx* c) {
    if (!c) return RT_ERR_INVALID;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);           // no kernel may still use the device arrays that `delete c` frees
    wavefront_destroy(c->wf);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev2) cudaEventDestroy(c->ev2);
    if (c->ev3) cudaEventDestroy(c->ev3);
    for (cudaEvent_t ev : c->ev_tune) if (ev) cudaEventDestroy(ev);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
    return RT_OK;
}

int rt_load_scene(rt_ctx* c, const char* json_path) {
    if (!c || !json_path) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    std::string err;
    int rc = c->scene.Load(json_path, err);
    int up = upload_scene(c);                                  // also after a partial load, like the reference
    ++c->radiance_key;
    rt_reset_accumulation(c);
    if (rc != RT_OK) return fail(c, rc, err);
    if (up != RT_OK) return up;
    return (int)c->scene.objects.size();
}

int rt_save_scene(rt_ctx* c, const char* json_path) {
    if (!c || !json_path) return RT_ERR_INVALID;
    std::string err;
    int rc = c->scene.SaveAs(json_path, err);
    return rc == RT_OK ? RT_OK : fail(c, rc, err);
}

int rt_set_scene(rt_ctx* c, const rt_object* objects, int n) {
    if (!c || n < 0 || (n > 0 && !objects)) return fail(c, RT_ERR_INVALID, "rt_set_scene: bad arguments");
    RT_CUDA(c, cudaSetDevice(c->device));
    // identical content (a host that re-submits its object array every frame): the device copy is still
    // refreshed, but the BVH and the back-end choice stay valid
    const bool same = (size_t)n == c->scene.objects.size() && c->bvh_valid && c->view.n_tri == 0 &&
                      (n == 0 || memcmp(objects, c->scene.objects.data(), (size_t)n * sizeof(rt_object)) == 0);
    c->scene.objects.assign(objects, objects + n);
    c->scene.names.resize((size_t)n);
    c->scene.meshes.assign((size_t)n, HostMesh());             // mesh data is attached afterwards (rt_set_mesh)
    for (rt_object& o : c->scene.objects) {                    // Color ctor clamp (Common.hpp:253-262)
        for (int k = 0; k < 3; ++k) {
            if (o.base[k] < 0) o.base[k] = 0;
            if (o.emissive[k] < 0) o.emissive[k] = 0;
            if (o.spec_color[k] < 0) o.spec_color[k] = 0;
        }
    }
    const int keep_tuned = same ? c->tuned_accel : -1, keep_pipe = same ? c->tuned_pipeline : -1;
    const bool keep_flat = same && c->flat_valid;
    int rc = upload_scene(c);
    ++c->radiance_key;
    if (rc != RT_OK) return rc;
    if (same) { c->bvh_valid = true; c->flat_valid = keep_flat; }
    c->tuned_accel = keep_tuned; c->tuned_pipeline = keep_pipe;
    return rt_reset_accumulation(c);
}

int rt_get_scene(rt_ctx* c, rt_object* out, int max_objects) {
    if (!c) return RT_ERR_INVALID;
    int n = (int)c->scene.objects.size();
    if (out) for (int i = 0; i < n && i < max_objects; ++i) out[i] = c->scene.objects[(size_t)i];
    return n;
}

int rt_scene_file_read(const char* json_path, rt_object* out, int max_objects, int* n_total, char* err_buf, int err_buf_len) {
    if (!json_path) return RT_ERR_INVALID;
    HostScene sc;
    std::string err;
    int rc = sc.Load(json_path, err);
    if (n_total) *n_total = (int)sc.objects.size();
    if (out) for (int i = 0; i < (int)sc.objects.size() && i < max_objects; ++i) out[i] = sc.objects[(size_t)i];
    if (err_buf && err_buf_len > 0) { strncpy(err_buf, err.c_str(), (size_t)err_buf_len - 1); err_buf[err_buf_len - 1] = 0; }
    return rc;
}

int rt_scene_file_read_names(const char* json_path, char* names_buf, int names_buf_len, char* scene_name, int scene_name_len) {
    if (!json_path) return RT_ERR_INVALID;
    HostScene sc;
    std::string err;
    sc.Load(json_path, err);
    size_t need = 0;
    for (const std::string& n : sc.names) need += n.size() + 1;
    if (names_buf && names_buf_len > 0) {
        size_t off = 0;
        for (const std::string& n : sc.names) {
            if (off + n.size() + 1 > (size_t)names_buf_len) break;
            memcpy(names_buf + off, n.c_str(), n.size() + 1);
            off += n.size() + 1;
        }
    }
    if (scene_name && scene_name_len > 0) { strncpy(scene_name, sc.scene_name.c_str(), (size_t)scene_name_len - 1); scene_name[scene_name_len - 1] = 0; }
    return (int)need;
}

int rt_scene_file_write(const char* json_path, const char* scene_name, const rt_object* objects, const char* const* names, int n) {
    if (!json_path || n < 0 || (n > 0 && !objects)) return RT_ERR_INVALID;
    HostScene sc;
    sc.scene_name = scene_name ? scene_name : "";
    for (int i = 0; i < n; ++i) sc.AddObject(objects[i], names && names[i] ? names[i] : "");
    std::string err;
    return sc.SaveAs(json_path, err);
}

const char* rt_object_name(rt_ctx* c, int index) {
    if (!c || index < 0 || (size_t)index >= c->scene.names.size()) return nullptr;
    return c->scene.names[(size_t)index].c_str();
}
int rt_set_object_name(rt_ctx* c, int index, const char* name) {
    if (!c || !name || index < 0 || (size_t)index >= c->scene.names.size()) return RT_ERR_INVALID;
    c->scene.names[(size_t)index] = name;
    return RT_OK;
}
const char* rt_scene_name(rt_ctx* c) { return c ? c->scene.scene_name.c_str() : nullptr; }

// ---- mesh extension ------------------------------------------------------------------------------
static int mesh_changed(rt_ctx* c) {
    int rc = upload_scene(c);
    ++c->radiance_key;
    if (rc != RT_OK) return rc;
    return rt_reset_accumulation(c);
}

int rt_set_mesh(rt_ctx* c, int object_index, const float* vertices_xyz, int n_vertices, const int32_t* indices, int n_triangles) {
    if (!c || object_index < 0 || (size_t)object_index >= c->scene.objects.size() || n_vertices < 0 || n_triangles < 0 ||
        (n_vertices > 0 && !vertices_xyz) || (n_triangles > 0 && !indices))
        return fail(c, RT_ERR_INVALID, "rt_set_mesh: bad arguments");
    if (c->scene.objects[(size_t)object_index].type != RT_OBJ_MESH) return fail(c, RT_ERR_INVALID, "rt_set_mesh: object is not of type RT_OBJ_MESH");
    for (int i = 0; i < 3 * n_triangles; ++i)
        if (indices[i] < 0 || indices[i] >= n_vertices) return fail(c, RT_ERR_INVALID, "rt_set_mesh: vertex index out of range");
    RT_CUDA(c, cudaSetDevice(c->device));
    c->scene.meshes.resize(c->scene.objects.size());
    HostMesh& m = c->scene.meshes[(size_t)object_index];
    m.vertices.assign(vertices_xyz, vertices_xyz + (size_t)3 * n_vertices);
    m.indices.assign(indices, indices + (size_t)3 * n_triangles);
    m.file.clear();
    return mesh_changed(c);
}

int rt_load_mesh_obj(rt_ctx* c, int object_index, const char* obj_path) {
    if (!c || !obj_path || object_index < 0 || (size_t)object_index >= c->scene.objects.size())
        return fail(c, RT_ERR_INVALID, "rt_load_mesh_obj: bad arguments");
    if (c->scene.objects[(size_t)object_index].type != RT_OBJ_MESH) return fail(c, RT_ERR_INVALID, "rt_load_mesh_obj: object is not of type RT_OBJ_MESH");
    RT_CUDA(c, cudaSetDevice(c->device));
    HostMesh m; std::string err;
    if (!load_obj(obj_path, m, err)) return fail(c, RT_ERR_IO, err);
    c->scene.meshes.resize(c->scene.objects.size());
    c->scene.meshes[(size_t)object_index] = std::move(m);
    return mesh_changed(c);
}

int rt_get_mesh_info(rt_ctx* c, int object_index, int* n_vertices, int* n_triangles) {
    if (!c || object_index < 0 || (size_t)object_index >= c->scene.objects.size()) return RT_ERR_INVALID;
    const HostMesh* m = (size_t)object_index < c->scene.meshes.size() ? &c->scene.meshes[(size_t)object_index] : nullptr;
    if (n_vertices) *n_vertices = m ? (int)(m->vertices.size() / 3) : 0;
    if (n_triangles) *n_triangles = m ? (int)(m->indices.size() / 3) : 0;
    return RT_OK;
}

int rt_set_camera(rt_ctx* c, const rt_camera* cam) {
    if (!c || !cam) return RT_ERR_INVALID;
    if (memcmp(&c->cam, cam, sizeof *cam) != 0) c->prim_valid = false;   // a host that re-submits the same pose every frame keeps the cache
    c->cam = *cam;
    c->frame_dirty = true;
    return RT_OK;
}

int rt_set_params(rt_ctx* c, const rt_params* p) {
    if (!c || !p) return RT_ERR_INVALID;
    if (p->width <= 0 || p->height <= 0 || (long long)p->width * p->height > (1ll << 28))
        return fail(c, RT_ERR_INVALID, "rt_set_params: bad resolution");
    if (p->mode != RT_MODE_PATH && p->mode != RT_MODE_PREVIEW) return fail(c, RT_ERR_INVALID, "rt_set_params: bad mode");
    bool resized = p->width != c->par.width || p->height != c->par.height;
    if (!(fabsf(p->eps) <= fabsf(c->par.eps))) { c->bvh_valid = false; c->flat_valid = false; }   // margins were derived for the old offset
    if (resized || p->max_bounces != c->par.max_bounces || p->mode != c->par.mode) c->tuned_accel = c->tuned_pipeline = -1;
    // the primary-hit cache keeps the environment colour of the pixels whose primary ray misses
    const bool env_changed = memcmp(p->sun_dir, c->par.sun_dir, sizeof p->sun_dir) || memcmp(p->sky, c->par.sky, sizeof p->sky) ||
                             memcmp(p->horizon, c->par.horizon, sizeof p->horizon) || memcmp(p->ground, c->par.ground, sizeof p->ground) ||
                             memcmp(p->sun, c->par.sun, sizeof p->sun);
    if (env_changed) c->prim_valid = false;
    // what changes the expected radiance ends a temporal history (the seed, selected_id and the pixel step do not)
    if (p->mode != c->par.mode || (p->max_bounces < 0 ? 0 : p->max_bounces) != c->par.max_bounces || env_changed ||
        memcmp(&p->dissipation, &c->par.dissipation, sizeof p->dissipation) || memcmp(&p->eps, &c->par.eps, sizeof p->eps)) ++c->radiance_key;
    c->par = *p;
    if (c->par.max_bounces < 0) c->par.max_bounces = 0;        // MAXBOUNCES = max(MAXBOUNCES, 0) Raytracer.cpp:475
    c->frame_dirty = true;
    if (resized) {
        RT_CUDA(c, cudaSetDevice(c->device));
        RT_CUDA(c, cudaStreamSynchronize(c->stream));
        // the frame buffers, the denoiser pair (32 B per pixel), a group's gather buffer (16 B per pixel) and the temporal set (88 B per
        // pixel, the history is gone with it) are sized for the old resolution
        c->d_accum.reset(); c->d_argb.reset(); c->d_gather.reset();
        for (int k = 0; k < 2; ++k) { c->d_denoise[k].reset(); c->d_tp_h[k].reset(); c->d_tp_nt[k].reset(); c->d_tp_id[k].reset(); }
        c->d_tp_prior.reset();
        c->tp_valid = false;
        ++c->accum_epoch;
        c->prim_valid = false;
        c->exch.ready = false;
        wavefront_release(c->wf);                              // sized for the old resolution (up to tens of GB)
    }
    return RT_OK;
}

int rt_set_option(rt_ctx* c, int option, int value) {
    if (!c) return RT_ERR_INVALID;
    auto bad = [&](const char* what) { return fail(c, RT_ERR_INVALID, std::string("rt_set_option: ") + what); };
    const int retune = -1;
    switch (option) {
        case RT_OPT_PIPELINE:
            if (value < RT_PIPELINE_AUTO || value > RT_PIPELINE_STREAM) return bad("RT_OPT_PIPELINE takes RT_PIPELINE_AUTO / REGEN / WAVEFRONT / STREAM");
            c->opt_pipeline = value; return RT_OK;
        case RT_OPT_ACCEL:
            if (value < RT_ACCEL_AUTO || value > RT_ACCEL_FLAT) return bad("RT_OPT_ACCEL takes RT_ACCEL_AUTO / BRUTE / BVH / FLAT");
            c->opt_accel = value; return RT_OK;
        case RT_OPT_BVH_THRESHOLD:
            if (value < 1) return bad("RT_OPT_BVH_THRESHOLD must be at least 1");
            c->opt_bvh_threshold = value; c->tuned_accel = retune; return RT_OK;
        case RT_OPT_BVH_SCHED:
            if (value != 0 && value != 1) return bad("RT_OPT_BVH_SCHED takes 0 or 1");
            c->opt_bvh_sched = value; return RT_OK;
        case RT_OPT_BVH_WIDE:
            if (value < 0 || value > 2) return bad("RT_OPT_BVH_WIDE takes 0, 1 or 2");
            c->opt_bvh_wide = value; c->bvh_valid = false; c->tuned_accel = c->tuned_pipeline = retune; return RT_OK;
        case RT_OPT_BVH_LEAF:
            if (value < 1 || value > 16) return bad("RT_OPT_BVH_LEAF takes 1 .. 16 primitives per leaf");
            c->opt_bvh_leaf = value; c->bvh_valid = false; c->tuned_accel = c->tuned_pipeline = retune; return RT_OK;
        case RT_OPT_PRIMARY_REUSE: c->opt_primary_reuse = value != 0; c->tuned_accel = c->tuned_pipeline = retune; return RT_OK;
        case RT_OPT_FLAT_COOP:
            if (value < 0 || value > 2) return bad("RT_OPT_FLAT_COOP takes 0, 1 or 2");
            c->opt_flat_coop = value; c->tuned_accel = c->tuned_pipeline = retune; return RT_OK;
        case RT_OPT_POOL_TILES:
            if (value < 0 || value > 32) return bad("RT_OPT_POOL_TILES takes 0 (automatic) .. 32");
            c->opt_pool_tiles = value; return RT_OK;
        case RT_OPT_WF_REFILL:
            if (value < 1 || value > 32) return bad("RT_OPT_WF_REFILL takes 1 .. 32 lanes");
            c->opt_wf_refill = value; return RT_OK;
        case RT_OPT_WF_NODE_MIN:
            if (value < 1 || value > 32) return bad("RT_OPT_WF_NODE_MIN takes 1 .. 32 lanes");
            c->opt_wf_node_min = value; return RT_OK;
        case RT_OPT_WF_WAVE_MPATHS:
            if (value < 0 || value > 1024) return bad("RT_OPT_WF_WAVE_MPATHS takes 0 (default) .. 1024");
            c->opt_wf_wave_mpaths = value; c->tuned_pipeline = retune; return RT_OK;
        case RT_OPT_BVH_WAIT_K:
            if (value < 1 || value > 32) return bad("RT_OPT_BVH_WAIT_K takes 1 .. 32 lanes");
            c->opt_bvh_wait_k = value; return RT_OK;
        case RT_OPT_TRAVERSAL_STATS: c->opt_trav_stats = value != 0; return RT_OK;
        case RT_OPT_BVH_QUANT: c->opt_bvh_quant = value != 0; c->bvh_valid = false; c->tuned_pipeline = retune; return RT_OK;
    }
    return fail(c, RT_ERR_INVALID, "rt_set_option: unknown option");
}

int rt_set_pixel_step(rt_ctx* c, int steps, int strip_columns) {
    if (!c || steps < 1 || strip_columns < 0) return fail(c, RT_ERR_INVALID, "rt_set_pixel_step: bad arguments");
    c->pixel_step = steps; c->strip_columns = strip_columns;
    return RT_OK;
}

int rt_reference_pixel_step(float screen_scale, float progressive_scaler) {
    return (int)ceil(1 / ((float)screen_scale * progressive_scaler));             // Raytracer.cpp:233
}

int rt_reference_strip_columns(int width) { return (int)ceil(width / 16) + 1; }   // Raytracer.cpp:28,330 (integer division first)

void rt_default_pixel_filter(rt_pixel_filter* f) {
    if (!f) return;
    memset(f, 0, sizeof *f);
    f->type = RT_FILTER_NONE; f->radius = 0.5f;
}

int rt_set_pixel_filter(rt_ctx* c, const rt_pixel_filter* f) {
    if (!c) return RT_ERR_INVALID;
    rt_pixel_filter v;
    rt_default_pixel_filter(&v);
    if (f) {
        if (f->type != RT_FILTER_NONE && f->type != RT_FILTER_BOX && f->type != RT_FILTER_TENT)
            return fail(c, RT_ERR_INVALID, "rt_set_pixel_filter: type takes RT_FILTER_NONE / BOX / TENT");
        if (!(std::isfinite(f->radius) && f->radius > 0.f && f->radius <= 4.f))
            return fail(c, RT_ERR_INVALID, "rt_set_pixel_filter: radius must be finite and in (0, 4]");
        if (f->reserved[0] != 0 || f->reserved[1] != 0) return fail(c, RT_ERR_INVALID, "rt_set_pixel_filter: reserved words must be 0");
        v = *f;
    }
    if (memcmp(&v, &c->filter, sizeof v) != 0) ++c->radiance_key;   // the expected radiance of a pixel changes: a temporal history ends
    c->filter = v;
    return RT_OK;
}

int rt_get_pixel_filter(rt_ctx* c, rt_pixel_filter* out) {
    if (!c || !out) return RT_ERR_INVALID;
    *out = c->filter;
    return RT_OK;
}

int rt_set_shard(rt_ctx* c, int rank, int world) {
    if (!c || world < 1 || rank < 0 || rank >= world) return fail(c, RT_ERR_INVALID, "rt_set_shard: bad rank/world");
    c->rank = rank; c->world = world;
    return RT_OK;
}

int rt_shard_range(int spp, int rank, int world, uint32_t next_sample, uint32_t* first, int* count) {
    if (spp < 0 || world < 1 || rank < 0 || rank >= world || !first || !count) return RT_ERR_INVALID;
    const int base = spp / world, rem = spp % world;          // the first `rem` ranks take one extra sample
    *count = base + (rank < rem ? 1 : 0);
    *first = next_sample + (uint32_t)(rank * base + (rank < rem ? rank : rem));
    return RT_OK;
}

int rt_reset_accumulation(rt_ctx* c) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    RT_CUDA(c, cudaMemsetAsync(c->d_accum.get(), 0, (size_t)c->par.width * c->par.height * sizeof(float4), c->stream));
    // counters: [0] segments since the last reset, [1] since rt_create (never cleared); [2], [3] the same for the
    // closest-hit queries actually executed (primary-hit reuse); [4..7] scratch for the autotuner; [8..12] BVH traversal
    // statistics since the last reset (RT_OPT_TRAVERSAL_STATS: queries, node visits, sphere / cube / triangle tests)
    RT_CUDA(c, cudaMemsetAsync(c->d_counters.get(), 0, sizeof(unsigned long long), c->stream));
    RT_CUDA(c, cudaMemsetAsync(c->d_counters.get() + 2, 0, sizeof(unsigned long long), c->stream));
    RT_CUDA(c, cudaMemsetAsync(c->d_counters.get() + 8, 0, 8 * sizeof(unsigned long long), c->stream));
    c->samples = 0; c->next_sample = 0; c->paths = 0;
    ++c->accum_epoch;
    return RT_OK;
}

// rt_render_spp; `frame` != nullptr (rt_render_frame): the launch may resolve the frame itself (FrameTarget::fused)
static int render_samples(rt_ctx* c, int spp, FrameTarget* frame) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (spp < 0) return fail(c, RT_ERR_INVALID, "rt_render_spp: negative spp");
    if (spp == 0) return RT_OK;
    const size_t px = (size_t)c->par.width * c->par.height;
    if (c->par.mode == RT_MODE_PATH && (rc = autotune_accel(c, spp)) != RT_OK) return rc;
    AccelSel ac;
    if ((rc = make_accel(c, want_accel(c), camera_extent(c), ac)) != RT_OK) return rc;
    c->used_accel = accel_of(ac);
    // a pixel filter applies to full-resolution path renders, which then run the megakernel's jittered forms (rt_set_pixel_filter)
    const bool filtered = c->filter.type != RT_FILTER_NONE && c->par.mode == RT_MODE_PATH && c->pixel_step == 1;
    const PixelFilter pf = {c->filter.type, c->filter.radius};
    if (c->par.mode == RT_MODE_PATH && !filtered && (rc = autotune_pipeline(c, ac, spp)) != RT_OK) return rc;
    RT_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    if (c->pixel_step > 1) {
        // SCREEN_SCALE / progressive resolution: one path per block, block-filled (Raytracer.cpp:233-248)
        int mine = 1; uint32_t first = 0;
        if (c->par.mode == RT_MODE_PATH) rt_shard_range(spp, c->rank, c->world, c->next_sample, &first, &mine);
        RT_CUDA(c, launch_render_blocks(c->view, ac, c->frame, c->d_accum.get(), first, mine, c->pixel_step, c->strip_columns, c->d_counters.get(), c->stream));
        const int sw = c->strip_columns > 0 && c->strip_columns < c->par.width ? c->strip_columns : c->par.width;
        uint64_t blocks = 0;
        for (int x0 = 0; x0 < c->par.width; x0 += sw) {
            const int len = (x0 + sw < c->par.width ? sw : c->par.width - x0);
            blocks += (uint64_t)((len + c->pixel_step - 1) / c->pixel_step);
        }
        blocks *= (uint64_t)((c->par.height + c->pixel_step - 1) / c->pixel_step);
        if (c->par.mode == RT_MODE_PREVIEW) { c->samples = 1; c->next_sample = 0; }
        else { c->next_sample += (uint32_t)spp; c->samples += (uint32_t)mine; }
        c->paths += blocks * (uint64_t)mine; c->total_paths += blocks * (uint64_t)mine;
        c->used_pipeline = RT_PIPELINE_REGEN;
    } else if (c->par.mode == RT_MODE_PREVIEW) {
        // SIMPLEDRAW: ACCUMULATIONFRAMES stays 1, every frame overwrites (Raytracer.cpp:66-67,589)
        RT_CUDA(c, launch_render_preview(c->view, ac, c->frame, c->d_accum.get(), c->d_counters.get(), c->stream));
        c->samples = 1; c->next_sample = 0; c->paths += px; c->total_paths += px;
    } else {
        // this rank's slice of the global sample indices [next, next+spp)
        int mine = 0; uint32_t first = 0;
        rt_shard_range(spp, c->rank, c->world, c->next_sample, &first, &mine);
        const int pipe = filtered ? RT_PIPELINE_REGEN
                       : c->opt_pipeline != RT_PIPELINE_AUTO ? c->opt_pipeline : (c->tuned_pipeline > 0 && mine >= kWavefrontMinSpp ? c->tuned_pipeline : RT_PIPELINE_REGEN);
        // the streaming kernel walks the binary BVH only; for other back ends RT_PIPELINE_STREAM runs the bounce-round kernels
        const bool streaming = pipe == RT_PIPELINE_STREAM && ac.kind == kAccelBvh && !ac.bvh.wnodes && c->opt_bvh_sched == 0;
        bool wavefront = (pipe == RT_PIPELINE_WAVEFRONT || pipe == RT_PIPELINE_STREAM) &&
                         (streaming || c->par.max_bounces <= 60);   // bounce rounds: one queue counter per round; deeper paths use the megakernel
        const bool scheduled = !wavefront && !filtered && ac.kind == kAccelBvh && c->opt_bvh_sched && c->view.n_tri == 0;   // experimental kernel, re-traces primaries
        PrimCache pc;
        if (c->opt_primary_reuse && !scheduled && !filtered && mine > 0 && (rc = ensure_prim_cache(c, ac)) != RT_OK) return rc;
        const PrimCache* prim = prim_cache_arg(c, pc);
        if (wavefront) {
            if (!c->wf) c->wf = wavefront_create();
            const cudaError_t we = launch_render_wavefront(c->wf, c->view, ac, c->frame, c->d_accum.get(), first, mine, prim, c->d_counters.get(), c->stream, c->opt_bvh_sched == 0,
                                                           c->opt_wf_refill, c->opt_wf_node_min, c->opt_wf_wave_mpaths, c->opt_trav_stats != 0, streaming);
            if (we == cudaErrorMemoryAllocation) {
                // not even one sample per pixel of path state fits next to what else lives on the device: the megakernel
                // needs no state and gives the same image (nothing was launched: allocation precedes the first kernel)
                wavefront = false;
                if (c->opt_pipeline == RT_PIPELINE_AUTO) c->tuned_pipeline = RT_PIPELINE_REGEN;
            } else {
                RT_CUDA(c, we);
                c->used_pipeline = streaming ? RT_PIPELINE_STREAM : RT_PIPELINE_WAVEFRONT;
            }
        }
        if (wavefront) {}
        else if (scheduled)
            RT_CUDA(c, launch_render_bvh(c->view, ac, c->frame, c->d_accum.get(), first, mine, c->d_counters.get(), c->opt_bvh_wait_k, c->stream));
        else {
            if (frame) frame->samples_after = c->samples + (uint32_t)mine;
            RT_CUDA(c, launch_render_regen(c->view, ac, c->frame, c->d_accum.get(), first, mine, prim, c->d_counters.get(), c->stream, c->opt_pool_tiles,
                                           c->opt_flat_coop == 2 ? (c->opt_accel == RT_ACCEL_AUTO ? c->tuned_flat_coop != 0 : c->view.n_box == 0) : c->opt_flat_coop != 0,
                                           c->opt_trav_stats != 0, c->world == 1 && mine > 0 ? frame : nullptr, filtered ? &pf : nullptr));
        }
        if (!wavefront) c->used_pipeline = RT_PIPELINE_REGEN;
        c->next_sample += (uint32_t)spp;
        c->samples += (uint32_t)mine;      // what THIS buffer holds; rt_set_sample_count after an external reduce
        c->paths += (uint64_t)mine * px; c->total_paths += (uint64_t)mine * px;
    }
    RT_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    c->render_timed = true;
    return RT_OK;
}

int rt_render_spp(rt_ctx* c, int spp) { return render_samples(c, spp, nullptr); }

// Device pointer of a page-locked host surface with a tight pitch, else nullptr. The kernels store to such a surface (rt_host_alloc)
// themselves, over PCIe (zero-copy): an interactive frame then has no separate device-to-host copy to set up and wait for.
// RTB200_ZEROCOPY=0 turns it off.
static uint32_t* mapped_surface(uint32_t* host_out, int pitch_bytes, int w) {
    static const bool zero_copy = [] { const char* v = getenv("RTB200_ZEROCOPY"); return !(v && v[0] == '0'); }();
    if (!zero_copy || pitch_bytes != w * 4) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host_out) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) return (uint32_t*)at.devicePointer;
    cudaGetLastError();
    return nullptr;
}

// the filter parameters of rt_denoise_rgba8 / rt_read_denoised / the temporal calls and log2 of the normal power
static int check_denoise_params(rt_ctx* c, const char* fn, const rt_denoise_params& p, int& pow_log2) {
    pow_log2 = 0;
    while (pow_log2 < 9 && (1 << pow_log2) != p.normal_power) ++pow_log2;
    if (p.passes < 0 || p.passes > kDenoiseMaxPasses) return fail(c, RT_ERR_INVALID, std::string(fn) + ": passes must be 0 .. 8");
    if (pow_log2 > 8) return fail(c, RT_ERR_INVALID, std::string(fn) + ": normal_power must be a power of two in 1 .. 256");
    // below kDenoiseSigmaMin the centre tap's weight, and with it every hit pixel, would be NaN (rt_denoise.cuh)
    if (!(p.sigma_color >= kDenoiseSigmaMin && p.sigma_color <= FLT_MAX) || !(p.sigma_depth >= kDenoiseSigmaMin && p.sigma_depth <= FLT_MAX))
        return fail(c, RT_ERR_INVALID, std::string(fn) + ": sigma_color and sigma_depth must be finite and at least 2^-16");
    return RT_OK;
}

static int check_temporal_params(rt_ctx* c, const char* fn, const rt_temporal_params& tp) {
    if (tp.max_history < 1 || tp.max_history > 4096) return fail(c, RT_ERR_INVALID, std::string(fn) + ": max_history must be 1 .. 4096");
    if (!(tp.tau_depth > 0.f && tp.tau_depth <= FLT_MAX)) return fail(c, RT_ERR_INVALID, std::string(fn) + ": tau_depth must be finite and positive");
    if (!(tp.tau_normal >= -1.f && tp.tau_normal <= 1.f)) return fail(c, RT_ERR_INVALID, std::string(fn) + ": tau_normal must be in -1 .. 1");
    return RT_OK;
}

}  // extern "C"

namespace rtb_capi {
int check_present(rt_ctx* c, const char* fn, const PresentOut& out, bool full, const rt_temporal_params* tp, const rt_denoise_params* dn,
                  int* pow_log2) {
    int rc, pw = 0;
    if (out.argb ? out.pitch_bytes < c->par.width * 4 : !out.rgba) return fail(c, RT_ERR_INVALID, std::string(fn) + ": bad output buffer");
    if (tp && !full) return fail(c, RT_ERR_INVALID, std::string(fn) + ": not supported on a shard (its buffer holds only part of the samples)");
    if (tp && (rc = check_temporal_params(c, fn, *tp)) != RT_OK) return rc;
    if (dn && (rc = check_denoise_params(c, fn, *dn, pw)) != RT_OK) return rc;
    if (pow_log2) *pow_log2 = pw;
    return RT_OK;
}

// Every call that presents an image. spp != NULL (rt_render_frame): *spp samples are rendered first, and for 1-2 samples the render
// kernel may resolve the frame itself. Then the image of the source: the plain resolve; with dn the filter of rt_denoise.cu, guided by
// the primary-hit cache; with tp the prior from the temporal history (rt_temporal.cuh) and the blend, filtered when dn has passes, and
// the new history. Apart from the render, read-only on the source, the accumulation buffer, the sample counter and the path statistics.
int present(rt_ctx* c, const char* fn, const PresentOut& out, const rt_temporal_params* tp, const rt_denoise_params* dn,
            const PresentSrc* src, const int* spp) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    const int w = c->par.width, h = c->par.height;
    const size_t px = (size_t)w * h;
    int pow_log2 = 0;
    if ((rc = check_present(c, fn, out, src ? src->full : c->world == 1, tp, dn, &pow_log2)) != RT_OK) return rc;
    // preview shading is deterministic: nothing to filter, and no history
    const bool preview = c->par.mode == RT_MODE_PREVIEW;
    const int passes = dn && !preview ? dn->passes : 0;
    // rt_read_denoised reads the filter's output also without passes: the plain mean
    const bool filter = passes > 0 || (dn && out.rgba && !tp);
    const int flip_y = out.flip_y ? 1 : 0;
    uint32_t* mapped = out.argb ? mapped_surface(out.argb, out.pitch_bytes, w) : nullptr;
    bool fused = false;
    if (spp) {
        static const bool fuse_on = [] { const char* v = getenv("RTB200_FRAME_FUSE"); return !(v && v[0] == '0'); }();
        FrameTarget ft;
        ft.surface = c->d_argb.get(); ft.mapped_host = mapped; ft.flip_y = flip_y;
        const bool candidate = fuse_on && c->par.mode == RT_MODE_PATH && c->pixel_step <= 1 && c->world == 1;
        if ((rc = render_samples(c, *spp, candidate ? &ft : nullptr)) != RT_OK) return rc;
        fused = ft.fused;
    }
    const PresentSrc s = src ? *src : PresentSrc{c->d_accum.get(), c->samples, c->world == 1};
    if (passes > 0 || (tp && !preview)) {
        AccelSel ac;
        if ((rc = make_accel(c, want_accel(c), camera_extent(c), ac)) != RT_OK) return rc;
        if ((rc = ensure_prim_cache(c, ac)) != RT_OK) return rc;
    }
    if (tp && c->d_tp_prior.capacity() < px) {
        RT_CUDA(c, cudaStreamSynchronize(c->stream));
        c->tp_valid = false;                                   // the history is gone with its arrays
        const cudaError_t e = reserve_all(px, c->d_tp_h[0], c->d_tp_nt[0], c->d_tp_id[0], c->d_tp_h[1], c->d_tp_nt[1], c->d_tp_id[1], c->d_tp_prior);
        if (e != cudaSuccess) return cuda_fail(c, e, "temporal history buffers");
    }
    if (filter && c->d_denoise[0].capacity() < px) {
        RT_CUDA(c, cudaStreamSynchronize(c->stream));
        const cudaError_t e = reserve_all(px, c->d_denoise[0], c->d_denoise[1]);
        if (e != cudaSuccess) return cuda_fail(c, e, "denoiser buffers");
    }

    TemporalLaunch t;
    const int cur = c->tp_cur ^ 1;                             // the half the new history goes to
    if (tp) {
        t.accum = s.sum; t.count = (float)s.samples;
        t.nt = preview ? nullptr : c->d_prim_nt.get(); t.id = preview ? nullptr : c->d_prim_id.get();
        t.width = w; t.height = h;
        t.cap = (float)tp->max_history; t.tau_z = tp->tau_depth; t.tau_n = tp->tau_normal;
        t.cur.o = c->frame.cam_pos; t.cur.u = c->frame.u_axis; t.cur.v = c->frame.v_axis; t.cur.f = c->frame.fwd;
        t.prev = c->tp_pose;
        tp_inverse(t.prev, t.m);
        // the prior: none without a history of the same radiance; rebuilt when the accumulation restarted or the pose moved
        const bool same_pose = memcmp(&t.cur, &t.prev, sizeof t.cur) == 0;
        if (preview || !c->tp_valid || c->tp_key != c->radiance_key) t.mode = kTpZero;
        else if (c->tp_epoch != c->accum_epoch || !same_pose) t.mode = same_pose ? kTpCopy : kTpReproject;
        else t.mode = kTpKeep;
        const int old = c->tp_cur;
        t.hist.h = c->d_tp_h[old].get(); t.hist.nt = c->d_tp_nt[old].get(); t.hist.id = c->d_tp_id[old].get();
        t.prior = c->d_tp_prior.get();
        t.h_out = c->d_tp_h[cur].get(); t.nt_out = c->d_tp_nt[cur].get(); t.id_out = c->d_tp_id[cur].get();
        t.next = passes > 0 ? c->d_denoise[1].get() : nullptr;
        t.argb = out.argb && passes == 0 ? c->d_argb.get() : nullptr; t.argb_host = t.argb ? mapped : nullptr; t.flip_y = flip_y;
        c->tp_valid = false;                                   // until the new history is complete
    }
    cudaError_t e = cudaSuccess;
    if (!fused) {
        cudaEventRecord(c->ev2, c->stream);
        if (tp) e = launch_temporal(t, c->stream);
        else if (!filter) e = launch_resolve(s.sum, s.samples, w, h, 0, w * h, flip_y, c->d_argb.get(), 0, c->stream, mapped);
        if (e == cudaSuccess && filter) {
            DenoiseLaunch d;
            d.accum = tp ? nullptr : s.sum; d.samples = tp ? 0 : s.samples;
            d.nt = c->d_prim_nt.get(); d.id = c->d_prim_id.get();
            d.width = w; d.height = h; d.passes = passes; d.pow_log2 = pow_log2;
            d.sigma_color = dn->sigma_color; d.sigma_depth = dn->sigma_depth;
            d.buf[0] = c->d_denoise[0].get(); d.buf[1] = c->d_denoise[1].get();
            d.argb = out.argb ? c->d_argb.get() : nullptr; d.argb_host = mapped; d.flip_y = flip_y;
            d.neff = tp ? t.h_out : nullptr;                   // the temporal form: the blend is the input, with its per-pixel count
            e = launch_denoise(d, c->stream);
        }
        cudaEventRecord(c->ev3, c->stream);
    }
    if (e == cudaSuccess && out.rgba) {
        const float4* img = tp && passes == 0 ? t.h_out : c->d_denoise[passes > 0 ? (passes - 1) & 1 : 0].get();
        e = cudaMemcpyAsync(out.rgba, img, px * sizeof(float4), cudaMemcpyDeviceToHost, c->stream);
    } else if (e == cudaSuccess && !mapped) {
        if (out.pitch_bytes == w * 4)                          // tightly packed surface: one linear copy
            e = cudaMemcpyAsync(out.argb, c->d_argb.get(), px * 4, cudaMemcpyDeviceToHost, c->stream);
        else
            e = cudaMemcpy2DAsync(out.argb, (size_t)out.pitch_bytes, c->d_argb.get(), (size_t)w * 4, (size_t)w * 4, (size_t)h, cudaMemcpyDeviceToHost, c->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return cuda_fail(c, e, fn);
    if (fused) c->last_resolve_ms = 0.f;                       // no separate resolve ran
    else cudaEventElapsedTime(&c->last_resolve_ms, c->ev2, c->ev3);
    if (tp) {
        c->tp_cur = cur;
        c->tp_valid = !preview;
        c->tp_pose = t.cur; c->tp_epoch = c->accum_epoch; c->tp_key = c->radiance_key;
    }
    return RT_OK;
}
}  // namespace rtb_capi
using rtb_capi::present;

extern "C" {

// One progressive frame: rt_render_spp(spp) + rt_resolve_rgba8(host_out) with the same result, as ONE call - which is what the
// reference's frame is (renderArea resolves every pixel as it is traced, Raytracer.cpp:63-76,223-257). For 1-2 samples per pixel the
// render kernel resolves the pixels it finishes and streams them to a page-locked surface while it is still tracing (FrameOut,
// rt_kernels.cu); every other case runs the two steps one after the other.
int rt_render_frame(rt_ctx* c, int spp, uint32_t* host_out, int pitch_bytes, int flip_y) {
    return present(c, "rt_render_frame", {host_out, pitch_bytes, flip_y, nullptr}, nullptr, nullptr, nullptr, &spp);
}

int rt_resolve_device(rt_ctx* c, const void* dev_accum, uint32_t samples, int first_pixel, int n_pixels, void* dev_out, int flip_y) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (!dev_accum || !dev_out || first_pixel < 0 || n_pixels < 0 ||
        (long long)first_pixel + n_pixels > (long long)c->par.width * c->par.height)
        return fail(c, RT_ERR_INVALID, "rt_resolve_device: bad arguments");
    RT_CUDA(c, launch_resolve((const float4*)dev_accum, samples, c->par.width, c->par.height, first_pixel, n_pixels, flip_y,
                              (uint32_t*)dev_out, 1, c->stream));
    return RT_OK;
}

int rt_resolve_rgba8(rt_ctx* c, uint32_t* host_out, int pitch_bytes, int flip_y) {
    return present(c, "rt_resolve_rgba8", {host_out, pitch_bytes, flip_y, nullptr}, nullptr, nullptr, nullptr);
}

void rt_default_denoise_params(rt_denoise_params* p) {
    if (!p) return;
    p->passes = 5; p->normal_power = 128; p->sigma_color = 2.0f; p->sigma_depth = 1.0f;   // DESIGN.md 8: sigma_color tuned at 4 spp
}

int rt_denoise_rgba8(rt_ctx* c, const rt_denoise_params* p, uint32_t* host_out, int pitch_bytes, int flip_y) {
    rt_denoise_params d;
    if (!p) rt_default_denoise_params(&d);
    return present(c, "rt_denoise_rgba8", {host_out, pitch_bytes, flip_y, nullptr}, nullptr, p ? p : &d, nullptr);
}

int rt_read_denoised(rt_ctx* c, const rt_denoise_params* p, float* host_rgba) {
    rt_denoise_params d;
    if (!p) rt_default_denoise_params(&d);
    return present(c, "rt_read_denoised", {nullptr, 0, 0, host_rgba}, nullptr, p ? p : &d, nullptr);
}

void rt_default_temporal_params(rt_temporal_params* p) {
    if (!p) return;
    p->max_history = 32; p->tau_depth = 0.02f; p->tau_normal = 0.9f; p->reserved = 0;   // DESIGN.md 8: chosen from a measured sweep
}

// dn NULL: no filter
int rt_temporal_rgba8(rt_ctx* c, const rt_temporal_params* p, const rt_denoise_params* dn, uint32_t* host_out, int pitch_bytes, int flip_y) {
    rt_temporal_params d;
    if (!p) rt_default_temporal_params(&d);
    return present(c, "rt_temporal_rgba8", {host_out, pitch_bytes, flip_y, nullptr}, p ? p : &d, dn, nullptr);
}

int rt_read_temporal(rt_ctx* c, const rt_temporal_params* p, const rt_denoise_params* dn, float* host_rgba) {
    rt_temporal_params d;
    if (!p) rt_default_temporal_params(&d);
    return present(c, "rt_read_temporal", {nullptr, 0, 0, host_rgba}, p ? p : &d, dn, nullptr);
}

int rt_reset_temporal(rt_ctx* c) {
    if (!c) return RT_ERR_INVALID;
    c->tp_valid = false;
    return RT_OK;
}

void* rt_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (bytes == 0 || cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}

void rt_host_free(void* p) { if (p) cudaFreeHost(p); }

int rt_read_accum(rt_ctx* c, float* host_rgba, uint32_t* samples) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (host_rgba)
        RT_CUDA(c, cudaMemcpyAsync(host_rgba, c->d_accum.get(), (size_t)c->par.width * c->par.height * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    if (samples) *samples = c->samples;
    return RT_OK;
}

int rt_write_accum(rt_ctx* c, const float* host_rgba, uint32_t samples) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (!host_rgba) return fail(c, RT_ERR_INVALID, "rt_write_accum: NULL input");
    RT_CUDA(c, cudaMemcpyAsync(c->d_accum.get(), host_rgba, (size_t)c->par.width * c->par.height * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    c->samples = samples; c->next_sample = samples;
    ++c->accum_epoch;
    return RT_OK;
}

int rt_read_aov(rt_ctx* c, int32_t* id, float* t, float* normal, float* point) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    const size_t px = (size_t)c->par.width * c->par.height;
    AccelSel ac;
    if ((rc = make_accel(c, want_accel(c), camera_extent(c), ac)) != RT_OK) return rc;
    DeviceArray<int> d_id; DeviceArray<float> d_t, d_n, d_p;
    cudaError_t e = cudaSuccess;
    if (id) e = d_id.reserve(px);
    if (e == cudaSuccess && t) e = d_t.reserve(px);
    if (e == cudaSuccess && normal) e = d_n.reserve(px * 3);
    if (e == cudaSuccess && point) e = d_p.reserve(px * 3);
    if (e == cudaSuccess) e = launch_primary_aov(c->view, ac, c->frame, d_id.get(), d_t.get(), d_n.get(), d_p.get(), c->stream);
    if (e == cudaSuccess && id) e = cudaMemcpyAsync(id, d_id.get(), px * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && t) e = cudaMemcpyAsync(t, d_t.get(), px * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && normal) e = cudaMemcpyAsync(normal, d_n.get(), px * 12, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && point) e = cudaMemcpyAsync(point, d_p.get(), px * 12, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return cuda_fail(c, e, "rt_read_aov");
    return RT_OK;
}

int rt_read_ray_dirs(rt_ctx* c, float* dirs) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (!dirs) return fail(c, RT_ERR_INVALID, "rt_read_ray_dirs: NULL output");
    const size_t px = (size_t)c->par.width * c->par.height;
    DeviceArray<float> d;
    cudaError_t e = d.reserve(px * 3);
    if (e == cudaSuccess) e = launch_ray_dirs(c->frame, d.get(), c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dirs, d.get(), px * 12, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return cuda_fail(c, e, "rt_read_ray_dirs");
    return RT_OK;
}

int rt_read_sample_dirs(rt_ctx* c, uint32_t sample, float* dirs) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (!dirs) return fail(c, RT_ERR_INVALID, "rt_read_sample_dirs: NULL output");
    const size_t px = (size_t)c->par.width * c->par.height;
    DeviceArray<float> d;
    cudaError_t e = d.reserve(px * 3);
    if (e == cudaSuccess) e = launch_sample_dirs(c->frame, PixelFilter{c->filter.type, c->filter.radius}, sample, d.get(), c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dirs, d.get(), px * 12, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return cuda_fail(c, e, "rt_read_sample_dirs");
    return RT_OK;
}

int rt_trace_rays(rt_ctx* c, const float* origins, const float* dirs, int n, int32_t* id, float* t, float* normal, float* point) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (n < 0 || (n > 0 && (!origins || !dirs || !id || !t || !normal || !point)))
        return fail(c, RT_ERR_INVALID, "rt_trace_rays: bad arguments");
    if (n == 0) return RT_OK;
    const size_t N = (size_t)n;
    // The conservativeness arguments of the BVH and the flat accelerator need unit-length directions (to
    // float rounding) and origins inside the extent their margins were derived for; anything else goes through
    // the brute-force loop.
    int kind = want_accel(c);
    float ext = 0.f;
    if (kind != RT_ACCEL_BRUTE) {
        for (size_t i = 0; i < N && kind != RT_ACCEL_BRUTE; ++i) {
            const float* d = dirs + 3 * i; const float* o = origins + 3 * i;
            float l2 = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
            if (!(fabsf(l2 - 1.f) <= 2e-6f)) kind = kind == RT_ACCEL_FLAT && fabsf(l2 - 1.f) <= 1e-3f ? RT_ACCEL_BVH : RT_ACCEL_BRUTE;
            for (int k = 0; k < 3; ++k) { if (!(fabsf(o[k]) < 1e14f)) kind = RT_ACCEL_BRUTE; ext = fmaxf(ext, fabsf(o[k])); }
        }
    }
    AccelSel ac;
    if ((rc = make_accel(c, kind, ext, ac)) != RT_OK) return rc;
    DeviceArray<float> arr;                                    // org3 dir3 n3 p3 t1 id1 = 14 words per ray
    cudaError_t e = arr.reserve(N * 14);
    float* buf = arr.get();
    float *d_o = buf, *d_d = buf + 3 * N, *d_n = buf + 6 * N, *d_p = buf + 9 * N, *d_t = buf + 12 * N;
    int* d_id = (int*)(buf + 13 * N);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_o, origins, N * 12, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_d, dirs, N * 12, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = launch_trace_rays(c->view, ac, d_o, d_d, n, d_id, d_t, d_n, d_p, c->stream, c->opt_trav_stats ? c->d_counters.get() : nullptr);
    if (e == cudaSuccess) e = cudaMemcpyAsync(id, d_id, N * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(t, d_t, N * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(normal, d_n, N * 12, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(point, d_p, N * 12, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return cuda_fail(c, e, "rt_trace_rays");
    return RT_OK;
}

int rt_pick(rt_ctx* c, int x, int y_window, int* id) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (!id) return fail(c, RT_ERR_INVALID, "rt_pick: NULL id");
    // y = SCREEN_HEIGHT - y (Raytracer.cpp:532); no bounds check, like the reference: the ray
    // through any (x, y) is well defined. One-thread launch through the same device raygen
    // and closest-hit code as the render path.
    const int y = c->par.height - y_window;
    int* d_id = (int*)c->d_scratch.get();
    AccelSel ac;
    if ((rc = make_accel(c, want_accel(c), camera_extent(c), ac)) != RT_OK) return rc;
    RT_CUDA(c, launch_pick(c->view, ac, c->frame, x, y, d_id, c->stream));
    RT_CUDA(c, cudaMemcpyAsync(id, d_id, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    return RT_OK;
}

int rt_env_color(rt_ctx* c, const float* dirs, int n, float* rgb) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (n < 0 || (n > 0 && (!dirs || !rgb))) return fail(c, RT_ERR_INVALID, "rt_env_color: bad arguments");
    if (n == 0) return RT_OK;
    const size_t N = (size_t)n;
    DeviceArray<float> arr;                                    // dir3 rgb3 per direction
    cudaError_t e = arr.reserve(N * 6);
    float* buf = arr.get();
    if (e == cudaSuccess) e = cudaMemcpyAsync(buf, dirs, N * 12, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = launch_env_color(c->frame, buf, n, buf + 3 * N, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(rgb, buf + 3 * N, N * 12, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return cuda_fail(c, e, "rt_env_color");
    return RT_OK;
}

int rt_philox_block(rt_ctx* c, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    if (!c || !ctr || !key || !out) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    RT_CUDA(c, launch_philox(ctr, key, c->d_scratch.get(), c->stream));
    RT_CUDA(c, cudaMemcpyAsync(out, c->d_scratch.get(), 16, cudaMemcpyDeviceToHost, c->stream));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    return RT_OK;
}

int rt_selftest(rt_ctx* c, int which, int* failures) {
    if (!c || !failures || which < 0 || which > 2) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    if (which == 0) RT_CUDA(c, launch_selftest_uniform((int*)c->d_scratch.get(), c->stream));
    else if (which == 1) RT_CUDA(c, launch_selftest_normalize((int*)c->d_scratch.get(), c->stream));
    else RT_CUDA(c, launch_selftest_packed((int*)c->d_scratch.get(), c->stream));
    RT_CUDA(c, cudaMemcpyAsync(failures, c->d_scratch.get(), sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    return RT_OK;
}

int rt_get_stats(rt_ctx* c, rt_stats* out) {
    if (!c || !out) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    unsigned long long counters[kCounters] = {};
    RT_CUDA(c, cudaMemcpy(counters, c->d_counters.get(), sizeof counters, cudaMemcpyDeviceToHost));
    if (c->render_timed) { cudaEventElapsedTime(&c->last_render_ms, c->ev0, c->ev1); }
    memset(out, 0, sizeof *out);
    out->paths = c->paths; out->segments = counters[0];
    out->samples = c->samples; out->n_objects = (uint32_t)c->scene.objects.size();
    out->last_render_ms = c->last_render_ms; out->last_resolve_ms = c->last_resolve_ms;
    out->total_paths = c->total_paths; out->total_segments = counters[1];
    out->traced_segments = counters[2]; out->total_traced_segments = counters[3];
    out->pipeline = c->used_pipeline; out->accel = c->used_accel; out->sm_count = c->sm_count;
    return RT_OK;
}

int rt_get_traversal_stats(rt_ctx* c, rt_traversal_stats* out) {
    if (!c || !out) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    unsigned long long counters[kCounters] = {};
    RT_CUDA(c, cudaMemcpy(counters, c->d_counters.get(), sizeof counters, cudaMemcpyDeviceToHost));
    memset(out, 0, sizeof *out);
    out->queries = counters[8]; out->node_visits = counters[9];
    out->sphere_tests = counters[10]; out->cube_tests = counters[11]; out->tri_tests = counters[12];
    out->prim_tests = counters[10] + counters[11] + counters[12];
    out->node_bytes = (uint32_t)sizeof(BvhNode);
    return RT_OK;
}

void* rt_accum_device_ptr(rt_ctx* c) {
    if (!c || prepare(c) != RT_OK) return nullptr;
    return c->d_accum.get();
}

void* rt_argb_device_ptr(rt_ctx* c) {
    if (!c || prepare(c) != RT_OK) return nullptr;
    return c->d_argb.get();
}

int rt_ipc_export(rt_ctx* c, int which, unsigned char handle[RT_IPC_HANDLE_BYTES]) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (!handle || which < 0 || which > 2) return fail(c, RT_ERR_INVALID, "rt_ipc_export: bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == RT_IPC_HANDLE_BYTES, "IPC handle size");
    cudaIpcMemHandle_t h;
    RT_CUDA(c, cudaIpcGetMemHandle(&h, which == 0 ? (void*)c->d_accum.get() : which == 1 ? (void*)c->d_argb.get() : (void*)c->d_flags.get()));
    memcpy(handle, &h, sizeof h);
    return RT_OK;
}

int rt_ipc_open(rt_ctx* c, const unsigned char handle[RT_IPC_HANDLE_BYTES], void** dev_ptr) {
    if (!c || !handle || !dev_ptr) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    RT_CUDA(c, cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return RT_OK;
}

int rt_ipc_close(rt_ctx* c, void* dev_ptr) {
    if (!c || !dev_ptr) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    RT_CUDA(c, cudaIpcCloseMemHandle(dev_ptr));
    return RT_OK;
}

int rt_resolve_fused(rt_ctx* c, const void* const* accum_ptrs, int world, uint32_t total_samples, int first_pixel, int n_pixels,
                     void* dst, int flip_y) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (!accum_ptrs || !dst || world < 1 || world > RT_MAX_PEERS || first_pixel < 0 || n_pixels < 0 ||
        (long long)first_pixel + n_pixels > (long long)c->par.width * c->par.height)
        return fail(c, RT_ERR_INVALID, "rt_resolve_fused: bad arguments");
    for (int r = 0; r < world; ++r) {
        if (!accum_ptrs[r]) return fail(c, RT_ERR_INVALID, "rt_resolve_fused: NULL peer buffer");
        if ((rc = enable_peer_access_to(c, accum_ptrs[r], "rt_resolve_fused: accumulation buffer")) != RT_OK) return rc;
    }
    if ((rc = enable_peer_access_to(c, dst, "rt_resolve_fused: destination surface")) != RT_OK) return rc;
    return rtb_capi::resolve_fused_unchecked(c, accum_ptrs, world, total_samples, first_pixel, n_pixels, dst, flip_y);
}

int rt_exchange_setup(rt_ctx* c, int rank, int world, void* const* accum_ptrs, void* const* flag_ptrs, void* dst) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    if (world < 1 || world > RT_MAX_PEERS || rank < 0 || rank >= world || !accum_ptrs || !flag_ptrs)
        return fail(c, RT_ERR_INVALID, "rt_exchange_setup: bad arguments");
    ExchangeState& x = c->exch;
    x.ready = false;
    // NOTE: every rank must run on its OWN device - the ranks wait for each other inside kernels, and kernels of two ranks on one
    // GPU are not guaranteed to run concurrently. This cannot be checked here: for a CUDA-IPC mapping cudaPointerGetAttributes
    // reports the importing context's device, not the exporter's. (Ranks sharing a device: rt_resolve_fused + host-side ordering.)
    for (int r = 0; r < world; ++r) {
        const void* a = r == rank && !accum_ptrs[r] ? (const void*)c->d_accum.get() : accum_ptrs[r];
        void* f = r == rank && !flag_ptrs[r] ? (void*)c->d_flags.get() : flag_ptrs[r];
        if (!a || !f) return fail(c, RT_ERR_INVALID, "rt_exchange_setup: NULL peer pointer");
        if ((rc = enable_peer_access_to(c, a, "rt_exchange_setup: accumulation buffer")) != RT_OK) return rc;
        if ((rc = enable_peer_access_to(c, f, "rt_exchange_setup: exchange flags")) != RT_OK) return rc;
        x.accum[r] = (const float4*)a; x.flags[r] = (ExchFlags*)f;
    }
    if (x.accum[rank] != c->d_accum.get() || x.flags[rank] != c->d_flags.get()) return fail(c, RT_ERR_INVALID, "rt_exchange_setup: entry `rank` is not this context's own buffer");
    if (!dst) dst = rank == 0 ? (void*)c->d_argb.get() : nullptr;
    if (!dst) return fail(c, RT_ERR_INVALID, "rt_exchange_setup: NULL destination surface");
    if ((rc = enable_peer_access_to(c, dst, "rt_exchange_setup: destination surface")) != RT_OK) return rc;
    x.dst = (uint32_t*)dst; x.rank = rank; x.world = world;
    x.ready = true;
    return RT_OK;
}

int rt_exchange_resolve(rt_ctx* c, uint32_t total_samples, int flip_y) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    ExchangeState& x = c->exch;
    if (!x.ready) return fail(c, RT_ERR_INVALID, "rt_exchange_resolve: rt_exchange_setup has not been called (or the frame buffers were reallocated since)");
    PeerPtrs pp; ExchPeers fl;
    memset(&pp, 0, sizeof pp); memset(&fl, 0, sizeof fl);
    for (int r = 0; r < x.world; ++r) { pp.p[r] = x.accum[r]; fl.f[r] = x.flags[r]; }
    const long long n_px = (long long)c->par.width * c->par.height;
    const int first = (int)(n_px * x.rank / x.world), count = (int)(n_px * (x.rank + 1) / x.world) - first;
    ++x.epoch;                                                 // every rank calls this the same number of times
    RT_CUDA(c, launch_resolve_fused_sync(pp, fl, x.rank, x.world, x.epoch, total_samples, c->par.width, c->par.height, first, count, flip_y, x.dst, c->stream));
    return RT_OK;
}

// a wait of the exchange timed out (a peer never signalled): reported by the calls that synchronise
static int check_exchange_error(rt_ctx* c) {
    if (!c->exch.ready) return RT_OK;
    uint32_t err = 0;
    RT_CUDA(c, cudaMemcpy(&err, &c->d_flags.get()->error, sizeof err, cudaMemcpyDeviceToHost));
    if (err) return fail(c, RT_ERR_CUDA, "exchange timed out: a peer rank did not signal within 4 s");
    return RT_OK;
}

int rt_read_surface(rt_ctx* c, uint32_t* host_out, int pitch_bytes) {
    int rc = prepare(c);
    if (rc != RT_OK) return rc;
    const int w = c->par.width, h = c->par.height;
    if (!host_out || pitch_bytes < w * 4) return fail(c, RT_ERR_INVALID, "rt_read_surface: bad output buffer");
    RT_CUDA(c, cudaMemcpy2DAsync(host_out, (size_t)pitch_bytes, c->d_argb.get(), (size_t)w * 4, (size_t)w * 4, (size_t)h, cudaMemcpyDeviceToHost, c->stream));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    return check_exchange_error(c);
}

int rt_set_stream(rt_ctx* c, void* cuda_stream) {
    if (!c) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
    return RT_OK;
}

int rt_sync(rt_ctx* c) {
    if (!c) return RT_ERR_INVALID;
    RT_CUDA(c, cudaSetDevice(c->device));
    RT_CUDA(c, cudaStreamSynchronize(c->stream));
    return check_exchange_error(c);
}

int rt_set_sample_count(rt_ctx* c, uint32_t samples) {
    if (!c) return RT_ERR_INVALID;
    c->samples = samples;
    ++c->accum_epoch;
    return RT_OK;
}

}  // extern "C"
