/* rt_b200.h - C-ABI of the B200-native path tracer (librt_b200.so).
 *
 * This is the drop-in boundary for the ONE hot path of JoshuaLim007/Software-Raytracer:
 * per-pixel ray generation -> closest hit over the Scene's object list -> scatter / shade ->
 * bounce loop -> progressive accumulation -> Reinhard resolve to ARGB8.
 *
 * The reference has no FFI; its seam is the set of free functions and globals that main()
 * and the 16 worker threads share (SURVEY.md 8b). Every entry point below names the reference
 * code it replaces as file:line under Raytracer/ of the reference tree. Plain pointers and
 * sizes only; no C++/torch types. All functions return 0 on success and a negative rt_status
 * on failure (the reference reports no errors at all: Scene.hpp:30-32,75-77 fail silently);
 * rt_last_error() gives the message. A context is used by one host thread at a time - the
 * reference's own rule ("thread safe after this point", Raytracer.cpp:373-385).
 *
 * There is NO CPU fallback: every compute entry point runs CUDA kernels on an sm_100a
 * device or fails with RT_ERR_CUDA.
 *
 * Conventions kept from the reference: image space is y-UP, row-major, pixel index
 * x + y*width (Raytracer.cpp:67); object id == index in the scene's object list == JSON
 * order (Raytracer.cpp:127-137); colours are linear float; the resolved surface is
 * 0xAARRGGBB with alpha byte 0 and rows flipped to y-down (Raytracer.cpp:64, Common.hpp:205).
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_B200_ABI_VERSION 4

typedef struct rt_ctx rt_ctx;

typedef enum {
    RT_OK = 0,
    RT_ERR_INVALID = -1,   /* bad argument / call order */
    RT_ERR_CUDA = -2,      /* no usable device, launch or copy failure */
    RT_ERR_IO = -3,        /* file missing / unreadable */
    RT_ERR_PARSE = -4,     /* malformed scene JSON or missing required key */
    RT_ERR_NOMEM = -5
} rt_status;

/* Object types: Scene.hpp:43-55 ("Sphere", "Cube", anything else -> never-hit Object). */
enum { RT_OBJ_NONE = 0, RT_OBJ_SPHERE = 1, RT_OBJ_CUBE = 2,
       RT_OBJ_MESH = 3 };   /* triangle mesh: an extension, the reference has no such type (rt_set_mesh below) */

/* One scene object: Object.transform.position + Sphere::radius | Box::size (half extents) +
 * Material (Common.hpp:293-319). 76 bytes, no padding. */
typedef struct {
    int32_t type;
    float pos[3];
    float radius;          /* spheres */
    float half[3];         /* cubes: half extents, axis aligned (Object.hpp:173-200,203) */
    float base[3];         /* Material.BaseColor      JSON "Color" */
    float emissive[3];     /* Material.EmissiveColor  JSON "Emissive" */
    float spec_color[3];   /* Material.SpecularColor  JSON "SpecularColor" */
    float smoothness;      /* Material.Smoothness */
    float spec_amount;     /* Material.SpecularAmount */
} rt_object;

/* Transform camera + FOV (Raytracer.cpp:295-297, :31). The basis is NOT re-orthonormalised,
 * exactly like the reference. fov_deg is the vertical field of view, an int like the reference's. */
typedef struct {
    float pos[3], right[3], up[3], forward[3];
    int32_t fov_deg;
} rt_camera;

enum { RT_MODE_PATH = 0, RT_MODE_PREVIEW = 1 };   /* SIMPLEDRAW false / true (Raytracer.cpp:35,147) */

/* Render parameters: the reference's compile-time #defines and mutable globals
 * (Raytracer.cpp:26-35, 55-59, 166, 177). rt_default_params() fills the reference's values. */
typedef struct {
    int32_t width, height;         /* SCREEN_WIDTH / SCREEN_HEIGHT */
    int32_t max_bounces;           /* MAXBOUNCES */
    int32_t mode;                  /* RT_MODE_* */
    int32_t selected_id;           /* selectedObject as an object id, -1 = none (preview highlight) */
    float sun_dir[3];              /* SunDirection after Normalized() (:55,:264) */
    float sky[3], horizon[3], ground[3], sun[3];   /* :56-59 */
    float dissipation;             /* lightEnergyDissipation 0.8 (:166) */
    float eps;                     /* secondary-origin offset 1e-5 (:177) */
    uint32_t seed_lo, seed_hi;     /* Philox key; the reference's srand(0) (:263) has no equivalent */
} rt_params;

typedef struct {
    uint64_t paths;                /* primary rays started since rt_reset_accumulation */
    uint64_t segments;             /* closest-hit queries traced (the metric's "path*bounces") */
    uint32_t samples;              /* samples per pixel accumulated so far (ACCUMULATIONFRAMES analogue) */
    uint32_t n_objects;
    float last_render_ms;          /* device time of the last rt_render_spp, CUDA events */
    float last_resolve_ms;
    int32_t pipeline;              /* RT_PIPELINE_* actually used by the last render */
    int32_t accel;                 /* RT_ACCEL_* actually used */
    int32_t sm_count;
    int32_t reserved;
    uint64_t total_paths;          /* since rt_create: never reset (benchmarks) */
    uint64_t total_segments;
    /* closest-hit queries actually executed. Equal to `segments` unless primary-hit reuse is on
     * (RT_OPT_PRIMARY_REUSE): the reference has no pixel jitter, so every sample of a pixel starts with the
     * same primary query; it is then run once per pixel per rt_render_spp call and its result reused. */
    uint64_t traced_segments;
    uint64_t total_traced_segments;
} rt_stats;

/* Tuning knobs that have no counterpart in the reference (they never change results). */
enum {
    RT_OPT_PIPELINE = 1,           /* RT_PIPELINE_* */
    RT_OPT_ACCEL = 2,              /* RT_ACCEL_* */
    RT_OPT_BVH_THRESHOLD = 3,      /* object count at which RT_ACCEL_AUTO switches to the BVH */
    RT_OPT_BVH_SCHED = 4,          /* 0 (default): megakernel per-ray BVH loop / wavefront intersect with ray refill + postponed leaves;
                                      1: experimental warp-scheduled BVH megakernel / wavefront intersect one ray per lane per batch */
    RT_OPT_BVH_WAIT_K = 5,         /* scheduled kernel: waiting lanes that trigger a shading pass (default 20) */
    RT_OPT_BVH_LEAF = 6,           /* BVH builder: maximum primitives per leaf (default 4) */
    RT_OPT_WF_REFILL = 8,          /* wavefront BVH intersect: free lanes that trigger a ray refill (default 8) */
    RT_OPT_WF_NODE_MIN = 9,        /* wavefront BVH intersect: lanes with inner-node work below which pending leaves are tested (default 8) */
    RT_OPT_POOL_TILES = 10,        /* megakernel, few samples per call: 8x4 pixel tiles per chunk a warp of the persistent pixel-pool kernel claims at a time;
                                      0 (default) automatic (2 for 1-spp calls), 1 one pixel per lane (no pool) */
    RT_OPT_FLAT_COOP = 11,         /* flat accelerator in the megakernel: 1 the warp pools the cluster culls and strict tests of its 32 rays, 0 every lane for itself,
                                      2 (default) pooled for scenes without cubes (open sphere scenes gain ~8 %, cube rooms lose ~10 %) */
    RT_OPT_WF_WAVE_MPATHS = 13,    /* wavefront pipeline: paths per wave in units of 2^20 (0 = default 128, i.e. ~15 GB of path state; at most 64 samples
                                      per pixel per wave and a third of the free device memory). Larger waves keep the late bounce rounds filled */
    RT_OPT_BVH_WIDE = 12,          /* BVH node format: 0 (default) 64-byte binary nodes; 1 scenes of 1024+ primitives traverse the 8-wide form with
                                      quantised child boxes (80-byte nodes, csrc/bvh_wide.h); 2 every BVH scene. Identical results; on B200 the
                                      wide form makes 2.2x fewer node visits but executes more instructions and measured slower (DESIGN.md) */
    RT_OPT_PRIMARY_REUSE = 7,      /* 1 (default): ONE primary closest-hit query per pixel, kept in a per-pixel cache of the context
                                      (id, t, normal) and reused by every sample of every rt_render_spp call until the camera, the
                                      scene, the resolution or the secondary-origin offset changes (identical ray: the reference has
                                      no pixel jitter, Raytracer.cpp:106-122); 0: re-trace it for every sample like the reference.
                                      Results are bit-identical. */
    RT_OPT_BVH_QUANT = 15,         /* 1 (default): BVHs traversed from global memory by the persistent kernels also get 32-byte nodes with 16-bit
                                      child planes on one grid per tree (conservative, identical results; falls back to the float nodes
                                      when the grid would be coarser than 1/8 of the median primitive extent); 0: float nodes only */
    RT_OPT_TRAVERSAL_STATS = 14    /* 1: BVH kernels count inner-node visits and primitive tests (rt_get_traversal_stats); a separate
                                      instantiation of the kernels, ~3 % slower. 0 (default): off */
};
enum { RT_PIPELINE_AUTO = 0, RT_PIPELINE_REGEN = 1, RT_PIPELINE_WAVEFRONT = 2, RT_PIPELINE_STREAM = 3 };
/* BRUTE: the reference's object loop. BVH: host-built BVH2. FLAT: two-level flat accelerator for scenes of up
 * to 255 objects (conservative culls with warp-uniform control flow, then the strict tests). All three give
 * bit-identical hits; AUTO measures them on the first rt_render_spp call of at least 64 samples after a scene or parameter
 * change (shorter calls, and camera moves, keep a heuristic choice: flat up to 255 objects, BVH from `bvh_threshold`).
 * RT_PIPELINE_AUTO is the regeneration megakernel, except that BVH scenes of 2048+ primitives also time the wavefront
 * pipeline (raygen / persistent-thread intersect / shade + ray compaction kernels, one pass over device queues per bounce)
 * and the streaming pipeline (RT_PIPELINE_STREAM: ONE persistent kernel per wave whose lanes claim path ids from a global
 * cursor, traverse with postponed leaves, shade their own hits and go on with the scattered ray - no per-bounce state in
 * HBM) on the first call of 8+ samples and keep the fastest for calls of 8+ samples; shorter calls always use the
 * megakernel. All pipelines give bit-identical accumulation buffers. */
enum { RT_ACCEL_AUTO = 0, RT_ACCEL_BRUTE = 1, RT_ACCEL_BVH = 2, RT_ACCEL_FLAT = 3 };

/* ---- lifetime: replaces the worker spawn/join (Raytracer.cpp:331-342, 598-607) -------- */
int rt_create(int cuda_device, rt_ctx** out);
int rt_destroy(rt_ctx* ctx);
const char* rt_last_error(const rt_ctx* ctx);   /* ctx may be NULL: last rt_create failure */
int rt_abi_version(void);

/* ---- scene: replaces Scene::Load/SaveAs + `ObjectsToRender = GetObjects()`
 *      (Scene.hpp:27-104, Raytracer.cpp:291-293,418-421) ------------------------------ */
int rt_load_scene(rt_ctx* ctx, const char* json_path);              /* returns object count (>= 0) */
int rt_save_scene(rt_ctx* ctx, const char* json_path);              /* Scene::SaveAs */
int rt_set_scene(rt_ctx* ctx, const rt_object* objects, int n);     /* host array -> device SoA */
int rt_get_scene(rt_ctx* ctx, rt_object* out, int max_objects);     /* returns count */

/* Host-only helpers over the same reader/writer (no device, no context): parse a scene file
 * into a caller array / write one with dump(4) formatting. *n_total receives the number of
 * objects parsed (also on RT_ERR_PARSE: the partial-load count). names may be NULL. */
int rt_scene_file_read(const char* json_path, rt_object* out, int max_objects, int* n_total,
                       char* err_buf, int err_buf_len);
/* Names of the same file: object names as consecutive NUL-terminated strings in names_buf (in object
 * order; returns the number of bytes needed), the scene's "SceneName" in scene_name. */
int rt_scene_file_read_names(const char* json_path, char* names_buf, int names_buf_len,
                             char* scene_name, int scene_name_len);
int rt_scene_file_write(const char* json_path, const char* scene_name, const rt_object* objects,
                        const char* const* names, int n);
/* Object / scene names travel with the scene (Object::name, Scene::sceneName). */
const char* rt_object_name(rt_ctx* ctx, int index);
int rt_set_object_name(rt_ctx* ctx, int index, const char* name);
const char* rt_scene_name(rt_ctx* ctx);

/* ---- triangle meshes: EXTENSION (BASELINE.json config 4) ---------------------------------
 * The reference's Scene holds Sphere and Box objects only (Scene.hpp:43-55); a mesh follows the same
 * Object contract: one scene object (one id, one Material, Transform.position as a translation) whose
 * Raytrace() reports the closest of its triangles (Object.hpp:21-23; csrc/mesh.h defines the intersector).
 * JSON: "Renderer": {"Type": "Mesh", "File": "mesh.obj"} (path relative to the scene file) or inline
 * "Vertices": [x,y,z,...] / "Triangles": [i,j,k,...]. Geometry is attached to an object of type RT_OBJ_MESH
 * AFTER rt_set_scene / rt_load_scene (which drop all mesh data); scenes with meshes use the BVH back end. */
int rt_set_mesh(rt_ctx* ctx, int object_index, const float* vertices_xyz, int n_vertices,
                const int32_t* indices, int n_triangles);
int rt_load_mesh_obj(rt_ctx* ctx, int object_index, const char* obj_path);
int rt_get_mesh_info(rt_ctx* ctx, int object_index, int* n_vertices, int* n_triangles);

/* ---- camera and parameters ----------------------------------------------------------- */
void rt_default_params(rt_params* p);                               /* Raytracer.cpp:26-35,55-59 */
void rt_default_camera(rt_camera* c);                               /* Raytracer.cpp:295-297 */
void rt_rotate_camera(rt_camera* c, float angle, const float axis[3]);  /* Transform::RotateAboutAxis, Common.hpp:287-291 */
int rt_set_camera(rt_ctx* ctx, const rt_camera* cam);
int rt_set_params(rt_ctx* ctx, const rt_params* p);
int rt_set_option(rt_ctx* ctx, int option, int value);

/* Block-filled frames - the reference's SCREEN_SCALE slider and progressive-resolution first frame
 * (Raytracer.cpp:30,47,233-248,576-590): with steps = ceil(1 / (SCREEN_SCALE * progressiveResolutionScaler)) > 1,
 * every rt_render_spp traces ONE path per steps x steps block (through the block's first pixel) and writes it
 * to all pixels of the block. Blocks start at the first column of each worker strip and are clipped to it:
 * strip_columns = 0 treats the image as one strip, rt_reference_strip_columns(width) gives the reference's 16
 * strips (ceil(width / 16) + 1 columns, :330). steps = 1 (default) is the full-resolution path; the C-ABI's
 * default is full resolution, the reference's default SCREEN_SCALE of .5 corresponds to steps = 2. */
int rt_set_pixel_step(rt_ctx* ctx, int steps, int strip_columns);
int rt_reference_pixel_step(float screen_scale, float progressive_scaler);
int rt_reference_strip_columns(int width);

/* Multi-GPU sharding by samples-per-pixel: rank r of `world` renders its slice of the global
 * sample indices of every rt_render_spp call, so the reduced image does not depend on the
 * GPU count (up to float summation order). Default (0, 1). */
int rt_set_shard(rt_ctx* ctx, int rank, int world);
/* The shard arithmetic itself (host only, no context): for a call adding `spp` global samples starting
 * at global index `next_sample`, rank r of `world` traces samples [*first, *first + *count). */
int rt_shard_range(int spp, int rank, int world, uint32_t next_sample, uint32_t* first, int* count);

/* ---- the hot path --------------------------------------------------------------------- */
/* `setFrame = true; ACCUMULATIONFRAMES = 1` (Raytracer.cpp:576-581). */
int rt_reset_accumulation(rt_ctx* ctx);

/* Adds `spp` samples per pixel (global count; this rank traces its shard) to the device float4
 * SUM buffer and advances the sample counter: renderArea frames (Raytracer.cpp:231-252) +
 * RaytraceScene (:141-213) + the accumulate half of SetScreenPixel (:65-71). The reference
 * keeps a running mean; sum/count is the same value up to rounding (DESIGN.md). Asynchronous
 * on the context's stream. */
int rt_render_spp(rt_ctx* ctx, int spp);

/* Reinhard c/(1+c), truncating 8-bit pack to 0xAARRGGBB (alpha 0), optional row flip to y-down:
 * the resolve half of SetScreenPixel (Raytracer.cpp:73-75, Common.hpp:189-206).
 * host_out: height rows of pitch_bytes. Synchronises. */
int rt_resolve_rgba8(rt_ctx* ctx, uint32_t* host_out, int pitch_bytes, int flip_y);

/* One progressive frame = rt_render_spp(ctx, spp) followed by rt_resolve_rgba8(ctx, host_out, pitch_bytes, flip_y), same
 * accumulation buffer, same surface bits, as ONE call: the reference's frame resolves every pixel the moment it is traced
 * (renderArea -> SetScreenPixel, Raytracer.cpp:63-76,223-257), and for 1-2 samples per pixel so does the render kernel here - pixels
 * are resolved as they finish and streamed to a page-locked surface (rt_host_alloc, tight pitch) while the rest of the frame is
 * still being traced, so the frame costs the render alone instead of render + resolve + copy. Other cases (more samples, block-
 * filled frames, preview, shards of a multi-GPU render) run the two steps back to back. Synchronises. */
int rt_render_frame(rt_ctx* ctx, int spp, uint32_t* host_out, int pitch_bytes, int flip_y);

/* Denoised resolve: an edge-avoiding a-trous filter (B3-spline taps at steps 1, 2, 4, ..) over the mean radiance, guided by the
 * primary-hit cache (object id, normal, t per pixel; RT_OPT_PRIMARY_REUSE), in front of the plain resolve. A pixel never takes colour
 * from another object or from the sky; within an object the normal and the relative depth stop it at creases; the colour tolerance
 * shrinks as sigma_color * 2^-pass / sqrt(samples), so a converged image is left almost untouched. Sky pixels come out exactly as
 * rt_resolve_rgba8 gives them. The guides describe the CURRENT camera and scene: denoise after rendering and before moving (a call
 * after rt_set_camera / rt_set_scene filters the buffer with the new pose's guides). If the cache is not valid (also with
 * RT_OPT_PRIMARY_REUSE 0) the call traces it first; those queries count in traced_segments. Neither call changes the accumulation
 * buffer, the sample counter, segments or paths; last_resolve_ms reports the device time of filter + pack. Preview mode, and
 * passes 0, give the plain resolve. Bad parameters: RT_ERR_INVALID. See DESIGN.md 5 for the filter's definition. */
typedef struct {
    int32_t passes;         /* 0..8; 0 = the plain resolve, bit for bit */
    int32_t normal_power;   /* P: 1, 2, 4, .. 256 */
    float sigma_color;      /* sigma_c: tolerance on Reinhard luminance at 1 spp; 2^-16 .. FLT_MAX */
    float sigma_depth;      /* sigma_z: relative depth tolerance per pixel of step; 2^-16 .. FLT_MAX */
} rt_denoise_params;        /* 16 bytes */
void rt_default_denoise_params(rt_denoise_params* p);
/* rt_resolve_rgba8 with the filter in front. NULL params = defaults. Synchronises. */
int rt_denoise_rgba8(rt_ctx* ctx, const rt_denoise_params* p, uint32_t* host_out, int pitch_bytes, int flip_y);
/* The filtered MEAN radiance, width*height float4 (r,g,b,0), y-up: rt_read_accum's layout. Synchronises. */
int rt_read_denoised(rt_ctx* ctx, const rt_denoise_params* p, float* host_rgba);

/* Temporal resolve: carries the presented image across camera moves. The context keeps a history after every temporal call:
 * per pixel the presented colour H and its weight W_H, that pose's primary-hit guides (object id, normal, t), the pose, the
 * accumulation epoch (it changes on rt_reset_accumulation, rt_write_accum, rt_set_sample_count and a resize) and the radiance key
 * (it changes on rt_set_scene, rt_load_scene, rt_set_mesh, rt_load_mesh_obj and any rt_set_params change of mode, max_bounces, the
 * environment colours, sun_dir, dissipation or eps; not on the seed, selected_id or the pixel step). It also keeps a prior per pixel,
 * colour P and weight w_P. A call
 *   1. drops the history (w_P = 0 everywhere) when there is none, after rt_reset_temporal, a resize or a radiance-key change;
 *   2. else, when the epoch or the pose (origin and axes of the rays) changed, rebuilds the prior: an identical pose copies it
 *      (P = H, w_P = min(W_H, max_history)); otherwise every pixel with a primary hit projects its hit point into the history's
 *      pose and takes the bilinear 2x2 history taps of the same object id within tau_depth * distance of the point and with
 *      normals n_p . n_q >= tau_normal (w_P = min(max_history, sum b_q W_H), 0 when none counts); sky pixels get w_P = 0;
 *   3. else keeps the prior (more samples were added, or the call was repeated);
 *   4. presents O = (S + w_P P) / (N + w_P) (S the sample sum, N the sample count) where w_P > 0 and the pixel has a hit and N > 0,
 *      elsewhere the plain mean, bit for bit rt_resolve_rgba8's; and stores (O, N + w_P) as the new history.
 * With filter parameters (dn non-NULL, passes > 0) the a-trous filter of rt_denoise_rgba8 runs over O, its colour tolerance per
 * pixel from N_eff = N + w_P instead of N; the history keeps the unfiltered O. Without a history the calls give exactly what
 * rt_resolve_rgba8 / rt_read_denoised / rt_denoise_rgba8 give. No colour crosses an object id. Moving objects need a scene edit,
 * which drops the history; mirror reflections lag by up to max_history frames. Preview mode gives the plain resolve and drops the
 * history. Neither call changes the accumulation buffer, the sample counter, segments or paths; an invalid primary-hit cache is
 * traced first (counted in traced_segments). last_resolve_ms reports the device time of reprojection, filter and pack. A shard
 * context (rt_set_shard world > 1) and bad parameters: RT_ERR_INVALID. Synchronise. See DESIGN.md 5. */
typedef struct {
    int32_t max_history;    /* cap of the prior's weight in samples: 1 .. 4096 */
    float tau_depth;        /* relative distance tolerance of a history tap, finite and > 0 */
    float tau_normal;       /* smallest n_p . n_q of a history tap, -1 .. 1 */
    int32_t reserved;
} rt_temporal_params;       /* 16 bytes */
void rt_default_temporal_params(rt_temporal_params* p);
/* The temporally reprojected frame as ARGB8 (NULL tp = defaults; dn NULL or passes 0: no filter). */
int rt_temporal_rgba8(rt_ctx* ctx, const rt_temporal_params* tp, const rt_denoise_params* dn, uint32_t* host_out, int pitch_bytes, int flip_y);
/* The same as width*height float4 (r, g, b, N_eff), y-up: rt_read_accum's layout (rgb filtered when dn asks for it). */
int rt_read_temporal(rt_ctx* ctx, const rt_temporal_params* tp, const rt_denoise_params* dn, float* host_rgba);
/* Forget the history: the next temporal call presents the plain (or filtered) mean. */
int rt_reset_temporal(rt_ctx* ctx);

/* Pixel filter: anti-aliased path renders. The reference shoots every sample through the pixel corner (GetRayDirection,
 * Raytracer.cpp:106-122), so however many samples accumulate, edges stay stair-stepped. With a filter every path-mode sample
 * traces its own primary ray, offset from the corner by a per-sample (jx, jy) drawn from Philox4x32-10 with counter (pixel, global
 * sample index, 0, 1) and the context's key: RT_FILTER_BOX uniform on [-radius, radius)^2, RT_FILTER_TENT the separable tent of
 * that radius. The footprint is centred on the corner, so the image does not shift against the unfiltered one. DESIGN.md 5 states
 * the arithmetic exactly; a zero offset gives GetRayDirection's bits.
 *   - rt_set_pixel_filter: RT_ERR_INVALID for an unknown type, a radius that is not finite or not in (0, 4], or nonzero reserved
 *     words; nothing changes then. NULL = RT_FILTER_NONE, which is the reference's render, bit for bit.
 *   - Changing the filter does not reset the accumulation (the host decides, as with rt_set_params); it changes the radiance key,
 *     so a temporal history is dropped.
 *   - With a filter, path-mode renders run the regeneration megakernel without primary-hit reuse: RT_PIPELINE_AUTO does not time
 *     the wavefront or streaming pipelines, and RT_PIPELINE_WAVEFRONT / RT_PIPELINE_STREAM or RT_OPT_BVH_SCHED 1 render with the
 *     megakernel too (rt_stats.pipeline reports RT_PIPELINE_REGEN). traced_segments == segments for such renders, plus the
 *     primary-hit cache pass when the cache is traced as a guide.
 *   - Preview mode and block-filled frames (rt_set_pixel_step > 1) ignore the filter: they are the reference's coarse interaction
 *     frames. rt_pick, rt_read_aov, rt_read_ray_dirs and the primary-hit cache stay the unjittered corner rays, so the denoised,
 *     temporal and group resolves work unchanged on an anti-aliased buffer, guided by the corner rays. */
enum { RT_FILTER_NONE = 0, RT_FILTER_BOX = 1, RT_FILTER_TENT = 2 };
typedef struct {
    int32_t type;           /* RT_FILTER_* */
    float radius;           /* half-width of the footprint in pixels, (0, 4] */
    int32_t reserved[2];    /* 0 */
} rt_pixel_filter;          /* 16 bytes */
void rt_default_pixel_filter(rt_pixel_filter* f);                  /* RT_FILTER_NONE, radius 0.5 (the box's natural width) */
int rt_set_pixel_filter(rt_ctx* ctx, const rt_pixel_filter* f);    /* NULL = none */
int rt_get_pixel_filter(rt_ctx* ctx, rt_pixel_filter* out);
/* The primary direction of global sample `sample` for every pixel (width*height*3 floats, y-up), from the same device function
 * the render kernels use; with RT_FILTER_NONE rt_read_ray_dirs' corner rays. */
int rt_read_sample_dirs(rt_ctx* ctx, uint32_t sample, float* dirs);

/* Page-locked host memory for the surface handed to rt_resolve_rgba8 / rt_read_surface: the device-to-host copy
 * then runs as one DMA instead of being staged by the driver (1280x720 frame loop: 0.30 ms instead of 0.44 ms per
 * frame). Any host pointer works; this is only faster. */
void* rt_host_alloc(size_t bytes);
void rt_host_free(void* p);

/* Mouse picking: GetClosestObject(camera.position, GetRayDirection(camera, x, H - y))
 * (Raytracer.cpp:530-541). x, y in window space (y-down). id = -1 on miss. */
int rt_pick(rt_ctx* ctx, int x, int y_window, int* id);

/* ---- test / inspection hooks ----------------------------------------------------------- */
/* Accumulated SUM image, width*height float4 (r,g,b,0), y-up; *samples = sample count. */
int rt_read_accum(rt_ctx* ctx, float* host_rgba, uint32_t* samples);
/* Checkpoint/resume of a long accumulation: upload a SUM image holding `samples` samples. */
int rt_write_accum(rt_ctx* ctx, const float* host_rgba, uint32_t samples);
/* Primary visibility AOVs (any pointer may be NULL): id int32 (-1 miss), t, normal[3], point[3]. */
int rt_read_aov(rt_ctx* ctx, int32_t* id, float* t, float* normal, float* point);
/* GetRayDirection for every pixel (Raytracer.cpp:106-122): width*height*3 floats. */
int rt_read_ray_dirs(rt_ctx* ctx, float* dirs);
/* GetClosestObject on arbitrary rays (Raytracer.cpp:123-140). */
int rt_trace_rays(rt_ctx* ctx, const float* origins, const float* dirs, int n,
                  int32_t* id, float* t, float* normal, float* point);
/* GetEnvironmentColor (Raytracer.cpp:77-89). */
int rt_env_color(rt_ctx* ctx, const float* dirs, int n, float* rgb);
/* Philox4x32-10 block as the device computes it (known-answer tests). */
int rt_philox_block(rt_ctx* ctx, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* Device self-tests of exact-equivalence shortcuts; *failures = number of mismatching inputs.
 * which = 0: unit_from_word, (float)((double)k * (1.0/32767.0)) == (float)k / 32767.0f for all 32768 k.
 * which = 1: normalize (Common.hpp:159-162) with one shared reciprocal == three IEEE divisions, 2^28 vectors.
 * which = 2: packed FP32 pairs (add / sub / mul / fma.rn.f32x2) == the scalar .rn ops on each half, 2^26 operand sets of
 *            random and edge values (subnormals, +-0, +-inf, near overflow, mixed exponents); two NaN results count as equal. */
int rt_selftest(rt_ctx* ctx, int which, int* failures);
int rt_get_stats(rt_ctx* ctx, rt_stats* out);
/* BVH traversal work actually executed by the render kernels since rt_reset_accumulation, counted on the device while
 * RT_OPT_TRAVERSAL_STATS is 1 (SURVEY.md 8d: bytes per segment = node bytes x <nodes visited> + primitive bytes x <primitives
 * tested>). The per-ray loop (rt_trace_rays, megakernel) visits exactly the nodes the CPU emulation of the same code visits
 * (tests/host_emu); the wavefront intersect kernel postpones leaves, so it visits a few more. */
typedef struct {
    uint64_t queries;              /* closest-hit queries that went through a counting BVH kernel */
    uint64_t node_visits;          /* inner nodes fetched (64 B each: both children's boxes + links) */
    uint64_t prim_tests;           /* leaf primitives tested with the strict intersectors */
    uint64_t sphere_tests, cube_tests, tri_tests;   /* prim_tests by type (16 B + 4 B id, 32 B + 4 B, 48 B + 4 B per test) */
    uint32_t node_bytes, reserved;
} rt_traversal_stats;
int rt_get_traversal_stats(rt_ctx* ctx, rt_traversal_stats* out);

/* ---- device-side interop (multi-GPU reduce, benchmarks) -------------------------------- */
void* rt_accum_device_ptr(rt_ctx* ctx);          /* float4[width*height] sum buffer, device memory */
int rt_set_stream(rt_ctx* ctx, void* cuda_stream);   /* cudaStream_t to launch on (default: own stream) */
int rt_sync(rt_ctx* ctx);
/* Tells the context that the accumulation buffer now holds `samples` samples per pixel
 * (after an external reduce added other ranks' sums). */
int rt_set_sample_count(rt_ctx* ctx, uint32_t samples);
/* Resolve any device float4 sum buffer (n_pixels of it, starting at first_pixel of the image)
 * into a device ARGB8 buffer - the per-rank slice step of reduce-scatter + resolve + gather. */
int rt_resolve_device(rt_ctx* ctx, const void* dev_accum_rgba, uint32_t samples,
                      int first_pixel, int n_pixels, void* dev_out_argb, int flip_y);

/* ---- multi-GPU: fused reduce + resolve over NVLink peer memory ----------------------------
 * With samples sharded over ranks the only exchange of the path is the sum of the accumulation
 * buffers before the resolve. Instead of an all-reduce followed by a resolve, every rank runs ONE
 * kernel over its slice of the pixels that loads that slice from every rank's buffer (its own and
 * the peers' through NVLink P2P mappings), adds them in rank order, applies Reinhard + ARGB8 pack
 * and stores the result straight into the destination surface (typically rank 0's, also
 * peer-mapped): 16 B read per pixel per rank, 4 B written, no intermediate buffer, deterministic
 * summation order. Buffers of other processes are mapped with the rt_ipc_* helpers (CUDA IPC);
 * buffers of other contexts in the same process can be passed as they are: rt_resolve_fused looks every
 * pointer up (cudaPointerGetAttributes) and enables peer access to its device, or fails with RT_ERR_CUDA
 * when the devices cannot reach each other. With rt_resolve_fused the CALLER makes sure every rank's render
 * has completed (a barrier) before launching, and again before reading dst; rt_exchange_* below and
 * rt_group_* do that ordering themselves. */
#define RT_IPC_HANDLE_BYTES 64
#define RT_MAX_PEERS 16
void* rt_argb_device_ptr(rt_ctx* ctx);                       /* uint32[width*height] resolved surface, device */
int rt_ipc_export(rt_ctx* ctx, int which /* 0 accumulation, 1 surface, 2 exchange flags */, unsigned char handle[RT_IPC_HANDLE_BYTES]);
int rt_ipc_open(rt_ctx* ctx, const unsigned char handle[RT_IPC_HANDLE_BYTES], void** dev_ptr);
int rt_ipc_close(rt_ctx* ctx, void* dev_ptr);
int rt_resolve_fused(rt_ctx* ctx, const void* const* accum_ptrs, int world, uint32_t total_samples,
                     int first_pixel, int n_pixels, void* dst_argb_whole_image, int flip_y);
/* Copies the context's device surface to the host (after a fused resolve wrote it). */
int rt_read_surface(rt_ctx* ctx, uint32_t* host_out, int pitch_bytes);

/* One process per GPU: the exchange step WITHOUT host synchronisation or a collective library. Every context owns a
 * small block of flags in device memory (rt_ipc_export(ctx, 2, ..)). rt_exchange_setup gives a context the peer-mapped
 * accumulation buffers and flag blocks of all ranks (rank order; its own entries may be NULL) and the destination
 * surface (rank 0's). rt_exchange_resolve is then stream-ordered and asynchronous:
 *   1. signal: "my samples are in my buffer" is stored into every peer's flag block (st.release.sys over NVLink);
 *   2. k_resolve_fused waits on its OWN flag block until every rank has signalled this epoch, then reduces + resolves
 *      its slice of the pixels from all ranks' buffers into the destination surface;
 *   3. the last CTA signals "my slice is written and I have finished reading your buffers" to every peer;
 *   4. a one-warp kernel waits until every rank has sent that, so whatever is enqueued next on the stream - rank 0's
 *      rt_read_surface, any rank's next rt_reset_accumulation - is ordered after the whole exchange.
 * Epochs only grow, nothing is reset. Every rank needs its OWN device (the ranks wait for each other inside kernels). A wait gives up after ~4 s (a peer died) and the next rt_sync / rt_read_surface
 * reports RT_ERR_CUDA. total_samples: samples per pixel summed over all ranks (the resolve's divisor). */
int rt_exchange_setup(rt_ctx* ctx, int rank, int world, void* const* accum_ptrs, void* const* flag_ptrs, void* dst_argb_whole_image);
int rt_exchange_resolve(rt_ctx* ctx, uint32_t total_samples, int flip_y);

/* ---- library-owned multi-GPU: replaces the worker spawn / join of the reference (Raytracer.cpp:331-342, 598-607) ----
 * SURVEY.md 8b: "rt_create(int device_count, const int* devices, ..) owns streams, device buffers and the exchange". One
 * host process, n devices: a group creates one context per device, enables peer access between them, shards every
 * rt_group_render_spp call by samples per pixel (rt_set_shard(i, n)) and resolves with the fused reduce + resolve
 * kernel, every device writing its slice of the pixels straight into device 0's surface; the ordering between the
 * devices' streams is done with CUDA events (no host synchronisation until the download). No torch, no NCCL, no IPC.
 * Setters are broadcast to every member; rt_group_ctx gives a member for anything else (options, statistics). */
typedef struct rt_group rt_group;
int rt_create_multi(int n_devices, const int* cuda_devices, rt_group** out);   /* cuda_devices NULL: 0 .. n-1 */
int rt_group_destroy(rt_group* g);
int rt_group_size(const rt_group* g);
rt_ctx* rt_group_ctx(rt_group* g, int index);
const char* rt_group_last_error(const rt_group* g);          /* g may be NULL: last rt_create_multi failure */
int rt_group_set_scene(rt_group* g, const rt_object* objects, int n);
int rt_group_load_scene(rt_group* g, const char* json_path);  /* returns object count */
int rt_group_set_mesh(rt_group* g, int object_index, const float* vertices_xyz, int n_vertices, const int32_t* indices, int n_triangles);
int rt_group_set_camera(rt_group* g, const rt_camera* cam);
int rt_group_set_params(rt_group* g, const rt_params* p);
int rt_group_set_option(rt_group* g, int option, int value);
int rt_group_reset_accumulation(rt_group* g);
int rt_group_render_spp(rt_group* g, int spp);               /* spp = GLOBAL samples per pixel, split over the devices */
int rt_group_resolve_rgba8(rt_group* g, uint32_t* host_out, int pitch_bytes, int flip_y);
/* The denoised and temporal resolves of the group's image: rt_denoise_rgba8 / rt_read_denoised / rt_temporal_rgba8 / rt_read_temporal /
 * rt_reset_temporal with the same parameters and NULL defaults, over the sum that rt_group_resolve_rgba8 presents - every member's
 * accumulation buffer added in member order - and the total of the members' sample counts. The sum is gathered into a buffer on device
 * 0 (16 B per pixel, allocated on the first call, freed on a resize) by one kernel per member over its slice of the pixels, in
 * the same arithmetic as the fused resolve; device 0 then filters / blends and packs it. So preview mode and passes 0 give
 * rt_group_resolve_rgba8's bits. Read-only on every member's accumulation buffer, sample counter and path statistics. The guides and
 * the temporal history (pose, accumulation epoch, radiance key) are member 0's: every setter is broadcast and
 * rt_group_reset_accumulation restarts member 0 too, so they describe the group. Bad parameters or output buffer: RT_ERR_INVALID,
 * checked before anything is launched (the history stays as it was). last_resolve_ms of member 0 (rt_group_get_stats) reports
 * filter + pack, not the reduce. Synchronise. */
int rt_group_denoise_rgba8(rt_group* g, const rt_denoise_params* p, uint32_t* host_out, int pitch_bytes, int flip_y);
int rt_group_read_denoised(rt_group* g, const rt_denoise_params* p, float* host_rgba);
int rt_group_temporal_rgba8(rt_group* g, const rt_temporal_params* tp, const rt_denoise_params* dn, uint32_t* host_out, int pitch_bytes, int flip_y);
int rt_group_read_temporal(rt_group* g, const rt_temporal_params* tp, const rt_denoise_params* dn, float* host_rgba);
int rt_group_reset_temporal(rt_group* g);
int rt_group_set_pixel_filter(rt_group* g, const rt_pixel_filter* f);   /* rt_set_pixel_filter on every member */
int rt_group_get_stats(rt_group* g, rt_stats* out);           /* sums over the members; last_render_ms = the slowest */

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
