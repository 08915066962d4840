// rt_host.hpp - C++ host-side mirror of the reference's interface for the hot path, over the C-ABI
// (include/rt_b200.h). Same names and argument meaning as the reference so its main loop ports by
// search-and-replace (INTEGRATION.md): Transform::RotateAboutAxis (Common.hpp:287-291), Material
// (Common.hpp:293-319), Object/Sphere/Box (Object.hpp:19-234), Scene::Load/Save/SaveAs/GetObjects/
// AddObject/RemoveObject/Unload (Scene.hpp:12-119), and a Raytracer class that owns what were the
// globals and free functions of Raytracer.cpp:26-61, 63-257 and the frame state machine :572-595.
// Header-only; links against librt_b200.so. No rendering happens on the CPU here.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/rt_b200.h"

namespace rtb200 {

struct float3 {
    float x = 0, y = 0, z = 0;
    float3() = default;
    float3(float x_, float y_, float z_) : x(x_), y(y_), z(z_) {}
    float3 operator+(const float3& o) const { return {x + o.x, y + o.y, z + o.z}; }
    float3 operator-(const float3& o) const { return {x - o.x, y - o.y, z - o.z}; }
    float3 operator*(float s) const { return {x * s, y * s, z * s}; }
    bool operator!=(const float3& o) const { return x != o.x || y != o.y || z != o.z; }
};
struct Color { float r = 0, g = 0, b = 0; Color() = default; Color(float r_, float g_, float b_) : r(r_ < 0 ? 0 : r_), g(g_ < 0 ? 0 : g_), b(b_ < 0 ? 0 : b_) {} };

struct Transform {                                   // Common.hpp:281-292
    float3 right{1, 0, 0}, up{0, 1, 0}, forward{0, 0, 1}, position{0, 0, 0};
    void RotateAboutAxis(float angle, float3 axis) {
        rt_camera c = ToCamera(0);
        const float ax[3] = {axis.x, axis.y, axis.z};
        rt_rotate_camera(&c, angle, ax);             // the reference's Rodrigues expression, in its order
        right = {c.right[0], c.right[1], c.right[2]}; up = {c.up[0], c.up[1], c.up[2]};
        forward = {c.forward[0], c.forward[1], c.forward[2]};
    }
    rt_camera ToCamera(int fov) const {
        rt_camera c;
        const float3* v[4] = {&position, &right, &up, &forward};
        float* d[4] = {c.pos, c.right, c.up, c.forward};
        for (int i = 0; i < 4; ++i) { d[i][0] = v[i]->x; d[i][1] = v[i]->y; d[i][2] = v[i]->z; }
        c.fov_deg = fov;
        return c;
    }
};

struct Material {                                    // Common.hpp:293-319
    float Smoothness = 0.5f, SpecularAmount = 0.0f;
    Color BaseColor{1, 1, 1}, EmissiveColor{0, 0, 0}, SpecularColor{1, 1, 1};
};

struct Object {                                      // Object.hpp:19-26 (+ Sphere :86, Box :170 as a tagged value)
    enum Type { None = RT_OBJ_NONE, SphereType = RT_OBJ_SPHERE, BoxType = RT_OBJ_CUBE } type = None;
    Transform transform; Material material; std::string name;
    float radius = 0; float3 size;
    static Object Sphere(float radius, float3 position) { Object o; o.type = SphereType; o.radius = radius; o.transform.position = position; return o; }
    static Object Box(float3 size) { Object o; o.type = BoxType; o.size = size; return o; }
    rt_object ToPod() const {
        rt_object p{};
        p.type = type;
        p.pos[0] = transform.position.x; p.pos[1] = transform.position.y; p.pos[2] = transform.position.z;
        p.radius = radius; p.half[0] = size.x; p.half[1] = size.y; p.half[2] = size.z;
        const Color* c[3] = {&material.BaseColor, &material.EmissiveColor, &material.SpecularColor};
        float* d[3] = {p.base, p.emissive, p.spec_color};
        for (int i = 0; i < 3; ++i) { d[i][0] = c[i]->r; d[i][1] = c[i]->g; d[i][2] = c[i]->b; }
        p.smoothness = material.Smoothness; p.spec_amount = material.SpecularAmount;
        return p;
    }
    static Object FromPod(const rt_object& p, const std::string& name) {
        Object o; o.type = (Type)p.type; o.name = name;
        o.transform.position = {p.pos[0], p.pos[1], p.pos[2]}; o.radius = p.radius; o.size = {p.half[0], p.half[1], p.half[2]};
        o.material.BaseColor = {p.base[0], p.base[1], p.base[2]}; o.material.EmissiveColor = {p.emissive[0], p.emissive[1], p.emissive[2]};
        o.material.SpecularColor = {p.spec_color[0], p.spec_color[1], p.spec_color[2]};
        o.material.Smoothness = p.smoothness; o.material.SpecularAmount = p.spec_amount;
        return o;
    }
};

class Scene {                                        // Scene.hpp:12-119
    std::string fileName;
    std::vector<Object> sceneObjects;
public:
    std::string sceneName;
    int lastStatus = RT_OK;                          // the reference fails silently; the status is kept here
    std::string lastError;
    explicit Scene(std::string file) : fileName(std::move(file)) {}
    std::vector<Object>& GetObjects() { return sceneObjects; }
    std::string GetFilePath() const { return fileName; }
    void Load() {                                    // Scene.hpp:27-80 (host-only reader of the C-ABI library)
        sceneObjects.clear();
        int n = 0; char err[512] = {0};
        lastStatus = rt_scene_file_read(fileName.c_str(), nullptr, 0, &n, err, sizeof err);
        std::vector<rt_object> pods((size_t)n);
        if (n) rt_scene_file_read(fileName.c_str(), pods.data(), n, &n, err, sizeof err);
        lastError = err;
        std::vector<char> names((size_t)rt_scene_file_read_names(fileName.c_str(), nullptr, 0, nullptr, 0) + 1);
        char sn[1024] = {0};
        rt_scene_file_read_names(fileName.c_str(), names.data(), (int)names.size(), sn, sizeof sn);
        sceneName = sn;
        const char* q = names.data();
        for (const rt_object& p : pods) { sceneObjects.push_back(Object::FromPod(p, q)); q += strlen(q) + 1; }
    }
    void Unload() { sceneObjects.clear(); }
    void Save() {                                    // Scene.hpp:88-100
        std::vector<rt_object> pods; std::vector<const char*> names;
        for (const Object& o : sceneObjects) { pods.push_back(o.ToPod()); names.push_back(o.name.c_str()); }
        lastStatus = rt_scene_file_write(fileName.c_str(), sceneName.c_str(), pods.data(), names.data(), (int)pods.size());
    }
    void SaveAs(std::string file) { fileName = std::move(file); Save(); }
    void AddObject(const Object& o) { sceneObjects.push_back(o); }
    void RemoveObject(size_t index) { if (index < sceneObjects.size()) sceneObjects.erase(sceneObjects.begin() + index); }
};

// What Raytracer.cpp keeps in globals and free functions, as one object over an rt_ctx.
class Raytracer {
    rt_ctx* ctx = nullptr;
    rt_params par;
    bool doSetFrame = true;
    static void check(int rc, rt_ctx* c) { if (rc < 0) throw std::runtime_error(rt_last_error(c)); }
public:
    int FOV = 55, MAXBOUNCES = 2, TARGETFRAMES = 4096, ACCUMULATIONFRAMES = 1;     // Raytracer.cpp:31-34
    bool SIMPLEDRAW = true;                                                         // :35
    int selectedObject = -1;                                                        // :53 (as an object index)
    int DENOISE_PASSES = 0;                         // > 0: frames are presented through the a-trous filter (rt_denoise_rgba8), 0: plain resolve
    int TEMPORAL_HISTORY = 0;                       // > 0: frames are presented through the temporal resolve (rt_temporal_rgba8) with this
                                                    // history cap (and DENOISE_PASSES as its filter), 0: off
    Transform camera;                                                               // :295-297

    Raytracer(int width = 1280, int height = 720, int device = 0) {                 // :26-27
        check(rt_create(device, &ctx), nullptr);
        rt_default_params(&par);
        par.width = width; par.height = height;
    }
    ~Raytracer() { if (ctx) rt_destroy(ctx); }
    Raytracer(const Raytracer&) = delete;
    Raytracer& operator=(const Raytracer&) = delete;
    rt_ctx* Context() { return ctx; }

    // `ObjectsToRender = scene1.GetObjects()` (Raytracer.cpp:293,421)
    void SetObjectsToRender(const std::vector<Object>& objs) {
        std::vector<rt_object> pods;
        for (const Object& o : objs) pods.push_back(o.ToPod());
        check(rt_set_scene(ctx, pods.data(), (int)pods.size()), ctx);
        doSetFrame = true;
    }
    // Scene files with the Mesh extension ("Renderer": {"Type": "Mesh", ...}, csrc/mesh.h) carry geometry the POD object
    // list cannot: load them inside the library. Returns the object count; throws on I/O or parse errors.
    int LoadSceneFile(const std::string& path) {
        int n = rt_load_scene(ctx, path.c_str());
        check(n, ctx);
        doSetFrame = true;
        return n;
    }
    // Attach triangles (object-space xyz, index triples) to object `index`, which must be of type RT_OBJ_MESH.
    void SetMesh(int index, const std::vector<float>& vertices, const std::vector<int32_t>& indices) {
        check(rt_set_mesh(ctx, index, vertices.data(), (int)(vertices.size() / 3), indices.data(), (int)(indices.size() / 3)), ctx);
        doSetFrame = true;
    }
    void Invalidate() { doSetFrame = true; }         // any edit: doSetFrame = true (Raytracer.cpp:393,422,454,...)

    float SCREEN_SCALE = .5f;                                                       // :30 (slider 0.25 .. 1.0, :479)
    bool pause = false;                                                             // :50 ('P')
    float progressiveResolutionScaler = 1;                                          // :47

    // One iteration of the main loop's render step (Raytracer.cpp:572-595 + the workers' frame :231-252): returns
    // false when nothing was rendered (paused, or the frame cap reached). As in the reference the first frame after
    // a change is traced at 1/4 of the render scale and overwrites (:576-581), the next one is at full render scale
    // and overwrites again (:585-587), and later frames accumulate; every frame is block-filled with
    // steps = ceil(1 / (SCREEN_SCALE * progressiveResolutionScaler)) over the reference's 16 column strips (:233,330).
    // One deviation, on purpose: the reference's running mean counts that second frame twice (ACCUMULATIONFRAMES is
    // already 2 when it overwrites); here every accumulated frame has the same weight.
    bool RenderFrame() {
        if (!BeginFrame()) return false;
        check(rt_render_spp(ctx, 1), ctx);
        return true;
    }
    // The same frame traced AND presented in one call (rt_render_frame): the reference's workers write the surface pixel by
    // pixel while they trace (SetScreenPixel inside renderArea, :63-76,250), and so does the render kernel for full-resolution
    // accumulation frames - with a page-locked surface the frame then costs the render alone.
    // With DENOISE_PASSES > 0 or TEMPORAL_HISTORY > 0 the frame is traced (rt_render_spp) and then presented through Present.
    bool RenderFrame(uint32_t* pixels, int pitch_bytes) {
        if (!BeginFrame()) return false;
        if (DENOISE_PASSES > 0 || TEMPORAL_HISTORY > 0) {
            check(rt_render_spp(ctx, 1), ctx);
            Present(pixels, pitch_bytes);
        } else {
            check(rt_render_frame(ctx, 1, pixels, pitch_bytes, 1), ctx);
        }
        return true;
    }
    // SDL surface update (the resolve half of SetScreenPixel, Raytracer.cpp:73-75): ARGB8, rows y-down. With DENOISE_PASSES > 0
    // through the edge-avoiding filter (rt_denoise_rgba8, the library's default tolerances); with TEMPORAL_HISTORY > 0 through the
    // temporal resolve (rt_temporal_rgba8: the library's default tolerances, TEMPORAL_HISTORY as the cap, the filter if asked for).
    void Present(uint32_t* pixels, int pitch_bytes) {
        rt_denoise_params dp;
        rt_default_denoise_params(&dp);
        dp.passes = DENOISE_PASSES;
        if (TEMPORAL_HISTORY > 0) {
            rt_temporal_params tp;
            rt_default_temporal_params(&tp);
            tp.max_history = TEMPORAL_HISTORY;
            check(rt_temporal_rgba8(ctx, &tp, DENOISE_PASSES > 0 ? &dp : nullptr, pixels, pitch_bytes, 1), ctx);
        } else if (DENOISE_PASSES > 0) {
            check(rt_denoise_rgba8(ctx, &dp, pixels, pitch_bytes, 1), ctx);
        } else {
            check(rt_resolve_rgba8(ctx, pixels, pitch_bytes, 1), ctx);
        }
    }
    // Mouse picking (Raytracer.cpp:530-541), window coordinates.
    int Pick(int x, int y) { int id = -1; check(rt_pick(ctx, x, y, &id), ctx); return id; }
    int Width() const { return par.width; }
    int Height() const { return par.height; }

private:
    // the frame state machine up to (not including) the trace: false when nothing is to be rendered
    bool BeginFrame() {
        if (pause || (!doSetFrame && ACCUMULATIONFRAMES == TARGETFRAMES)) return false;     // :572
        par.max_bounces = MAXBOUNCES; par.mode = SIMPLEDRAW ? RT_MODE_PREVIEW : RT_MODE_PATH; par.selected_id = selectedObject;
        check(rt_set_params(ctx, &par), ctx);
        rt_camera cam = camera.ToCamera(FOV);
        check(rt_set_camera(ctx, &cam), ctx);
        bool setFrame;
        // :576-581; the 1/4-scale first frame only shows something quickly, which the reprojected history does with TEMPORAL_HISTORY > 0
        if (doSetFrame) { setFrame = true; ACCUMULATIONFRAMES = 1; progressiveResolutionScaler = TEMPORAL_HISTORY > 0 ? 1.0f : 1.0f / 4.0f; doSetFrame = false; }
        else {
            setFrame = progressiveResolutionScaler != 1;                            // :584-587
            progressiveResolutionScaler = 1;
            ACCUMULATIONFRAMES += SIMPLEDRAW ? 0 : 1;                               // :589
        }
        if (setFrame) check(rt_reset_accumulation(ctx), ctx);
        check(rt_set_pixel_step(ctx, rt_reference_pixel_step(SCREEN_SCALE, progressiveResolutionScaler), rt_reference_strip_columns(par.width)), ctx);
        return true;
    }
};

}  // namespace rtb200
