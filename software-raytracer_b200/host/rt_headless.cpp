// rt_headless - headless driver over the C-ABI: the reference's main loop without SDL/ImGui.
//   rt_headless --scene Scenes/Scene1.json [--width 1280 --height 720 --spp 64 --bounces 8]
//               [--preview] [--scale S] [--out frame.ppm] [--interactive N] [--gpus G] [--denoise K] [--temporal CAP] [--orbit DEG]
// --gpus G (G > 1): the library-owned multi-GPU group (rt_create_multi): the spp are sharded over G devices of this
// process and one fused reduce + resolve kernel per frame writes device 0's surface (path mode, full resolution).
// --scale S: the reference's SCREEN_SCALE (render scale slider, default here 1.0 = every pixel; the reference's is 0.5).
// --interactive N: N frames of 1 spp + resolve + download each (the viewer's per-frame work,
// BASELINE config 5) and prints p50/p99 frame latency.
// --denoise K: the final image, and every --interactive frame, is presented through K passes of the edge-avoiding a-trous
// filter (rt_denoise_rgba8; single GPU only).
// --temporal CAP: frames are presented through the temporal resolve (rt_temporal_rgba8, history cap CAP, --denoise K as its filter;
// single GPU only). --orbit DEG: the camera turns DEG degrees about its up axis before every --interactive frame (a fly-through).
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <vector>

#include "rt_host.hpp"

// A page-locked ARGB8 surface (rt_host_alloc): downloads are one DMA, and rt_render_frame writes it from the render kernel.
struct Pinned {
    uint32_t* p; size_t n;
    explicit Pinned(size_t count) : p(static_cast<uint32_t*>(rt_host_alloc(count * 4))), n(count) { if (!p) throw std::runtime_error("rt_host_alloc failed"); }
    ~Pinned() { rt_host_free(p); }
    Pinned(const Pinned&) = delete;
    Pinned& operator=(const Pinned&) = delete;
    uint32_t* data() { return p; }
    uint32_t* begin() { return p; }
    uint32_t* end() { return p + n; }
};

int main(int argc, char** argv) {
    std::string scene_path, out_path;
    int w = 1280, h = 720, spp = 64, bounces = 8, interactive = 0, gpus = 1, denoise = 0, temporal = 0;
    bool preview = false;
    float scale = 1.0f;
    double orbit = 0.0;
    for (int i = 1; i < argc; ++i) {
        auto arg = [&](const char* n) { return !strcmp(argv[i], n) && i + 1 < argc; };
        if (arg("--scene")) scene_path = argv[++i];
        else if (arg("--width")) w = atoi(argv[++i]);
        else if (arg("--height")) h = atoi(argv[++i]);
        else if (arg("--spp")) spp = atoi(argv[++i]);
        else if (arg("--bounces")) bounces = atoi(argv[++i]);
        else if (arg("--out")) out_path = argv[++i];
        else if (arg("--interactive")) interactive = atoi(argv[++i]);
        else if (arg("--scale")) scale = (float)atof(argv[++i]);
        else if (arg("--gpus")) gpus = atoi(argv[++i]);
        else if (arg("--denoise")) denoise = atoi(argv[++i]);
        else if (arg("--temporal")) temporal = atoi(argv[++i]);
        else if (arg("--orbit")) orbit = atof(argv[++i]);
        else if (!strcmp(argv[i], "--preview")) preview = true;
        else { fprintf(stderr, "unknown argument %s\n", argv[i]); return 2; }
    }
    if (scene_path.empty()) { fprintf(stderr, "usage: rt_headless --scene file.json [options]\n"); return 2; }
    if (denoise < 0 || denoise > 8) { fprintf(stderr, "rt_headless: --denoise takes 0 .. 8 passes\n"); return 2; }
    if (gpus > 1 && denoise > 0) {
        fprintf(stderr, "rt_headless: --denoise is not supported with --gpus > 1 (a member's buffer holds only its shard of the samples)\n");
        return 2;
    }
    if (temporal < 0 || temporal > 4096) { fprintf(stderr, "rt_headless: --temporal takes a history cap of 0 .. 4096\n"); return 2; }
    if (gpus > 1 && temporal > 0) {
        fprintf(stderr, "rt_headless: --temporal is not supported with --gpus > 1 (a member's buffer holds only its shard of the samples)\n");
        return 2;
    }
    if (gpus > 1) {
        // what the reference does with 16 worker threads, across devices: spawn (rt_create_multi), frames (rt_group_render_spp),
        // join + present (rt_group_resolve_rgba8)
        rt_group* g = nullptr;
        auto die = [&](const char* what) { fprintf(stderr, "rt_headless: %s: %s\n", what, rt_group_last_error(g)); if (g) rt_group_destroy(g); return 1; };
        if (rt_create_multi(gpus, nullptr, &g) != RT_OK) return die("rt_create_multi");
        if (rt_group_load_scene(g, scene_path.c_str()) < 0) return die("rt_group_load_scene");
        rt_params par; rt_default_params(&par);
        par.width = w; par.height = h; par.max_bounces = bounces; par.mode = RT_MODE_PATH;
        rt_camera cam; rt_default_camera(&cam);
        if (rt_group_set_params(g, &par) != RT_OK || rt_group_set_camera(g, &cam) != RT_OK || rt_group_reset_accumulation(g) != RT_OK) return die("setup");
        Pinned surface((size_t)w * h);
        using clk = std::chrono::steady_clock;
        if (rt_group_render_spp(g, spp) != RT_OK || rt_group_resolve_rgba8(g, surface.data(), w * 4, 1) != RT_OK) return die("warm-up frame");   // builds, tunes
        if (rt_group_reset_accumulation(g) != RT_OK) return die("reset");
        auto t0 = clk::now();
        if (rt_group_render_spp(g, spp) != RT_OK) return die("rt_group_render_spp");
        if (rt_group_resolve_rgba8(g, surface.data(), w * 4, 1) != RT_OK) return die("rt_group_resolve_rgba8");
        const double ms = std::chrono::duration<double, std::milli>(clk::now() - t0).count();
        rt_stats st;
        if (rt_group_get_stats(g, &st) != RT_OK) return die("rt_group_get_stats");
        printf("{\"gpus\": %d, \"objects\": %u, \"spp\": %u, \"paths\": %llu, \"segments\": %llu, \"wall_ms\": %.3f, \"slowest_render_ms\": %.3f}\n", gpus, st.n_objects,
               st.samples, (unsigned long long)st.paths, (unsigned long long)st.segments, ms, st.last_render_ms);
        if (!out_path.empty()) {
            std::ofstream f(out_path, std::ios::binary);
            f << "P6\n" << w << " " << h << "\n255\n";
            for (uint32_t p : surface) { char rgb[3] = {(char)(p >> 16), (char)(p >> 8), (char)p}; f.write(rgb, 3); }
        }
        rt_group_destroy(g);
        return 0;
    }
    try {
        rtb200::Scene scene1(scene_path);
        scene1.Load();
        if (scene1.lastStatus != RT_OK) fprintf(stderr, "scene load: %s (continuing with %zu objects, like the reference)\n",
                                                scene1.lastError.c_str(), scene1.GetObjects().size());
        rtb200::Raytracer rt(w, h);
        rt.SetObjectsToRender(scene1.GetObjects());
        rt.SIMPLEDRAW = preview; rt.MAXBOUNCES = bounces; rt.TARGETFRAMES = 1 << 30; rt.SCREEN_SCALE = scale;
        rt.DENOISE_PASSES = denoise;
        rt.TEMPORAL_HISTORY = temporal;
        const float orbit_rad = (float)(orbit * M_PI / 180.0);
        Pinned surface((size_t)w * h);                          // interactive frames are streamed into it by the render kernel itself (rt_render_frame)
        using clk = std::chrono::steady_clock;
        if (interactive > 0) {
            std::vector<double> ms;
            for (int f = 0; f < interactive + 10; ++f) {
                if (orbit != 0.0) { rt.camera.RotateAboutAxis(orbit_rad, rt.camera.up); rt.Invalidate(); }
                auto t0 = clk::now();
                rt.RenderFrame(surface.data(), w * 4);
                double d = std::chrono::duration<double, std::milli>(clk::now() - t0).count();
                if (f >= 10) ms.push_back(d);
            }
            std::sort(ms.begin(), ms.end());
            printf("{\"frames\": %d, \"width\": %d, \"height\": %d, \"p50_ms\": %.4f, \"p99_ms\": %.4f, \"mean_ms\": %.4f}\n", interactive, w, h,
                   ms[ms.size() / 2], ms[(size_t)(ms.size() * 0.99)], [&] { double s = 0; for (double v : ms) s += v; return s / ms.size(); }());
        } else {
            auto t0 = clk::now();
            rt.RenderFrame();                                        // first frame after a change: 1/4 scale, overwrite
            rt.RenderFrame();                                        // second frame: full render scale, overwrite
            if (!preview && spp > 1) {                               // the rest of the accumulation in one call
                if (rt_render_spp(rt.Context(), spp - 1) < 0) throw std::runtime_error(rt_last_error(rt.Context()));
                rt.ACCUMULATIONFRAMES = spp;
            }
            rt.Present(surface.data(), w * 4);
            double ms = std::chrono::duration<double, std::milli>(clk::now() - t0).count();
            rt_stats st; rt_get_stats(rt.Context(), &st);
            printf("{\"objects\": %u, \"spp\": %u, \"paths\": %llu, \"segments\": %llu, \"wall_ms\": %.3f, \"render_ms\": %.3f}\n", st.n_objects,
                   st.samples, (unsigned long long)st.paths, (unsigned long long)st.segments, ms, st.last_render_ms);
        }
        if (!out_path.empty()) {                                     // binary PPM of the ARGB surface
            std::ofstream f(out_path, std::ios::binary);
            f << "P6\n" << w << " " << h << "\n255\n";
            for (uint32_t p : surface) { char rgb[3] = {(char)(p >> 16), (char)(p >> 8), (char)p}; f.write(rgb, 3); }
        }
    } catch (const std::exception& e) { fprintf(stderr, "rt_headless: %s\n", e.what()); return 1; }
    return 0;
}
