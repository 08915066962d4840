// rt_viewer - the optional SDL2 / Dear ImGui front end over the C-ABI (SURVEY.md 8 f-4): what main() of the reference
// does around its hot path (Raytracer.cpp:259-615), with the path tracing on the B200 behind host/rt_host.hpp.
//
//   window + streaming surface      Raytracer.cpp:265-270, 543-550   (SDL window, ARGB8 surface uploaded every frame)
//   fly camera                      :388-396 (right mouse: yaw about WORLDUP, pitch about camera.right), :499-524 (WASD/QE, shift)
//   inspector                       :398-487 (scene open / save, create cube / sphere, object properties, settings)
//   object properties               Object.hpp:44-78, 148-152, 207-217 (name, position, colours, smoothness, specular, radius / size)
//   delete / picking                :491-497, :525-542
//   title bar                       :552-562 (fps, accumulated seconds, ACCUMULATIONFRAMES)
//   frame state machine             :568-590 -> rtb200::Raytracer::RenderFrame (1/4-scale first frame, overwrite, accumulate)
//
// Built only where SDL2 and the Dear ImGui sources (1.89.x, with the SDL2 + SDL_Renderer back ends) exist:
//   make -C software-raytracer_b200 viewer IMGUI_DIR=/path/to/imgui          (needs sdl2-config on PATH)
// Neither is in this image, so the target is skipped there; tests/test_capi_cpu.py compiles this file against declaration-only
// stubs (tests/viewer_stubs) so that it cannot rot. The reference's native file dialogs (tinyfiledialogs) are replaced by
// path fields in the inspector.
#include <SDL.h>

#include <chrono>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "imgui.h"
#include "imgui_impl_sdl2.h"
#include "imgui_impl_sdlrenderer.h"
#include "rt_host.hpp"

namespace {

using rtb200::float3;
using rtb200::Object;

const float3 WORLDUP(0, 1, 0);                                // Common.hpp: WORLDUP

// Object::OnGUI + Sphere::OnGUI + Box::OnGUI (Object.hpp:44-78,148-152,207-217). Returns true when anything changed.
bool ObjectGUI(Object& o) {
    const Object before = o;
    char nameBuffer[256];
    snprintf(nameBuffer, sizeof nameBuffer, "%s", o.name.c_str());
    ImGui::InputText("Name", nameBuffer, sizeof nameBuffer);
    o.name = nameBuffer;
    float v[3] = {o.transform.position.x, o.transform.position.y, o.transform.position.z};
    ImGui::DragFloat3("Position", v, 0.1f);
    o.transform.position = float3(v[0], v[1], v[2]);
    if (ImGui::CollapsingHeader("Base Color")) {
        float c[3] = {o.material.BaseColor.r, o.material.BaseColor.g, o.material.BaseColor.b};
        ImGui::ColorPicker3("Color", c);
        o.material.BaseColor = rtb200::Color(c[0], c[1], c[2]);
    }
    float e[3] = {o.material.EmissiveColor.r, o.material.EmissiveColor.g, o.material.EmissiveColor.b};
    ImGui::InputFloat3("Emissive Color", e);
    o.material.EmissiveColor = rtb200::Color(e[0], e[1], e[2]);
    ImGui::SliderFloat("Smoothness", &o.material.Smoothness, 0, 1);
    ImGui::SliderFloat("Specular Amount", &o.material.SpecularAmount, 0, 1);
    ImGui::NewLine();
    if (o.type == Object::SphereType) {
        ImGui::InputFloat("Sphere Radius", &o.radius);
        ImGui::NewLine();
    } else if (o.type == Object::BoxType) {
        float s[3] = {o.size.x, o.size.y, o.size.z};
        ImGui::DragFloat3("Cube Size", s, 0.1f);
        o.size = float3(s[0], s[1], s[2]);
    }
    const rt_object a = before.ToPod(), b = o.ToPod();
    return memcmp(&a, &b, sizeof a) != 0 || before.name != o.name;
}

}  // namespace

int main(int argc, char** argv) {
    int width = 1280, height = 720, device = 0;              // SCREEN_WIDTH / SCREEN_HEIGHT (Raytracer.cpp:26-27)
    std::string scenePath = "./Scenes/Scene1.json";           // :291
    for (int i = 1; i < argc; ++i) {
        if (!strcmp(argv[i], "--scene") && i + 1 < argc) scenePath = argv[++i];
        else if (!strcmp(argv[i], "--width") && i + 1 < argc) width = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--height") && i + 1 < argc) height = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--device") && i + 1 < argc) device = atoi(argv[++i]);
        else { fprintf(stderr, "usage: rt_viewer [--scene file.json] [--width W --height H] [--device N]\n"); return 2; }
    }
    if (SDL_Init(SDL_INIT_VIDEO) != 0) { fprintf(stderr, "SDL_Init: %s\n", SDL_GetError()); return 1; }
    SDL_Window* window = SDL_CreateWindow("Raytracer", SDL_WINDOWPOS_CENTERED, SDL_WINDOWPOS_CENTERED, width, height, 0);
    SDL_Renderer* renderer = SDL_CreateRenderer(window, -1, SDL_RENDERER_ACCELERATED);
    // the reference fills an SDL surface on the CPU and makes a texture of it every frame (:543); here the resolved ARGB8
    // surface comes from the device and is streamed into one texture
    SDL_Texture* renderTexture = SDL_CreateTexture(renderer, SDL_PIXELFORMAT_ARGB8888, SDL_TEXTUREACCESS_STREAMING, width, height);
    if (!window || !renderer || !renderTexture) { fprintf(stderr, "SDL: %s\n", SDL_GetError()); return 1; }

    IMGUI_CHECKVERSION();
    ImGui::CreateContext();
    ImGuiIO& io = ImGui::GetIO();
    io.ConfigDragClickToInputText = true;
    ImGui::StyleColorsDark();
    ImGui_ImplSDL2_InitForSDLRenderer(window, renderer);
    ImGui_ImplSDLRenderer_Init(renderer);

    int rc = 0;
    try {
        rtb200::Scene scene1(scenePath);
        scene1.Load();
        if (scene1.lastStatus != RT_OK) fprintf(stderr, "scene load: %s (continuing with %zu objects, like the reference)\n", scene1.lastError.c_str(), scene1.GetObjects().size());
        rtb200::Raytracer rt(width, height, device);
        rt.SetObjectsToRender(scene1.GetObjects());
        uint32_t* surface = static_cast<uint32_t*>(rt_host_alloc((size_t)width * height * 4));     // page-locked: one DMA per frame
        if (!surface) throw std::runtime_error("rt_host_alloc failed");

        int selected = -1;                                    // selectedObject as an index into scene1.GetObjects()
        bool sceneDirty = false;
        float delta = 0, mouseSpeed = .08f, moveSpeed = 1;
        double totalframetime = 0;
        char savePath[512], loadPath[512];
        snprintf(savePath, sizeof savePath, "%s", scene1.GetFilePath().c_str());
        snprintf(loadPath, sizeof loadPath, "%s", scene1.GetFilePath().c_str());
        auto t1 = std::chrono::steady_clock::now();
        bool running = true, mouseRight = false;
        while (running) {
            int mouseDX = 0, mouseDY = 0;
            bool leftDown = false, keyP = false, keyDelete = false;
            SDL_Event e;
            while (SDL_PollEvent(&e)) {
                ImGui_ImplSDL2_ProcessEvent(&e);
                if (e.type == SDL_QUIT || (e.type == SDL_WINDOWEVENT && e.window.event == SDL_WINDOWEVENT_CLOSE)) running = false;
                else if (e.type == SDL_MOUSEMOTION) { mouseDX += e.motion.xrel; mouseDY += e.motion.yrel; }
                else if (e.type == SDL_MOUSEBUTTONDOWN && e.button.button == SDL_BUTTON_LEFT) leftDown = true;
                else if (e.type == SDL_MOUSEBUTTONDOWN && e.button.button == SDL_BUTTON_RIGHT) mouseRight = true;
                else if (e.type == SDL_MOUSEBUTTONUP && e.button.button == SDL_BUTTON_RIGHT) mouseRight = false;
                else if (e.type == SDL_KEYDOWN && !e.key.repeat) {
                    if (e.key.keysym.scancode == SDL_SCANCODE_P) keyP = true;
                    if (e.key.keysym.scancode == SDL_SCANCODE_DELETE) keyDelete = true;
                }
            }
            if (keyP) rt.pause = !rt.pause;                                                       // :386-388
            if (mouseRight) {                                                                     // :390-394
                rt.Invalidate();
                rt.camera.RotateAboutAxis(mouseDX * mouseSpeed * 0.03f, WORLDUP);
                rt.camera.RotateAboutAxis(mouseDY * mouseSpeed * 0.03f, rt.camera.right);
            }

            ImGui_ImplSDLRenderer_NewFrame();
            ImGui_ImplSDL2_NewFrame();
            ImGui::NewFrame();
            std::vector<Object>& objects = scene1.GetObjects();
            ImGui::Begin("Inspector");
            if (ImGui::BeginMenu("Scene File")) {                                                 // :401-435
                ImGui::InputText("Open path", loadPath, sizeof loadPath);
                if (ImGui::MenuItem("Open..", "Ctrl+O")) {
                    scene1.Unload();
                    scene1 = rtb200::Scene(std::string(loadPath));
                    scene1.Load();
                    sceneDirty = true; selected = -1;
                }
                ImGui::InputText("Save path", savePath, sizeof savePath);
                if (ImGui::MenuItem("Save", "Ctrl+S")) scene1.SaveAs(savePath);
                ImGui::EndMenu();
            }
            if (ImGui::BeginMenu("Create")) {                                                     // :436-451
                const float3 at = rt.camera.position + rt.camera.forward * 5;
                if (ImGui::MenuItem("Cube")) {
                    Object o = Object::Box(float3(1, 1, 1));
                    o.transform.position = at;
                    scene1.AddObject(o); selected = (int)objects.size() - 1; sceneDirty = true;
                }
                if (ImGui::MenuItem("Sphere")) {
                    scene1.AddObject(Object::Sphere(.5f, at)); selected = (int)objects.size() - 1; sceneDirty = true;
                }
                ImGui::EndMenu();
            }
            if (selected >= 0 && selected < (int)objects.size() && ImGui::CollapsingHeader("Object Properties")) {   // :452-457
                // the reference restarts the accumulation on every frame this header is open; here only when a value changed
                if (ObjectGUI(objects[(size_t)selected])) sceneDirty = true;
            }
            if (ImGui::CollapsingHeader("Settings")) {                                            // :458-483
                if (ImGui::Button("Switch Render Mode")) { rt.SIMPLEDRAW = !rt.SIMPLEDRAW; rt.Invalidate(); }
                ImGui::InputInt("Max Frames", &rt.TARGETFRAMES);
                int v = rt.FOV;
                ImGui::SliderInt("FOV", &v, 15, 103);
                if (v != rt.FOV) { rt.FOV = v; rt.Invalidate(); }
                v = rt.MAXBOUNCES;
                ImGui::InputInt("Light Bounces", &v);
                if (v != rt.MAXBOUNCES) { rt.MAXBOUNCES = v < 0 ? 0 : v; rt.Invalidate(); }
                const float scaleBefore = rt.SCREEN_SCALE;
                ImGui::SliderFloat("Render Scale", &rt.SCREEN_SCALE, 0.25f, 1.0f);
                if (rt.SIMPLEDRAW) rt.SCREEN_SCALE = rt.SCREEN_SCALE < 0.25f ? 0.25f : rt.SCREEN_SCALE > 0.5f ? 0.5f : rt.SCREEN_SCALE;
                if (rt.SCREEN_SCALE != scaleBefore) rt.Invalidate();      // block size changes: mixing would blur (the reference keeps accumulating)
                ImGui::SliderInt("Denoise passes", &rt.DENOISE_PASSES, 0, 8);  // presentation only: the accumulation goes on
                ImGui::SliderInt("Temporal history", &rt.TEMPORAL_HISTORY, 0, 256);   // 0: off; > 0: the image survives camera moves
            }
            ImGui::Text("Application average %.3f \nms/frame (%.1f FPS)", 1000.0f / io.Framerate, io.Framerate);
            ImGui::End();

            if (!io.WantCaptureMouse && !io.WantCaptureKeyboard) {                                 // :489-542
                if (selected >= 0 && keyDelete) {
                    scene1.RemoveObject((size_t)selected);
                    selected = -1; sceneDirty = true;
                }
                const Uint8* keys = SDL_GetKeyboardState(nullptr);
                float speed = moveSpeed * delta;
                const float3 previousPos = rt.camera.position;
                if (keys[SDL_SCANCODE_LSHIFT]) speed = 2 * delta;
                if (keys[SDL_SCANCODE_W]) rt.camera.position = rt.camera.position + rt.camera.forward * speed;
                if (keys[SDL_SCANCODE_D]) rt.camera.position = rt.camera.position + rt.camera.right * speed;
                if (keys[SDL_SCANCODE_A]) rt.camera.position = rt.camera.position - rt.camera.right * speed;
                if (keys[SDL_SCANCODE_S]) rt.camera.position = rt.camera.position - rt.camera.forward * speed;
                if (keys[SDL_SCANCODE_E]) rt.camera.position = rt.camera.position + rt.camera.up * speed;
                if (keys[SDL_SCANCODE_Q]) rt.camera.position = rt.camera.position - rt.camera.up * speed;
                if (rt.camera.position != previousPos) rt.Invalidate();
                if (leftDown) {                                                                   // :525-541
                    if (selected >= 0) selected = -1;
                    else {
                        int x, y;
                        SDL_GetMouseState(&x, &y);
                        selected = rt.Pick(x, y);                                                 // window coordinates; -1 on a miss
                    }
                    if (rt.SIMPLEDRAW) rt.Invalidate();                                           // the highlight is part of the preview image
                }
            }
            if (sceneDirty) {                                   // `ObjectsToRender = scene1.GetObjects()` (:421) after any edit
                rt.SetObjectsToRender(scene1.GetObjects());
                sceneDirty = false;
            }
            rt.selectedObject = selected;

            // the render step of the loop (:568-590) + the surface update, then present
            rt.RenderFrame(surface, width * 4);               // traced and presented in one call (rt_render_frame)
            SDL_UpdateTexture(renderTexture, nullptr, surface, width * 4);
            ImGui::Render();
            SDL_RenderSetScale(renderer, io.DisplayFramebufferScale.x, io.DisplayFramebufferScale.y);
            SDL_RenderClear(renderer);
            SDL_RenderCopy(renderer, renderTexture, nullptr, nullptr);
            ImGui_ImplSDLRenderer_RenderDrawData(ImGui::GetDrawData());
            SDL_RenderPresent(renderer);

            const auto t2 = std::chrono::steady_clock::now();                                     // :552-565
            const double frametime = std::chrono::duration<double, std::milli>(t2 - t1).count();
            delta = (float)(frametime / 1000.0);
            totalframetime += rt.SIMPLEDRAW ? 0 : delta;
            if (rt.ACCUMULATIONFRAMES <= 1) totalframetime = 0;
            char title[256];
            snprintf(title, sizeof title, "fps: %f | total time (seconds): %f | ACCUMULATIONFRAMES: %d | ", frametime > 0 ? 1000.0 / frametime : 0.0, totalframetime, rt.ACCUMULATIONFRAMES);
            SDL_SetWindowTitle(window, title);
            t1 = std::chrono::steady_clock::now();
        }
        rt_host_free(surface);
    } catch (const std::exception& ex) {
        fprintf(stderr, "rt_viewer: %s\n", ex.what());
        rc = 1;
    }
    ImGui_ImplSDLRenderer_Shutdown();
    ImGui_ImplSDL2_Shutdown();
    ImGui::DestroyContext();
    SDL_DestroyTexture(renderTexture);
    SDL_DestroyRenderer(renderer);
    SDL_DestroyWindow(window);
    SDL_Quit();
    return rc;
}
