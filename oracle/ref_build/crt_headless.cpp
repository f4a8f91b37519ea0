// crt_headless.cpp — a headless twin of ChameleonRT's app loop (TEST INFRASTRUCTURE).
//
// Does what the reference's main.cpp:113-345 does minus SDL / ImGui widgets / OpenGL: same CLI
// flags, loads lib crt_<backend>.so through the REFERENCE'S OWN RenderPlugin class
// (util/render_plugin.cpp, compiled from /root/reference where it lies), builds the scene with
// the reference's own loaders (util/scene.cpp), derives the camera vectors with the
// reference's ArcballCamera, then initialize -> set_scene -> render x N. It proves that
// libcrt_cuda.so is a drop-in for `./chameleonrt cuda <scene>` on a box without SDL2/GL.
//
//   crt_headless <backend> <scene.obj|.gltf|.glb|.crts> [-eye x y z] [-center x y z] [-up x y z]
//                [-fov deg] [-spp n] [-img w h] [-mat-mode white_diffuse] [-benchmark-frames n]
//                [-validation prefix] [-accum out.f32]
#include <chrono>
#include <cstdio>
#include <dlfcn.h>
#include <fstream>
#include <iostream>
#include <memory>
#include <string>
#include <vector>
#include "arcball_camera.h"
#include "imgui.h"
#include "render_plugin.h"
#include "scene.h"
#include "scene_native_load.h"
#include "stb_image_write.h"
#include "util.h"

int main(int argc, const char **argv)
{
    const std::vector<std::string> args(argv, argv + argc);
    if (args.size() < 3) {
        std::cout << "usage: crt_headless <backend> <scene> [options]\n";
        return 1;
    }
    int win_width = 1280, win_height = 720;  // main.cpp:35-36
    std::string scene_file;
    glm::vec3 eye(0, 0, 5), center(0), up(0, 1, 0);
    float fov_y = 65.f;
    uint32_t samples_per_pixel = 1;
    size_t camera_id = 0, benchmark_frames = 1;
    bool got_camera_args = false;
    std::string validation_img_prefix, accum_out;
    MaterialMode material_mode = MaterialMode::DEFAULT;
    for (size_t i = 2; i < args.size(); ++i) {  // main.cpp:131-168
        if (args[i] == "-eye") {
            eye = glm::vec3(std::stof(args[i + 1]), std::stof(args[i + 2]), std::stof(args[i + 3]));
            i += 3;
            got_camera_args = true;
        } else if (args[i] == "-center") {
            center = glm::vec3(std::stof(args[i + 1]), std::stof(args[i + 2]), std::stof(args[i + 3]));
            i += 3;
            got_camera_args = true;
        } else if (args[i] == "-up") {
            up = glm::vec3(std::stof(args[i + 1]), std::stof(args[i + 2]), std::stof(args[i + 3]));
            i += 3;
            got_camera_args = true;
        } else if (args[i] == "-fov") {
            fov_y = std::stof(args[++i]);
            got_camera_args = true;
        } else if (args[i] == "-spp") {
            samples_per_pixel = std::stoi(args[++i]);
        } else if (args[i] == "-camera") {
            camera_id = std::stol(args[++i]);
        } else if (args[i] == "-validation") {
            validation_img_prefix = args[++i];
        } else if (args[i] == "-img") {
            win_width = std::stoi(args[++i]);
            win_height = std::stoi(args[++i]);
        } else if (args[i] == "-mat-mode") {
            if (args[++i] == "white_diffuse") {
                material_mode = MaterialMode::WHITE_DIFFUSE;
            }
        } else if (args[i] == "-benchmark-frames") {
            benchmark_frames = std::stoi(args[++i]);
        } else if (args[i] == "-accum") {
            accum_out = args[++i];
        } else if (args[i][0] != '-') {
            scene_file = args[i];
            canonicalize_path(scene_file);
        }
    }

    // The reference looks for lib crt_<backend>.so next to the executable (util/render_plugin.cpp:7-18): every plugin,
    // the product's libcrt_cuda.so included, is built into oracle/_ref/ beside this harness.
    // main.cpp:65-66, :94-100
    auto plugin = std::make_unique<RenderPlugin>("crt_" + args[1]);
    ImGuiContext *ctx = ImGui::CreateContext();
    plugin->set_imgui_context(ctx);
    std::unique_ptr<Display> display = plugin->make_display(nullptr);
    {
        std::unique_ptr<RenderBackend> renderer = plugin->make_renderer(display.get());
        display->resize(win_width, win_height);
        renderer->initialize(win_width, win_height);
        {
            // CRT_NATIVE_LOADER=1: the line a maintainer would put in main.cpp:186 instead (backends/cuda/scene_native_load.h)
            const char *native = std::getenv("CRT_NATIVE_LOADER");
            const auto load_t0 = std::chrono::steady_clock::now();
            Scene scene = (native && native[0] == '1') ? crt_cuda::load_scene_native(scene_file, material_mode) : Scene(scene_file, material_mode);
            std::cout << "scene load: " << std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - load_t0).count()
                      << " ms (" << ((native && native[0] == '1') ? "native loader" : "Scene constructor") << ")\n";
            scene.samples_per_pixel = samples_per_pixel;
            std::cout << "Scene '" << scene_file << "': tris " << scene.total_tris() << " geometries "
                      << scene.num_geometries() << " instances " << scene.instances.size() << " materials "
                      << scene.materials.size() << " textures " << scene.textures.size() << " lights "
                      << scene.lights.size() << " spp " << scene.samples_per_pixel << "\n";
            renderer->set_scene(scene);
            if (!got_camera_args && !scene.cameras.empty()) {
                eye = scene.cameras[camera_id].position;
                center = scene.cameras[camera_id].center;
                up = scene.cameras[camera_id].up;
                fov_y = scene.cameras[camera_id].fov_y;
            }
        }  // the Scene is destroyed here, as in main.cpp:214
        ArcballCamera camera(eye, center, up);
        std::cout << "backend: " << renderer->name() << "\n";
        {
            // exact (hex-float) camera vectors handed to render(), so a harness can replay them
            const glm::vec3 e = camera.eye(), d = camera.dir(), u = camera.up();
            char buf[512];
            std::snprintf(buf, sizeof(buf), "camera: %a %a %a %a %a %a %a %a %a %a\n", e.x, e.y, e.z, d.x, d.y, d.z, u.x,
                          u.y, u.z, fov_y);
            std::cout << buf;
        }
        float render_time = 0.f, rays_per_second = 0.f;
        bool camera_changed = true;
        for (size_t frame_id = 0; frame_id < benchmark_frames; ++frame_id) {
            const bool need_readback = !validation_img_prefix.empty() || frame_id + 1 == benchmark_frames;
            RenderStats stats = renderer->render(camera.eye(), camera.dir(), camera.up(), fov_y, camera_changed,
                                                 need_readback);  // main.cpp:300-301
            camera_changed = false;
            render_time += stats.render_time;
            rays_per_second += stats.rays_per_second;
            if (!validation_img_prefix.empty()) {
                const std::string img_name =
                    validation_img_prefix + args[1] + "-f" + std::to_string(frame_id) + ".png";
                stbi_write_png(img_name.c_str(), win_width, win_height, 4, renderer->img.data(), 4 * win_width);
            }
        }
        stbi_write_png("chameleonrt.png", win_width, win_height, 4, renderer->img.data(), 4 * win_width);
        // main.cpp:334-343
        std::cout << "Benchmark results: " << render_time / benchmark_frames << " ms/frame ("
                  << 1000.f / (render_time / benchmark_frames) << " FPS)\n";
        if (rays_per_second > 0) {
            std::cout << "Rays/s (mean of per-frame rates): "
                      << pretty_print_count(rays_per_second / benchmark_frames) << "\n";
        }
        {
            // the other extra export of the cuda / oracle plugins: per-stage times and counters of the last frame
            using GetStatsFn = int (*)(RenderBackend *, float *, int, uint64_t *, int);
            const std::string sym = "crt_" + args[1] + "_get_stats";
            GetStatsFn fn = reinterpret_cast<GetStatsFn>(dlsym(RTLD_DEFAULT, sym.c_str()));
            if (!fn) {
                void *h = dlopen((std::string(SDL_GetBasePath()) + "libcrt_" + args[1] + ".so").c_str(), RTLD_LAZY | RTLD_NOLOAD);
                fn = h ? reinterpret_cast<GetStatsFn>(dlsym(h, sym.c_str())) : nullptr;
            }
            float stage_ms[7] = {0, 0, 0, 0, 0, 0, 0};
            uint64_t counters[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            if (fn && fn(renderer.get(), stage_ms, 7, counters, 8) == 0) {
                std::cout << "last frame: stage ms";
                for (float v : stage_ms) {
                    std::cout << " " << v;
                }
                std::cout << " | counters";
                for (uint64_t v : counters) {
                    std::cout << " " << v;
                }
                std::cout << "\n";
            }
        }
        if (!accum_out.empty()) {
            // the extra export of the cuda / oracle plugins (not part of the reference API)
            const std::string sym = "crt_" + args[1] + "_read_accum";
            using ReadAccumFn = int (*)(RenderBackend *, float *);
            ReadAccumFn fn = reinterpret_cast<ReadAccumFn>(dlsym(RTLD_DEFAULT, sym.c_str()));
            if (!fn) {
                void *h = dlopen((std::string(SDL_GetBasePath()) + "libcrt_" + args[1] + ".so").c_str(),
                                 RTLD_LAZY | RTLD_NOLOAD);
                fn = h ? reinterpret_cast<ReadAccumFn>(dlsym(h, sym.c_str())) : nullptr;
            }
            if (!fn) {
                std::cerr << "plugin does not export " << sym << "\n";
                return 2;
            }
            std::vector<float> accum(static_cast<size_t>(win_width) * win_height * 3);
            fn(renderer.get(), accum.data());
            std::ofstream f(accum_out, std::ios::binary);
            f.write(reinterpret_cast<const char *>(accum.data()), accum.size() * sizeof(float));
        }
    }
    display = nullptr;
    ImGui::DestroyContext(ctx);
    return 0;
}
