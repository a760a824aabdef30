// gs_viewer_headless -- the reference viewer's command line (apps/viewer/main.cpp:12-98) without a window:
//   gs_viewer_headless [-d DEVICE] [-w WIDTH] [-h HEIGHT] [-v] [--frames N] [--camera x,y,z[,qw,qx,qy,qz]]
//                      [--fov DEG] [--camera-path poses.txt] [--mode exact|fast] [--cull [LEVEL]] [--out image.ppm]
//                      [--float-out image.pfm] [--alpha-out alpha.pfm] [--depth-out depth.pfm] scene.ply
// --camera-path: one pose per line `x y z qw qx qy qz [fov]` (# comments); `--frames` frames are rendered at each pose
// and one JSON line is printed per pose (SURVEY 8d: record M for every timed camera).
// Loads the .ply through GSScene, renders N frames through Renderer::draw() (B8G8R8A8 like the swapchain),
// prints the six per-stage timers + `instances` (Renderer.cpp:85-100,540) as one JSON line per run and
// optionally writes the last frame as a binary PPM (8-bit, what the swapchain would show) and / or as a PFM (float32 RGB, the
// unquantised blend render.comp:98 stores: what the 1e-4 parity tolerance is defined on).  The first JSON line also carries
// the load times (file read + activation, upload + cov3D ingest).  --alpha-out / --depth-out write the opacity (1 - final
// transmittance) and the un-normalised expected depth of one Renderer::renderAux frame as greyscale PFMs ("Pf", bottom to top).  Environment: VKGS_PHYSICAL_DEVICE like the viewer.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

#include "Renderer.h"

static void usage() {
    std::puts("usage: gs_viewer_headless [-d device] [-w width] [-h height] [-v] [--frames n] [--camera x,y,z[,qw,qx,qy,qz]]\n"
              "                          [--fov deg] [--camera-path poses.txt] [--mode exact|fast] [--cull [0|1|2]] [--out image.ppm]\n"
              "                          [--float-out image.pfm] [--alpha-out alpha.pfm] [--depth-out depth.pfm] scene.ply");
}

int main(int argc, char** argv) {
    Renderer::Configuration cfg;
    std::string out_path, float_path, alpha_path, depth_path, scene, path_file;
    int cull_level = 0;
    uint32_t frames = 1;
    bool verbose = false, cull = false;
    float cam[7] = {0, 0, 0, 1, 0, 0, 0};
    float fov = 45.0f;
    if (const char* env = std::getenv("VKGS_PHYSICAL_DEVICE")) cfg.physicalDeviceId = static_cast<uint8_t>(std::atoi(env));
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto next = [&]() -> const char* {
            if (i + 1 >= argc) {
                usage();
                std::exit(1);
            }
            return argv[++i];
        };
        if (a == "-d" || a == "--device") cfg.physicalDeviceId = static_cast<uint8_t>(std::atoi(next()));
        else if (a == "-w" || a == "--width") cfg.width = static_cast<uint32_t>(std::atoi(next()));
        else if (a == "-h" || a == "--height") cfg.height = static_cast<uint32_t>(std::atoi(next()));
        else if (a == "-v" || a == "--verbose") verbose = true;
        else if (a == "--frames") frames = static_cast<uint32_t>(std::atoi(next()));
        else if (a == "--fov") fov = static_cast<float>(std::atof(next()));
        else if (a == "--mode") cfg.mode = std::string(next()) == "fast" ? GSB_MODE_FAST : GSB_MODE_EXACT;
        else if (a == "--cull") {
            cull = true;
            cull_level = 1;
            if (i + 1 < argc && std::strlen(argv[i + 1]) == 1 && argv[i + 1][0] >= '0' && argv[i + 1][0] <= '2') cull_level = argv[++i][0] - '0';
        } else if (a == "--float-out") float_path = next();
        else if (a == "--alpha-out") alpha_path = next();
        else if (a == "--depth-out") depth_path = next();
        else if (a == "--out") out_path = next();
        else if (a == "--camera-path") path_file = next();
        else if (a == "--camera") {
            int k = 0;
            for (char* tok = std::strtok(const_cast<char*>(next()), ","); tok && k < 7; tok = std::strtok(nullptr, ",")) cam[k++] = static_cast<float>(std::atof(tok));
        } else if (a == "--help") {
            usage();
            return 0;
        } else scene = a;
    }
    if (scene.empty()) {
        usage();
        return 1;
    }
    cfg.scene = scene;
    try {  // the viewer catches at top level and logs (main.cpp:94-105)
        Renderer renderer(cfg);
        const auto t0 = std::chrono::steady_clock::now();
        renderer.initialize();
        const double load_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (cull && gsb_set_tile_cull(renderer.context(), cull_level) != GSB_OK) throw std::runtime_error("gsb_set_tile_cull failed");
        struct Pose {
            float v[7];
            float fov;
        };
        std::vector<Pose> poses;
        if (path_file.empty()) {
            poses.push_back(Pose{{cam[0], cam[1], cam[2], cam[3], cam[4], cam[5], cam[6]}, fov});
        } else {
            std::ifstream pf(path_file);
            if (!pf) throw std::runtime_error("cannot open camera path: " + path_file);
            std::string line;
            while (std::getline(pf, line)) {
                if (line.empty() || line[0] == '#') continue;
                Pose p{{0, 0, 0, 1, 0, 0, 0}, fov};
                const int got = std::sscanf(line.c_str(), "%f %f %f %f %f %f %f %f", &p.v[0], &p.v[1], &p.v[2], &p.v[3], &p.v[4], &p.v[5], &p.v[6], &p.fov);
                if (got < 7) throw std::runtime_error("bad camera path line: " + line);
                poses.push_back(p);
            }
            if (poses.empty()) throw std::runtime_error("camera path is empty: " + path_file);
        }
        if (verbose) std::fprintf(stderr, "loaded %llu Gaussians in %.1f ms\n", (unsigned long long)renderer.getScene()->getNumVertices(), load_ms);
        for (size_t pi = 0; pi < poses.size(); pi++) {
            const Pose& po = poses[pi];
            renderer.camera.position = {po.v[0], po.v[1], po.v[2]};
            renderer.camera.rotation = {po.v[3], po.v[4], po.v[5], po.v[6]};
            renderer.camera.fov = po.fov;
            const auto t1 = std::chrono::steady_clock::now();
            renderer.run(frames);
            const double wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count();
            const gsb_stats s = renderer.retrieveTimestamps();
            std::printf("{\"scene\": \"%s\", \"pose\": %zu, \"gaussians\": %llu, \"load_ms\": %.1f, \"read_activate_ms\": %.1f, \"upload_ms\": %.1f, "
                        "\"width\": %u, \"height\": %u, \"frames\": %u, \"fps_wall\": %.2f, "
                        "\"instances\": %llu, \"instances_aabb\": %llu, \"visible\": %llu, \"preprocess_ms\": %.4f, \"prefix_sum_ms\": %.4f, "
                        "\"preprocess_sort_ms\": %.4f, \"sort_ms\": %.4f, \"tile_boundary_ms\": %.4f, \"render_ms\": %.4f, \"frame_ms\": %.4f}\n",
                        scene.c_str(), pi, (unsigned long long)s.num_gaussians, load_ms, renderer.getScene()->lastReadMs,
                        renderer.getScene()->lastUploadMs, cfg.width, cfg.height, frames, 1000.0 * frames / wall_ms,
                        (unsigned long long)s.num_instances, (unsigned long long)s.num_instances_aabb, (unsigned long long)s.num_visible,
                        s.preprocess_ms, s.prefix_sum_ms, s.preprocess_sort_ms, s.sort_ms, s.tile_boundary_ms, s.render_ms, s.frame_ms);
        }
        if (!out_path.empty()) {
            const auto& px = renderer.frame();  // B8G8R8A8
            std::ofstream f(out_path, std::ios::binary);
            f << "P6\n" << cfg.width << " " << cfg.height << "\n255\n";
            std::vector<unsigned char> rgb(static_cast<size_t>(cfg.width) * cfg.height * 3);
            for (size_t p = 0; p < static_cast<size_t>(cfg.width) * cfg.height; p++) {
                rgb[p * 3 + 0] = px[p * 4 + 2];
                rgb[p * 3 + 1] = px[p * 4 + 1];
                rgb[p * 3 + 2] = px[p * 4 + 0];
            }
            f.write(reinterpret_cast<const char*>(rgb.data()), static_cast<std::streamsize>(rgb.size()));
        }
        if (!float_path.empty()) {  // PFM: "PF", width height, -1.0 (little endian), rows bottom to top, float32 RGB
            const float* px = static_cast<const float*>(renderer.render(cfg.width, cfg.height, GSB_FORMAT_RGBA32F));
            std::ofstream f(float_path, std::ios::binary);
            f << "PF\n" << cfg.width << " " << cfg.height << "\n-1.0\n";
            std::vector<float> row(static_cast<size_t>(cfg.width) * 3);
            for (uint32_t y = cfg.height; y-- > 0;) {
                for (uint32_t x = 0; x < cfg.width; x++)
                    for (int c = 0; c < 3; c++) row[x * 3 + c] = px[(static_cast<size_t>(y) * cfg.width + x) * 4 + c];
                f.write(reinterpret_cast<const char*>(row.data()), static_cast<std::streamsize>(row.size() * sizeof(float)));
            }
        }
        if (!alpha_path.empty() || !depth_path.empty()) {  // one renderAux frame: (opacity, expected depth) per pixel
            const float* aux = renderer.renderAux(cfg.width, cfg.height, cfg.format);
            for (int plane = 0; plane < 2; plane++) {
                const std::string& path = plane == 0 ? alpha_path : depth_path;
                if (path.empty()) continue;
                std::ofstream f(path, std::ios::binary);  // greyscale PFM: "Pf", rows bottom to top like --float-out
                f << "Pf\n" << cfg.width << " " << cfg.height << "\n-1.0\n";
                std::vector<float> row(cfg.width);
                for (uint32_t y = cfg.height; y-- > 0;) {
                    for (uint32_t x = 0; x < cfg.width; x++) row[x] = aux[(static_cast<size_t>(y) * cfg.width + x) * 2 + plane];
                    f.write(reinterpret_cast<const char*>(row.data()), static_cast<std::streamsize>(row.size() * sizeof(float)));
                }
            }
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "critical: %s\n", e.what());
        return 2;
    }
    return 0;
}
