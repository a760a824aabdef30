// capi.cpp -- C bridge over Renderer / GSScene (see gs_b200_host.h) + host-only helpers.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "GSScene.h"
#include "Renderer.h"
#include "gs_b200_host.h"

namespace {
thread_local std::string g_err;
template <typename F>
int guard(F&& f) {
    try {
        f();
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}
}  // namespace

struct gsh_renderer {
    std::unique_ptr<Renderer> r;
};

extern "C" {

const char* gsh_last_error(void) { return g_err.c_str(); }

gsh_renderer* gsh_initialize(const char* scene_path, int device, uint32_t width, uint32_t height, int format, int mode) {
    gsh_renderer* h = nullptr;
    const int rc = guard([&] {
        Renderer::Configuration cfg;
        cfg.scene = scene_path ? scene_path : "";
        if (device >= 0) cfg.physicalDeviceId = static_cast<uint8_t>(device);
        cfg.width = width;
        cfg.height = height;
        cfg.format = static_cast<gsb_format>(format);
        cfg.mode = static_cast<gsb_mode>(mode);
        auto holder = std::make_unique<gsh_renderer>();
        holder->r = std::make_unique<Renderer>(cfg);
        holder->r->initialize();
        h = holder.release();
    });
    return rc == 0 ? h : nullptr;
}

int gsh_draw(gsh_renderer* r) {
    return guard([&] { r->r->draw(); });
}
int gsh_pan_translation(gsh_renderer* r, float x, float y) {
    return guard([&] {
        Renderer::Input in;
        in.cursor_dx = x;
        in.cursor_dy = y;
        r->r->handleInput(in);
    });
}
int gsh_movement(gsh_renderer* r, float x, float y, float z) {
    return guard([&] { r->r->camera.translate({x, y, z}); });
}
int gsh_key_input(gsh_renderer* r, const int keys[6]) {
    return guard([&] {
        Renderer::Input in;
        for (int k = 0; k < 6; k++) in.keys[k] = keys[k] != 0;
        r->r->handleInput(in);
    });
}
void gsh_cleanup(gsh_renderer* r) {
    if (!r) return;
    r->r->stop();
    delete r;
}
int gsh_set_camera(gsh_renderer* r, const float pos[3], const float q[4], float fov, float near_plane, float far_plane) {
    return guard([&] {
        auto& c = r->r->camera;
        c.position = {pos[0], pos[1], pos[2]};
        c.rotation = {q[0], q[1], q[2], q[3]};
        c.fov = fov;
        c.nearPlane = near_plane;
        c.farPlane = far_plane;
    });
}
int gsh_get_camera(gsh_renderer* r, float pos[3], float q[4], float* fov) {
    return guard([&] {
        const auto& c = r->r->camera;
        pos[0] = c.position.x;
        pos[1] = c.position.y;
        pos[2] = c.position.z;
        q[0] = c.rotation.w;
        q[1] = c.rotation.x;
        q[2] = c.rotation.y;
        q[3] = c.rotation.z;
        if (fov) *fov = c.fov;
    });
}
int gsh_render(gsh_renderer* r, uint32_t width, uint32_t height, int format, void* out, size_t out_bytes) {
    return guard([&] {
        const void* px = r->r->render(width, height, static_cast<gsb_format>(format));
        const size_t need = r->r->frame().size();
        if (out) {
            if (out_bytes < need) throw std::runtime_error("gsh_render: output buffer too small");
            std::memcpy(out, px, need);
        }
    });
}
int gsh_render_aux(gsh_renderer* r, uint32_t width, uint32_t height, int format, void* out, size_t out_bytes, float* aux,
                   size_t aux_bytes) {
    return guard([&] {
        const float* planes = r->r->renderAux(width, height, static_cast<gsb_format>(format));
        const size_t need = r->r->frame().size(), need_aux = r->r->auxFrame().size();
        if ((out && out_bytes < need) || (aux && aux_bytes < need_aux)) throw std::runtime_error("gsh_render_aux: output buffer too small");
        if (out) std::memcpy(out, r->r->frame().data(), need);
        if (aux) std::memcpy(aux, planes, need_aux);
    });
}
const void* gsh_frame(gsh_renderer* r, size_t* bytes) {
    if (bytes) *bytes = r->r->frame().size();
    return r->r->frame().data();
}
int gsh_stats(gsh_renderer* r, gsb_stats* out) {
    return guard([&] { *out = r->r->retrieveTimestamps(); });
}
uint64_t gsh_num_vertices(gsh_renderer* r) { return r->r->getScene() ? r->r->getScene()->getNumVertices() : 0; }
gsb_ctx* gsh_context(gsh_renderer* r) { return r->r->context(); }

void gsh_uniforms_from_camera(const float pos[3], const float q[4], float fov, float near_plane, float far_plane,
                              uint32_t width, uint32_t height, gsb_uniforms* out) {
    Renderer::Camera c{{pos[0], pos[1], pos[2]}, {q[0], q[1], q[2], q[3]}, fov, near_plane, far_plane};
    const Renderer::UniformBuffer u = Renderer::makeUniforms(c, width, height);
    std::memcpy(out, &u, sizeof *out);
}

void gsh_camera_translate(float pos[3], const float q[4], const float t[3]) {
    Renderer::Camera c{{pos[0], pos[1], pos[2]}, {q[0], q[1], q[2], q[3]}, 45.f, 0.1f, 1000.f};
    c.translate({t[0], t[1], t[2]});
    pos[0] = c.position.x;
    pos[1] = c.position.y;
    pos[2] = c.position.z;
}

void gsh_activate_records(const float* records, uint64_t n, float* vertices) {
    GSScene::activateRecords(records, n, reinterpret_cast<GSScene::Vertex*>(vertices));
}

float* gsh_load_ply(const char* path, uint64_t* n_out) {
    float* out = nullptr;
    const int rc = guard([&] {
        GSScene scene(path);
        scene.loadToHost();
        const uint64_t n = scene.getNumVertices();
        out = static_cast<float*>(std::malloc(std::max<size_t>(1, n * sizeof(GSScene::Vertex))));
        if (!out) throw std::runtime_error("out of memory");
        std::memcpy(out, scene.vertices().data(), n * sizeof(GSScene::Vertex));
        if (n_out) *n_out = n;
    });
    return rc == 0 ? out : nullptr;
}
void gsh_free(void* p) { std::free(p); }

int gsh_write_ply(const char* path, const float* records, uint64_t n) {
    return guard([&] {
        std::ofstream f(path, std::ios::binary);
        if (!f) throw std::runtime_error(std::string("cannot open for writing: ") + path);
        f << "ply\nformat binary_little_endian 1.0\nelement vertex " << n << "\n";
        for (const char* p : {"x", "y", "z", "nx", "ny", "nz"}) f << "property float " << p << "\n";
        for (int k = 0; k < 3; k++) f << "property float f_dc_" << k << "\n";
        for (int k = 0; k < 45; k++) f << "property float f_rest_" << k << "\n";
        f << "property float opacity\n";
        for (int k = 0; k < 3; k++) f << "property float scale_" << k << "\n";
        for (int k = 0; k < 4; k++) f << "property float rot_" << k << "\n";
        f << "end_header\n";
        f.write(reinterpret_cast<const char*>(records), static_cast<std::streamsize>(n * 62 * sizeof(float)));
        if (!f) throw std::runtime_error(std::string("write failed: ") + path);
    });
}

// ---- synthetic scenes ----
void gsh_synth_default_params(gsh_synth_params* p) {
    *p = gsh_synth_params{{0.f, 0.f, 0.f}, {3.f, 3.f, 3.f}, std::log(0.01f), std::log(0.15f), -2.f, 4.f, 1.f, 0.1f};
}

static inline uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

void gsh_synth_records(uint64_t seed, uint64_t first, uint64_t n, const gsh_synth_params* p, float* records) {
    auto work = [&](uint64_t b, uint64_t e) {
        for (uint64_t k = b; k < e; k++) {
            const uint64_t i = first + k;
            const uint64_t base = splitmix64(seed) ^ (i * 128ull);
            auto bits = [&](uint32_t c) { return splitmix64(base + (uint64_t)c * 0x632BE59BD9B4E019ull); };
            auto uni = [&](uint32_t c) { return (double)(bits(c) >> 11) * (1.0 / 9007199254740992.0); };  // [0,1)
            auto nrm = [&](uint32_t c) {  // Box-Muller on counters (2c, 2c+1) of the normal stream
                const double u1 = ((double)(bits(16 + 2 * c) >> 11) + 1.0) * (1.0 / 9007199254740992.0);  // (0,1]
                const double u2 = (double)(bits(17 + 2 * c) >> 11) * (1.0 / 9007199254740992.0);
                return std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586476925 * u2);
            };
            float* r = records + k * 62;
            for (int a = 0; a < 3; a++) r[a] = (float)(p->center[a] + p->half_extent[a] * (2.0 * uni(a) - 1.0));
            r[3] = r[4] = r[5] = 0.0f;                                                      // normals (GSScene.cpp:56-58 asserts 0)
            for (int a = 0; a < 3; a++) r[6 + a] = (float)(p->sh_dc_range * (2.0 * uni(3 + a) - 1.0));  // f_dc
            for (int a = 0; a < 45; a++) r[9 + a] = (float)(p->sh_rest_sigma * nrm(4 + a));  // f_rest
            r[54] = (float)(p->opacity_min + (p->opacity_max - p->opacity_min) * uni(6));
            for (int a = 0; a < 3; a++)
                r[55 + a] = (float)(p->log_scale_min + (p->log_scale_max - p->log_scale_min) * uni(7 + a));
            for (int a = 0; a < 4; a++) r[58 + a] = (float)nrm(a);  // un-normalised quaternion; the loader normalises
        }
    };
    unsigned threads = std::max(1u, std::min(std::thread::hardware_concurrency(), 32u));
    if (n < 65536) threads = 1;
    if (threads == 1) {
        work(0, n);
        return;
    }
    std::vector<std::thread> pool;
    const uint64_t per = (n + threads - 1) / threads;
    for (unsigned t = 0; t < threads; t++) {
        const uint64_t b = std::min<uint64_t>(n, t * per), e = std::min<uint64_t>(n, b + per);
        if (b < e) pool.emplace_back(work, b, e);
    }
    for (auto& th : pool) th.join();
}

}  // extern "C"
