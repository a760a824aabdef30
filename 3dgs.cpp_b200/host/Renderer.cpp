// Renderer.cpp -- see Renderer.h.  Error convention of the reference is kept: every failure is a
// std::runtime_error (SURVEY 8b); the C ABI's error codes are converted here.
#include "Renderer.h"

#include <cmath>
#include <stdexcept>

using namespace gsmath;

Renderer::Renderer(Configuration cfg) : configuration(std::move(cfg)) {}

void Renderer::HostFrame::resize(size_t n) {
    if (n > capacity) {
        if (ptr) gsb_host_free(ptr);
        ptr = nullptr;
        capacity = 0;
        void* p = nullptr;
        if (gsb_host_alloc(&p, n) != GSB_OK) throw std::runtime_error("gsb_host_alloc failed (page-locked frame buffer)");
        ptr = static_cast<unsigned char*>(p);
        capacity = n;
    }
    bytes = n;
}

Renderer::HostFrame::~HostFrame() {
    if (ptr) gsb_host_free(ptr);
}

Renderer::~Renderer() {
    if (ctx) gsb_destroy(ctx);
}

void Renderer::check(int rc, const char* what) {
    if (rc != GSB_OK) throw std::runtime_error(std::string(what) + " failed: " + gsb_last_error(ctx));
}

void Renderer::initialize() {
    // Renderer::initialize (Renderer.cpp:19-31): device, scene, pipelines.  Pipelines/buffers live in libgsb200.
    scene = std::make_shared<GSScene>(configuration.scene);  // throws if the file does not exist
    const int device = configuration.physicalDeviceId.has_value() ? static_cast<int>(*configuration.physicalDeviceId) : 0;
    const int rc = gsb_create(device, &ctx);
    if (rc != GSB_OK) throw std::runtime_error(std::string("gsb_create failed: ") + gsb_last_error(nullptr));
    check(gsb_set_mode(ctx, configuration.mode), "gsb_set_mode");
    scene->load(ctx);
    scene->releaseHostCopy();
}

void Renderer::handleInput(const Input& in) {
    // rotate camera (Renderer.cpp:43-50)
    if (in.cursor_dx != 0.0 || in.cursor_dy != 0.0) {
        camera.rotation = rotate(camera.rotation, static_cast<float>(in.cursor_dx) * 0.005f, vec3{0.0f, -1.0f, 0.0f});
        camera.rotation = rotate(camera.rotation, static_cast<float>(in.cursor_dy) * 0.005f, vec3{-1.0f, 0.0f, 0.0f});
    }
    // move camera (Renderer.cpp:53-81)
    vec3 direction{0.0f, 0.0f, 0.0f};
    if (in.keys[0]) direction = direction + vec3{0.0f, 0.0f, -1.0f};
    if (in.keys[1]) direction = direction + vec3{-1.0f, 0.0f, 0.0f};
    if (in.keys[2]) direction = direction + vec3{0.0f, 0.0f, 1.0f};
    if (in.keys[3]) direction = direction + vec3{1.0f, 0.0f, 0.0f};
    if (in.keys[4]) direction = direction + vec3{0.0f, 1.0f, 0.0f};
    if (in.keys[5]) direction = direction + vec3{0.0f, -1.0f, 0.0f};
    if (direction.x != 0.0f || direction.y != 0.0f || direction.z != 0.0f) {
        const float inv = 1.0f / std::sqrt(direction.x * direction.x + direction.y * direction.y + direction.z * direction.z);
        direction = direction * inv;
        // (mat4_cast(rotation) * vec4(direction, 1)).xyz * 0.3
        const mat4 r = mat4_cast(camera.rotation);
        vec3 moved;
        moved.x = ((r.at(0, 0) * direction.x + r.at(1, 0) * direction.y) + r.at(2, 0) * direction.z) + r.at(3, 0);
        moved.y = ((r.at(0, 1) * direction.x + r.at(1, 1) * direction.y) + r.at(2, 1) * direction.z) + r.at(3, 1);
        moved.z = ((r.at(0, 2) * direction.x + r.at(1, 2) * direction.y) + r.at(2, 2) * direction.z) + r.at(3, 2);
        camera.position = camera.position + moved * 0.3f;
    }
}

Renderer::UniformBuffer Renderer::makeUniforms(const Camera& camera, uint32_t width, uint32_t height) {
    UniformBuffer data{};
    data.width = width;
    data.height = height;
    data.camera_position[0] = camera.position.x;
    data.camera_position[1] = camera.position.y;
    data.camera_position[2] = camera.position.z;
    data.camera_position[3] = 1.0f;

    const mat4 rotation = mat4_cast(camera.rotation);
    const mat4 translation = translate(mat4{}, camera.position);
    mat4 view = inverse(translation * rotation);

    const float tan_fovx = static_cast<float>(std::tan(static_cast<double>(radians(camera.fov)) / 2.0));
    const float tan_fovy = tan_fovx * static_cast<float>(height) / static_cast<float>(width);
    mat4 proj = perspective(std::atan(tan_fovy) * 2.0f, static_cast<float>(width) / static_cast<float>(height),
                            camera.nearPlane, camera.farPlane) *
                view;
    // the shaders work in a y-down, z-forward camera frame: flip rows y,z of view and row y of proj
    for (int c = 0; c < 4; c++) {
        view.at(c, 1) *= -1.0f;
        view.at(c, 2) *= -1.0f;
        proj.at(c, 1) *= -1.0f;
    }
    std::memcpy(data.view_mat, view.m, sizeof view.m);
    std::memcpy(data.proj_mat, proj.m, sizeof proj.m);
    data.tan_fovx = tan_fovx;
    data.tan_fovy = tan_fovy;
    return data;
}

const void* Renderer::render(uint32_t width, uint32_t height, gsb_format format) {
    if (!ctx) throw std::runtime_error("Renderer::render before initialize()");
    const UniformBuffer ubo = makeUniforms(camera, width, height);
    const size_t bpp = format == GSB_FORMAT_RGBA32F ? 16 : 4;
    hostFrame.resize(static_cast<size_t>(width) * height * bpp);
    gsb_uniforms u;
    std::memcpy(&u, &ubo, sizeof u);
    check(gsb_render(ctx, &u, 0, UINT32_MAX, hostFrame.data(), 0, GSB_MEM_HOST, format, nullptr), "gsb_render");
    return hostFrame.data();
}

const float* Renderer::renderAux(uint32_t width, uint32_t height, gsb_format format) {
    if (!ctx) throw std::runtime_error("Renderer::renderAux before initialize()");
    const UniformBuffer ubo = makeUniforms(camera, width, height);
    const size_t bpp = format == GSB_FORMAT_RGBA32F ? 16 : 4;
    hostFrame.resize(static_cast<size_t>(width) * height * bpp);
    hostAux.resize(static_cast<size_t>(width) * height * 2 * sizeof(float));
    gsb_uniforms u;
    std::memcpy(&u, &ubo, sizeof u);
    check(gsb_render_aux(ctx, &u, 0, UINT32_MAX, hostFrame.data(), 0, reinterpret_cast<float*>(hostAux.data()), 0, GSB_MEM_HOST,
                         format, nullptr),
          "gsb_render_aux");
    return reinterpret_cast<const float*>(hostAux.data());
}

void Renderer::draw() { render(configuration.width, configuration.height, configuration.format); }

void Renderer::run(uint32_t frames) {
    running = true;
    for (uint32_t f = 0; f < frames && running; f++) draw();
}

void Renderer::stop() { running = false; }

gsb_stats Renderer::retrieveTimestamps() {
    gsb_stats s{};
    if (!ctx) throw std::runtime_error("Renderer::retrieveTimestamps before initialize()");
    check(gsb_get_stats(ctx, &s), "gsb_get_stats");
    return s;
}
