// Renderer -- host-side frame orchestration with the reference's surface (src/Renderer.h:19-85):
// public mutable `camera`, initialize(), draw(), stop(); plus the render(width,height) -> RGBA
// buffer entry BASELINE.json's north_star asks for (the reference can only store into a
// swapchain image, render.comp:98).  All Vulkan objects are gone: the per-frame work is one
// gsb_render() call into libgsb200 (include/gs_b200.h).
#pragma once
#include <atomic>
#include <cstdint>
#include <memory>
#include <optional>
#include <string>
#include <vector>

#include "GSScene.h"
#include "gs_b200.h"
#include "gsmath.h"

class Renderer {
public:
    // VulkanSplatting::RendererConfiguration (include/3dgs/3dgs.h:13-25) minus the window/Vulkan knobs.
    struct Configuration {
        std::string scene;
        std::optional<uint8_t> physicalDeviceId = std::nullopt;  // -d / VKGS_PHYSICAL_DEVICE -> CUDA device
        uint32_t width = 1280;                                   // viewer defaults, apps/viewer/main.cpp:88-89
        uint32_t height = 720;
        float fov = 45.0f;  // 3dgs.h:19-21: present but never read by the reference either
        float near = 0.2f;
        float far = 1000.0f;
        gsb_format format = GSB_FORMAT_BGRA8;  // the reference swapchain format (Swapchain.cpp:24)
        gsb_mode mode = GSB_MODE_EXACT;
    };

    // src/Renderer.h:21-29
    struct alignas(16) UniformBuffer {
        float camera_position[4];
        float proj_mat[16];
        float view_mat[16];
        uint32_t width;
        uint32_t height;
        float tan_fovx;
        float tan_fovy;
    };
    static_assert(sizeof(UniformBuffer) == sizeof(gsb_uniforms), "UBO layout");

    // src/Renderer.h:40-50
    struct Camera {
        gsmath::vec3 position;
        gsmath::quat rotation;
        float fov;
        float nearPlane;
        float farPlane;
        void translate(gsmath::vec3 translation) { position = position + gsmath::rotate(rotation, translation); }
    };

    // Headless stand-in for Window::getCursorTranslation/getKeys (Renderer::handleInput, Renderer.cpp:33-83)
    struct Input {
        double cursor_dx = 0, cursor_dy = 0;
        bool keys[6] = {false, false, false, false, false, false};  // W A S D space shift
    };

    explicit Renderer(Configuration configuration);
    ~Renderer();
    Renderer(const Renderer&) = delete;
    Renderer& operator=(const Renderer&) = delete;

    void initialize();                // create the CUDA context, load + upload the scene
    void handleInput(const Input&);   // same camera updates as Renderer.cpp:43-82
    void draw();                      // one frame at the configured size/format into frame()
    void run(uint32_t frames);        // draw() loop (the viewer's run() without a window)
    void stop();

    // Render at an explicit size; returns tightly packed RGBA32F / RGBA8 / BGRA8 pixels owned by the renderer.
    const void* render(uint32_t width, uint32_t height, gsb_format format);
    const void* render(uint32_t width, uint32_t height) { return render(width, height, GSB_FORMAT_RGBA32F); }
    // render() plus the frame's per-pixel (opacity, expected depth) planes (gsb_render_aux): the pixels go to frame() as with
    // render(); returns width * height float2, page-locked and owned by the renderer (auxFrame()).
    const float* renderAux(uint32_t width, uint32_t height, gsb_format format);
    // The last frame.  The buffer is page-locked (gsb_host_alloc): gsb_render's blend stores the pixels straight into it over
    // PCIe while it runs -- the analogue of the reference's host-visible swapchain image (render.comp:98) -- instead of a
    // device frame + a pageable cudaMemcpy (measured 16 ms per 3200x1400 BGRA8 frame through a std::vector).
    struct HostFrame {
        unsigned char* ptr = nullptr;
        size_t bytes = 0, capacity = 0;
        const unsigned char* data() const { return ptr; }
        unsigned char* data() { return ptr; }
        size_t size() const { return bytes; }
        const unsigned char& operator[](size_t i) const { return ptr[i]; }
        void resize(size_t n);
        ~HostFrame();
        HostFrame() = default;
        HostFrame(const HostFrame&) = delete;
        HostFrame& operator=(const HostFrame&) = delete;
    };
    const HostFrame& frame() const { return hostFrame; }
    const HostFrame& auxFrame() const { return hostAux; }  // planes of the last renderAux()

    // Renderer::updateUniforms (Renderer.cpp:719-754), exposed so tests can pin it.
    static UniformBuffer makeUniforms(const Camera& camera, uint32_t width, uint32_t height);

    gsb_stats retrieveTimestamps();  // QueryManager analogue (Renderer.cpp:85-100)
    gsb_ctx* context() const { return ctx; }
    const GSScene* getScene() const { return scene.get(); }

    Camera camera{
        .position = {0.0f, 0.0f, 0.0f},
        .rotation = {1.0f, 0.0f, 0.0f, 0.0f},
        .fov = 45.0f,
        .nearPlane = 0.1f,
        .farPlane = 1000.0f,
    };

private:
    Configuration configuration;
    gsb_ctx* ctx = nullptr;
    std::shared_ptr<GSScene> scene;
    HostFrame hostFrame;
    HostFrame hostAux;
    std::atomic<bool> running{true};
    void check(int rc, const char* what);
};
