// gsb_ctx.cuh -- the context object behind the C ABI and the frame-orchestration helpers shared by gsb_api.cu (single
// GPU) and gsb_shard.cu (frame sharded over several GPUs).  Not part of the public ABI.
#pragma once
#include <algorithm>
#include <string>

#include "gsb_internal.cuh"

namespace gsb {
struct ShardState;  // gsb_shard.cu
}
using gsb::Control;

// Captured CUDA graph of the "middle" of a frame (depth sort, key emission, tile sort: 9-10 kernels whose arguments do
// not depend on the camera).  Replaces recordRenderCommandBuffer's pre-recorded command buffer (src/Renderer.cpp:532-717).
struct MiddleKey {
    uint32_t tiles_x = 0, num_tiles = 0, nv_q = 0, m_q = 0, cull = 0, tag = 0, cs = 0;
    uint64_t alloc_gen = 0;
    bool operator==(const MiddleKey& o) const {
        return tiles_x == o.tiles_x && num_tiles == o.num_tiles && nv_q == o.nv_q && m_q == o.m_q && cull == o.cull && tag == o.tag &&
               cs == o.cs && alloc_gen == o.alloc_gen;
    }
};
struct MiddleGraph {
    MiddleKey key;
    cudaGraphExec_t exec = nullptr;
    uint64_t last_use = 0;
};


struct gsb_ctx {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    std::string err;

    // scene
    uint64_t n = 0;
    float4* pos_op = nullptr;
    float4* cov_a = nullptr;
    float2* cov_b = nullptr;
    float* sh = nullptr;        // [n][48] fp32, or [n][48] fp16 when sh_half
    bool sh_half = false;       // gsb_set_sh_storage(1): takes effect at the next gsb_scene_upload
    bool scene_sh_half = false; // storage of the uploaded scene

    // frame state
    Control* ctl = nullptr;
    Control* ctl_host = nullptr;  // pinned mirror, filled at the end of each frame
    uint32_t* project_status = nullptr;        // k_project look-back words (one per 256-Gaussian chunk)
    unsigned long long* emit_status = nullptr;  // k_emit look-back words
    float4* recs = nullptr;
    uint32_t* dkeys[2] = {nullptr, nullptr};  // Gaussian-level sort: depth bits
    uint32_t* dvals[2] = {nullptr, nullptr};  //                       compact ids
    uint64_t capacity = 0;
    uint32_t* keys[2] = {nullptr, nullptr};   // instance-level sort: tile ids
    uint32_t* vals[2] = {nullptr, nullptr};   //                      compact ids
    unsigned long long* sort_status = nullptr;
    uint32_t sort_status_tiles = 0;
    uint32_t epoch = 8;
    uint2* ranges = nullptr;
    uint32_t ranges_tiles = 0;
    void* fb = nullptr;
    size_t fb_bytes = 0;
    void* aux_fb = nullptr;  // gsb_render_aux: device staging of a pageable host aux plane
    size_t aux_fb_bytes = 0;

    int mode = GSB_MODE_EXACT;
    bool debug = false;
    bool timers = true;
    int tile_cull = 0;          // gsb_set_tile_cull level: 0 reference-equivalent lists, 1 exact per-tile culling, 2 coarse bins
    uint32_t coarse_shift = 2;  // level 2 bins are 2^shift x 2^shift tiles (GSB_COARSE_SHIFT)
    cudaEvent_t ev[8] = {};
    cudaEvent_t ev_sort[9] = {};  // instance sort: after hist, after each pass
    cudaEvent_t ev_done = nullptr;
    bool frame_pending = false;
    bool have_frame = false;
    bool frame_debug = false;   // the last frame ran with gsb_set_debug on (its debug buffers and sorted keys exist)
    bool frame_timers = false;  // the last frame recorded the stage events (gsb_get_stats may read them)
    bool host_direct = true;    // gsb_render to page-locked host memory: blend straight into it (GSB_HOST_DIRECT=0: always stage)
    int blend_variant = 2;      // GSB_BLEND_VARIANT=1 selects the round-1 one-pixel-per-thread kernel (A/B only)
    bool use_graph = true;      // replay the sorts + key emission from a captured CUDA graph when timers and debug are off
    uint64_t alloc_gen = 0;     // bumped by every (re)allocation a captured graph could point into
    uint64_t graph_clock = 0;
    uint32_t frames_since_epoch_clear = 0;
    MiddleGraph graphs[4] = {};
    uint32_t m_hint = 0;
    uint32_t nv_hint = 0;
    uint32_t regrow_count = 0;

    // description of the last frame (for stats / debug download)
    uint32_t last_w = 0, last_h = 0, last_tiles_x = 0, last_tiles_y = 0, last_passes = 0, last_depth_passes = 0, last_final = 0;

    // debug copies
    uint32_t* dbg_tiles = nullptr;
    uint4* dbg_aabb = nullptr;
    uint32_t* dbg_keys_unsorted = nullptr;
    uint32_t* dbg_vals_unsorted = nullptr;
    uint64_t dbg_m = 0;
    unsigned long long* dbg_offsets = nullptr;  // N: k_emit's exclusive scan value per depth-sorted survivor

    // frame sharding over several GPUs (gsb_shard.cu); null for a plain context
    gsb::ShardState* shard = nullptr;
    uint32_t middle_tag = 0;  // distinguishes captured graphs that read different record buffers (the shard exchange parity)
};


namespace gsb {

int fail(gsb_ctx* c, int code, const char* what, cudaError_t e = cudaSuccess);

#define CK(call)                                                       \
    do {                                                               \
        cudaError_t e_ = (call);                                       \
        if (e_ != cudaSuccess) return gsb::fail(ctx, e_ == cudaErrorMemoryAllocation ? GSB_ERR_OOM : GSB_ERR_CUDA, #call, e_); \
    } while (0)

template <typename T>
cudaError_t dev_alloc(T** p, size_t count) {
    return cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(count, 1) * sizeof(T));
}
template <typename T>
void dev_free(T*& p) {
    if (p) cudaFree(p);
    p = nullptr;
}

struct FramePlan {
    uint32_t W, H, tiles_x, tiles_y, T, rb, re;
    uint32_t cs, bins_x, bins;  // instance-sort bins: 2^cs x 2^cs tile blocks (cs = 0: the tiles themselves, bins == T)
    uint32_t nv_q, m_q, depth_passes, passes;
    int fin;
};

void drop_graphs(gsb_ctx* ctx);
int ensure_sort_status(gsb_ctx* ctx, uint64_t items);
int ensure_arena(gsb_ctx* ctx, uint64_t capacity);
uint32_t bits_for(uint32_t count);
uint32_t quantise_hint(uint64_t hint);
size_t bytes_per_pixel(int fmt);
int wait_frame(gsb_ctx* ctx);
int ensure_ranges(gsb_ctx* ctx, uint32_t W, uint32_t H);
// fills the size-derived fields of a plan, (re)allocates the tile ranges and handles the look-back epoch wrap
int plan_frame(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t rb, uint32_t re, cudaStream_t stream, FramePlan* out);
int enqueue_middle(gsb_ctx* ctx, const FramePlan& fp, cudaStream_t stream, bool events);
int launch_middle_graph(gsb_ctx* ctx, const FramePlan& fp, cudaStream_t stream);
int enqueue_blend(gsb_ctx* ctx, const FramePlan& fp, uint32_t b0, uint32_t b1, void* band_out, size_t pitch, int fmt,
                  cudaStream_t stream, void* const* peer_frames = nullptr, int num_peer_frames = 0, void* band_aux = nullptr,
                  size_t aux_pitch = 0);
int enqueue_tail(gsb_ctx* ctx, const FramePlan& fp, cudaStream_t stream);
int check_render_args(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t& rb, uint32_t& re, const void* out, size_t& pitch, int fmt);

// gsb_shard.cu
void shard_destroy(gsb_ctx* ctx);

}  // namespace gsb
