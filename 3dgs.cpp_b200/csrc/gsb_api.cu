// gsb_api.cu -- the C ABI of libgsb200.so (include/gs_b200.h): context, scene upload, frame
// orchestration.  This is the dispatch glue that replaces Renderer::draw / record*CommandBuffer /
// create*Pipeline (src/Renderer.cpp:166-364,366-426,468-717): stream ordering instead of
// pipeline barriers, kernel arguments instead of descriptor sets, and no mid-frame host sync.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <thread>
#include <vector>

#include "gsb_ctx.cuh"

using namespace gsb;

namespace {
thread_local std::string g_create_error;
}  // namespace

namespace gsb {

int fail(gsb_ctx* c, int code, const char* what, cudaError_t e) {
    if (c) {
        c->err = what;
        if (e != cudaSuccess) {
            c->err += ": ";
            c->err += cudaGetErrorString(e);
        }
    }
    return code;
}

int free_arena(gsb_ctx* ctx) {
    dev_free(ctx->keys[0]);
    dev_free(ctx->keys[1]);
    dev_free(ctx->vals[0]);
    dev_free(ctx->vals[1]);
    dev_free(ctx->sort_status);
    ctx->capacity = 0;
    ctx->sort_status_tiles = 0;
    return GSB_OK;
}

void drop_graphs(gsb_ctx* ctx) {
    for (auto& g : ctx->graphs) {
        if (g.exec) cudaGraphExecDestroy(g.exec);
        g = MiddleGraph{};
    }
}

int ensure_sort_status(gsb_ctx* ctx, uint64_t items) {
    const uint32_t tiles = (uint32_t)((items + sort_tile_items() - 1) / sort_tile_items());
    if (tiles <= ctx->sort_status_tiles) return GSB_OK;
    dev_free(ctx->sort_status);
    ctx->sort_status_tiles = 0;
    ctx->alloc_gen++;
    CK(dev_alloc(&ctx->sort_status, (size_t)tiles * 256));
    // Epoch tag 0 = "never published".  The frames run on ctx->stream (non-blocking) or on a caller's stream, neither of
    // which is ordered against the legacy default stream a plain cudaMemset uses: clear on our stream and wait.
    CK(cudaMemsetAsync(ctx->sort_status, 0, (size_t)tiles * 256 * sizeof(unsigned long long), ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->sort_status_tiles = tiles;
    return GSB_OK;
}

int ensure_arena(gsb_ctx* ctx, uint64_t capacity) {
    if (capacity <= ctx->capacity) return GSB_OK;
    if (capacity >= (1ull << 30)) return fail(ctx, GSB_ERR_OVERFLOW, "instance arena limited to 2^30 - 1 entries");
    dev_free(ctx->keys[0]);
    dev_free(ctx->keys[1]);
    dev_free(ctx->vals[0]);
    dev_free(ctx->vals[1]);
    ctx->capacity = 0;
    ctx->alloc_gen++;
    // + 16 entries: the blend's TMA segments are 16-B granular and may read up to 3 entries past the end of the last run
    CK(dev_alloc(&ctx->keys[0], capacity + 16));
    CK(dev_alloc(&ctx->keys[1], capacity + 16));
    CK(dev_alloc(&ctx->vals[0], capacity + 16));
    CK(dev_alloc(&ctx->vals[1], capacity + 16));
    int rc = ensure_sort_status(ctx, std::max<uint64_t>(capacity, ctx->n));
    if (rc != GSB_OK) return rc;
    ctx->capacity = capacity;
    return GSB_OK;
}

uint32_t bits_for(uint32_t count) {  // bits needed to represent 0 .. count-1
    uint32_t b = 0;
    while (b < 32 && (1ull << b) < count) b++;
    return b;
}

// Grid sizes come from the previous frame's counts; quantised to powers of two so that consecutive frames launch the
// same grids (any grid size is correct: every count-dependent kernel is a ticket / grid-stride loop) and a captured
// graph stays valid while the camera moves.
uint32_t quantise_hint(uint64_t hint) {
    uint64_t q = 4096;
    while (q < hint && q < (1ull << 31)) q <<= 1;
    return (uint32_t)q;
}

size_t bytes_per_pixel(int fmt) { return fmt == GSB_FORMAT_RGBA32F ? 16 : 4; }

int wait_frame(gsb_ctx* ctx) {
    if (ctx->frame_pending) {
        CK(cudaEventSynchronize(ctx->ev_done));
        ctx->frame_pending = false;
        ctx->m_hint = ctx->ctl_host->num_instances;
        ctx->nv_hint = ctx->ctl_host->num_visible;
    }
    return GSB_OK;
}

static __global__ void k_frame_init(Control* ctl, uint32_t* __restrict__ project_status, uint32_t project_chunks,
                                    unsigned long long* __restrict__ emit_status, uint32_t emit_chunks, uint2* __restrict__ ranges,
                                    uint32_t num_tiles, uint32_t* __restrict__ extra_words, uint32_t num_extra_words) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    uint32_t* w = reinterpret_cast<uint32_t*>(ctl);
    for (uint32_t k = i; k < sizeof(Control) / 4; k += stride) {
        if (k == offsetof(Control, overflow_sticky) / 4) continue;  // reported (and cleared) by the host, not per frame
        if (k == offsetof(Control, epoch) / 4) w[k] += 16u;          // fresh look-back tags for this frame's two sorts
        else w[k] = 0u;
    }
    // the two look-back arrays have different lengths on a sharded context (local slice vs. the band's whole survivor list)
    for (uint32_t k = i; k < project_chunks; k += stride) project_status[k] = 0u;
    for (uint32_t k = i; k < emit_chunks; k += stride) emit_status[k] = 0ull;
    for (uint32_t k = i; k < num_tiles; k += stride) ranges[k] = make_uint2(0xffffffffu, 0xffffffffu);  // tile_boundary's fillBuffer (Renderer.cpp:633)
    for (uint32_t k = i; k < num_extra_words; k += stride) extra_words[k] = 0u;  // frame sharding: k_route's look-back words
}

cudaError_t launch_frame_init(Control* ctl, uint32_t* project_status, uint32_t project_chunks, unsigned long long* emit_status,
                              uint32_t emit_chunks, uint2* ranges, uint32_t num_tiles, cudaStream_t s, uint32_t* extra_words,
                              uint32_t num_extra_words) {
    const uint32_t work = std::max<uint32_t>(std::max(std::max(std::max(project_chunks, emit_chunks), num_tiles), num_extra_words),
                                             (uint32_t)(sizeof(Control) / 4));
    const uint32_t blocks = std::min<uint32_t>((work + 255) / 256, 148u * 4u);
    k_frame_init<<<blocks, 256, 0, s>>>(ctl, project_status, project_chunks, emit_status, emit_chunks, ranges, num_tiles, extra_words,
                                        num_extra_words);
    return cudaGetLastError();
}

// depth sort -> key emission -> tile sort: everything between k_project and k_blend.  No argument depends on the camera,
// so the sequence is captured once per (frame size, grid sizes, allocation generation) and replayed.
int enqueue_middle(gsb_ctx* ctx, const FramePlan& fp, cudaStream_t stream, bool events) {
    // ---- Gaussian-level Onesweep: the 32 depth bits (the reference's passes 0-3), N_v elements ----
    SortParams sa{};
    sa.keys[0] = ctx->dkeys[0];
    sa.keys[1] = ctx->dkeys[1];
    sa.vals[0] = ctx->dvals[0];
    sa.vals[1] = ctx->dvals[1];
    sa.key_bytes = 4;
    sa.d_m = &ctx->ctl->num_visible;
    sa.m_hint = fp.nv_q;
    sa.key_bits = 32;
    sa.status = ctx->sort_status;
    sa.status_tiles = ctx->sort_status_tiles;
    sa.d_epoch = &ctx->ctl->epoch;
    sa.epoch_base = 0;
    sa.sc = &ctx->ctl->sort_depth;
    sa.num_sms = ctx->num_sms;
    sa.events = nullptr;
    sa.ranges = nullptr;
    sa.discard_sorted_keys = true;  // k_emit reads the sorted compact ids only
    uint32_t depth_passes = 0;
    CK(launch_sort(sa, &depth_passes, stream));
    const int fin_a = depth_passes & 1;
    if (events) CK(cudaEventRecord(ctx->ev[2], stream));

    // ---- k_emit: scan of tile counts + (tile id, payload) emission in depth order ----
    EmitParams ep{};
    ep.sorted_cid = ctx->dvals[fin_a];
    ep.nv_hint = fp.nv_q;
    ep.tiles_x = fp.bins_x;
    ep.coarse_shift = fp.cs;
    ep.keys = ctx->keys[0];
    ep.vals = ctx->vals[0];
    ep.capacity = (uint32_t)ctx->capacity;
    ep.status = ctx->emit_status;
    ep.ctl = ctx->ctl;
    ep.num_sms = ctx->num_sms;
    ep.recs = ctx->recs;
    ep.cull = (ctx->tile_cull >= 1 && fp.cs == 0) ? 1 : 0;  // level 2 falls back to level 1 where coarse bins are unavailable
    ep.dbg_offsets = ctx->debug ? ctx->dbg_offsets : nullptr;
    CK(launch_emit(ep, stream));
    if (events) CK(cudaEventRecord(ctx->ev[3], stream));

    if (ctx->debug) {  // keep the emitted (not yet tile-sorted) pairs: the reference's sort buffers after its pass 3
        CK(cudaStreamSynchronize(stream));
        uint32_t m = 0;
        CK(cudaMemcpy(&m, &ctx->ctl->num_instances, sizeof m, cudaMemcpyDeviceToHost));
        dev_free(ctx->dbg_keys_unsorted);
        dev_free(ctx->dbg_vals_unsorted);
        CK(dev_alloc(&ctx->dbg_keys_unsorted, m));
        CK(dev_alloc(&ctx->dbg_vals_unsorted, m));
        CK(cudaMemcpyAsync(ctx->dbg_keys_unsorted, ctx->keys[0], (size_t)m * 4, cudaMemcpyDeviceToDevice, stream));
        CK(cudaMemcpyAsync(ctx->dbg_vals_unsorted, ctx->vals[0], (size_t)m * 4, cudaMemcpyDeviceToDevice, stream));
        ctx->dbg_m = m;
    }

    // ---- instance-level Onesweep: the tile-id bits (the reference's passes 4-7), M elements ----
    SortParams sp{};
    sp.keys[0] = ctx->keys[0];
    sp.keys[1] = ctx->keys[1];
    sp.vals[0] = ctx->vals[0];
    sp.vals[1] = ctx->vals[1];
    sp.key_bytes = 4;
    sp.d_m = &ctx->ctl->num_instances;
    sp.m_hint = fp.m_q;
    sp.key_bits = bits_for(fp.bins);
    sp.status = ctx->sort_status;
    sp.status_tiles = ctx->sort_status_tiles;
    sp.d_epoch = &ctx->ctl->epoch;
    sp.epoch_base = 4;
    sp.sc = &ctx->ctl->sort_tile;
    sp.num_sms = ctx->num_sms;
    sp.events = events ? ctx->ev_sort : nullptr;
    sp.ranges = ctx->ranges;  // the last pass writes the tile ranges (tile_boundary.comp fused)
    // the fully sorted keys are read by gsb_debug_download(GSB_BUF_KEYS) and, with coarse bins, by the blend (tile masks)
    sp.discard_sorted_keys = !ctx->debug && fp.cs == 0;
    sp.range_key_mask = fp.cs ? 0xffffu : 0u;
    uint32_t passes = 0;
    CK(launch_sort(sp, &passes, stream));
    if (events) CK(cudaEventRecord(ctx->ev[4], stream));
    if (passes == 0) CK(launch_ranges_single_tile(sp.d_m, ctx->ranges, stream));  // one tile: nothing to sort
    if (events) CK(cudaEventRecord(ctx->ev[5], stream));
    if (depth_passes != fp.depth_passes || passes != fp.passes) return fail(ctx, GSB_ERR_CUDA, "internal: pass count mismatch");
    return GSB_OK;
}

// The same sequence replayed from a captured graph (4-entry LRU over MiddleKey).
int launch_middle_graph(gsb_ctx* ctx, const FramePlan& fp, cudaStream_t stream) {
    MiddleKey key;
    key.tiles_x = fp.tiles_x;
    key.num_tiles = fp.T;
    key.nv_q = fp.nv_q;
    key.m_q = fp.m_q;
    key.cull = (uint32_t)ctx->tile_cull;
    key.cs = fp.cs;
    key.tag = ctx->middle_tag;
    key.alloc_gen = ctx->alloc_gen;
    MiddleGraph* slot = nullptr;
    for (auto& g : ctx->graphs)
        if (g.exec && g.key == key) slot = &g;
    if (!slot) {
        slot = &ctx->graphs[0];
        for (auto& g : ctx->graphs)
            if (!g.exec || (slot->exec && g.last_use < slot->last_use)) slot = &g;
        if (slot->exec) cudaGraphExecDestroy(slot->exec);
        *slot = MiddleGraph{};
        // capture on the context's own stream (a caller's stream may be in use by its owner); the graph is launched on `stream`
        cudaGraph_t graph = nullptr;
        CK(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue_middle(ctx, fp, ctx->stream, false);
        cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
        if (rc != GSB_OK) {
            if (graph) cudaGraphDestroy(graph);
            return rc;
        }
        if (e != cudaSuccess) return fail(ctx, GSB_ERR_CUDA, "cudaStreamEndCapture", e);
        e = cudaGraphInstantiate(&slot->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) {
            slot->exec = nullptr;
            return fail(ctx, GSB_ERR_CUDA, "cudaGraphInstantiate", e);
        }
        slot->key = key;
    }
    slot->last_use = ++ctx->graph_clock;
    CK(cudaGraphLaunch(slot->exec, stream));
    return GSB_OK;
}

// Tile ranges for a W x H frame.  cudaMalloc / cudaFree may wait for every device that has this one peer-mapped, so a
// group that drives several GPUs from one host thread calls this for every rank BEFORE enqueuing any rank's frame (a rank
// already spinning in k_shard_wait for a peer whose enqueue is stuck behind an allocation would only leave by timeout).
int ensure_ranges(gsb_ctx* ctx, uint32_t W, uint32_t H) {
    const uint32_t T = ((W + GSB_TILE - 1) / GSB_TILE) * ((H + GSB_TILE - 1) / GSB_TILE);
    if (T > ctx->ranges_tiles) {
        dev_free(ctx->ranges);
        ctx->ranges_tiles = 0;
        ctx->alloc_gen++;
        CK(dev_alloc(&ctx->ranges, T));
        ctx->ranges_tiles = T;
    }
    return GSB_OK;
}

int plan_frame(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t rb, uint32_t re, cudaStream_t stream, FramePlan* out) {
    FramePlan fp{};
    fp.W = ubo->width;
    fp.H = ubo->height;
    fp.tiles_x = (fp.W + GSB_TILE - 1) / GSB_TILE;
    fp.tiles_y = (fp.H + GSB_TILE - 1) / GSB_TILE;
    fp.T = fp.tiles_x * fp.tiles_y;
    fp.rb = rb;
    fp.re = re;
    {
        int rc = ensure_ranges(ctx, fp.W, fp.H);
        if (rc != GSB_OK) return rc;
    }
    const uint32_t n = (uint32_t)ctx->n;
    fp.nv_q = std::min<uint32_t>(quantise_hint(ctx->nv_hint ? ctx->nv_hint : n), quantise_hint(n));
    fp.m_q = quantise_hint(ctx->m_hint ? ctx->m_hint : std::min<uint64_t>(ctx->capacity, 4u * 1024 * 1024));
    // gsb_set_tile_cull level 2: the instance sort bins by blocks of 2^cs x 2^cs tiles; every tile of a block walks the block's
    // list and keeps the records whose AABB holds the tile (k_blend2).  Debug downloads expose per-tile lists: level 2 is off then.
    fp.cs = (ctx->tile_cull == 2 && !ctx->debug && ctx->blend_variant == 2) ? ctx->coarse_shift : 0u;
    fp.bins_x = (fp.tiles_x + (1u << fp.cs) - 1) >> fp.cs;
    fp.bins = fp.bins_x * ((fp.tiles_y + (1u << fp.cs) - 1) >> fp.cs);
    if (fp.cs && fp.bins > 65536u) {  // the block id must fit the 16 key bits below the tile mask (8K x 4K frames still do)
        fp.cs = 0;
        fp.bins_x = fp.tiles_x;
        fp.bins = fp.T;
    }
    fp.depth_passes = 4;
    fp.passes = (bits_for(fp.bins) + 7) / 8;
    fp.fin = (int)(fp.passes & 1);
    if (++ctx->frames_since_epoch_clear >= (1u << 27)) {  // epoch wrap (2^32 / 16 frames): clear the look-back tags once
        CK(cudaMemsetAsync(ctx->sort_status, 0, (size_t)ctx->sort_status_tiles * 256 * sizeof(unsigned long long), stream));
        CK(cudaMemsetAsync(&ctx->ctl->epoch, 0, sizeof(uint32_t), stream));
        ctx->frames_since_epoch_clear = 0;
    }
    *out = fp;
    return GSB_OK;
}

// frame start + k_project + middle.  After this the tile ranges and sorted payloads of the frame are in flight on `stream`.
static int enqueue_front(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t rb, uint32_t re, cudaStream_t stream, FramePlan* out) {
    FramePlan fp{};
    int rc = plan_frame(ctx, ubo, rb, re, stream, &fp);
    if (rc != GSB_OK) return rc;
    const uint32_t n = (uint32_t)ctx->n;
    const uint32_t chunks = (n + 255) / 256;
    const bool timers = ctx->timers;
    CK(launch_frame_init(ctx->ctl, ctx->project_status, std::max(chunks, 1u), ctx->emit_status, std::max(chunks, 1u), ctx->ranges, fp.T, stream));
    if (timers) CK(cudaEventRecord(ctx->ev[0], stream));

    // ---- k_project: preprocess.comp + survivor compaction ----
    ProjectParams pp{};
    pp.pos_op = ctx->pos_op;
    pp.cov_a = ctx->cov_a;
    pp.cov_b = ctx->cov_b;
    pp.sh = ctx->sh;
    pp.sh_half = ctx->scene_sh_half ? 1 : 0;
    pp.n = n;
    pp.index_base = 0;
    pp.ubo = *ubo;
    pp.tile_row_begin = rb;
    pp.tile_row_end = re;
    pp.recs = ctx->recs;
    pp.dkeys = ctx->dkeys[0];
    pp.dvals = ctx->dvals[0];
    pp.status = ctx->project_status;
    pp.ctl = ctx->ctl;
    pp.dbg_tiles = ctx->dbg_tiles;
    pp.dbg_aabb = ctx->dbg_aabb;
    CK(launch_project(pp, ctx->debug, stream));
    if (timers) CK(cudaEventRecord(ctx->ev[1], stream));

    if (ctx->use_graph && !timers && !ctx->debug) rc = launch_middle_graph(ctx, fp, stream);
    else rc = enqueue_middle(ctx, fp, stream, timers);
    if (rc != GSB_OK) return rc;
    *out = fp;
    return GSB_OK;
}

// k_blend over tile rows [b0, b1) of the frame; `band_out` is the first pixel row of the frame's band [fp.rb, fp.re).
int enqueue_blend(gsb_ctx* ctx, const FramePlan& fp, uint32_t b0, uint32_t b1, void* band_out, size_t pitch, int fmt,
                  cudaStream_t stream, void* const* peer_frames, int num_peer_frames, void* band_aux, size_t aux_pitch) {
    BlendParams bp{};
    bp.recs = ctx->recs;
    bp.vals = ctx->vals[fp.fin];
    bp.keys = ctx->keys[fp.fin];
    bp.ranges = ctx->ranges;
    bp.width = fp.W;
    bp.height = fp.H;
    bp.tiles_x = fp.tiles_x;
    bp.coarse_shift = fp.cs;
    bp.bins_x = fp.bins_x;
    bp.tile_row_begin = b0;
    bp.tile_row_end = b1;
    bp.out = static_cast<unsigned char*>(band_out) + (size_t)(b0 - fp.rb) * GSB_TILE * pitch;
    bp.out_first_row = b0 * GSB_TILE;
    // frame sharding: the band is stored into the WHOLE-frame buffers of every rank (peer memory over NVLink) instead
    bp.num_peers = num_peer_frames;
    for (int k = 0; k < num_peer_frames && k < GSB_MAX_SHARDS; k++) bp.peer_frames[k] = peer_frames[k];
    if (num_peer_frames > 0) bp.out_first_row = 0;
    bp.row_pitch_bytes = pitch;
    bp.format = fmt;
    bp.mode = ctx->mode;
    bp.variant = ctx->blend_variant;
    bp.stats = ctx->debug ? 2 : (ctx->timers ? 1 : 0);  // 2 also counts blend_pixel_hits (a few % of the kernel)
    bp.one = 1.0f;
    bp.ctl = ctx->ctl;
    if (band_aux) {  // gsb_render_aux: the (opacity, depth) plane, same band layout as `band_out`
        bp.aux = reinterpret_cast<float2*>(static_cast<unsigned char*>(band_aux) + (size_t)(b0 - fp.rb) * GSB_TILE * aux_pitch);
        bp.aux_pitch = aux_pitch;
    }
    CK(launch_blend(bp, stream));
    return GSB_OK;
}

// stats copy + completion event; latches what gsb_get_stats / gsb_debug_download may read about this frame
int enqueue_tail(gsb_ctx* ctx, const FramePlan& fp, cudaStream_t stream) {
    if (ctx->timers) CK(cudaEventRecord(ctx->ev[6], stream));
    CK(cudaMemcpyAsync(ctx->ctl_host, ctx->ctl, offsetof(Control, sort_depth), cudaMemcpyDeviceToHost, stream));
    CK(cudaEventRecord(ctx->ev_done, stream));
    ctx->frame_pending = true;
    ctx->have_frame = true;
    ctx->frame_debug = ctx->debug;
    ctx->frame_timers = ctx->timers;
    ctx->last_w = fp.W;
    ctx->last_h = fp.H;
    ctx->last_tiles_x = fp.tiles_x;
    ctx->last_tiles_y = fp.tiles_y;
    ctx->last_passes = fp.passes;
    ctx->last_depth_passes = fp.depth_passes;
    ctx->last_final = (uint32_t)fp.fin;
    return GSB_OK;
}

// Enqueue one whole frame on `stream`; out_dev (and aux_dev, if not null) is device memory.
static int enqueue_frame(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t rb, uint32_t re, void* out_dev, size_t pitch, int fmt,
                  cudaStream_t stream, void* aux_dev = nullptr, size_t aux_pitch = 0) {
    FramePlan fp{};
    int rc = enqueue_front(ctx, ubo, rb, re, stream, &fp);
    if (rc != GSB_OK) return rc;
    rc = enqueue_blend(ctx, fp, rb, re, out_dev, pitch, fmt, stream, nullptr, 0, aux_dev, aux_pitch);
    if (rc != GSB_OK) return rc;
    return enqueue_tail(ctx, fp, stream);
}

int check_render_args(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t& rb, uint32_t& re, const void* out, size_t& pitch,
                      int fmt) {
    if (!ctx) return GSB_ERR_INVALID;
    if (!ubo || !out) return fail(ctx, GSB_ERR_INVALID, "null argument");
    if (!ctx->pos_op) return fail(ctx, GSB_ERR_NO_SCENE, "no scene uploaded");
    if (fmt < GSB_FORMAT_RGBA32F || fmt > GSB_FORMAT_BGRA8) return fail(ctx, GSB_ERR_INVALID, "bad format");
    const uint32_t W = ubo->width, H = ubo->height;
    if (W == 0 || H == 0 || W > 16u * 65535u || H > 16u * 65535u) return fail(ctx, GSB_ERR_INVALID, "bad image size");
    const uint32_t tiles_y = (H + GSB_TILE - 1) / GSB_TILE;
    if (re > tiles_y) re = tiles_y;
    if (rb >= re) return fail(ctx, GSB_ERR_INVALID, "empty tile-row band");
    const size_t tight = (size_t)W * bytes_per_pixel(fmt);
    if (pitch == 0) pitch = tight;
    if (pitch < tight || (pitch % (fmt == GSB_FORMAT_RGBA32F ? 16 : 4)) != 0) return fail(ctx, GSB_ERR_INVALID, "bad row pitch");
    return GSB_OK;
}

}  // namespace gsb

extern "C" {

int gsb_abi_version(void) { return GSB_ABI_VERSION; }

int gsb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char* gsb_last_error(const gsb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int gsb_create(int device, gsb_ctx** out) {
    if (!out) return GSB_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        g_create_error = "no usable CUDA device (libgsb200 has no CPU path)";
        if (e != cudaSuccess) g_create_error += std::string(": ") + cudaGetErrorString(e);
        return GSB_ERR_NO_DEVICE;
    }
    gsb_ctx* ctx = new (std::nothrow) gsb_ctx();
    if (!ctx) return GSB_ERR_OOM;
    ctx->device = device;
    auto bail = [&](const char* what, cudaError_t err) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
        gsb_destroy(ctx);
        return GSB_ERR_CUDA;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
    // The library carries sm_100a SASS only (arch-specific, no forward-compatible PTX): any other device would pass
    // here and fail at its first launch with "no kernel image".  Probe a kernel image instead of trusting major/minor.
    cudaFuncAttributes fa;
    if (prop.major != 10 || prop.minor != 0 || cudaFuncGetAttributes(&fa, k_frame_init) != cudaSuccess) {
        cudaGetLastError();
        g_create_error = "libgsb200 is built for sm_100a (B200, compute capability 10.0) only; device is sm_" +
                         std::to_string(prop.major) + std::to_string(prop.minor);
        gsb_destroy(ctx);
        return GSB_ERR_NO_DEVICE;
    }
    ctx->num_sms = prop.multiProcessorCount;
    if (const char* v = getenv("GSB_BLEND_VARIANT")) ctx->blend_variant = atoi(v) == 1 ? 1 : 2;
    if (const char* v = getenv("GSB_HOST_DIRECT")) ctx->host_direct = atoi(v) != 0;
    if (const char* v = getenv("GSB_COARSE_SHIFT")) ctx->coarse_shift = (uint32_t)std::min(2, std::max(1, atoi(v)));  // 2x2 or 4x4 tiles: the mask has 16 bits
    if ((e = sort_prepare()) != cudaSuccess) return bail("sort_prepare", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    if ((e = dev_alloc(&ctx->ctl, 1)) != cudaSuccess) return bail("cudaMalloc", e);
    if ((e = cudaMemset(ctx->ctl, 0, sizeof(Control))) != cudaSuccess) return bail("cudaMemset", e);  // epoch and overflow_sticky start at 0
    if ((e = cudaDeviceSynchronize()) != cudaSuccess) return bail("cudaDeviceSynchronize", e);
    if ((e = cudaMallocHost(reinterpret_cast<void**>(&ctx->ctl_host), sizeof(Control))) != cudaSuccess) return bail("cudaMallocHost", e);
    memset(ctx->ctl_host, 0, sizeof(Control));
    for (auto& ev : ctx->ev)
        if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (auto& ev : ctx->ev_sort)
        if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&ctx->ev_done, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    *out = ctx;
    return GSB_OK;
}

void gsb_destroy(gsb_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    cudaDeviceSynchronize();
    drop_graphs(ctx);
    shard_destroy(ctx);
    dev_free(ctx->dbg_offsets);
    dev_free(ctx->pos_op);
    dev_free(ctx->cov_a);
    dev_free(ctx->cov_b);
    dev_free(ctx->sh);
    dev_free(ctx->ctl);
    if (ctx->ctl_host) cudaFreeHost(ctx->ctl_host);
    dev_free(ctx->project_status);
    dev_free(ctx->emit_status);
    dev_free(ctx->recs);
    dev_free(ctx->dkeys[0]);
    dev_free(ctx->dkeys[1]);
    dev_free(ctx->dvals[0]);
    dev_free(ctx->dvals[1]);
    free_arena(ctx);
    dev_free(ctx->ranges);
    if (ctx->fb) cudaFree(ctx->fb);
    if (ctx->aux_fb) cudaFree(ctx->aux_fb);
    dev_free(ctx->dbg_tiles);
    dev_free(ctx->dbg_aabb);
    dev_free(ctx->dbg_keys_unsorted);
    dev_free(ctx->dbg_vals_unsorted);
    for (auto& ev : ctx->ev)
        if (ev) cudaEventDestroy(ev);
    for (auto& ev : ctx->ev_sort)
        if (ev) cudaEventDestroy(ev);
    if (ctx->ev_done) cudaEventDestroy(ctx->ev_done);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int gsb_scene_upload(gsb_ctx* ctx, const float* vertices, uint64_t n, gsb_memory mem) {
    if (!ctx) return GSB_ERR_INVALID;
    if (n && !vertices) return fail(ctx, GSB_ERR_INVALID, "null vertices");
    if (n >= (1ull << 30)) return fail(ctx, GSB_ERR_INVALID, "scene limited to 2^30 - 1 Gaussians");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->frame_pending = false;
    ctx->have_frame = false;
    dev_free(ctx->pos_op);
    dev_free(ctx->cov_a);
    dev_free(ctx->cov_b);
    dev_free(ctx->sh);
    dev_free(ctx->recs);
    dev_free(ctx->dkeys[0]);
    dev_free(ctx->dkeys[1]);
    dev_free(ctx->dvals[0]);
    dev_free(ctx->dvals[1]);
    dev_free(ctx->project_status);
    dev_free(ctx->emit_status);
    dev_free(ctx->dbg_tiles);
    dev_free(ctx->dbg_aabb);
    dev_free(ctx->dbg_offsets);
    ctx->n = 0;
    ctx->alloc_gen++;
    drop_graphs(ctx);
    CK(dev_alloc(&ctx->pos_op, n));
    CK(dev_alloc(&ctx->cov_a, n));
    CK(dev_alloc(&ctx->cov_b, n));
    ctx->scene_sh_half = ctx->sh_half;
    CK(dev_alloc(&ctx->sh, n * (ctx->scene_sh_half ? 24 : 48)));
    CK(dev_alloc(&ctx->recs, n * GSB_REC_F4));
    CK(dev_alloc(&ctx->dkeys[0], n));
    CK(dev_alloc(&ctx->dkeys[1], n));
    CK(dev_alloc(&ctx->dvals[0], n));
    CK(dev_alloc(&ctx->dvals[1], n));
    CK(dev_alloc(&ctx->project_status, (n + 255) / 256));
    CK(dev_alloc(&ctx->emit_status, (n + 255) / 256));
    if (ctx->debug) {
        CK(dev_alloc(&ctx->dbg_tiles, n));
        CK(dev_alloc(&ctx->dbg_aabb, n));
        CK(dev_alloc(&ctx->dbg_offsets, n));
    }
    // Stream the AoS records to the device in chunks (C5: 50 M x 240 B = 12 GB on the host) through a ring of two page-locked
    // host buffers + two device staging buffers: while chunk k is copied (cudaMemcpyAsync from pinned memory: DMA at PCIe
    // speed) and ingested by k_ingest_cov3d, the host threads copy chunk k + 1 out of the caller's pageable memory into the
    // other pinned buffer.  A caller buffer that is already page-locked (gsb_host_alloc / cudaHostRegister) is DMA'd directly.
    // Replaces vertexBuffer->uploadFrom + GSScene::precomputeCov3D (GSScene.cpp:61,157-184).
    if (mem == GSB_MEM_DEVICE) {
        const uint64_t chunk = std::min<uint64_t>(std::max<uint64_t>(n, 1), 1u << 20);
        for (uint64_t off = 0; off < n; off += chunk) {
            const uint64_t cnt = std::min(chunk, n - off);
            // scale_factor = 1.0f: GSScene.cpp:176
            cudaError_t e = launch_cov3d(vertices + off * 60, cnt, off, ctx->pos_op, ctx->cov_a, ctx->cov_b, ctx->sh, 1.0f, ctx->stream, ctx->scene_sh_half);
            if (e != cudaSuccess) return fail(ctx, GSB_ERR_CUDA, "cov3d precompute", e);
        }
        CK(cudaStreamSynchronize(ctx->stream));
    } else if (n) {
        cudaPointerAttributes pa{};
        const bool caller_pinned = cudaPointerGetAttributes(&pa, vertices) == cudaSuccess && pa.type == cudaMemoryTypeHost;
        cudaGetLastError();
        const uint64_t chunk = std::min<uint64_t>(n, 1u << 18);  // 256 K vertices = 63 MB per ring slot
        float* dev_stage[2] = {nullptr, nullptr};
        float* pin_stage[2] = {nullptr, nullptr};
        cudaEvent_t slot_free[2] = {nullptr, nullptr};
        cudaError_t e = cudaSuccess;
        for (int k = 0; k < 2 && e == cudaSuccess; k++) {
            e = dev_alloc(&dev_stage[k], chunk * 60);
            if (e == cudaSuccess && !caller_pinned) e = cudaMallocHost(reinterpret_cast<void**>(&pin_stage[k]), chunk * 60 * sizeof(float));
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&slot_free[k], cudaEventDisableTiming);
        }
        const unsigned hw = std::max(1u, std::min(std::thread::hardware_concurrency(), 8u));
        uint64_t idx = 0;
        for (uint64_t off = 0; off < n && e == cudaSuccess; off += chunk, idx++) {
            const int k = (int)(idx & 1);
            const uint64_t cnt = std::min(chunk, n - off);
            const float* src = vertices + off * 60;
            if (idx >= 2) e = cudaEventSynchronize(slot_free[k]);  // the slot's previous copy + ingest are done
            if (e != cudaSuccess) break;
            if (!caller_pinned) {  // pageable -> pinned by a few host threads (one memcpy thread tops out well below PCIe 5)
                const size_t bytes = cnt * 60 * sizeof(float);
                const unsigned nt = bytes >= (8u << 20) ? hw : 1u;
                std::vector<std::thread> pool;
                const size_t per = (bytes / nt + 63) & ~size_t(63);
                for (unsigned t = 1; t < nt; t++) {
                    const size_t b = std::min(bytes, t * per), en = std::min(bytes, b + per);
                    if (b < en) pool.emplace_back([=] { memcpy(reinterpret_cast<char*>(pin_stage[k]) + b, reinterpret_cast<const char*>(src) + b, en - b); });
                }
                memcpy(pin_stage[k], src, std::min(bytes, per));
                for (auto& th : pool) th.join();
                src = pin_stage[k];
            }
            e = cudaMemcpyAsync(dev_stage[k], src, cnt * 60 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
            if (e == cudaSuccess) e = launch_cov3d(dev_stage[k], cnt, off, ctx->pos_op, ctx->cov_a, ctx->cov_b, ctx->sh, 1.0f, ctx->stream, ctx->scene_sh_half);
            if (e == cudaSuccess) e = cudaEventRecord(slot_free[k], ctx->stream);
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        else cudaStreamSynchronize(ctx->stream);
        for (int k = 0; k < 2; k++) {
            if (dev_stage[k]) cudaFree(dev_stage[k]);
            if (pin_stage[k]) cudaFreeHost(pin_stage[k]);
            if (slot_free[k]) cudaEventDestroy(slot_free[k]);
        }
        if (e != cudaSuccess) return fail(ctx, e == cudaErrorMemoryAllocation ? GSB_ERR_OOM : GSB_ERR_CUDA, "scene upload", e);
    }
    ctx->n = n;
    ctx->m_hint = 0;
    ctx->nv_hint = 0;
    {
        int rc = ensure_sort_status(ctx, std::max<uint64_t>(n, ctx->capacity));
        if (rc != GSB_OK) return rc;
    }
    // the reference starts the sort arena at N entries (sortBufferSizeMultiplier = 1, Renderer.cpp:235-242)
    if (ctx->capacity == 0) {
        int rc = ensure_arena(ctx, std::max<uint64_t>(n, 1024));
        if (rc != GSB_OK) return rc;
    }
    return GSB_OK;
}

uint64_t gsb_scene_size(const gsb_ctx* ctx) { return ctx ? ctx->n : 0; }

int gsb_set_mode(gsb_ctx* ctx, gsb_mode mode) {
    if (!ctx || (mode != GSB_MODE_EXACT && mode != GSB_MODE_FAST)) return GSB_ERR_INVALID;
    ctx->mode = mode;
    return GSB_OK;
}

int gsb_set_sh_storage(gsb_ctx* ctx, int half_precision) {
    if (!ctx) return GSB_ERR_INVALID;
    ctx->sh_half = half_precision != 0;  // the next gsb_scene_upload stores the coefficients that way
    return GSB_OK;
}

int gsb_set_debug(gsb_ctx* ctx, int debug) {
    if (!ctx) return GSB_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    ctx->debug = debug != 0;
    if (ctx->debug && ctx->n && !ctx->dbg_tiles) {
        CK(dev_alloc(&ctx->dbg_tiles, ctx->n));
        CK(dev_alloc(&ctx->dbg_aabb, ctx->n));
        CK(dev_alloc(&ctx->dbg_offsets, ctx->n));
    }
    return GSB_OK;
}

int gsb_set_graph(gsb_ctx* ctx, int enabled) {
    if (!ctx) return GSB_ERR_INVALID;
    ctx->use_graph = enabled != 0;
    return GSB_OK;
}

int gsb_host_alloc(void** out, size_t bytes) {
    if (!out) return GSB_ERR_INVALID;
    *out = nullptr;
    cudaError_t e = cudaMallocHost(out, bytes ? bytes : 1);
    if (e != cudaSuccess) {
        cudaGetLastError();
        g_create_error = std::string("cudaMallocHost: ") + cudaGetErrorString(e);
        return e == cudaErrorMemoryAllocation ? GSB_ERR_OOM : GSB_ERR_CUDA;
    }
    return GSB_OK;
}

void gsb_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

int gsb_set_tile_cull(gsb_ctx* ctx, int level) {
    if (!ctx || level < 0 || level > 2) return GSB_ERR_INVALID;
    ctx->tile_cull = level;
    return GSB_OK;
}

int gsb_set_timers(gsb_ctx* ctx, int enabled) {
    if (!ctx) return GSB_ERR_INVALID;
    ctx->timers = enabled != 0;
    return GSB_OK;
}

int gsb_reserve_instances(gsb_ctx* ctx, uint64_t capacity) {
    if (!ctx) return GSB_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    int rc = wait_frame(ctx);
    if (rc != GSB_OK) return rc;
    return ensure_arena(ctx, capacity);
}

int gsb_render_async(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t rb, uint32_t re, void* out_device, size_t pitch,
                     gsb_format fmt, void* stream) {
    int rc = check_render_args(ctx, ubo, rb, re, out_device, pitch, fmt);
    if (rc != GSB_OK) return rc;
    CK(cudaSetDevice(ctx->device));
    if (ctx->frame_pending && cudaEventQuery(ctx->ev_done) == cudaSuccess) {  // opportunistic hint refresh
        ctx->frame_pending = false;
        ctx->m_hint = ctx->ctl_host->num_instances;
        ctx->nv_hint = ctx->ctl_host->num_visible;
    }
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return enqueue_frame(ctx, ubo, rb, re, out_device, pitch, fmt, s);
}

// Where the blend stores a HOST buffer of `need` bytes: a page-locked buffer (gsb_host_alloc / cudaHostAlloc / cudaHostRegister)
// is written in place through its device alias; pageable memory goes through the device staging buffer (*buf, *bytes), grown
// on demand, and one cudaMemcpy2D after the frame.
static int host_target(gsb_ctx* ctx, void* host, size_t need, void** buf, size_t* bytes, void** dev, bool* staged) {
    cudaPointerAttributes pa{};
    const bool pinned = ctx->host_direct && cudaPointerGetAttributes(&pa, host) == cudaSuccess && pa.type == cudaMemoryTypeHost &&
                        pa.devicePointer != nullptr;
    cudaGetLastError();
    *staged = !pinned;
    if (pinned) {
        *dev = pa.devicePointer;
        return GSB_OK;
    }
    if (need > *bytes) {
        if (*buf) cudaFree(*buf);
        *buf = nullptr;
        *bytes = 0;
        CK(cudaMalloc(buf, need));
        *bytes = need;
    }
    *dev = *buf;
    return GSB_OK;
}

// gsb_render and gsb_render_aux: one synchronous frame, regrown and re-rendered on arena overflow.  aux == null: colour only.
static int render_sync(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t rb, uint32_t re, void* out, size_t pitch, gsb_memory out_mem,
                       gsb_format fmt, void* stream, void* aux, size_t aux_pitch) {
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    const uint32_t H = ubo->height;
    const uint32_t rows = std::min(H, re * GSB_TILE) - rb * GSB_TILE;
    const size_t tight = (size_t)ubo->width * bytes_per_pixel(fmt);
    const size_t aux_tight = (size_t)ubo->width * sizeof(float2);
    int rc;

    // Host output.  If `out` is page-locked (gsb_host_alloc / cudaHostAlloc / cudaHostRegister) the blend stores the frame
    // straight into it over PCIe: k_blend2 writes whole 64-B tile rows, the stores are posted and the kernel is issue-bound,
    // so the 17.9 MB of a 3200x1400 BGRA8 frame leave the GPU while the blend is still running and no copy is left at the
    // end (the reference likewise stores into a host-visible swapchain image, render.comp:98).  Pageable memory goes
    // through a device staging frame and one cudaMemcpy2D.  The aux plane is decided on its own: out and aux may differ.
    void* dev_out = out;
    size_t dev_pitch = pitch;
    bool staged = false;
    void* dev_aux = aux;
    size_t dev_aux_pitch = aux_pitch;
    bool aux_staged = false;
    if (out_mem == GSB_MEM_HOST) {
        rc = host_target(ctx, out, tight * rows, &ctx->fb, &ctx->fb_bytes, &dev_out, &staged);
        if (rc != GSB_OK) return rc;
        if (staged) dev_pitch = tight;
        if (aux) {
            rc = host_target(ctx, aux, aux_tight * rows, &ctx->aux_fb, &ctx->aux_fb_bytes, &dev_aux, &aux_staged);
            if (rc != GSB_OK) return rc;
            if (aux_staged) dev_aux_pitch = aux_tight;
        }
    }
    for (int attempt = 0;; attempt++) {
        rc = enqueue_frame(ctx, ubo, rb, re, dev_out, dev_pitch, fmt, s, dev_aux, dev_aux_pitch);
        if (rc != GSB_OK) return rc;
        rc = wait_frame(ctx);
        if (rc != GSB_OK) return rc;
        if (!ctx->ctl_host->overflow) break;
        // arena overflow: grow like the reference's sortBufferSizeMultiplier retry (Renderer.cpp:541-563)
        if (attempt >= 3) return fail(ctx, GSB_ERR_OVERFLOW, "instance arena overflow persists after regrow");
        const uint64_t want = ctx->ctl_host->instances_total + ctx->ctl_host->instances_total / 4 + 4096;
        rc = ensure_arena(ctx, want);
        if (rc != GSB_OK) return rc;
        CK(cudaMemsetAsync(&ctx->ctl->overflow_sticky, 0, sizeof(uint32_t), s));  // this overflow is being handled right here
        ctx->regrow_count++;
    }
    if (staged) CK(cudaMemcpy2DAsync(out, pitch, dev_out, dev_pitch, tight, rows, cudaMemcpyDeviceToHost, s));
    if (aux_staged) CK(cudaMemcpy2DAsync(aux, aux_pitch, dev_aux, dev_aux_pitch, aux_tight, rows, cudaMemcpyDeviceToHost, s));
    if (staged || aux_staged) CK(cudaStreamSynchronize(s));
    return GSB_OK;
}

int gsb_render(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t rb, uint32_t re, void* out, size_t pitch, gsb_memory out_mem,
               gsb_format fmt, void* stream) {
    int rc = check_render_args(ctx, ubo, rb, re, out, pitch, fmt);
    if (rc != GSB_OK) return rc;
    return render_sync(ctx, ubo, rb, re, out, pitch, out_mem, fmt, stream, nullptr, 0);
}

int gsb_render_aux(gsb_ctx* ctx, const gsb_uniforms* ubo, uint32_t rb, uint32_t re, void* out, size_t pitch, float* aux,
                   size_t aux_pitch, gsb_memory out_mem, gsb_format fmt, void* stream) {
    if (!ctx) return GSB_ERR_INVALID;
    if (!aux) return fail(ctx, GSB_ERR_INVALID, "null aux buffer");
    if (ctx->shard) return fail(ctx, GSB_ERR_INVALID, "gsb_render_aux: aux planes are not available on a sharded context");
    int rc = check_render_args(ctx, ubo, rb, re, out, pitch, fmt);
    if (rc != GSB_OK) return rc;
    const size_t aux_tight = (size_t)ubo->width * sizeof(float2);
    if (aux_pitch == 0) aux_pitch = aux_tight;
    if (aux_pitch < aux_tight || aux_pitch % sizeof(float2) != 0) return fail(ctx, GSB_ERR_INVALID, "bad aux row pitch");
    return render_sync(ctx, ubo, rb, re, out, pitch, out_mem, fmt, stream, aux, aux_pitch);
}

int gsb_get_stats(gsb_ctx* ctx, gsb_stats* out) {
    if (!ctx || !out) return GSB_ERR_INVALID;
    memset(out, 0, sizeof *out);
    if (!ctx->have_frame) return fail(ctx, GSB_ERR_INVALID, "no frame rendered yet");
    CK(cudaSetDevice(ctx->device));
    if (ctx->frame_pending) {
        int rc = wait_frame(ctx);
        if (rc != GSB_OK) return rc;
    } else {
        CK(cudaEventSynchronize(ctx->ev_done));
    }
    const Control* c = ctx->ctl_host;
    out->num_gaussians = ctx->n;
    out->num_visible = c->num_visible;
    out->num_instances = c->instances_total;
    out->num_instances_aabb = c->candidates_total;
    out->blend_consumed = c->blend_consumed;
    out->blend_warp_visits = c->blend_walked;
    out->blend_pixel_hits = c->blend_hits;
    out->blend_staged = c->blend_staged;
    out->instance_capacity = ctx->capacity;
    out->sort_passes = ctx->last_passes;
    out->sort_depth_passes = ctx->last_depth_passes;
    out->regrow_count = ctx->regrow_count;
    if (ctx->frame_timers) {  // latched per frame: toggling gsb_set_timers between frames must not read stale events
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
        out->preprocess_ms = ms;  // k_project
        CK(cudaEventElapsedTime(&ms, ctx->ev[1], ctx->ev[2]));
        out->sort_depth_ms = ms;  // Gaussian-level Onesweep (histogram + 4 passes over N_v)
        CK(cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]));
        out->preprocess_sort_ms = ms;  // k_emit (scan + key emission); prefix_sum_ms stays 0: fused here
        CK(cudaEventElapsedTime(&ms, ctx->ev[3], ctx->ev[4]));
        out->sort_tile_ms = ms;  // instance-level Onesweep
        out->sort_ms = out->sort_depth_ms + out->sort_tile_ms;
        if (ctx->last_passes) {
            CK(cudaEventElapsedTime(&ms, ctx->ev[3], ctx->ev_sort[0]));
            out->sort_hist_ms = ms;
            for (uint32_t p = 0; p < ctx->last_passes && p < 8; p++) {
                CK(cudaEventElapsedTime(&ms, ctx->ev_sort[p], ctx->ev_sort[p + 1]));
                out->sort_pass_ms[p] = ms;
            }
        }
        CK(cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]));
        out->tile_boundary_ms = ms;
        CK(cudaEventElapsedTime(&ms, ctx->ev[5], ctx->ev[6]));
        out->render_ms = ms;
        CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[6]));
        out->frame_ms = ms;
        if (ctx->shard) {
            CK(cudaEventElapsedTime(&ms, ctx->ev[5], ctx->ev[7]));
            out->shard_blend_ms = ms;
            CK(cudaEventElapsedTime(&ms, ctx->ev[7], ctx->ev[6]));
            out->shard_wait_ms = ms;
        }
    }
    if (c->overflow || c->overflow_sticky) {
        // sticky: set by ANY frame since the last report (pipelined gsb_render_async frames overwrite the per-frame flag)
        CK(cudaMemsetAsync(&ctx->ctl->overflow_sticky, 0, sizeof(uint32_t), ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->ctl_host->overflow_sticky = 0;
        return fail(ctx, GSB_ERR_OVERFLOW, c->overflow ? "last frame overflowed the instance arena (gsb_render regrows; gsb_render_async does not)"
                                                       : "an earlier gsb_render_async frame overflowed the instance arena (its image is incomplete)");
    }
    return GSB_OK;
}

size_t gsb_debug_size(gsb_ctx* ctx, gsb_buffer which) {
    if (!ctx) return 0;
    const uint64_t n = ctx->n;
    if (which == GSB_BUF_COV3D) return (size_t)n * 6 * sizeof(float);
    if (!ctx->have_frame || !ctx->debug || !ctx->frame_debug) return 0;
    if (wait_frame(ctx) != GSB_OK) return 0;
    const uint64_t m = ctx->ctl_host->num_instances;
    switch (which) {
        case GSB_BUF_ATTR: return (size_t)n * sizeof(gsb_vertex_attribute);
        case GSB_BUF_TILES_OVERLAP:
        case GSB_BUF_PREFIX_SUM: return (size_t)n * 4;
        case GSB_BUF_KEYS_UNSORTED:
        case GSB_BUF_KEYS_SORTED: return (size_t)m * 8;
        case GSB_BUF_VALS_UNSORTED:
        case GSB_BUF_VALS_SORTED: return (size_t)m * 4;
        case GSB_BUF_TILE_BOUNDARY: return (size_t)ctx->last_tiles_x * ctx->last_tiles_y * 8;
        case GSB_BUF_DEPTH_ORDER: return (size_t)ctx->ctl_host->num_visible * 4;
        case GSB_BUF_EMIT_OFFSETS: return (size_t)ctx->ctl_host->num_visible * 8;
        default: return 0;
    }
}

int gsb_debug_download(gsb_ctx* ctx, gsb_buffer which, void* dst, size_t bytes) {
    if (!ctx || !dst) return GSB_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const size_t need = gsb_debug_size(ctx, which);
    if (need == 0 && which != GSB_BUF_COV3D) return fail(ctx, GSB_ERR_INVALID, "debug buffer unavailable (enable gsb_set_debug before rendering)");
    if (bytes < need) return fail(ctx, GSB_ERR_INVALID, "destination too small");
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaDeviceSynchronize());
    const uint64_t n = ctx->n;
    const uint32_t nv = ctx->have_frame ? ctx->ctl_host->num_visible : 0;
    const uint64_t m = ctx->have_frame ? ctx->ctl_host->num_instances : 0;
    switch (which) {
        case GSB_BUF_COV3D: {
            std::vector<float4> a(n);
            std::vector<float2> b(n);
            if (n) {
                CK(cudaMemcpy(a.data(), ctx->cov_a, n * sizeof(float4), cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(b.data(), ctx->cov_b, n * sizeof(float2), cudaMemcpyDeviceToHost));
            }
            float* o = static_cast<float*>(dst);
            for (uint64_t i = 0; i < n; i++) {
                o[i * 6 + 0] = a[i].x;
                o[i * 6 + 1] = a[i].y;
                o[i * 6 + 2] = a[i].z;
                o[i * 6 + 3] = a[i].w;
                o[i * 6 + 4] = b[i].x;
                o[i * 6 + 5] = b[i].y;
            }
            return GSB_OK;
        }
        case GSB_BUF_ATTR: {
            std::vector<float4> recs((size_t)nv * GSB_REC_F4);
            std::vector<uint4> aabb(n);
            if (nv) CK(cudaMemcpy(recs.data(), ctx->recs, recs.size() * sizeof(float4), cudaMemcpyDeviceToHost));
            if (n) CK(cudaMemcpy(aabb.data(), ctx->dbg_aabb, n * sizeof(uint4), cudaMemcpyDeviceToHost));
            gsb_vertex_attribute* o = static_cast<gsb_vertex_attribute*>(dst);
            memset(o, 0, n * sizeof(gsb_vertex_attribute));
            for (uint32_t c = 0; c < nv; c++) {
                const float4 r0 = recs[(size_t)c * GSB_REC_F4], r1 = recs[(size_t)c * GSB_REC_F4 + 1], r2 = recs[(size_t)c * GSB_REC_F4 + 2],
                             r3 = recs[(size_t)c * GSB_REC_F4 + 3];
                uint32_t i;
                memcpy(&i, &r3.y, 4);
                if (i >= n) return fail(ctx, GSB_ERR_CUDA, "corrupt compact record");
                gsb_vertex_attribute& a = o[i];
                a.conic_opacity[0] = r0.z;
                a.conic_opacity[1] = r0.w;
                a.conic_opacity[2] = r1.x;
                a.conic_opacity[3] = r1.y;
                a.color_radii[0] = r2.x;
                a.color_radii[1] = r2.y;
                a.color_radii[2] = r2.z;
                a.color_radii[3] = r3.x;
                a.aabb[0] = aabb[i].x;
                a.aabb[1] = aabb[i].y;
                a.aabb[2] = aabb[i].z;
                a.aabb[3] = aabb[i].w;
                a.uv[0] = r0.x;
                a.uv[1] = r0.y;
                a.depth = r2.w;
                a.magic = 0x4d415449u;  // common.glsl:14
            }
            return GSB_OK;
        }
        case GSB_BUF_TILES_OVERLAP:
            if (n) CK(cudaMemcpy(dst, ctx->dbg_tiles, n * 4, cudaMemcpyDeviceToHost));
            return GSB_OK;
        case GSB_BUF_PREFIX_SUM: {  // derived on the host: the device scans in depth order inside k_emit
            uint32_t* o = static_cast<uint32_t*>(dst);
            if (n) CK(cudaMemcpy(o, ctx->dbg_tiles, n * 4, cudaMemcpyDeviceToHost));
            uint32_t run = 0;
            for (uint64_t i = 0; i < n; i++) {
                run += o[i];
                o[i] = run;
            }
            return GSB_OK;
        }
        case GSB_BUF_KEYS_UNSORTED:
        case GSB_BUF_KEYS_SORTED:
        case GSB_BUF_VALS_UNSORTED:
        case GSB_BUF_VALS_SORTED: {
            // device pairs are (u32 tile id, u32 compact id); rebuild the reference's (tile << 32 | depth, Gaussian index)
            const bool sorted = which == GSB_BUF_KEYS_SORTED || which == GSB_BUF_VALS_SORTED;
            const bool want_keys = which == GSB_BUF_KEYS_UNSORTED || which == GSB_BUF_KEYS_SORTED;
            std::vector<float4> recs((size_t)nv * GSB_REC_F4);
            if (nv) CK(cudaMemcpy(recs.data(), ctx->recs, recs.size() * sizeof(float4), cudaMemcpyDeviceToHost));
            std::vector<uint32_t> tk(m), cv(m);
            const uint32_t* ksrc = sorted ? ctx->keys[ctx->last_final] : ctx->dbg_keys_unsorted;
            const uint32_t* vsrc = sorted ? ctx->vals[ctx->last_final] : ctx->dbg_vals_unsorted;
            if (m) {
                CK(cudaMemcpy(tk.data(), ksrc, m * 4, cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(cv.data(), vsrc, m * 4, cudaMemcpyDeviceToHost));
            }
            for (uint64_t k = 0; k < m; k++) {
                if (cv[k] >= nv) return fail(ctx, GSB_ERR_CUDA, "corrupt payload");
                const float4 r2 = recs[(size_t)cv[k] * GSB_REC_F4 + 2], r3 = recs[(size_t)cv[k] * GSB_REC_F4 + 3];
                uint32_t depth_bits, orig;
                memcpy(&depth_bits, &r2.w, 4);
                memcpy(&orig, &r3.y, 4);
                if (want_keys) static_cast<uint64_t*>(dst)[k] = ((uint64_t)tk[k] << 32) | depth_bits;
                else static_cast<uint32_t*>(dst)[k] = orig;
            }
            return GSB_OK;
        }
        case GSB_BUF_DEPTH_ORDER: {  // the Gaussian-level sort's output: survivors in (depth bits, index) order, as Gaussian indices
            std::vector<float4> recs((size_t)nv * GSB_REC_F4);
            std::vector<uint32_t> cid(nv);
            if (nv) {
                CK(cudaMemcpy(recs.data(), ctx->recs, recs.size() * sizeof(float4), cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(cid.data(), ctx->dvals[ctx->last_depth_passes & 1], (size_t)nv * 4, cudaMemcpyDeviceToHost));
            }
            for (uint32_t j = 0; j < nv; j++) {
                if (cid[j] >= nv) return fail(ctx, GSB_ERR_CUDA, "corrupt depth order");
                memcpy(static_cast<uint32_t*>(dst) + j, &recs[(size_t)cid[j] * GSB_REC_F4 + 3].y, 4);
            }
            return GSB_OK;
        }
        case GSB_BUF_EMIT_OFFSETS:  // k_emit's device scan: exclusive instance offset of each depth-sorted survivor
            if (nv) CK(cudaMemcpy(dst, ctx->dbg_offsets, (size_t)nv * 8, cudaMemcpyDeviceToHost));
            return GSB_OK;
        case GSB_BUF_TILE_BOUNDARY: {  // device encoding (start, ~end), untouched = all ones -> the reference's (start, end) / (0, 0)
            CK(cudaMemcpy(dst, ctx->ranges, need, cudaMemcpyDeviceToHost));
            uint32_t* o = static_cast<uint32_t*>(dst);
            for (size_t t = 0; t < need / 8; t++) {
                if (o[2 * t] == 0xffffffffu) o[2 * t] = o[2 * t + 1] = 0u;
                else o[2 * t + 1] = ~o[2 * t + 1];
            }
            return GSB_OK;
        }
        default: return fail(ctx, GSB_ERR_INVALID, "unknown buffer id");
    }
}

// shared body of gsb_sort_pairs (u64 keys) and gsb_sort_pairs32 (u32 keys)
static int sort_pairs_impl(gsb_ctx* ctx, void* keys, uint32_t* vals, void* keys_tmp, uint32_t* vals_tmp, uint64_t m,
                           uint32_t key_bits, int key_bytes, void* stream, const char* what) {
    if (!ctx) return GSB_ERR_INVALID;
    if (m == 0) return GSB_OK;
    if (!keys || !vals || !keys_tmp || !vals_tmp || key_bits == 0 || key_bits > 8u * (uint32_t)key_bytes) return fail(ctx, GSB_ERR_INVALID, "bad argument");
    if (m >= (1ull << 30)) return fail(ctx, GSB_ERR_INVALID, "sort limited to 2^30 - 1 pairs");
    CK(cudaSetDevice(ctx->device));
    int rc = wait_frame(ctx);
    if (rc != GSB_OK) return rc;
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    // private look-back storage sized for m (the frame path uses the arena's)
    const uint32_t tiles = (uint32_t)((m + sort_tile_items() - 1) / sort_tile_items());
    unsigned long long* status = nullptr;
    CK(dev_alloc(&status, (size_t)tiles * 256));
    cudaError_t e = cudaMemsetAsync(status, 0, (size_t)tiles * 256 * 8, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(&ctx->ctl->sort_tile, 0, sizeof(SortCtl), s);  // not the whole block: epoch / overflow_sticky persist
    const uint32_t m32 = (uint32_t)m;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&ctx->ctl->num_instances, &m32, 4, cudaMemcpyHostToDevice, s);
    SortParams sp{};
    sp.keys[0] = keys;
    sp.keys[1] = keys_tmp;
    sp.key_bytes = key_bytes;
    sp.vals[0] = vals;
    sp.vals[1] = vals_tmp;
    sp.d_m = &ctx->ctl->num_instances;
    sp.m_hint = m32;
    sp.key_bits = key_bits;
    sp.status = status;
    sp.status_tiles = tiles;
    sp.d_epoch = nullptr;
    sp.epoch_base = 8;
    sp.sc = &ctx->ctl->sort_tile;
    sp.num_sms = ctx->num_sms;
    sp.events = nullptr;
    sp.ranges = nullptr;
    uint32_t passes = 0;
    if (e == cudaSuccess) e = launch_sort(sp, &passes, s);
    if (e == cudaSuccess && (passes & 1)) {  // odd pass count: bring the result back to the "Even" buffers
        e = cudaMemcpyAsync(keys, keys_tmp, m * (size_t)key_bytes, cudaMemcpyDeviceToDevice, s);
        if (e == cudaSuccess) e = cudaMemcpyAsync(vals, vals_tmp, m * 4, cudaMemcpyDeviceToDevice, s);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);  // m32/status lifetime
    cudaFree(status);
    if (e != cudaSuccess) return fail(ctx, GSB_ERR_CUDA, what, e);
    return GSB_OK;
}

int gsb_sort_pairs(gsb_ctx* ctx, uint64_t* keys, uint32_t* vals, uint64_t* keys_tmp, uint32_t* vals_tmp, uint64_t m,
                   uint32_t key_bits, void* stream) {
    return sort_pairs_impl(ctx, keys, vals, keys_tmp, vals_tmp, m, key_bits, 8, stream, "gsb_sort_pairs");
}

int gsb_sort_pairs32(gsb_ctx* ctx, uint32_t* keys, uint32_t* vals, uint32_t* keys_tmp, uint32_t* vals_tmp, uint64_t m,
                     uint32_t key_bits, void* stream) {
    return sort_pairs_impl(ctx, keys, vals, keys_tmp, vals_tmp, m, key_bits, 4, stream, "gsb_sort_pairs32");
}

}  // extern "C"
