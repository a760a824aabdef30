/*
 * gs_b200.h -- C ABI of libgsb200.so: the B200 (sm_100a) CUDA replacement for the per-frame
 * compute path of shg8/3DGS.cpp (project+SH -> bin -> sort -> blend).
 *
 * The reference has no plugin/FFI seam for this path; the seam is compile-time inside
 * Renderer/GSScene (SURVEY.md 8b).  Every entry point below therefore names the reference
 * code it replaces (paths relative to /root/reference).  A maintainer swaps the Vulkan
 * dispatch for these calls as shown in INTEGRATION.md.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; every function returns
 * GSB_OK (0) or a negative gsb_status and never throws; gsb_last_error() gives the text.
 * A context is single-owner: one CUDA device, calls from one thread at a time (the reference
 * is single-threaded with FRAMES_IN_FLIGHT = 1, src/vulkan/VulkanContext.h:6).
 * There is NO CPU fallback: without a CUDA device gsb_create() fails with GSB_ERR_NO_DEVICE.
 */
#ifndef GS_B200_H
#define GS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSB_ABI_VERSION 3

typedef struct gsb_ctx gsb_ctx;

typedef enum gsb_status {
    GSB_OK = 0,
    GSB_ERR_INVALID = -1,   /* bad argument */
    GSB_ERR_NO_DEVICE = -2, /* no usable CUDA device (the product has no CPU path) */
    GSB_ERR_CUDA = -3,      /* CUDA runtime error, see gsb_last_error */
    GSB_ERR_NO_SCENE = -4,  /* render before gsb_scene_upload */
    GSB_ERR_OOM = -5,       /* device allocation failed */
    GSB_ERR_OVERFLOW = -6   /* instance arena could not be grown enough */
} gsb_status;

/* Renderer::UniformBuffer -- src/Renderer.h:21-29 == preprocess.comp:16-24 (std140, 160 bytes,
 * column-major mat4).  Produced on the host by Renderer::updateUniforms (src/Renderer.cpp:719-754). */
typedef struct gsb_uniforms {
    float camera_position[4];
    float proj_mat[16];
    float view_mat[16];
    uint32_t width;
    uint32_t height;
    float tan_fovx;
    float tan_fovy;
} gsb_uniforms;

/* VertexAttribute -- src/shaders/common.glsl:42-49 == Renderer.h:31-38; only used by
 * gsb_debug_download(GSB_BUF_ATTR) so intermediates can be diffed against the reference layout. */
typedef struct gsb_vertex_attribute {
    float conic_opacity[4];
    float color_radii[4];
    uint32_t aabb[4];
    float uv[2];
    float depth;
    uint32_t magic;
} gsb_vertex_attribute;

/* Output image formats.  The reference stores vec4(c,1) into a B8G8R8A8_UNORM swapchain image
 * (render.comp:98, src/vulkan/Swapchain.cpp:24); RGBA32F is the un-quantised value of that store. */
typedef enum gsb_format {
    GSB_FORMAT_RGBA32F = 0, /* float4 per pixel, 16 B */
    GSB_FORMAT_RGBA8 = 1,   /* UNORM8, R,G,B,A byte order */
    GSB_FORMAT_BGRA8 = 2    /* UNORM8, B,G,R,A byte order (the reference swapchain format) */
} gsb_format;

/* Arithmetic mode of the blend stage.
 * EXACT: every fp32 op is a single IEEE operation in render.comp's order and exp() is the fixed
 *        operation sequence documented in DESIGN.md; bit-identical to oracle exp-mode 1.
 * FAST : FMA contraction + ex2.approx; same algorithm, results within ~1e-6 of EXACT except at
 *        the shader's own step functions. */
typedef enum gsb_mode { GSB_MODE_EXACT = 0, GSB_MODE_FAST = 1 } gsb_mode;

typedef enum gsb_memory { GSB_MEM_HOST = 0, GSB_MEM_DEVICE = 1 } gsb_memory;

/* Buffers retrievable with gsb_debug_download, in the REFERENCE's layouts (SURVEY Appendix B). */
typedef enum gsb_buffer {
    GSB_BUF_COV3D = 0,         /* scene->cov3DBuffer: N * 6 float                 (GSScene.cpp:158) */
    GSB_BUF_ATTR = 1,          /* vertexAttributeBuffer: N * gsb_vertex_attribute (Renderer.cpp:169); culled entries zero */
    GSB_BUF_TILES_OVERLAP = 2, /* tileOverlapBuffer: N * u32                      (Renderer.cpp:170) */
    GSB_BUF_PREFIX_SUM = 3,    /* inclusive scan in Gaussian-index order: N * u32 (Renderer.cpp:215); derived on the
                                  host from TILES_OVERLAP -- the device scans in depth order inside k_emit */
    GSB_BUF_KEYS_UNSORTED = 4, /* sortKBuffer after the reference's radix pass 3 (bits 0-31 = depth sorted, tile
                                  bits not yet): M * u64.  Equals preprocess_sort's output stably sorted by depth;
                                  this implementation emits the instances directly in that order (DESIGN.md) */
    GSB_BUF_VALS_UNSORTED = 5, /* the payloads (Gaussian indices) that go with KEYS_UNSORTED: M * u32 */
    GSB_BUF_KEYS_SORTED = 6,   /* sortKBufferEven after the 8 passes: M * u64 */
    GSB_BUF_VALS_SORTED = 7,   /* sortVBufferEven after the 8 passes: M * u32 (Gaussian indices) */
    GSB_BUF_TILE_BOUNDARY = 8, /* tileBoundaryBuffer: T * 2 u32                   (Renderer.cpp:321) */
    /* No reference counterpart: the two device results the two-level sort adds (DESIGN.md section 3), exposed so the
     * device scan and the Gaussian-level sort are pinned directly and not only through the key placement. */
    GSB_BUF_DEPTH_ORDER = 9,   /* N_v * u32: Gaussian indices of the cull survivors in (depth bits, index) order */
    GSB_BUF_EMIT_OFFSETS = 10  /* N_v * u64: k_emit's exclusive scan of the tile counts in that order = the slot of each
                                  survivor's first instance (prefix_sum.comp's job, in depth order) */
} gsb_buffer;

/* The reference's six timestamp pairs (src/Renderer.cpp:484-699) + its "instances" text metric
 * (:540).  Mapping: preprocess_ms = k_project; preprocess_sort_ms = k_emit (tile-count scan + key
 * emission, so prefix_sum_ms is 0); sort_ms = Gaussian-level depth sort + instance-level tile sort. */
typedef struct gsb_stats {
    uint64_t num_gaussians;     /* N */
    uint64_t num_visible;       /* N_v: survivors of the three culls */
    uint64_t num_instances;     /* M: (Gaussian, tile) instances emitted and sorted this frame */
    uint64_t num_instances_aabb; /* AABB instances = the reference's "instances" (Renderer.cpp:540); equals
                                   num_instances unless gsb_set_tile_cull is on */
    uint64_t blend_consumed;    /* sum over tiles of run entries read before the tile terminated */
    uint64_t instance_capacity; /* current arena capacity in instances */
    uint32_t sort_passes;       /* radix passes of the instance-level (tile id) sort = ceil(log2(T) / 8) */
    uint32_t regrow_count;      /* times the arena was regrown and the frame re-rendered so far */
    float preprocess_ms, prefix_sum_ms, preprocess_sort_ms, sort_ms, tile_boundary_ms, render_ms;
    float frame_ms;         /* first kernel to last kernel of the frame */
    float sort_depth_ms;    /* Onesweep over the N_v visible Gaussians, 32-bit depth keys (histogram + passes) */
    float sort_tile_ms;     /* Onesweep over the M instances, tile-id keys (histogram + passes) */
    float sort_hist_ms;     /* the histogram kernel of the instance sort */
    float sort_pass_ms[8];  /* each pass kernel of the instance sort (first sort_passes entries) */
    uint32_t sort_depth_passes; /* passes of the Gaussian-level sort (4) */
    uint32_t pad_;
    uint64_t blend_warp_visits; /* (warp, record) visits of the blend's inner loop = evaluated pixel-pair x Gaussian work / 64
                                   (each visit evaluates 64 pixels); counted only while timers or debug are on */
    uint64_t blend_pixel_hits;  /* (pixel, Gaussian) pairs of those visits that passed render.comp:68-80 (power <= 0 and
                                   alpha >= 1/255): hits / (64 * visits) = SIMT lane utilisation of the blend's walk; counted on
                                   gsb_set_debug frames only (0 otherwise) */
    uint64_t blend_staged;      /* records gathered into shared memory by the blend (with coarse bins: this tile's entries among the
                                   blend_consumed list entries it scanned; otherwise equal to the entries read) */
    float shard_blend_ms;       /* frame sharding only: this rank's blend kernel alone (render_ms also holds the wait below) */
    float shard_wait_ms;        /* frame sharding only: from the end of this rank's blend until every rank's band has landed */
} gsb_stats;

/* ---- lifetime: replaces Renderer::initializeVulkan + create*Pipeline (Renderer.cpp:119-155,166-364) ---- */
int gsb_abi_version(void);
int gsb_device_count(void);
int gsb_create(int device, gsb_ctx **out);
void gsb_destroy(gsb_ctx *ctx);
/* Text of the last error on ctx (ctx == NULL: last gsb_create error on this thread). */
const char *gsb_last_error(const gsb_ctx *ctx);

/* ---- scene: replaces vertexBuffer->uploadFrom + GSScene::precomputeCov3D (GSScene.cpp:61,157-184) ----
 * vertices: n records of GSScene::Vertex (src/GSScene.h:41-46): 60 floats =
 * position(xyz,1) scale_opacity(exp(s),sigmoid(o)) rotation(w,x,y,z normalised) sh[48] (RGB-interleaved),
 * i.e. exactly what GSScene::load (GSScene.cpp:36-59) stages.  mem says where `vertices` lives.
 * Precomputes cov3D on the device (precomp_cov3d.comp:25-48, scale_factor 1.0 as GSScene.cpp:176). */
int gsb_scene_upload(gsb_ctx *ctx, const float *vertices, uint64_t n, gsb_memory mem);
uint64_t gsb_scene_size(const gsb_ctx *ctx);

/* Storage of the 48 SH coefficients, chosen BEFORE gsb_scene_upload (default 0 = fp32, 192 B per Gaussian).  1 = fp16 (96 B):
 * NOT a parity mode -- colours come from coefficients rounded to half precision (relative 2^-11), so pixels differ from the
 * reference / oracle by up to ~1e-3; geometry, culling, instance lists and sort order are unaffected.  It halves the
 * dominant term of k_project's HBM traffic (SURVEY 8f row 2 "optional fp16 SH storage mode (non-parity)"). */
int gsb_set_sh_storage(gsb_ctx *ctx, int half_precision);

/* ---- configuration ---- */
int gsb_set_mode(gsb_ctx *ctx, gsb_mode mode);
/* debug != 0: keep every intermediate so gsb_debug_download works (extra HBM traffic). */
int gsb_set_debug(gsb_ctx *ctx, int debug);
/* How the per-tile lists are produced (default 0).  The IMAGE is bit-identical at every level.
 *   0  reference-equivalent: one (Gaussian, tile) instance per tile of the AABB (preprocess_sort.comp:47-58); M, keys,
 *      payloads and tile ranges equal the reference's.
 *   1  exact instance culling: an instance is dropped at key emission if the Gaussian provably stays below the shader's
 *      own alpha < 1/255 cut on every pixel of the tile; M and the key / payload / tile-range buffers are an ordered
 *      subset of the reference's.  Trades a per-candidate test for fewer instances to sort.
 *   2  coarse bins: the instance sort runs over blocks of 4 x 4 tiles (one entry per (Gaussian, block), the key carrying
 *      the mask of the block's tiles inside the Gaussian's tile AABB); every tile then walks its block's depth-ordered
 *      list and keeps the entries whose mask has its bit -- exactly the tile's own list of level 0, in the same order.
 *      ~3x fewer instances to emit and sort.  num_instances then counts (Gaussian, block) entries; num_instances_aabb
 *      stays the reference's count.  Unavailable (falls back to 1) with gsb_set_debug, whose downloads are per tile,
 *      and for frames of more than 65536 blocks. */
int gsb_set_tile_cull(gsb_ctx *ctx, int level);
/* per-stage cudaEvent timers (the QueryManager analogue, Renderer.cpp:85-100). Default on. */
int gsb_set_timers(gsb_ctx *ctx, int enabled);
/* Replay the camera-independent middle of the frame (both sorts + key emission) from a captured CUDA graph instead of
 * ~10 separate launches -- the analogue of the reference's pre-recorded renderCommandBuffer (Renderer.cpp:532-717).
 * Default on; only used while timers and debug are off (both need per-kernel host calls). */
int gsb_set_graph(gsb_ctx *ctx, int enabled);
/* Page-locked host memory for frames / vertex data handed to gsb_render / gsb_scene_upload: copies to and from it are
 * asynchronous DMA (the reference's host-visible staging buffers, Buffer::staging, src/vulkan/Buffer.cpp). */
int gsb_host_alloc(void **out, size_t bytes);
void gsb_host_free(void *p);
/* Pre-size the (tile,depth) instance arena (the reference's sortBufferSizeMultiplier,
 * Renderer.cpp:541-563, grows N*k on overflow; this does the same between frames). */
int gsb_reserve_instances(gsb_ctx *ctx, uint64_t capacity);

/* ---- the frame: replaces Renderer::draw()'s two submits (Renderer.cpp:388-405), i.e.
 * preprocess.comp -> prefix_sum.comp x(log2N+1) -> preprocess_sort.comp -> 8x(hist.comp, sort.comp)
 * -> tile_boundary.comp -> render.comp, without the mid-frame fence + host read of M (:391,:538).
 *
 * Renders tile rows [tile_row_begin, tile_row_end) of the (ubo->width x ubo->height) frame
 * (pass 0, UINT32_MAX for the whole frame; a sub-range is the multi-GPU band of SURVEY 8e).
 * `out` receives pixel rows [16*tile_row_begin, min(H, 16*tile_row_end)) densely, row-major,
 * `row_pitch_bytes` apart (0 = tight).  out_mem says whether `out` is host or device memory.
 * `stream` is a cudaStream_t (NULL = the context's own stream).  The call returns when the frame
 * (and, for host output, the copy) has completed.  If the instance arena overflows, the arena is
 * regrown and the frame re-rendered transparently (the reference's retry, Renderer.cpp:397-399). */
int gsb_render(gsb_ctx *ctx, const gsb_uniforms *ubo, uint32_t tile_row_begin, uint32_t tile_row_end,
               void *out, size_t row_pitch_bytes, gsb_memory out_mem, gsb_format fmt, void *stream);

/* gsb_render plus two per-pixel planes of the same frame, for compositing and depth testing (no reference counterpart:
 * render.comp:98 stores vec4(c, 1) and drops the transmittance).  `out` receives exactly what gsb_render writes.  `aux`
 * receives one float2 (x = opacity, y = expected depth) per pixel for the same pixel rows, `aux_row_pitch_bytes` apart
 * (0 = tight, 8 * width; otherwise >= 8 * width and a multiple of 8).  out_mem applies to both buffers; each one may be
 * page-locked or pageable on its own.  Walking the tile's list as render.comp:61-89 does, a Gaussian i is *accumulated*
 * when it reaches :87 (passes :68-70 and :78-80 and does not trigger the break at :83-85); T_i is T just before it:
 *   opacity = 1 - T_end (one fp32 subtraction), T_end = T after the last accumulated Gaussian; in [0, 0.9999], 0 if none;
 *   depth   = D, D = D + (depth_i * alpha_i) * T_i in list order (the shape of :87), depth_i = VertexAttribute.depth (the
 *             view-space z of GSB_BUF_ATTR).  D is NOT normalised: the mean depth of the covered part is depth / opacity.
 * The colour is premultiplied, so the frame over a background B is c + (1 - opacity) * B.  EXACT mode: both planes are
 * bit-identical to the oracle with exp mode 1 and the colour to gsb_render's; FAST mode accumulates D = fma(depth, alpha*T, D).
 * Errors: GSB_ERR_INVALID for a null aux, a bad aux pitch, or a context of a sharded frame (gsb_create_sharded,
 * gsb_group_context); everything else as gsb_render. */
int gsb_render_aux(gsb_ctx *ctx, const gsb_uniforms *ubo, uint32_t tile_row_begin, uint32_t tile_row_end,
                   void *out, size_t row_pitch_bytes, float *aux, size_t aux_row_pitch_bytes,
                   gsb_memory out_mem, gsb_format fmt, void *stream);

/* Enqueue-only variant for pipelined callers (bench e2e): never synchronises, never regrows;
 * overflow is reported by the next gsb_get_stats()/gsb_render().  out must be device memory. */
int gsb_render_async(gsb_ctx *ctx, const gsb_uniforms *ubo, uint32_t tile_row_begin,
                     uint32_t tile_row_end, void *out_device, size_t row_pitch_bytes, gsb_format fmt,
                     void *stream);

/* Waits for the last frame and fills stats (the retrieveTimestamps analogue, Renderer.cpp:85-100). */
int gsb_get_stats(gsb_ctx *ctx, gsb_stats *out);

/* Size in bytes of a debug buffer for the last frame (0 if unavailable), and its download. */
size_t gsb_debug_size(gsb_ctx *ctx, gsb_buffer which);
int gsb_debug_download(gsb_ctx *ctx, gsb_buffer which, void *dst, size_t bytes);

/* ---- standalone stage entry points (device pointers), used by tests/bench to pin each kernel ---- */
/* Onesweep LSD radix sort of (u64 key, u32 value) pairs over the low `key_bits` bits; stable.
 * Replaces the 8x(hist.comp + sort.comp) loop (Renderer.cpp:598-629).  Sorted data ends in
 * keys/vals (the "Even" buffers, Renderer.cpp:641); keys_tmp/vals_tmp are the "Odd" buffers. */
int gsb_sort_pairs(gsb_ctx *ctx, uint64_t *keys, uint32_t *vals, uint64_t *keys_tmp, uint32_t *vals_tmp,
                   uint64_t m, uint32_t key_bits, void *stream);
/* The same operator over u32 keys (key_bits <= 32): the instantiation the frame itself runs twice -- depth
 * bits over the visible Gaussians, tile ids over the instances (the reference's passes 0-3 and 4-7 of the same
 * loop, Renderer.cpp:598-629). */
int gsb_sort_pairs32(gsb_ctx *ctx, uint32_t *keys, uint32_t *vals, uint32_t *keys_tmp, uint32_t *vals_tmp,
                     uint64_t m, uint32_t key_bits, void *stream);

/* ---- one frame over several GPUs of an NVSwitch domain (SURVEY 8b `gs_create_sharded`, 8e) ----
 * No reference counterpart (the reference is single-GPU).  The scene is sharded by Gaussian index (rank r holds and
 * projects slice r), the frame by tile rows (rank d sorts and blends band d); survivors travel from their slice's rank
 * to their band's rank(s) and the blended bands to every rank's whole-frame buffer by stores into peer-mapped memory
 * (NVLink), ordered by mailbox words -- no collective call in the frame.  Every rank ends the frame holding the whole
 * framebuffer, bit-identical to a single-GPU gsb_render of the same scene and camera.
 *
 * (a) one process drives all GPUs.  `devices` = ndev CUDA device ids (NULL: 0 .. ndev-1); an id may repeat (several
 *     ranks on one GPU -- how the single-GPU tests cover the protocol).  vertices = all n GSScene::Vertex records. */
typedef struct gsb_group gsb_group;
int gsb_group_create(int ndev, const int *devices, gsb_group **out);
void gsb_group_destroy(gsb_group *g);
int gsb_group_size(const gsb_group *g);
gsb_ctx *gsb_group_context(gsb_group *g, int rank); /* per-rank context: gsb_set_mode / _tile_cull / _timers, gsb_get_stats */
const char *gsb_group_last_error(const gsb_group *g);
int gsb_group_scene_upload(gsb_group *g, const float *vertices, uint64_t n, gsb_memory mem);
/* Renders the frame on all GPUs and waits; grows instance arenas and re-renders on overflow like gsb_render.  `out` (may be
 * NULL) receives the whole frame from rank 0's copy; gsb_shard_frame(gsb_group_context(g, r)) is rank r's device copy. */
int gsb_group_render(gsb_group *g, const gsb_uniforms *ubo, void *out, size_t row_pitch_bytes, gsb_memory out_mem, gsb_format fmt);
int gsb_group_render_async(gsb_group *g, const gsb_uniforms *ubo, gsb_format fmt); /* enqueue only, never synchronises */

/* (b) one process per GPU (torchrun / MPI).  Rank 0 calls gsb_shard_unique_id and the host program distributes the 128
 *     bytes by any means; NCCL (dlopen'ed libnccl.so.2, used only here) bootstraps the group and carries the cudaIpc handles
 *     of the exchange windows.  GSB_SHARD_GATHER=nccl reassembles the framebuffer with one in-place ncclAllGather instead
 *     of the blend's peer stores (the baseline the fused path is measured against). */
typedef struct gsb_shard_id { unsigned char bytes[128]; } gsb_shard_id;
int gsb_shard_unique_id(gsb_shard_id *out);
const char *gsb_shard_last_error(void); /* text of the last gsb_shard_unique_id / gsb_create_sharded / gsb_group_create error */
int gsb_create_sharded(int device, int rank, int world, const gsb_shard_id *id, gsb_ctx **out); /* gsb_destroy frees it */
int gsb_shard_rank(const gsb_ctx *ctx);
int gsb_shard_world(const gsb_ctx *ctx);
/* Slice of rank `rank`: Gaussians [first, first + count) with S = ceil(n_total / world), first = rank * S. */
int gsb_shard_slice(uint64_t n_total, int rank, int world, uint64_t *first, uint64_t *count);
/* Tile rows [begin, end) of the frame this rank blends at image height `height` (equal-height bands). */
int gsb_shard_band(const gsb_ctx *ctx, uint32_t height, uint32_t *row_begin, uint32_t *row_end);
/* slice_vertices = this rank's slice only (gsb_shard_slice), n_total = size of the whole scene. */
int gsb_scene_upload_sharded(gsb_ctx *ctx, const float *slice_vertices, uint64_t n_total, gsb_memory mem);
/* Collective: every rank calls it with the same ubo / fmt.  Waits for the frame; `out` (may be NULL) receives this rank's
 * copy of the WHOLE frame.  The first call at a new frame size (re)allocates and re-exchanges the windows. */
int gsb_render_sharded(gsb_ctx *ctx, const gsb_uniforms *ubo, void *out, size_t row_pitch_bytes, gsb_memory out_mem,
                       gsb_format fmt, void *stream);
int gsb_render_sharded_async(gsb_ctx *ctx, const gsb_uniforms *ubo, gsb_format fmt, void *stream);
/* This rank's device copy of the last whole frame (tight pitch); valid until the second-next render call. */
const void *gsb_shard_frame(const gsb_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* GS_B200_H */
