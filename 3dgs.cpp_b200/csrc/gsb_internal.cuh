// gsb_internal.cuh -- shared declarations of libgsb200 (not part of the public ABI).
//
// Device data layout (HBM), all fp32:
//   scene   pos_op[N]  float4 (x, y, z, opacity)            16 B  coalesced LDG.128
//           cov_a[N]   float4 (S00, S01, S02, S11)          16 B
//           cov_b[N]   float2 (S12, S22)                     8 B
//           sh[N][48]  RGB-interleaved degree-3 SH         192 B  read by cull survivors only
//   frame   recs[Nv][4] float4  compacted per-survivor record, 64 B, 64-B aligned (GSB_REC_F4 float4):
//               q0 = (uv.x, uv.y, conic.x, conic.y)                  \ first 32-B sector: all k_emit reads
//               q1 = (conic.z, opacity, bits(x0 | y0 << 16), bits(w | h << 16))  / (tile AABB, band-clipped)
//               q2 = (color.r, color.g, color.b, depth)              the blend reads q0, q1.xy, q2.xyz
//               q3 = (radius, bits(original index), -, -)            debug downloads only
//           dkeys[2][Nv] u32 bits(depth), dvals[2][Nv] u32 compact id      -- Gaussian-level sort
//           keys[2][cap] u32 tile id,     vals[2][cap] u32 compact id      -- instance-level sort
//           ranges[T] uint2 (start, ~end) per tile; (0xFFFFFFFF, 0xFFFFFFFF) = empty
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "gs_b200.h"

#define GSB_TILE 16
#define GSB_REC_F4 4  // float4 per survivor record
#define GSB_MAX_SHARDS 8  // GPUs of one NVSwitch domain a frame can be sharded over

namespace gsb {

// control words of one Onesweep sort (device memory, zeroed at frame start)
struct SortCtl {
    uint32_t ticket[8];     // tile tickets, one per radix pass
    uint32_t hist[8][256];  // global digit histograms
};

// ---- per-frame control block (device memory, zeroed by k_frame_init at frame start, except overflow_sticky) ----
struct Control {
    uint32_t project_ticket;   // chunk tickets of k_project
    uint32_t emit_ticket;      // chunk tickets of k_emit
    uint32_t num_visible;      // N_v
    uint32_t num_instances;    // M clamped to the arena capacity
    uint32_t overflow;         // 1 if M_total > capacity in THIS frame
    uint32_t overflow_sticky;  // OR of `overflow` over every frame since it was last reported; survives k_frame_init
    uint32_t epoch;            // look-back epoch of this frame's sorts: += 16 per frame by k_frame_init, never zeroed
    uint32_t pad0;
    unsigned long long instances_total;  // unclamped M
    unsigned long long blend_consumed;
    unsigned long long candidates_total;  // AABB instances before tile culling (the reference's M)
    unsigned long long blend_walked;      // (warp, record) visits of the blend's inner loop (k_blend2 with stats on)
    unsigned long long blend_hits;        // (pixel, Gaussian) pairs of those visits that passed the shader's tests
    unsigned long long blend_staged;      // records gathered into shared memory by the blend
    SortCtl sort_depth;        // Gaussian-level sort (32-bit depth keys)
    SortCtl sort_tile;         // instance-level sort (tile-id keys); also used by gsb_sort_pairs
    // frame sharding (gsb_shard.cu): k_route's chunk tickets and per-destination-band survivor totals
    uint32_t route_ticket;
    uint32_t route_total[GSB_MAX_SHARDS];
};

struct ProjectParams {
    const float4* pos_op;
    const float4* cov_a;
    const float2* cov_b;
    const float* sh;
    int sh_half;          // sh holds 48 fp16 per Gaussian (gsb_set_sh_storage; non-parity)
    uint32_t n;
    uint32_t index_base;  // global index of this context's first Gaussian (frame sharding: the rank's slice; else 0)
    gsb_uniforms ubo;
    uint32_t tile_row_begin, tile_row_end;  // band clip (multi-GPU); [0, tiles_y) = whole frame
    // outputs (compacted by survivor rank)
    float4* recs;
    uint32_t* dkeys;
    uint32_t* dvals;
    uint32_t* status;  // decoupled look-back words, one per 256-Gaussian chunk
    Control* ctl;
    // debug outputs (may be null)
    uint32_t* dbg_tiles;  // N
    uint4* dbg_aabb;      // N
    // frame sharding (route_world > 0): instead of compacting into recs / dkeys, every survivor is delivered -- its 64-B record
    // with the tile AABB clipped to the band, and its depth key -- into the exchange buffers of each rank whose band (band_rows
    // tile rows per rank) its AABB touches; route_dst_* point at THIS source's region inside rank d's buffers (peer memory)
    int route_world;
    uint32_t band_rows;
    uint32_t* route_status;  // [chunks][GSB_MAX_SHARDS] look-back words, one column per destination
    float4* route_dst_recs[GSB_MAX_SHARDS];
    uint32_t* route_dst_dkeys[GSB_MAX_SHARDS];
};

struct EmitParams {
    const uint32_t* sorted_cid;  // survivors in (depth, index) order
    uint32_t nv_hint;            // host estimate of N_v (sizes the grid only)
    uint32_t tiles_x;
    uint32_t* keys;              // tile ids
    uint32_t* vals;              // compact ids
    uint32_t capacity;
    unsigned long long* status;  // decoupled look-back words, one per 256-survivor chunk
    Control* ctl;
    int num_sms;
    const float4* recs;          // survivor records: tile AABB (+ centre, conic, opacity for the optional instance culling)
    int cull;                    // gsb_set_tile_cull level 1: exact per-tile instance culling (k_emit_cull)
    uint32_t coarse_shift;       // gsb_set_tile_cull level 2: bin by 2^shift x 2^shift tile blocks (tiles_x = bins per row); 0 = by tile
    unsigned long long* dbg_offsets;  // debug (may be null): exclusive instance offset of each depth-sorted survivor
};

cudaError_t launch_cov3d(const float* vtx_aos, uint64_t count, uint64_t dst_offset, float4* pos_op,
                         float4* cov_a, float2* cov_b, float* sh, float scale_factor, cudaStream_t s, bool sh_half = false);
cudaError_t launch_project(const ProjectParams& p, bool debug, cudaStream_t s);
cudaError_t launch_emit(const EmitParams& p, cudaStream_t s);

struct SortParams {
    void* keys[2];             // u32 or u64 keys (key_bytes)
    uint32_t* vals[2];
    int key_bytes;             // 4 or 8
    const uint32_t* d_m;       // device pointer to the element count
    uint32_t m_hint;           // host estimate of the count (sizes the grids only; any value is correct)
    uint32_t key_bits;
    unsigned long long* status;  // epoch-tagged look-back words [tiles][256]
    uint32_t status_tiles;     // capacity of status in tiles
    const uint32_t* d_epoch;   // device word added to the epoch (the frame counter of Control; null = 0)
    uint32_t epoch_base;       // pass p tags its look-back words with *d_epoch + epoch_base + p: unique per (frame, sort, pass)
    SortCtl* sc;               // must be zero on entry
    int num_sms;
    cudaEvent_t* events;       // optional: events[0] after the histogram, events[1 + p] after pass p
    uint2* ranges;             // optional (u32 keys): the last pass also produces the tile ranges (start, ~end)
    uint32_t range_key_mask;   // bits of a key that index `ranges` (0 = all; coarse bins keep a tile mask above bit 15)
    bool discard_sorted_keys;  // the last pass writes payloads only (the caller never reads the sorted keys)
};
// Returns the number of passes P via *passes; sorted data ends in keys[P & 1].
cudaError_t launch_sort(const SortParams& p, uint32_t* passes, cudaStream_t s);
uint32_t sort_tile_items();

// One kernel instead of four memsets: zeroes the control block (keeping overflow_sticky) and the look-back words of
// k_project / k_emit, and fills the tile ranges with (0xFFFFFFFF, 0xFFFFFFFF) = empty.
cudaError_t launch_frame_init(Control* ctl, uint32_t* project_status, uint32_t project_chunks, unsigned long long* emit_status,
                              uint32_t emit_chunks, uint2* ranges, uint32_t num_tiles, cudaStream_t s, uint32_t* extra_words = nullptr,
                              uint32_t num_extra_words = 0);
cudaError_t sort_prepare();  // one-time function attributes (dynamic shared memory opt-in) of the Onesweep kernels
cudaError_t launch_ranges_single_tile(const uint32_t* d_m, uint2* ranges, cudaStream_t s);

struct BlendParams {
    const float4* recs;
    const uint32_t* vals;
    const uint32_t* keys;   // coarse bins only: the sorted keys (block id | tile mask << 16)
    const uint2* ranges;
    uint32_t width, height, tiles_x;
    uint32_t coarse_shift, bins_x;  // the sorted lists and `ranges` are per 2^shift x 2^shift tile block (0: per tile), bins_x blocks per row
    uint32_t tile_row_begin, tile_row_end;
    void* out;              // pixel row `out_first_row` of the frame lives at out + 0
    uint32_t out_first_row; // 16 * tile_row_begin for a band buffer, 0 for a whole-frame buffer
    int num_peers;          // > 0: store the band into these whole-frame buffers instead of `out` (one per rank, peer memory)
    void* peer_frames[GSB_MAX_SHARDS];
    size_t row_pitch_bytes;
    int format;             // gsb_format
    int mode;               // gsb_mode
    int variant;            // 2 = k_blend2 (two pixels per thread, packed fp32; default), 1 = k_blend
    int stats;              // 1: count blend_consumed / blend_walked (~4 instructions per record); 2: blend_hits as well
    float one;              // 1.0f, passed as data so that ptxas cannot fold it (gsb_blend.cu, add2_of_product)
    Control* ctl;
    // gsb_render_aux: per-pixel (opacity, expected depth) plane, laid out like `out` (pixel row `out_first_row` at aux + 0,
    // rows aux_pitch bytes apart); null = colour only.  Single-context frames only (num_peers == 0).
    float2* aux;
    size_t aux_pitch;
};
cudaError_t launch_blend(const BlendParams& p, cudaStream_t s);

}  // namespace gsb
