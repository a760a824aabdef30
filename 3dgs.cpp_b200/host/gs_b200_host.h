/*
 * gs_b200_host.h -- C bridge over the C++ host classes (Renderer / GSScene), in the spirit of the
 * reference's only C-style FFI, the vkgs_* bridging functions of the Apple app
 * (apps/apple/VulkanSplatting/VulkanSplatting-Bridging-Header.h:9-37: vkgs_initialize, vkgs_draw,
 * vkgs_pan_translation, vkgs_movement, vkgs_cleanup).  Handle based instead of a static singleton
 * so tests can hold several renderers.  Errors: 0 = ok, negative = failure, text via
 * gsh_last_error() (the C++ side throws std::runtime_error like the reference; caught here).
 * Host-only helpers (PLY I/O, activations, uniforms, synthetic scenes) need no GPU.
 */
#ifndef GS_B200_HOST_H
#define GS_B200_HOST_H
#include <stddef.h>
#include <stdint.h>

#include "gs_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gsh_renderer gsh_renderer;

const char *gsh_last_error(void);

/* ---- vkgs_* analogues ---- */
/* vkgs_initialize: construct Renderer(config) + initialize(). device < 0 = default (0). */
gsh_renderer *gsh_initialize(const char *scene_path, int device, uint32_t width, uint32_t height,
                             int format /*gsb_format*/, int mode /*gsb_mode*/);
int gsh_draw(gsh_renderer *r);                                     /* vkgs_draw */
int gsh_pan_translation(gsh_renderer *r, float x, float y);        /* vkgs_pan_translation -> cursor delta */
int gsh_movement(gsh_renderer *r, float x, float y, float z);      /* vkgs_movement -> Camera::translate */
void gsh_cleanup(gsh_renderer *r);                                 /* vkgs_cleanup */

/* camera + render(width, height) -> RGBA buffer (north_star API) */
int gsh_set_camera(gsh_renderer *r, const float pos[3], const float quat_wxyz[4], float fov_deg,
                   float near_plane, float far_plane);
int gsh_get_camera(gsh_renderer *r, float pos[3], float quat_wxyz[4], float *fov_deg);
int gsh_key_input(gsh_renderer *r, const int keys[6]); /* W A S D space shift for one handleInput() */
int gsh_render(gsh_renderer *r, uint32_t width, uint32_t height, int format, void *out, size_t out_bytes);
/* Renderer::renderAux: gsh_render + the width*height float2 (opacity, expected depth) planes of gsb_render_aux into aux
 * (aux_bytes >= 8 * width * height; either buffer may be NULL to leave it in the renderer) */
int gsh_render_aux(gsh_renderer *r, uint32_t width, uint32_t height, int format, void *out, size_t out_bytes, float *aux,
                   size_t aux_bytes);
const void *gsh_frame(gsh_renderer *r, size_t *bytes); /* pixels of the last draw()/render() */
int gsh_stats(gsh_renderer *r, gsb_stats *out);
uint64_t gsh_num_vertices(gsh_renderer *r);
gsb_ctx *gsh_context(gsh_renderer *r);

/* ---- host-only helpers (no GPU) ---- */
/* Renderer::updateUniforms (src/Renderer.cpp:719-754) */
void gsh_uniforms_from_camera(const float pos[3], const float quat_wxyz[4], float fov_deg, float near_plane,
                              float far_plane, uint32_t width, uint32_t height, gsb_uniforms *out);
/* Camera::translate (src/Renderer.h:47-49) */
void gsh_camera_translate(float pos[3], const float quat_wxyz[4], const float t[3]);
/* GSScene::load record activation (src/GSScene.cpp:36-59): n*62 floats -> n*60 floats */
void gsh_activate_records(const float *records, uint64_t n, float *vertices);
/* GSScene(path).loadToHost(); returns malloc'd n*60 floats (free with gsh_free) or NULL */
float *gsh_load_ply(const char *path, uint64_t *n_out);
void gsh_free(void *p);
/* write n 62-float records as an Inria-format binary PLY */
int gsh_write_ply(const char *path, const float *records, uint64_t n);

/* Deterministic synthetic scene (SURVEY 8d): counter-based splitmix64; record i depends only on (seed, i). */
typedef struct gsh_synth_params {
    float center[3];       /* positions U[center - half_extent, center + half_extent] */
    float half_extent[3];
    float log_scale_min;   /* log-scales U[min, max] per axis */
    float log_scale_max;
    float opacity_min;     /* opacity logits U[min, max] */
    float opacity_max;
    float sh_dc_range;     /* SH DC U[-r, r] */
    float sh_rest_sigma;   /* SH rest N(0, sigma) */
} gsh_synth_params;
void gsh_synth_default_params(gsh_synth_params *p); /* config 1: box 3, ln0.01..ln0.15, logits -2..4, DC 1, rest 0.1 */
void gsh_synth_records(uint64_t seed, uint64_t first, uint64_t n, const gsh_synth_params *p, float *records);

#ifdef __cplusplus
}
#endif
#endif
