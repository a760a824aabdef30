/* aux_oracle.c -- CPU reference for gsb_render_aux's per-pixel planes (test infrastructure, built by tests/aux_oracle.py).
 *
 * gso_blend (oracle/gs_oracle.c, render.comp:30-99) restated with the two extra accumulators.  Walking a tile's list in
 * order, a Gaussian is *accumulated* when it reaches render.comp:87; T_i is T just before it:
 *   aux[.., 0] = 1.0f - T_end   (T after the last accumulated Gaussian; the Gaussian that triggers the break is not one)
 *   aux[.., 1] = D, D = D + (depth_i * alpha_i) * T_i in list order (depth_i = VertexAttribute.depth), not normalised.
 * rgba receives exactly what gso_blend writes (tests/test_aux_oracle.py pins that bit for bit), so the colour loop below
 * must stay gso_blend's operation for operation.  Built with the oracle's flags (-ffp-contract=off, no fast math). */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#define TILE 16

typedef struct attr_t { /* gso_attr == VertexAttribute, 64 B */
    float conic_opacity[4];
    float color_radii[4];
    uint32_t aabb[4];
    float uv[2];
    float depth;
    uint32_t magic;
} attr_t;

float gso_exp_shared(float x); /* liboracle.so: the shared-definition exp the CUDA kernel reproduces (exp mode 1) */

void aux_blend(const attr_t *attr, const uint32_t *vals, const uint32_t *ranges, uint32_t width, uint32_t height,
               uint32_t tile_row_begin, uint32_t tile_row_end, int exp_mode, float *rgba, float *aux) {
    const uint32_t tiles_x = (width + TILE - 1) / TILE, tiles_y = (height + TILE - 1) / TILE;
    if (tile_row_end > tiles_y) tile_row_end = tiles_y;
    const int64_t t0 = (int64_t)tile_row_begin * tiles_x, t1 = (int64_t)tile_row_end * tiles_x;
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 4)
#endif
    for (int64_t tt = t0; tt < t1; tt++) {
        const uint32_t tile_x = (uint32_t)(tt % tiles_x), tile_y = (uint32_t)(tt / tiles_x);
        const uint32_t start = ranges[tt * 2], end = ranges[tt * 2 + 1];
        for (uint32_t ly = 0; ly < TILE; ly++)
            for (uint32_t lx = 0; lx < TILE; lx++) {
                const uint32_t px = tile_x * TILE + lx, py = tile_y * TILE + ly;
                if (px >= width || py >= height) continue;
                float T = 1.0f, c0 = 0.0f, c1 = 0.0f, c2 = 0.0f, d = 0.0f;
                const float fx = (float)px, fy = (float)py;
                for (uint32_t i = start; i < end; i++) {
                    const attr_t *a = &attr[vals[i]];
                    float dx = a->uv[0] - fx, dy = a->uv[1] - fy;
                    const float *co = a->conic_opacity;
                    float power = -0.5f * ((co[0] * dx) * dx + (co[2] * dy) * dy) - (co[1] * dx) * dy;
                    if (power > 0.0f) continue;
                    const float e = exp_mode == 1 ? gso_exp_shared(power) : expf(power);
                    float alpha = fminf(0.99f, co[3] * e);
                    if (alpha < 1.0f / 255.0f) continue;
                    float test_T = T * (1.0f - alpha);
                    if (test_T < 0.0001f) break;
                    c0 = c0 + (a->color_radii[0] * alpha) * T;
                    c1 = c1 + (a->color_radii[1] * alpha) * T;
                    c2 = c2 + (a->color_radii[2] * alpha) * T;
                    d = d + (a->depth * alpha) * T; /* :87's shape */
                    T = test_T;                     /* the break leaves T as it was: T_end */
                }
                const size_t p = (size_t)py * width + px;
                rgba[p * 4 + 0] = c0;
                rgba[p * 4 + 1] = c1;
                rgba[p * 4 + 2] = c2;
                rgba[p * 4 + 3] = 1.0f;
                aux[p * 2 + 0] = 1.0f - T;
                aux[p * 2 + 1] = d;
            }
    }
}
