// gsb_blend.cu -- per-16x16-tile front-to-back alpha blending.
// Replaces render.comp:30-99 (dispatch src/Renderer.cpp:654-677).  The reference makes every
// pixel thread gather idx + uv + conic + colour from global memory for every Gaussian of the
// tile's run (render.comp:62-65,87; README.md:87 lists staging as a TODO).  Here one CTA owns one
// tile and
//   * stages the run in batches of 256 compact 48-B records into shared memory once;
//   * while staging, each thread classifies its Gaussian against the eight 8x4-pixel blocks of
//     the tile (one block per warp): a block whose best-case exponent is below the shader's own
//     alpha < 1/255 cut (with an fp32 error margin) can never contribute, so that warp never
//     touches the record (bit-identical result: those pairs hit `continue` in render.comp:78);
//   * each warp compacts the batch with one ballot per 32 records and walks only its survivors,
//     reading each record as a shared-memory broadcast; the walk is branch-free per lane (the
//     shader's `continue`s and `break` are predicates on the four state updates).
// The per-pixel `break` (render.comp:83-85) becomes a per-lane done flag + warp / block votes.
//
// EXACT mode: -fmad=false, ops in render.comp's order, exp = the fixed IEEE sequence below
// (bit-identical to oracle exp-mode 1).  FAST mode: explicit FMA + ex2.approx.
#include "gsb_cull.cuh"
#include "gsb_internal.cuh"
#include "gsb_tma.cuh"

namespace gsb {

namespace {

constexpr int BLEND_THREADS = 256;
constexpr unsigned FULL = 0xffffffffu;

// Bit-defined exp for x in [-87, 0]; mirrors gso_exp_shared() in oracle/gs_oracle.c op for op: Cody-Waite
// reduction, degree-5 Horner with the constant term 1, 2^n applied through the exponent bits (13 instructions).
__device__ __forceinline__ float exp_shared(float x) {
    x = fmaxf(x, -87.0f);
    const float t = __fmul_rn(x, 1.44269504088896341f);
    const float tm = __fadd_rn(t, 12582912.0f);  // low mantissa bits = rint(t) in two's complement
    const float n = __fsub_rn(tm, 12582912.0f);
    float r = __fmaf_rn(n, -0.693359375f, x);
    r = __fmaf_rn(n, 2.12194440e-4f, r);
    float p = __fmaf_rn(8.290082216262817e-3f, r, 4.1899293661117554e-2f);
    p = __fmaf_rn(p, r, 1.6667647659778595e-1f);
    p = __fmaf_rn(p, r, 4.9999138712882996e-1f);
    p = __fmaf_rn(p, r, 9.999997019767761e-1f);
    p = __fmaf_rn(p, r, 1.0f);
    return __uint_as_float(__float_as_uint(p) + (__float_as_uint(tm) << 23));
}

#if GSB_BLEND_TDONE
// same sequence without the clamp: only evaluated results with power in [cut, 0] are used (identity there)
__device__ __forceinline__ float exp_shared_inrange(float x) {
    const float t = __fmul_rn(x, 1.44269504088896341f);
    const float tm = __fadd_rn(t, 12582912.0f);
    const float n = __fsub_rn(tm, 12582912.0f);
    float r = __fmaf_rn(n, -0.693359375f, x);
    r = __fmaf_rn(n, 2.12194440e-4f, r);
    float p = __fmaf_rn(8.290082216262817e-3f, r, 4.1899293661117554e-2f);
    p = __fmaf_rn(p, r, 1.6667647659778595e-1f);
    p = __fmaf_rn(p, r, 4.9999138712882996e-1f);
    p = __fmaf_rn(p, r, 9.999997019767761e-1f);
    p = __fmaf_rn(p, r, 1.0f);
    return __uint_as_float(__float_as_uint(p) + (__float_as_uint(tm) << 23));
}
#endif

// shared-memory loads by 32-bit shared-window address (one LDS each, immediate offsets, no generic-pointer arithmetic)
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

__device__ __forceinline__ uint32_t unorm8(float v) {
    v = fminf(fmaxf(v, 0.0f), 1.0f);  // NaN -> 0
    return __float2uint_rn(v * 255.0f);
}

// Bit w set <=> warp w's 8x4 pixel block may receive a contribution from this Gaussian (gsb_cull.cuh).
__device__ __forceinline__ uint32_t block_mask(float ux, float uy, float A, float B, float C, float cut, float tile_x0, float tile_y0) {
    if (!(A > 0.0f) || !(C > 0.0f)) return 0xffu;  // not positive definite / NaN: never cull
    const float inv_a = __frcp_rn(A), inv_c = __frcp_rn(C);
    uint32_t mask = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) {
        const float x0 = tile_x0 + (float)((w & 1) * 8), y0 = tile_y0 + (float)((w >> 1) * 4);
        if (rect_may_contribute(ux, uy, A, B, C, inv_a, inv_c, x0, y0, 8.0f, 4.0f, cut)) mask |= 1u << w;
    }
    return mask;
}

// one staged record (48 B): three 16-B slots so the inner loop addresses it with one byte offset
struct __align__(16) StagedRec {
    float4 r0;  // uv.x uv.y -conic.x/2 -conic.y      (exact sign / power-of-two scalings: render.comp:66 becomes
    float4 r1;  // -conic.z/2 power_cut opacity r       ((-A/2 dx) dx + (-C/2 dy) dy) + ((-B) dx) dy, bit for bit)
    float4 r2;  // g b - -
};

#ifndef GSB_BLEND_CHECK
#define GSB_BLEND_CHECK 8  // records walked between two "is the whole warp done" votes (measured: 8 -> 0.673 ms, 16 -> 0.685, 32 -> 0.733)
#endif
#ifndef GSB_BLEND_TDONE
#define GSB_BLEND_TDONE 0  // 1: a finished pixel is T == 0 (no separate flag in the walk); needs GSB_BLEND_PREDICATED
#endif
#ifndef GSB_BLEND_PREDICATED
#define GSB_BLEND_PREDICATED 1
#endif
#ifndef GSB_BLEND_MIN_BLOCKS
#define GSB_BLEND_MIN_BLOCKS 5  // <= 51 registers, 5 CTAs per SM (measured: 0.873 ms; 4 CTAs 0.886, 6 CTAs 0.891, 80 registers 0.972)
#endif
template <int MODE>
__global__ void __launch_bounds__(BLEND_THREADS, GSB_BLEND_MIN_BLOCKS) k_blend(const __grid_constant__ BlendParams P) {
    __shared__ StagedRec s_rec[BLEND_THREADS];
    __shared__ uint32_t s_mask[BLEND_THREADS];
    __shared__ uint16_t s_list[BLEND_THREADS / 32][BLEND_THREADS];  // per warp: byte offsets of the records it must visit
    __shared__ uint32_t s_used;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tx = blockIdx.x % P.tiles_x;
    const uint32_t ty = P.tile_row_begin + blockIdx.x / P.tiles_x;
    uint2 range = P.ranges[ty * P.tiles_x + tx];  // render.comp:43-44; stored as (start, ~end), empty = all ones
    range.y = ~range.y;
    // warp w owns the 8x4 pixel block at (8 * (w & 1), 4 * (w >> 1)) of the tile
    const uint32_t px = tx * GSB_TILE + (warp & 1) * 8 + (lane & 7);
    const uint32_t py = ty * GSB_TILE + (warp >> 1) * 4 + (lane >> 3);
    const bool inside = px < P.width && py < P.height;  // :37-39
    const float fx = (float)px, fy = (float)py;
    const float tile_x0 = (float)(tx * GSB_TILE), tile_y0 = (float)(ty * GSB_TILE);
    if (tid == 0) s_used = 0;
    __syncthreads();

    float T = 1.0f, c0 = 0.0f, c1 = 0.0f, c2 = 0.0f;
#if GSB_BLEND_TDONE
    if (!inside) T = 0.0f;
#define BLEND_DONE (T == 0.0f)
#else
    bool done = !inside;
#define BLEND_DONE done
#endif
    uint32_t used = 0;
    const uint32_t rec_sh = (uint32_t)__cvta_generic_to_shared(&s_rec[0]);  // < 64 KiB: fits the u16 list entries

    for (uint32_t base = range.x; base < range.y; base += BLEND_THREADS) {
        const uint32_t cnt = min((uint32_t)BLEND_THREADS, range.y - base);
        if ((uint32_t)tid < cnt) {
            const uint32_t cid = __ldg(P.vals + base + tid);
            const float4* rec = P.recs + (size_t)cid * GSB_REC_F4;
            const float4 a = __ldg(rec), col = __ldg(rec + 2);
            const float2 b = __ldg(reinterpret_cast<const float2*>(rec + 1));  // conic.z, opacity
            const float cut = power_cut(b.y);
            s_rec[tid].r0 = make_float4(a.x, a.y, -0.5f * a.z, -a.w);
            s_rec[tid].r1 = make_float4(-0.5f * b.x, cut, b.y, col.x);
            s_rec[tid].r2 = make_float4(col.y, col.z, 0.f, 0.f);
            s_mask[tid] = block_mask(a.x, a.y, a.z, a.w, b.x, cut, tile_x0, tile_y0);
        }
        __syncthreads();
        if (!__all_sync(FULL, BLEND_DONE)) {
#if GSB_BLEND_TDONE
            const bool was_done = BLEND_DONE;
#endif
            // compact this warp's survivors of the batch into a list of shared-memory addresses (one ballot per 32 records)
            uint32_t n = 0;
            for (uint32_t c = 0; c < cnt; c += 32) {
                const bool mine = (c + lane < cnt) && ((s_mask[c + lane] >> warp) & 1u);
                const unsigned bits = __ballot_sync(FULL, mine);
                if (mine) s_list[warp][n + __popc(bits & ((1u << lane) - 1u))] = (uint16_t)(rec_sh + (c + lane) * sizeof(StagedRec));
                n += __popc(bits);
            }
            __syncwarp();
            // The walk is branch-free per lane: the shader's `continue`s (render.comp:68-70, :78-80) and `break` (:83-85)
            // become the predicate `ok`; only the every-16 "whole warp done" test is a (warp-uniform) branch.
            const uint32_t list_sh = (uint32_t)__cvta_generic_to_shared(&s_list[warp][0]);
            uint32_t fin_k = 0xffffffffu;
            for (uint32_t k0 = 0; k0 < n; k0 += GSB_BLEND_CHECK) {
                if (__all_sync(FULL, BLEND_DONE)) break;
                const uint32_t k1 = min(n, k0 + (uint32_t)GSB_BLEND_CHECK);
                for (uint32_t k = k0; k < k1; k++) {
                    const uint32_t addr = lds_u16(list_sh + 2u * k);
                    const float4 a = lds_f4(addr);
                    const float4 b = lds_f4(addr + 16u);
                    const float2 gb = lds_f2(addr + 32u);
                    const float dx = a.x - fx, dy = a.y - fy;  // :64
                    float power, alpha;
                    if (MODE == GSB_MODE_EXACT) {
                        power = ((a.z * dx) * dx + (b.x * dy) * dy) + (a.w * dx) * dy;  // :66 (pre-scaled conic)
#if GSB_BLEND_TDONE
                        alpha = fminf(0.99f, b.z * exp_shared_inrange(power));             // :77
#else
                        alpha = fminf(0.99f, b.z * exp_shared(power));                     // :77
#endif
                    } else {
                        power = fmaf(a.z * dx, dx, fmaf(b.x * dy, dy, (a.w * dx) * dy));
                        alpha = fminf(0.99f, b.z * __expf(power));
                    }
#if GSB_BLEND_TDONE
                    // A finished pixel carries T == 0 (a live one has T >= 1e-4): its test_T is 0, so it "finishes" again at
                    // every record it would touch and never accumulates; fin_k keeps the FIRST such record.  A NaN power
                    // fails both comparisons and is skipped, as in the oracle (its exp clamps NaN to exp(-87)).
                    bool ok = (power <= 0.0f && power >= b.y) && !(alpha < 1.0f / 255.0f);  // :68-70, :78-80
                    const float test_T = T * (1.0f - alpha);                               // :82
                    const bool fin = ok && test_T < 0.0001f;                               // :83-85
                    fin_k = fin ? min(fin_k, k) : fin_k;
                    ok = ok && !fin;
#else
                    // :68-70 and, below the Gaussian's cut, alpha < 1/255 (:78); a NaN power passes like in the shader
                    bool ok = !done && !(power > 0.0f || power < b.y) && !(alpha < 1.0f / 255.0f);  // :78-80
                    const float test_T = T * (1.0f - alpha);  // :82
                    if (ok && test_T < 0.0001f) {             // :83-85
                        done = true;
                        fin_k = k;
                        ok = false;
                    }
#endif
#if GSB_BLEND_PREDICATED
                    // select form: the products are computed unconditionally, only the four state updates are predicated
                    if (MODE == GSB_MODE_EXACT) {
                        const float n0 = c0 + (b.w * alpha) * T, n1 = c1 + (gb.x * alpha) * T, n2 = c2 + (gb.y * alpha) * T;  // :87
                        c0 = ok ? n0 : c0;
                        c1 = ok ? n1 : c1;
                        c2 = ok ? n2 : c2;
                    } else {
                        const float w = alpha * T;
                        c0 = ok ? fmaf(b.w, w, c0) : c0;
                        c1 = ok ? fmaf(gb.x, w, c1) : c1;
                        c2 = ok ? fmaf(gb.y, w, c2) : c2;
                    }
#if GSB_BLEND_TDONE
                    T = fin ? 0.0f : (ok ? test_T : T);  // :88, and the break
#else
                    T = ok ? test_T : T;  // :88
#endif
#else
                    if (ok) {
                        if (MODE == GSB_MODE_EXACT) {
                            c0 = c0 + (b.w * alpha) * T;  // :87
                            c1 = c1 + (gb.x * alpha) * T;
                            c2 = c2 + (gb.y * alpha) * T;
                        } else {
                            const float w = alpha * T;
                            c0 = fmaf(b.w, w, c0);
                            c1 = fmaf(gb.x, w, c1);
                            c2 = fmaf(gb.y, w, c2);
                        }
                        T = test_T;  // :88
                    }
#endif
                }
            }
#if GSB_BLEND_TDONE
            if (!was_done && fin_k != 0xffffffffu) used = base - range.x + (s_list[warp][fin_k] - rec_sh) / (uint32_t)sizeof(StagedRec) + 1;
            else if (!BLEND_DONE) used = base - range.x + cnt;
#else
            if (fin_k != 0xffffffffu) used = base - range.x + (s_list[warp][fin_k] - rec_sh) / (uint32_t)sizeof(StagedRec) + 1;
            else if (!done) used = base - range.x + cnt;
#endif
        }
        if (__syncthreads_and(BLEND_DONE)) break;
    }

    if (inside) {
        atomicMax(&s_used, used);
        const uint32_t row = py - P.out_first_row;
        unsigned char* dst = static_cast<unsigned char*>(P.out) + (size_t)row * P.row_pitch_bytes;
        if (P.format == GSB_FORMAT_RGBA32F) {
            reinterpret_cast<float4*>(dst)[px] = make_float4(c0, c1, c2, 1.0f);  // :98 vec4(c, 1)
        } else {
            const uint32_t r = unorm8(c0), g = unorm8(c1), b = unorm8(c2);
            const uint32_t v = (P.format == GSB_FORMAT_BGRA8) ? (b | (g << 8) | (r << 16) | 0xff000000u)
                                                              : (r | (g << 8) | (b << 16) | 0xff000000u);
            reinterpret_cast<uint32_t*>(dst)[px] = v;
        }
    }
    __syncthreads();
    if (tid == 0 && s_used) atomicAdd(&P.ctl->blend_consumed, (unsigned long long)s_used);
}


// ------------------------------------------------------------------------------------------------------------------
// k_blend2 -- two pixels per thread, packed fp32 (Blackwell FMUL2 / FADD2 / FFMA2 = PTX *.f32x2).
//
// One CTA of 128 threads owns one 16x16 tile; warp w owns the 8x8 pixel block at (8 (w & 1), 8 (w >> 1)) and lane
// (lx = lane & 7, ly = lane >> 3) owns the two pixels (lx, ly) and (lx, ly + 4) of it.  Every arithmetic step of
// render.comp:64-88 is issued once for both pixels as one packed instruction; each half of a packed instruction is the
// same single correctly rounded IEEE operation as its scalar form, so EXACT mode stays bit-identical to the oracle.
// Measured on B200 (tools/ubench/f32x2.cu): FMUL2 / FADD2 issue at the scalar rate (2x the lanes per issue slot), FFMA2
// at half of it (same lanes per cycle as FFMA) -- the kernel is issue-bound, so what counts is that the per-record loop
// drops from 51.5 instructions per 32 pixels to ~66 per 64 pixels.  The comparisons and selects of the shader's
// `continue` / `break` logic have no packed form and stay per pixel.
// Staged records are stored pre-broadcast ((ux, ux), (A', A'), ...) so that every packed operand is an aligned register
// pair straight out of an LDS.128: no MOVs in the loop.  Per-warp survivor lists, per-block conservative culling
// (8x8 blocks) and the batch pipeline are those of k_blend.
// ------------------------------------------------------------------------------------------------------------------
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(u64 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
    u64 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
    u64 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 sub2(u64 a, u64 b) {
    u64 d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
    u64 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
// EXACT-mode add whose first operand is a packed PRODUCT.  ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even
// though both carry .rn (it honours .rn for scalar f32; -fmad=false, volatile asm and a constant 1.0 multiplier do not
// stop it -- checked in SASS), which would change the rounding of render.comp:66/:87.  Two ways to keep the two roundings:
//   GSB_BLEND2_ADD == 1: a + b = fma(a, 1.0, b) with the 1.0 coming from a kernel argument (opaque to ptxas), one FFMA2
//                        with a uniform-register operand;
//   GSB_BLEND2_ADD == 0: two scalar add.rn.f32 on the halves.
#ifndef GSB_BLEND2_ADD
#define GSB_BLEND2_ADD 0  // measured on the bench scene: k_blend2 0.597 ms with the scalar adds, 0.665 ms with FFMA2 (half-rate on B200)
#endif
#ifndef GSB_BLEND2_PRED
#define GSB_BLEND2_PRED 1  // colour / transmittance updates: 1 = predicated scalar adds, 0 = packed adds + selects
#endif
__device__ __forceinline__ u64 add2_of_product(u64 prod, u64 b, u64 one2) {
#if GSB_BLEND2_ADD
    return fma2(prod, one2, b);
#else
    float p0, p1, b0, b1;
    upk2(prod, p0, p1);
    upk2(b, b0, b1);
    return pk2(__fadd_rn(p0, b0), __fadd_rn(p1, b1));
#endif
}
// two 64-bit register pairs out of one LDS.128
__device__ __forceinline__ void lds_2x64(uint32_t addr, u64& a, u64& b) {
    asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr));
}

#ifndef GSB_BLEND2_BATCH
#define GSB_BLEND2_BATCH 256  // records staged per batch (2 per thread)
#endif
#ifndef GSB_BLEND2_MIN_BLOCKS
#define GSB_BLEND2_MIN_BLOCKS 8
#endif
#ifndef GSB_BLEND2_CHECK
#define GSB_BLEND2_CHECK 8
#endif
#ifndef GSB_BLEND_TMA
#define GSB_BLEND_TMA 1  // coarse bins: list segments staged by TMA bulk copies (0: per-thread __ldg)
#endif
constexpr int B2_THREADS = 128;
constexpr int B2_SEG = 4 * B2_THREADS;  // list entries scanned per batch at most
constexpr int B2_BATCH = GSB_BLEND2_BATCH;
constexpr int B2_WARPS = B2_THREADS / 32;

struct __align__(16) StagedRec2 {  // 80 B: five 16-B slots = five LDS.128 per visited record
    float4 q0;  // ux ux uy uy
    float4 q1;  // -A/2 -A/2 -B -B       (exact power-of-two / sign scalings of the conic, as in k_blend)
    float4 q2;  // -C/2 -C/2 opacity opacity
    float4 q3;  // r r g g
    float4 q4;  // b b power_cut bits(index in batch)
};
struct __align__(16) StagedRec2Aux {  // 96 B (gsb_render_aux): StagedRec2 + a sixth slot
    float4 q0, q1, q2, q3, q4;
    float4 q5;  // depth depth - -     (view-space z = VertexAttribute.depth, pre-broadcast like the others)
};
template <bool AUX> struct StagedRec2Of { typedef StagedRec2 type; };
template <> struct StagedRec2Of<true> { typedef StagedRec2Aux type; };

#ifndef GSB_BLEND2_AUX_MIN_BLOCKS
#define GSB_BLEND2_AUX_MIN_BLOCKS 7  // AUX: 72-register cap (the colour-only kernels sit at the 64-register cap of 8 CTAs/SM)
#endif

__device__ __forceinline__ uint32_t block_mask2(float ux, float uy, float A, float B, float C, float cut, float tile_x0, float tile_y0) {
    if (!(A > 0.0f) || !(C > 0.0f)) return 0xfu;  // not positive definite / NaN: never cull
    const float inv_a = __frcp_rn(A), inv_c = __frcp_rn(C);
    uint32_t mask = 0;
#pragma unroll
    for (int w = 0; w < B2_WARPS; w++) {
        const float x0 = tile_x0 + (float)((w & 1) * 8), y0 = tile_y0 + (float)((w >> 1) * 8);
        if (rect_may_contribute(ux, uy, A, B, C, inv_a, inv_c, x0, y0, 8.0f, 8.0f, cut)) mask |= 1u << w;
    }
    return mask;
}

// exp for both pixels; same operation sequence as exp_shared without the clamp at -87 (identity on [cut, 0] with
// cut >= -87, and results for powers outside that range are never selected)
__device__ __forceinline__ void exp_shared2(u64 x, u64 one2, float& e0, float& e1) {
    const u64 L2E = pk2(1.44269504088896341f, 1.44269504088896341f), MAGIC = pk2(12582912.0f, 12582912.0f);
    const u64 t = mul2(x, L2E);
    const u64 tm = add2_of_product(t, MAGIC, one2);
    const u64 n = sub2(tm, MAGIC);
    u64 r = fma2(n, pk2(-0.693359375f, -0.693359375f), x);
    r = fma2(n, pk2(2.12194440e-4f, 2.12194440e-4f), r);
    u64 p = fma2(pk2(8.290082216262817e-3f, 8.290082216262817e-3f), r, pk2(4.1899293661117554e-2f, 4.1899293661117554e-2f));
    p = fma2(p, r, pk2(1.6667647659778595e-1f, 1.6667647659778595e-1f));
    p = fma2(p, r, pk2(4.9999138712882996e-1f, 4.9999138712882996e-1f));
    p = fma2(p, r, pk2(9.999997019767761e-1f, 9.999997019767761e-1f));
    p = fma2(p, r, pk2(1.0f, 1.0f));
    float p0, p1, m0, m1;
    upk2(p, p0, p1);
    upk2(tm, m0, m1);
    e0 = __uint_as_float(__float_as_uint(p0) + (__float_as_uint(m0) << 23));
    e1 = __uint_as_float(__float_as_uint(p1) + (__float_as_uint(m1) << 23));
}

// COARSE (gsb_set_tile_cull level 2): the list is that of a block of 2^cs x 2^cs tiles and every entry's key carries the mask
// of the block's tiles inside the Gaussian's tile AABB.  Staging becomes a stream compaction: the CTA scans the list 128
// entries at a time (keys + payloads only, coalesced), keeps the entries whose mask has this tile's bit -- in list order, so
// the tile's own (depth, index) order is preserved -- and gathers records only for those, until the batch holds up to
// B2_BATCH of them.  The walk is unchanged.
// AUX (gsb_render_aux): the walk also accumulates D += (depth * alpha) * T next to the colour and keeps the transmittance after
// the last accumulated Gaussian (T itself is overwritten with 0 at the break); every pixel then stores (1 - T_end, D).  All
// of it sits behind `if constexpr (AUX)`: the colour-only instantiations are unchanged.
template <int MODE, bool STATS, bool COARSE, bool AUX>
__global__ void __launch_bounds__(B2_THREADS, AUX ? GSB_BLEND2_AUX_MIN_BLOCKS : GSB_BLEND2_MIN_BLOCKS)
    k_blend2(const __grid_constant__ BlendParams P) {
    typedef typename StagedRec2Of<AUX>::type Rec;
    __shared__ Rec s_rec[B2_BATCH];
    __shared__ uint8_t s_mask[B2_BATCH];
    __shared__ uint32_t s_wc[B2_WARPS];
#if GSB_BLEND_TMA
    // COARSE: the next segment of the block's (key, payload) run, fetched by TMA (cp.async.bulk) while the current batch is
    // gathered and walked: BASELINE north_star's "TMA bulk staging of per-tile Gaussian runs into shared memory"
    __shared__ alignas(16) uint32_t s_seg[COARSE ? 2 : 1][COARSE ? B2_SEG + 4 : 4];
    __shared__ unsigned long long s_bar;
#endif
    __shared__ alignas(16) uint16_t s_list[B2_WARPS][B2_BATCH];  // per warp: shared-window addresses of the records it must visit
    // COARSE: compact id and list position of the batch's entries.  They live in the same 2 KB as the per-warp lists: written
    // by the fill, read by the record gather, and only then (a barrier later) do the warps build their lists; the barrier at
    // the end of the batch separates the walk from the next fill.  (27 KB instead of 29 KB per CTA = 8 instead of 7 per SM.)
    static_assert(sizeof(uint16_t) * B2_WARPS * B2_BATCH >= 2 * sizeof(uint32_t) * B2_BATCH, "s_cid + s_eidx alias s_list");
    uint32_t* const s_cid = reinterpret_cast<uint32_t*>(&s_list[0][0]);
    uint32_t* const s_eidx = s_cid + B2_BATCH;
    __shared__ uint32_t s_used, s_walked, s_hits;
    static_assert(sizeof(Rec) * B2_BATCH < 65536, "u16 list entries hold shared-window addresses");

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tx = blockIdx.x % P.tiles_x;
    const uint32_t ty = P.tile_row_begin + blockIdx.x / P.tiles_x;
    // render.comp:43-44; stored as (start, ~end), empty = all ones.  With coarse bins (gsb_set_tile_cull level 2) the list is
    // that of the 2^cs x 2^cs tile block holding this tile: still in (depth, index) order, and the staging below keeps exactly
    // the records whose tile AABB holds (tx, ty) = the tile's own list in the reference.
    const uint32_t cs = P.coarse_shift;
    uint2 range = P.ranges[(ty >> cs) * P.bins_x + (tx >> cs)];
    range.y = ~range.y;
    const uint32_t px = tx * GSB_TILE + (warp & 1) * 8 + (lane & 7);
    const uint32_t py0 = ty * GSB_TILE + (warp >> 1) * 8 + (lane >> 3), py1 = py0 + 4;
    const bool in0 = px < P.width && py0 < P.height, in1 = px < P.width && py1 < P.height;  // :37-39
    const u64 fx2 = pk2((float)px, (float)px), fy2 = pk2((float)py0, (float)py1);
    const u64 one2 = pk2(P.one, P.one);  // 1.0f the compiler cannot see (add2_of_product)
    const float tile_x0 = (float)(tx * GSB_TILE), tile_y0 = (float)(ty * GSB_TILE);
    if (tid == 0) {
        s_used = 0;
        s_walked = 0;
        s_hits = 0;
    }
    __syncthreads();

    // transmittance (0 = finished or outside the image) and colour a/b/c of pixel 0/1
    float T0 = in0 ? 1.0f : 0.0f, T1 = in1 ? 1.0f : 0.0f, ca0 = 0.f, ca1 = 0.f, cb0 = 0.f, cb1 = 0.f, cc0 = 0.f, cc1 = 0.f;
#define B2_DONE (T0 == 0.0f && T1 == 0.0f)
    // AUX: expected depth and the transmittance after the last accumulated Gaussian (T0 / T1 become 0 at the break)
    float d0 = 0.f, d1 = 0.f, tl0 = 1.0f, tl1 = 1.0f;
    uint32_t used = 0, walked = 0, hits = 0, staged = 0;
    const uint32_t rec_sh = (uint32_t)__cvta_generic_to_shared(&s_rec[0]);
    const uint32_t list_sh = (uint32_t)__cvta_generic_to_shared(&s_list[warp][0]);

    const uint32_t tbit = 16u + (((ty & ((1u << cs) - 1u)) << cs) | (tx & ((1u << cs) - 1u)));  // this tile's bit in a coarse key
    uint32_t cursor = range.x;  // COARSE: next list entry to scan
#if GSB_BLEND_TMA
    uint32_t seg_a = range.x & ~3u, seg_parity = 0u;
    bool seg_pending = COARSE && range.x < range.y;  // a bulk copy into s_seg is in flight
    if (COARSE) {
        if (tid == 0) {
            mbar_init(&s_bar, 1);
            mbar_fence_init();
            if (range.x < range.y) {
                const uint32_t bytes = (((min(range.y, range.x + (uint32_t)B2_SEG) - seg_a) + 3u) & ~3u) * 4u;
                mbar_expect_tx(&s_bar, 2u * bytes);
                tma_load(s_seg[0], P.keys + seg_a, bytes, &s_bar);
                tma_load(s_seg[1], P.vals + seg_a, bytes, &s_bar);
            }
        }
        __syncthreads();  // the barrier object is initialised before anyone waits on it
    }
#endif
    for (uint32_t base = range.x; COARSE ? (cursor < range.y) : (base < range.y); base += B2_BATCH) {
        uint32_t cnt;
        if constexpr (COARSE) {
            // ---- fill: scan up to 4 x 128 entries (loads issued together), compact this tile's entries in list order ----
            constexpr int STEPS = 4;
            uint32_t kk[STEPS], vv[STEPS];
#if GSB_BLEND_TMA
            // the segment that starts at `cursor` (16-B aligned start seg_a <= cursor).  One warp polls the mbarrier, the others
            // sleep on the hardware barrier: 128 threads spinning on try_wait cost issue slots the other CTAs' walks need
            if (warp == 0) mbar_wait(&s_bar, seg_parity);
            __syncthreads();
            seg_parity ^= 1u;
            seg_pending = false;
#pragma unroll
            for (int j = 0; j < STEPS; j++) {
                const uint32_t e = cursor + (uint32_t)(j * B2_THREADS + tid);
                kk[j] = 0u;
                vv[j] = 0u;
                if (e < range.y) {
                    kk[j] = s_seg[0][e - seg_a];
                    vv[j] = s_seg[1][e - seg_a];
                }
            }
#else
#pragma unroll
            for (int j = 0; j < STEPS; j++) {
                const uint32_t e = cursor + (uint32_t)(j * B2_THREADS + tid);
                kk[j] = 0u;
                vv[j] = 0u;
                if (e < range.y) {
                    kk[j] = __ldg(P.keys + e);
                    vv[j] = __ldg(P.vals + e);
                }
            }
#endif
            uint32_t nfill = 0, steps = 0;
#pragma unroll
            for (int j = 0; j < STEPS; j++) {
                if (cursor + (uint32_t)(j * B2_THREADS) >= range.y || nfill > (uint32_t)(B2_BATCH - B2_THREADS)) break;  // uniform
                const bool match = (kk[j] >> tbit) & 1u;
                const unsigned bits = __ballot_sync(FULL, match);
                if (lane == 0) s_wc[warp] = __popc(bits);
                __syncthreads();
                uint32_t off = nfill + __popc(bits & ((1u << lane) - 1u)), tot = 0;
#pragma unroll
                for (int w = 0; w < B2_WARPS; w++) {
                    const uint32_t c = s_wc[w];
                    if (w < warp) off += c;
                    tot += c;
                }
                if (match) {
                    s_cid[off] = vv[j];
                    s_eidx[off] = cursor - range.x + (uint32_t)(j * B2_THREADS + tid);
                }
                nfill += tot;
                steps++;
                __syncthreads();  // s_wc is reused by the next step; s_cid / s_eidx are read below
            }
            cursor = min(range.y, cursor + steps * (uint32_t)B2_THREADS);
            cnt = nfill;
#if GSB_BLEND_TMA
            // every thread has read its entries (the barriers of the steps above): fetch the next segment now, it lands while
            // this batch's records are gathered and walked
            if (cursor < range.y) {
                seg_a = cursor & ~3u;
                seg_pending = true;
                if (tid == 0) {
                    const uint32_t bytes = (((min(range.y, cursor + (uint32_t)B2_SEG) - seg_a) + 3u) & ~3u) * 4u;
                    fence_proxy_async();
                    mbar_expect_tx(&s_bar, 2u * bytes);
                    tma_load(s_seg[0], P.keys + seg_a, bytes, &s_bar);
                    tma_load(s_seg[1], P.vals + seg_a, bytes, &s_bar);
                }
            }
#endif
        } else {
            cnt = min((uint32_t)B2_BATCH, range.y - base);
        }
        if (STATS) staged += cnt;
#pragma unroll
        for (int j = 0; j < B2_BATCH / B2_THREADS; j++) {
            const uint32_t li = (uint32_t)(j * B2_THREADS + tid);
            if (li < cnt) {
                const uint32_t cid = COARSE ? s_cid[li] : __ldg(P.vals + base + li);
                const float4* rec = P.recs + (size_t)cid * GSB_REC_F4;
                const float4 a = __ldg(rec), col = __ldg(rec + 2);
                const float2 b = __ldg(reinterpret_cast<const float2*>(rec + 1));  // conic.z, opacity
                const float cut = power_cut(b.y);
                const uint32_t m = block_mask2(a.x, a.y, a.z, a.w, b.x, cut, tile_x0, tile_y0);
                if (m) {
                    const float na = -0.5f * a.z, nb = -a.w, nc = -0.5f * b.x;
                    s_rec[li].q0 = make_float4(a.x, a.x, a.y, a.y);
                    s_rec[li].q1 = make_float4(na, na, nb, nb);
                    s_rec[li].q2 = make_float4(nc, nc, b.y, b.y);
                    s_rec[li].q3 = make_float4(col.x, col.x, col.y, col.y);
                    // q4.w: position in the list relative to the batch's base offset (the consumed-entries statistic)
                    s_rec[li].q4 = make_float4(col.z, col.z, cut, __uint_as_float(COARSE ? s_eidx[li] : li));
                    if constexpr (AUX) s_rec[li].q5 = make_float4(col.w, col.w, 0.f, 0.f);  // q2.w of the record: view-space depth
                }
                s_mask[li] = (uint8_t)m;
            }
        }
        __syncthreads();
        if (!__all_sync(FULL, B2_DONE)) {
            uint32_t n = 0;
            for (uint32_t c = 0; c < cnt; c += 32) {  // one ballot per 32 records
                const bool mine = (c + lane < cnt) && ((s_mask[c + lane] >> warp) & 1u);
                const unsigned bits = __ballot_sync(FULL, mine);
                if (mine) s_list[warp][n + __popc(bits & ((1u << lane) - 1u))] = (uint16_t)(rec_sh + (c + lane) * sizeof(Rec));
                n += __popc(bits);
            }
            __syncwarp();
            const uint32_t base_off = COARSE ? 0u : base - range.x;
            uint32_t k0 = 0;
            for (; k0 < n; k0 += GSB_BLEND2_CHECK) {
                if (__all_sync(FULL, B2_DONE)) break;
                const uint32_t k1 = min(n, k0 + (uint32_t)GSB_BLEND2_CHECK);
                for (uint32_t k = k0; k < k1; k++) {
                    const uint32_t addr = lds_u16(list_sh + 2u * k);
                    u64 ux2, uy2, A2, B2, C2, op2, r2, g2, b2, misc;
                    lds_2x64(addr, ux2, uy2);
                    lds_2x64(addr + 16u, A2, B2);
                    lds_2x64(addr + 32u, C2, op2);
                    lds_2x64(addr + 48u, r2, g2);
                    lds_2x64(addr + 64u, b2, misc);
                    float cut, idxf;
                    upk2(misc, cut, idxf);
                    const u64 dx2 = sub2(ux2, fx2), dy2 = sub2(uy2, fy2);  // :64
                    float pw0, pw1, al0, al1;
                    u64 alpha2;
                    if (MODE == GSB_MODE_EXACT) {
                        // :66 with the pre-scaled conic: ((A' dx) dx + (C' dy) dy) + (B' dx) dy
                        const u64 s2 = add2_of_product(mul2(mul2(A2, dx2), dx2), mul2(mul2(C2, dy2), dy2), one2);
                        const u64 pw2 = add2_of_product(mul2(mul2(B2, dx2), dy2), s2, one2);  // s + t3 == t3 + s (commutative, one rounding)
                        upk2(pw2, pw0, pw1);
                        float e0, e1;
                        exp_shared2(pw2, one2, e0, e1);
                        float o0, o1;
                        upk2(mul2(op2, pk2(e0, e1)), o0, o1);  // :77
                        al0 = fminf(0.99f, o0);
                        al1 = fminf(0.99f, o1);
                    } else {
                        const u64 pw2 = fma2(mul2(A2, dx2), dx2, fma2(mul2(C2, dy2), dy2, mul2(mul2(B2, dx2), dy2)));
                        upk2(pw2, pw0, pw1);
                        float o0, o1;
                        upk2(op2, o0, o1);
                        al0 = fminf(0.99f, o0 * __expf(pw0));
                        al1 = fminf(0.99f, o1 * __expf(pw1));
                    }
                    alpha2 = pk2(al0, al1);
                    // A finished (or out-of-image) pixel carries T == 0 (a live one has T >= 1e-4): its test_T is 0, so it
                    // "finishes" again at every record it would touch, never accumulates, and needs no separate flag.
                    // in0 / in1: :68-70 and, below the Gaussian's cut, alpha < 1/255 (:78); a NaN power passes like in the shader
                    const bool in0k = !(pw0 > 0.0f || pw0 < cut) && !(al0 < 1.0f / 255.0f);  // :78-80
                    const bool in1k = !(pw1 > 0.0f || pw1 < cut) && !(al1 < 1.0f / 255.0f);
                    float tt0, tt1;
                    const u64 T2 = pk2(T0, T1);
                    upk2(mul2(T2, sub2(pk2(1.0f, 1.0f), alpha2)), tt0, tt1);  // :82
                    const bool ok0 = in0k && !(tt0 < 0.0001f), ok1 = in1k && !(tt1 < 0.0001f);  // :83-85 (the break)
                    if (STATS) {
                        const uint32_t u = base_off + __float_as_uint(idxf) + 1u;
                        used = ((in0k && !ok0 && T0 != 0.0f) || (in1k && !ok1 && T1 != 0.0f)) ? max(used, u) : used;
                        if (P.stats > 1) hits += (in0k && T0 != 0.0f ? 1u : 0u) + (in1k && T1 != 0.0f ? 1u : 0u);  // debug frames only
                    }
                    if constexpr (AUX) {
                        u64 z2, zpad;
                        lds_2x64(addr + 80u, z2, zpad);
                        float wd0, wd1;
                        if (MODE == GSB_MODE_EXACT) {
                            upk2(mul2(mul2(z2, alpha2), T2), wd0, wd1);  // (depth * alpha) * T, :87's shape
                            if (ok0) d0 = __fadd_rn(d0, wd0);
                            if (ok1) d1 = __fadd_rn(d1, wd1);
                        } else {
                            float z, z_;
                            upk2(z2, z, z_);
                            upk2(mul2(alpha2, T2), wd0, wd1);
                            if (ok0) d0 = fmaf(z, wd0, d0);
                            if (ok1) d1 = fmaf(z, wd1, d1);
                        }
                        tl0 = ok0 ? tt0 : tl0;  // :88 without the break's 0
                        tl1 = ok1 ? tt1 : tl1;
                    }
#if GSB_BLEND2_PRED
                    // predicated scalar accumulates (FMA pipe) instead of packed adds + selects (the half-rate ALU pipe is
                    // this kernel's bottleneck: profiles/)
                    float w0a, w1a, w0b, w1b, w0c, w1c;
                    if (MODE == GSB_MODE_EXACT) {
                        upk2(mul2(mul2(r2, alpha2), T2), w0a, w1a);  // :87
                        upk2(mul2(mul2(g2, alpha2), T2), w0b, w1b);
                        upk2(mul2(mul2(b2, alpha2), T2), w0c, w1c);
                    } else {
                        const u64 w2 = mul2(alpha2, T2);
                        upk2(mul2(r2, w2), w0a, w1a);
                        upk2(mul2(g2, w2), w0b, w1b);
                        upk2(mul2(b2, w2), w0c, w1c);
                    }
                    if (ok0) {
                        ca0 = __fadd_rn(ca0, w0a);
                        cb0 = __fadd_rn(cb0, w0b);
                        cc0 = __fadd_rn(cc0, w0c);
                    }
                    if (ok1) {
                        ca1 = __fadd_rn(ca1, w1a);
                        cb1 = __fadd_rn(cb1, w1b);
                        cc1 = __fadd_rn(cc1, w1c);
                    }
                    if (in0k) T0 = ok0 ? tt0 : 0.0f;  // :88, or the break
                    if (in1k) T1 = ok1 ? tt1 : 0.0f;
#else
                    float na0, na1, nb0, nb1, nc0, nc1;
                    if (MODE == GSB_MODE_EXACT) {
                        upk2(add2_of_product(mul2(mul2(r2, alpha2), T2), pk2(ca0, ca1), one2), na0, na1);  // :87
                        upk2(add2_of_product(mul2(mul2(g2, alpha2), T2), pk2(cb0, cb1), one2), nb0, nb1);
                        upk2(add2_of_product(mul2(mul2(b2, alpha2), T2), pk2(cc0, cc1), one2), nc0, nc1);
                    } else {
                        const u64 w2 = mul2(alpha2, T2);
                        upk2(fma2(r2, w2, pk2(ca0, ca1)), na0, na1);
                        upk2(fma2(g2, w2, pk2(cb0, cb1)), nb0, nb1);
                        upk2(fma2(b2, w2, pk2(cc0, cc1)), nc0, nc1);
                    }
                    ca0 = ok0 ? na0 : ca0;
                    cb0 = ok0 ? nb0 : cb0;
                    cc0 = ok0 ? nc0 : cc0;
                    T0 = in0k ? (ok0 ? tt0 : 0.0f) : T0;  // :88, or the break
                    ca1 = ok1 ? na1 : ca1;
                    cb1 = ok1 ? nb1 : cb1;
                    cc1 = ok1 ? nc1 : cc1;
                    T1 = in1k ? (ok1 ? tt1 : 0.0f) : T1;
#endif
                }
            }
            if (STATS) {
                walked += min(k0, n);
                if (!B2_DONE) used = COARSE ? cursor - range.x : base_off + cnt;  // a live pixel read the whole batch
            }
        }
        if (__syncthreads_and(B2_DONE)) break;
    }
#undef B2_DONE
#if GSB_BLEND_TMA
    if (COARSE && seg_pending) mbar_wait(&s_bar, seg_parity);  // never leave with a bulk copy still writing this CTA's shared memory
#endif

    if (STATS) {
        if (in0 || in1) atomicMax(&s_used, used);
        if (lane == 0 && walked) atomicAdd(&s_walked, walked);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) hits += __shfl_xor_sync(FULL, hits, o);
        if (lane == 0 && hits) atomicAdd(&s_hits, hits);
    }
    // Destinations: the caller's buffer, or -- frame sharding -- the whole-frame buffer of EVERY rank (peer memory over
    // NVLink; posted stores, so the framebuffer exchange rides under the blend instead of following it as a collective).
    const int ndst = P.num_peers > 0 ? P.num_peers : 1;
    const uint32_t row0 = py0 - P.out_first_row;
    if (P.format == GSB_FORMAT_RGBA32F) {
        for (int d = 0; d < ndst; d++) {
            unsigned char* band = static_cast<unsigned char*>(P.num_peers > 0 ? P.peer_frames[d] : P.out);
            if (in0) reinterpret_cast<float4*>(band + (size_t)row0 * P.row_pitch_bytes)[px] = make_float4(ca0, cb0, cc0, 1.0f);  // :98 vec4(c, 1)
            if (in1) reinterpret_cast<float4*>(band + (size_t)(row0 + 4) * P.row_pitch_bytes)[px] = make_float4(ca1, cb1, cc1, 1.0f);
        }
    } else {
        // 8-bit formats: transpose the tile through shared memory so that every warp store covers whole 64-B tile rows
        // (also what lets gsb_render write a pinned host frame directly at a good PCIe payload size)
        __syncthreads();  // everyone is out of the batch loop: s_rec can be reused
        uint32_t* s_tile = reinterpret_cast<uint32_t*>(&s_rec[0]);  // [16][16]
        const bool bgra = P.format == GSB_FORMAT_BGRA8;
        {
            const uint32_t r0 = unorm8(ca0), g0 = unorm8(cb0), b0 = unorm8(cc0), r1 = unorm8(ca1), g1 = unorm8(cb1), b1 = unorm8(cc1);
            const uint32_t lx = (warp & 1) * 8 + (lane & 7), ly = (warp >> 1) * 8 + (lane >> 3);
            s_tile[ly * 16 + lx] = bgra ? (b0 | (g0 << 8) | (r0 << 16) | 0xff000000u) : (r0 | (g0 << 8) | (b0 << 16) | 0xff000000u);
            s_tile[(ly + 4) * 16 + lx] = bgra ? (b1 | (g1 << 8) | (r1 << 16) | 0xff000000u) : (r1 | (g1 << 8) | (b1 << 16) | 0xff000000u);
        }
        __syncthreads();
        if (tid < 64) {  // thread -> (row = tid / 4, 4 pixels at x = 4 (tid % 4)): 4 consecutive threads = one 64-B tile row
            const uint32_t ry = (uint32_t)tid >> 2, rx = ((uint32_t)tid & 3u) * 4u;
            const uint32_t gy = ty * GSB_TILE + ry, gx = tx * GSB_TILE + rx;
            if (gy < P.height && gx < P.width) {
                const uint4 v = *reinterpret_cast<const uint4*>(&s_tile[ry * 16 + rx]);
                for (int d = 0; d < ndst; d++) {
                    unsigned char* band = static_cast<unsigned char*>(P.num_peers > 0 ? P.peer_frames[d] : P.out);
                    uint32_t* dst = reinterpret_cast<uint32_t*>(band + (size_t)(gy - P.out_first_row) * P.row_pitch_bytes) + gx;
                    if (gx + 3 < P.width && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
                        *reinterpret_cast<uint4*>(dst) = v;
                    } else {  // ragged right edge (W not a multiple of 4) or an unaligned pitch
                        const uint32_t e[4] = {v.x, v.y, v.z, v.w};
                        for (uint32_t q = 0; q < 4 && gx + q < P.width; q++) dst[q] = e[q];
                    }
                }
            }
        }
    }
    if constexpr (AUX) {  // one 8-B store per pixel: the 8 lanes of a pixel row cover 64 contiguous bytes
        unsigned char* abase = reinterpret_cast<unsigned char*>(P.aux);
        if (in0) reinterpret_cast<float2*>(abase + (size_t)row0 * P.aux_pitch)[px] = make_float2(__fsub_rn(1.0f, tl0), d0);
        if (in1) reinterpret_cast<float2*>(abase + (size_t)(row0 + 4) * P.aux_pitch)[px] = make_float2(__fsub_rn(1.0f, tl1), d1);
    }
    if (STATS) {
        __syncthreads();
        if (tid == 0) {
            if (s_used) atomicAdd(&P.ctl->blend_consumed, (unsigned long long)s_used);
            if (s_walked) atomicAdd(&P.ctl->blend_walked, (unsigned long long)s_walked);
            if (s_hits) atomicAdd(&P.ctl->blend_hits, (unsigned long long)s_hits);
            if (staged) atomicAdd(&P.ctl->blend_staged, (unsigned long long)staged);
        }
    }
}

template <bool AUX>
void launch_blend2(const BlendParams& p, uint32_t blocks, cudaStream_t s) {
    if (p.coarse_shift) {
        if (p.stats) {
            if (p.mode == GSB_MODE_EXACT) k_blend2<GSB_MODE_EXACT, true, true, AUX><<<blocks, B2_THREADS, 0, s>>>(p);
            else k_blend2<GSB_MODE_FAST, true, true, AUX><<<blocks, B2_THREADS, 0, s>>>(p);
        } else {
            if (p.mode == GSB_MODE_EXACT) k_blend2<GSB_MODE_EXACT, false, true, AUX><<<blocks, B2_THREADS, 0, s>>>(p);
            else k_blend2<GSB_MODE_FAST, false, true, AUX><<<blocks, B2_THREADS, 0, s>>>(p);
        }
    } else if (p.stats) {
        if (p.mode == GSB_MODE_EXACT) k_blend2<GSB_MODE_EXACT, true, false, AUX><<<blocks, B2_THREADS, 0, s>>>(p);
        else k_blend2<GSB_MODE_FAST, true, false, AUX><<<blocks, B2_THREADS, 0, s>>>(p);
    } else {
        if (p.mode == GSB_MODE_EXACT) k_blend2<GSB_MODE_EXACT, false, false, AUX><<<blocks, B2_THREADS, 0, s>>>(p);
        else k_blend2<GSB_MODE_FAST, false, false, AUX><<<blocks, B2_THREADS, 0, s>>>(p);
    }
}

}  // namespace

cudaError_t launch_blend(const BlendParams& p, cudaStream_t s) {
    const uint32_t rows = p.tile_row_end - p.tile_row_begin;
    const uint32_t blocks = rows * p.tiles_x;
    if (blocks == 0) return cudaSuccess;
    if (p.aux) {  // gsb_render_aux (single context only): k_blend2, the round-1 kernel has no aux planes
        launch_blend2<true>(p, blocks, s);
    } else if (p.variant == 1 && p.num_peers == 0 && p.coarse_shift == 0) {  // round-1 kernel (one pixel per thread), kept for A/B: GSB_BLEND_VARIANT=1
        if (p.mode == GSB_MODE_EXACT) k_blend<GSB_MODE_EXACT><<<blocks, BLEND_THREADS, 0, s>>>(p);
        else k_blend<GSB_MODE_FAST><<<blocks, BLEND_THREADS, 0, s>>>(p);
    } else {
        launch_blend2<false>(p, blocks, s);
    }
    return cudaGetLastError();
}

}  // namespace gsb
