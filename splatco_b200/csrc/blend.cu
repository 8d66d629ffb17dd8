// Per-tile front-to-back alpha blend, forward and backward.  Replaces upstream renderCUDA<3> fwd/bwd
// [SURVEY.md Appendix A.4, A.5; reference call site gaussian_renderer/__init__.py:163-171 and the
// autograd backward triggered at train.py:240].
//
// One CTA per 16x16 tile, one thread per pixel; warps cover 8x4-pixel patches.  ncu showed these kernels to be
// instruction-issue bound from the first version on (81 % issue-active, DRAM < 1 % of peak), so the design goal is
// the fewest instructions per LIVE (pixel, splat) pair.  Common to every kernel here:
//  * splats are staged through shared memory in batches of 512 (two per thread); the staging thread precomputes, once
//    per (tile, splat), the conic pre-scaled into the log2 domain (P2 = log2(e) * power, evaluated from
//    (dx, dy) exactly like the reference so threshold decisions keep full fp32 precision) and
//    log2(opacity), which is folded into the exponent so the alpha >= 1/255 cut is a compare BEFORE the
//    ex2 (culled pairs never touch the SFU);
//  * a warp leaves as soon as all its pixels are saturated, the CTA when every warp has; CTAs run longest tile first.
// Two generations are kept behind splatco_blend_set_impl (A/B timing; the tests compare them):
//  round 1  blend_fwd_kernel / blend_bwd_kernel: the splat's alpha >= 1/255 bounding box against the 8 patches -> one
//           mask word per (warp, 32 splats); warps walk their set bits in list order, one splat per warp step.  The
//           backward forms nine partial sums per visit and reduces them through a per-warp transposition buffer.
//  round 2  blend_fwd2_kernel (per-row alpha >= 1/255 spans -> per-PIXEL candidate bit lists; every lane walks its own
//           list) and blend_bwd2_kernel (same walk as round 1, two parked values per visit and a matrix-form reduction
//           with constant weights).  The defaults; see the comments at the kernels.
#include "common.cuh"
#include <stdlib.h>
#include <type_traits>

namespace splatco {

constexpr int BLEND_THREADS = TILE * TILE;   // 256
constexpr int BLEND_BATCH = 2 * BLEND_THREADS;   // splats staged per barrier (two per thread): half the barriers of a
                                                 // 256-splat batch, and the per-warp work imbalance averages out better
constexpr int BLEND_WORDS = BLEND_BATCH / 32;    // 16 mask words per patch warp
constexpr int RB_SLOTS = 3, RB_ROWS = 9 * RB_SLOTS, RB_STRIDE = 36;     // backward reduction buffer (see blend_bwd_kernel)
constexpr size_t BWD_SMEM = (size_t)BLEND_BATCH * 48 + (size_t)(BLEND_THREADS / 32) * RB_ROWS * RB_STRIDE * sizeof(float);
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLog2Inv255 = -7.994353436858858f;     // log2(1/255)

__device__ __forceinline__ void pixel_of_thread(int tile_x, int tile_y, int &px, int &py, float &u, float &v) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lx = (warp & 1) * 8 + (lane & 7), ly = (warp >> 1) * 4 + (lane >> 3);
    px = tile_x * TILE + lx;
    py = tile_y * TILE + ly;
    u = (float)lx - 7.5f;      // tile-centred pixel coordinates
    v = (float)ly - 7.5f;
}

struct SplatCoef {
    float4 k0;    // sx, sy, a2, b2        (centre relative to the tile centre; log2-domain conic)
    float4 k1;    // c2, log2(opacity), r, g
    uint32_t mask8;
};

// P2 = log2(e) * power = a2 dx^2 + b2 dx dy + c2 dy^2   (a2 = -0.5 log2e A, b2 = -log2e B, c2 = -0.5 log2e C)
__device__ __forceinline__ float eval_p2(const float4 &k0, float c2, float u, float v, float &dx, float &dy) {
    dx = k0.x - u; dy = k0.y - v;
    const float t = fmaf(k0.z, dx, k0.w * dy);
    return fmaf(c2 * dy, dy, t * dx);
}

// Both cull filters (the bounding box below, the row spans of splat_patch_words) solve the conic's quadratic from
// det = a2 c2 - b2^2 / 4.  For needle-shaped splats that is a cancellation: its relative error, and that of the pair
// test's own p2 evaluation, is about eps * a2 c2 / det, which outgrows the fixed margins of the solutions (0.2 % of
// tau2, 0.02 px) -- on needles of screen sigma 1000 px and more the row spans dropped pairs the per-pixel test
// accepts, far out on the needle's flank (tests/test_blend_filters_gpu.py).  Above det / (a2 c2) = 2^-10 the error is
// about 6e-5, 30x inside the margin; conics worse than that are not culled.
constexpr float kMinDetRatio = 1.0f / 1024.0f;
__device__ __forceinline__ bool conic_cullable(float a2, float c2, float det) {
    return det > 0.f && det > kMinDetRatio * (a2 * c2);
}

// sx, sy: splat centre relative to the tile centre.  Returns the log2-domain coefficients and the
// 8-bit patch mask (bit w = warp w's 8x4 patch may see alpha >= 1/255).
__device__ __forceinline__ SplatCoef splat_setup(float sx, float sy, float A, float B, float C, float op, float r,
                                                 float g) {
    SplatCoef s;
    const float a2 = -0.5f * kLog2e * A, c2 = -0.5f * kLog2e * C, b2 = -kLog2e * B;
    const float lo = op > 0.f ? __log2f(op) : -1e30f;
    s.k0 = make_float4(sx, sy, a2, b2);
    s.k1 = make_float4(c2, lo, r, g);
    // bounding box of { d : -P2(d) <= tau2 },  tau2 = log2(255 * opacity)
    const float tau2 = lo - kLog2Inv255;
    uint32_t m = 0;
    const float det = a2 * c2 - 0.25f * b2 * b2;        // > 0 for a valid conic
    if (tau2 > 0.f && conic_cullable(a2, c2, det)) {
        const float t = tau2 * 1.002f + 1e-3f;
        const float inv = t / det;
        const float ex = sqrtf(fmaxf(-c2 * inv, 0.f)) + 0.02f;
        const float ey = sqrtf(fmaxf(-a2 * inv, 0.f)) + 0.02f;
        const float x0 = sx - ex, x1 = sx + ex, y0 = sy - ey, y1 = sy + ey;
        const uint32_t xb = ((x1 >= -7.5f && x0 <= -0.5f) ? 1u : 0u) | ((x1 >= 0.5f && x0 <= 7.5f) ? 2u : 0u);
        uint32_t yb = 0;
#pragma unroll
        for (int h = 0; h < 4; ++h) yb |= (y1 >= -7.5f + 4.f * h && y0 <= -4.5f + 4.f * h) ? (1u << h) : 0u;
#pragma unroll
        for (int w = 0; w < 8; ++w) m |= (((xb >> (w & 1)) & 1u) & ((yb >> (w >> 1)) & 1u)) << w;
    } else if (tau2 > 0.f) {
        m = 0xffu;                                      // degenerate or ill-conditioned conic: never cull
    }
    s.mask8 = m;
    return s;
}

// turn the per-splat 8-bit masks of one staging warp into 8 ballot words s_mask[w][word]
template <int WORDS>
__device__ __forceinline__ void publish_masks(uint32_t mask8, uint32_t (*s_mask)[WORDS], int word) {
    const int lane = threadIdx.x & 31;
    uint32_t mine = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        const uint32_t b = __ballot_sync(0xffffffffu, (mask8 >> w) & 1u);
        if (lane == w) mine = b;
    }
    if (lane < 8) s_mask[lane][word] = mine;
}

__global__ void __launch_bounds__(BLEND_THREADS, 6)
blend_fwd_kernel(const int2 *__restrict__ ranges, const uint32_t *__restrict__ point_list,
                 const float4 *__restrict__ rec, int W, int H, int gx, const float *__restrict__ bg,
                 float *__restrict__ out_color, float *__restrict__ final_T,
                 int32_t *__restrict__ n_contrib, const uint32_t *__restrict__ order) {
    __shared__ float4 s_k0[BLEND_BATCH];
    __shared__ float4 s_k1[BLEND_BATCH];
    __shared__ float s_b[BLEND_BATCH];
    __shared__ uint32_t s_mask[8][BLEND_WORDS];          // [patch warp][32 splats]
    const int tile = order ? (int)order[blockIdx.x] : (int)blockIdx.x;
    const int tile_x = tile % gx, tile_y = tile / gx;
    int px, py;
    float u, v;
    pixel_of_thread(tile_x, tile_y, px, py, u, v);
    const bool inside = px < W && py < H;
    const int2 range = ranges[tile];
    const float cx = (float)(tile_x * TILE) + 7.5f, cy = (float)(tile_y * TILE) + 7.5f;
    int todo = range.y - range.x;
    bool done = !inside;
    float T = 1.0f, C0 = 0.f, C1 = 0.f, C2 = 0.f;
    int last_contributor = 0;
    const int warp = threadIdx.x >> 5;

    for (int base = range.x; todo > 0; base += BLEND_BATCH, todo -= BLEND_BATCH) {
        if (__syncthreads_and(done)) break;
#pragma unroll
        for (int h = 0; h < 2; ++h) {                   // slot j = h * 256 + tid; its mask word = h * 8 + warp
            const int j = h * BLEND_THREADS + (int)threadIdx.x;
            uint32_t mask8 = 0;
            if (j < todo) {
                const uint32_t id = point_list[base + j];
                const float4 r0 = rec[3 * (size_t)id], r1 = rec[3 * (size_t)id + 1], r2 = rec[3 * (size_t)id + 2];
                const SplatCoef sc = splat_setup(r0.x - cx, r0.y - cy, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w);
                s_k0[j] = sc.k0; s_k1[j] = sc.k1; s_b[j] = r2.x;
                mask8 = sc.mask8;
            }
            publish_masks<BLEND_WORDS>(mask8, s_mask, h * 8 + warp);
        }
        __syncthreads();
        if (__all_sync(0xffffffffu, done)) continue;
        const int pos0 = base - range.x + 1;
        const int nwords = min(BLEND_WORDS, (todo + 31) >> 5);
#pragma unroll 1
        for (int word = 0; word < nwords; ++word) {
            uint32_t bits = s_mask[warp][word];
            while (bits) {
                const int j = word * 32 + __ffs(bits) - 1;
                bits &= bits - 1;
                const float4 k0 = s_k0[j];
                const float4 k1 = s_k1[j];
                float dx, dy;
                const float p2 = eval_p2(k0, k1.x, u, v, dx, dy);
                const float e = p2 + k1.y;
                // power > 0 (invalid conic) and alpha < 1/255 skips; `done` pixels take no part
                const bool live = !done && p2 <= 0.f && e >= kLog2Inv255;
                if (__any_sync(0xffffffffu, live)) {
                    if (live) {
                        const float alpha = fminf(0.99f, ex2_approx(e));
                        const float test_T = T * (1.0f - alpha);
                        if (test_T < 0.0001f) {
                            done = true;
                        } else {
                            const float w = alpha * T;
                            C0 = fmaf(k1.z, w, C0); C1 = fmaf(k1.w, w, C1); C2 = fmaf(s_b[j], w, C2);
                            T = test_T;
                            last_contributor = pos0 + j;
                        }
                    }
                    if (__all_sync(0xffffffffu, done)) { bits = 0; word = nwords; }
                }
            }
        }
    }
    if (inside) {
        const size_t pid = (size_t)py * W + px, HW = (size_t)H * W;
        final_T[pid] = T;
        n_contrib[pid] = last_contributor;
        out_color[pid] = C0 + T * bg[0];
        out_color[HW + pid] = C1 + T * bg[1];
        out_color[2 * HW + pid] = C2 + T * bg[2];
    }
}

// ---- forward, per-pixel candidate lists (v2) -----------------------------------------------------------
// The warp-synchronous walk above evaluates a splat on all 32 pixels of a patch as soon as its bounding box touches the
// patch; a census of the C2 view shows 14 of 32 lanes live per visit on average and 42 % of the (tile, splat) instances
// with no live pixel at all.  Here the staging thread solves, per splat and per pixel row of the tile, the quadratic
// alpha >= 1/255 for the column span [x0, x1] (conservatively widened; degenerate conics get the whole row), packs the
// spans into the 8 patch words of the splat and the staging warp transposes the [32 splats x 32 pixels] bit matrices with
// shuffles, so that every PIXEL owns, per 32-splat word, the bit list of the splats that may be live on it.  Each lane
// then walks its own list: different lanes of a warp evaluate different splats in the same step (the front-to-back
// order only binds per pixel, and the forward has no cross-lane reduction), which packs the lanes 74 % full instead of
// 45 %.  The lane still evaluates the exponent exactly as before from (dx, dy), so every skip decision -- and therefore
// the image, final_T and n_contrib -- is unchanged; the bit lists are only a superset filter.
__device__ __forceinline__ float sqrt_approx(float x) {
    float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
}
__device__ __forceinline__ uint32_t transpose32(uint32_t x) {        // lane p returns the word whose bit s is bit p of lane s's x
    const uint32_t lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const uint32_t lowmask = d == 16 ? 0x0000ffffu : d == 8 ? 0x00ff00ffu : d == 4 ? 0x0f0f0f0fu : d == 2 ? 0x33333333u : 0x55555555u;
        const uint32_t y = __shfl_xor_sync(0xffffffffu, x, d);
        const bool up = lane & d;
        const uint32_t keep = up ? ~lowmask : lowmask;
        const uint32_t t = up ? (y >> d) : (y << d);
        x = (x & keep) | (t & ~keep);
    }
    return x;
}

// 8 patch words (bit ly*8+lx of word w = pixel (lx, ly) of patch w) of the pixels on which the splat can reach alpha >= 1/255
__device__ __forceinline__ void splat_patch_words(float sx, float sy, float a2, float b2, float c2, float lo, uint32_t (&pm)[8]) {
    const float tau2 = lo - kLog2Inv255;
    const float det = a2 * c2 - 0.25f * b2 * b2;
    uint32_t rows2[8];                                   // row masks, two 16-bit rows per word
    if (!(tau2 > 0.f)) {
#pragma unroll
        for (int w = 0; w < 8; ++w) pm[w] = 0;
        return;
    }
    if (conic_cullable(a2, c2, det) && a2 < 0.f) {
        const float t = tau2 * 1.002f + 1e-3f;
        const float inv_a = rcp_approx(-a2);             // 1 / alpha, alpha = -a2 > 0
        const float at = -a2 * t;
        const float kb = -0.5f * b2 * inv_a;             // span centre: dx_c = -kb * dy, column u_c = sx - dx_c
        const float sy8 = sy + 7.5f, sx8 = sx + 7.5f;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const float dy = sy8 - (float)r;
            const float q = fmaf(-det, dy * dy, at);     // alpha t - det dy^2 (< 0: the row misses the ellipse)
            const float hw = fmaf(sqrt_approx(fmaxf(q, 0.f)), inv_a, 0.02f);
            const float uc = fmaf(kb, dy, sx8);          // span centre in column units
            const int k0 = max(0, __float2int_ru(uc - hw)), k1 = min(15, __float2int_rd(uc + hw));
            const uint32_t m = (q >= 0.f && k1 >= k0) ? (2u << k1) - (1u << k0) : 0u;
            if (r & 1) rows2[r >> 1] |= m << 16; else rows2[r >> 1] = m;
        }
    } else {
#pragma unroll
        for (int w = 0; w < 8; ++w) rows2[w] = 0xffffffffu;       // degenerate or ill-conditioned conic: never cull
    }
#pragma unroll
    for (int yq = 0; yq < 4; ++yq) {                    // rows 4yq..4yq+3: low bytes -> left patch, high bytes -> right patch
        pm[2 * yq] = __byte_perm(rows2[2 * yq], rows2[2 * yq + 1], 0x6420);
        pm[2 * yq + 1] = __byte_perm(rows2[2 * yq], rows2[2 * yq + 1], 0x7531);
    }
}

//
// DA (depth / alpha maps): the view-space depth z of each staged splat rides next to its blue channel (one float2 load
// per live pair instead of one float), D = sum z alpha T is accumulated like a fourth colour channel with background 0,
// and the kernel also writes depth[pid] = D and alpha[pid] = 1 - T.  Same walk, same decisions: colour, final_T and
// n_contrib are those of blend_fwd2_kernel<false>.
template <bool DA>
__global__ void __launch_bounds__(BLEND_THREADS, 5)
blend_fwd2_kernel(const int2 *__restrict__ ranges, const uint32_t *__restrict__ point_list,
                  const float4 *__restrict__ rec, int W, int H, int gx, const float *__restrict__ bg,
                  float *__restrict__ out_color, float *__restrict__ final_T,
                  int32_t *__restrict__ n_contrib, const uint32_t *__restrict__ order,
                  float *__restrict__ out_depth = nullptr, float *__restrict__ out_alpha = nullptr) {
    using BZ = std::conditional_t<DA, float2, float>;           // blue (and z)
    __shared__ float4 s_k0[BLEND_BATCH];
    __shared__ float4 s_k1[BLEND_BATCH];
    __shared__ BZ s_b[BLEND_BATCH];
    __shared__ uint32_t s_cand[BLEND_WORDS][BLEND_THREADS];      // [32-splat word][pixel thread]
    const int tile = order ? (int)order[blockIdx.x] : (int)blockIdx.x;
    const int tile_x = tile % gx, tile_y = tile / gx;
    int px, py;
    float u, v;
    pixel_of_thread(tile_x, tile_y, px, py, u, v);
    const bool inside = px < W && py < H;
    const int2 range = ranges[tile];
    const float cx = (float)(tile_x * TILE) + 7.5f, cy = (float)(tile_y * TILE) + 7.5f;
    int todo = range.y - range.x;
    bool done = !inside;
    float T = 1.0f, C0 = 0.f, C1 = 0.f, C2 = 0.f, D = 0.f;
    int last_contributor = 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    for (int base = range.x; todo > 0; base += BLEND_BATCH, todo -= BLEND_BATCH) {
        if (__syncthreads_and(done)) break;
#pragma unroll
        for (int h = 0; h < 2; ++h) {                   // slot j = h * 256 + tid is bit `lane` of word h * 8 + warp
            const int j = h * BLEND_THREADS + (int)threadIdx.x;
            uint32_t pm[8];
#pragma unroll
            for (int w = 0; w < 8; ++w) pm[w] = 0;
            if (j < todo) {
                const uint32_t id = point_list[base + j];
                const float4 r0 = rec[3 * (size_t)id], r1 = rec[3 * (size_t)id + 1], r2 = rec[3 * (size_t)id + 2];
                const float sx = r0.x - cx, sy = r0.y - cy;
                const float a2 = -0.5f * kLog2e * r0.z, c2 = -0.5f * kLog2e * r1.x, b2 = -kLog2e * r0.w;
                const float lo = r1.y > 0.f ? __log2f(r1.y) : -1e30f;
                s_k0[j] = make_float4(sx, sy, a2, b2); s_k1[j] = make_float4(c2, lo, r1.z, r1.w);
                if constexpr (DA) s_b[j] = make_float2(r2.x, r2.y); else s_b[j] = r2.x;
                splat_patch_words(sx, sy, a2, b2, c2, lo, pm);
            }
#pragma unroll
            for (int w = 0; w < 8; ++w) s_cand[h * 8 + warp][w * 32 + lane] = transpose32(pm[w]);
        }
        __syncthreads();
        if (!done) {
            uint32_t summ = 0;                          // words with a candidate for this pixel
#pragma unroll
            for (int w = 0; w < BLEND_WORDS; ++w) summ |= (s_cand[w][threadIdx.x] != 0u ? 1u : 0u) << w;
            const int pos0 = base - range.x + 1;
            uint32_t bits = 0;
            int wbase = 0;
            while (true) {
                {                                       // next non-empty word when this one is used up (branch-free: the
                    const int w = (__ffs(summ) - 1) & (BLEND_WORDS - 1);      // load is harmless when it is not needed)
                    const uint32_t nb = s_cand[w][threadIdx.x];
                    if (bits == 0) {
                        if (summ == 0) break;
                        bits = nb; wbase = w * 32; summ &= summ - 1;
                    }
                }
                const int j = wbase + __ffs(bits) - 1;
                bits &= bits - 1;
                const float4 k0 = s_k0[j];
                const float4 k1 = s_k1[j];
                float dx, dy;
                const float p2 = eval_p2(k0, k1.x, u, v, dx, dy);
                const float e = p2 + k1.y;
                if (p2 <= 0.f && e >= kLog2Inv255) {    // power > 0 (invalid conic) and alpha < 1/255 skip
                    const float alpha = fminf(0.99f, ex2_approx(e));
                    const float test_T = T * (1.0f - alpha);
                    if (test_T < 0.0001f) { done = true; break; }
                    const float wgt = alpha * T;
                    if constexpr (DA) {
                        const float2 bz = s_b[j];
                        C0 = fmaf(k1.z, wgt, C0); C1 = fmaf(k1.w, wgt, C1); C2 = fmaf(bz.x, wgt, C2);
                        D = fmaf(bz.y, wgt, D);
                    } else {
                        C0 = fmaf(k1.z, wgt, C0); C1 = fmaf(k1.w, wgt, C1); C2 = fmaf(s_b[j], wgt, C2);
                    }
                    T = test_T;
                    last_contributor = pos0 + j;
                }
            }
        }
    }
    if (inside) {
        const size_t pid = (size_t)py * W + px, HW = (size_t)H * W;
        final_T[pid] = T;
        n_contrib[pid] = last_contributor;
        out_color[pid] = C0 + T * bg[0];
        out_color[HW + pid] = C1 + T * bg[1];
        out_color[2 * HW + pid] = C2 + T * bg[2];
        if constexpr (DA) {
            out_depth[pid] = D;
            out_alpha[pid] = 1.0f - T;
        }
    }
}

// ---- backward ---------------------------------------------------------------------------------------
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ float2 lds64(uint32_t a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
    return v;
}

// Staged splat record of the backward: 48 bytes = 3 x float4  (the conic itself is recovered from its log2-domain
// form at flush time: A = a2 * (-2 / log2 e), B = -b2 / log2 e, C = c2 * (-2 / log2 e))
//   [0] sx, sy, a2, b2   [1] c2, log2(op), r, g   [2] b, id(bits), 1/opacity, 0
//
// Per (pixel, splat) pair the lanes only form the six moments of D = dL/dG * G about the splat centre
// (D, D dx, D dy, D dx^2, D dx dy, D dy^2) and the three colour terms; D = dL/dalpha * ex2(e) because
// o * G = ex2(p2 + log2 o) is the (unclamped) alpha the forward exponent already gives.  The conic / opacity
// factors of the reference's per-pixel formulas are per-splat constants, so they are applied ONCE per
// (warp, splat) after the warp reduction, by the lanes that own the reduced sums:
//   dmean2D.x = -0.5 W (A Sx + B Sy)   dmean2D.y = -0.5 H (C Sy + B Sx)
//   dconic    = -0.5 (Sxx, Sxy, Syy)   dopacity  = S / o   dcolour = (c0, c1, c2)
__global__ void __launch_bounds__(BLEND_THREADS)
blend_bwd_kernel(const int2 *__restrict__ ranges, const uint32_t *__restrict__ point_list,
                 const float4 *__restrict__ rec, int W, int H, int gx, const float *__restrict__ bg,
                 const float *__restrict__ final_T, const int32_t *__restrict__ n_contrib,
                 const float *__restrict__ dL_dpix, float *__restrict__ dL_dmean2D,
                 float *__restrict__ dL_dconic, float *__restrict__ dL_dopacity,
                 float *__restrict__ dL_dcolor, const uint32_t *__restrict__ order) {
    // dynamic shared memory (BWD_SMEM bytes): the staged records, then the per-warp transposition buffers of the
    // gradient partials: RB_SLOTS buffered (warp, splat) visits x 9 sums x 32 lanes, rows padded to 36 floats so
    // that both the lane-wise stores and the row-wise 16-byte loads are bank-conflict free
    extern __shared__ float4 s_dyn4[];
    float4 *const s_rec = s_dyn4;                                             // [BLEND_BATCH * 3]
    float *const s_buf_all = reinterpret_cast<float *>(s_dyn4 + BLEND_BATCH * 3);   // [8][RB_ROWS * RB_STRIDE]
    __shared__ uint32_t s_mask[8][BLEND_WORDS];
    __shared__ int s_max[BLEND_THREADS / 32];
    __shared__ int s_meta[BLEND_THREADS / 32][RB_SLOTS];
    const int tile = order ? (int)order[blockIdx.x] : (int)blockIdx.x;
    const int tile_x = tile % gx, tile_y = tile / gx;
    int px, py;
    float u, v;
    pixel_of_thread(tile_x, tile_y, px, py, u, v);
    const bool inside = px < W && py < H;
    const float cx = (float)(tile_x * TILE) + 7.5f, cy = (float)(tile_y * TILE) + 7.5f;
    const int2 range = ranges[tile];
    const size_t pid = (size_t)py * W + px, HW = (size_t)H * W;
    const float T_final = inside ? final_T[pid] : 0.f;
    const int last = inside ? n_contrib[pid] : 0;
    float T = T_final;
    float dp0 = 0.f, dp1 = 0.f, dp2 = 0.f;
    if (inside) { dp0 = dL_dpix[pid]; dp1 = dL_dpix[HW + pid]; dp2 = dL_dpix[2 * HW + pid]; }
    const float neg_Tf_bg = -T_final * (bg[0] * dp0 + bg[1] * dp1 + bg[2] * dp2);
    float ar0 = 0.f, ar1 = 0.f, ar2 = 0.f, lc0 = 0.f, lc1 = 0.f, lc2 = 0.f, last_alpha = 0.f;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t a_rec = (uint32_t)__cvta_generic_to_shared(s_rec);
    float *const buf = s_buf_all + warp * (RB_ROWS * RB_STRIDE);

    // deepest contributor over the tile: nothing behind it receives gradient
    const int warp_last = __reduce_max_sync(0xffffffffu, last);
    if (lane == 0) s_max[warp] = warp_last;
    __syncthreads();
    int tile_last = 0;
#pragma unroll
    for (int w = 0; w < BLEND_THREADS / 32; ++w) tile_last = max(tile_last, s_max[w]);

    // Flush role of this lane: row = lane of the buffer = (slot, sum kind).  kind: 0 S, 1 Sx, 2 Sy, 3 Sxx, 4 Sxy, 5 Syy,
    // 6..8 colour.  Destination rows have stride 3 (mean2D, conic, colour) or 1 (opacity).
    const int f_slot = lane / 9, f_kind = lane - 9 * f_slot;
    const float half_w = -0.5f * (float)W, half_h = -0.5f * (float)H;
    int nbuf = 0;                                     // buffered visits (warp-uniform)

    auto flush = [&]() {
        __syncwarp();
        if (lane < RB_ROWS && f_slot < nbuf) {
            const float4 *row = reinterpret_cast<const float4 *>(buf + lane * RB_STRIDE);
            float4 acc = row[0];
#pragma unroll
            for (int q = 1; q < 8; ++q) { const float4 t = row[q]; acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w; }
            const float sum = (acc.x + acc.y) + (acc.z + acc.w);
            if (sum != 0.f) {
                const uint32_t addr = a_rec + (uint32_t)s_meta[warp][f_slot] * 48u;
                const float4 q2 = lds128(addr + 32);                       // b, id, 1/opacity, -
                const uint32_t id = __float_as_uint(q2.y);
                if (f_kind == 0) atomicAdd(dL_dopacity + id, sum * q2.z);
                else if (f_kind < 3) {
                    const float4 q0 = lds128(addr);                        // sx, sy, a2, b2
                    const float conA = q0.z * (-2.0f / kLog2e), conB = q0.w * (-1.0f / kLog2e);
                    const float conC = lds128(addr + 16).x * (-2.0f / kLog2e);
                    if (f_kind == 1) { atomicAdd(dL_dmean2D + 3u * id, half_w * conA * sum); atomicAdd(dL_dmean2D + 3u * id + 1, half_h * conB * sum); }
                    else { atomicAdd(dL_dmean2D + 3u * id, half_w * conB * sum); atomicAdd(dL_dmean2D + 3u * id + 1, half_h * conC * sum); }
                }
                else if (f_kind < 6) atomicAdd(dL_dconic + 3u * id + (f_kind - 3), -0.5f * sum);
                else atomicAdd(dL_dcolor + 3u * id + (f_kind - 6), sum);
            }
        }
        __syncwarp();
        nbuf = 0;
    };

    // walk positions tile_last-1 .. 0 in batches, back to front; slot j holds position hi-1-j
    for (int hi = tile_last; hi > 0; hi -= BLEND_BATCH) {
        const int nb = min(BLEND_BATCH, hi);
        __syncthreads();                        // every warp is done with the previous batch (and has flushed)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int j = h * BLEND_THREADS + (int)threadIdx.x;
            uint32_t mask8 = 0;
            if (j < nb) {
                const uint32_t id = point_list[range.x + hi - 1 - j];
                const float4 r0 = rec[3 * (size_t)id], r1 = rec[3 * (size_t)id + 1], r2 = rec[3 * (size_t)id + 2];
                const float sx = r0.x - cx, sy = r0.y - cy;
                const SplatCoef sc = splat_setup(sx, sy, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w);
                s_rec[3 * j] = sc.k0; s_rec[3 * j + 1] = sc.k1;
                s_rec[3 * j + 2] = make_float4(r2.x, __uint_as_float(id), r1.y > 0.f ? 1.0f / r1.y : 0.f, 0.f);
                mask8 = sc.mask8;
            }
            publish_masks<BLEND_WORDS>(mask8, s_mask, h * 8 + warp);
        }
        __syncthreads();
        // slots whose position is at or behind this warp's deepest contributor cannot receive gradient:
        // position = hi-1-j >= warp_last  <=>  j < hi - warp_last
        const int skip = hi - warp_last;
        const int nwords = (nb + 31) >> 5;
#pragma unroll 1
        for (int word = 0; word < nwords; ++word) {
            uint32_t bits = s_mask[warp][word];
            const int lo = word * 32;
            if (skip >= lo + 32) bits = 0;
            else if (skip > lo) bits &= ~((1u << (skip - lo)) - 1u);
            while (bits) {
                const int j = lo + __ffs(bits) - 1;
                bits &= bits - 1;
                const uint32_t addr = a_rec + (uint32_t)j * 48u;
                const float4 k0 = lds128(addr);
                const float4 k1 = lds128(addr + 16);
                float dx, dy;
                const float p2 = eval_p2(k0, k1.x, u, v, dx, dy);
                const float e = p2 + k1.y;
                const bool live = (hi - 1 - j) < last && p2 <= 0.f && e >= kLog2Inv255;   // same decisions as the forward
                if (!__any_sync(0xffffffffu, live)) continue;
                float gS = 0.f, gx_ = 0.f, gy_ = 0.f, gxx = 0.f, gxy = 0.f, gyy = 0.f, gc0 = 0.f, gc1 = 0.f, gc2 = 0.f;
                if (live) {
                    const float au = ex2_approx(e);            // o * G
                    const float alpha = fminf(0.99f, au);
                    const float rcp = rcp_approx(1.0f - alpha);         // 1 - alpha >= 0.01
                    T *= rcp;
                    const float dch = alpha * T;
                    const float c0 = k1.z, c1 = k1.w, c2 = lds64(addr + 32).x;
                    const float om = 1.f - last_alpha;
                    ar0 = fmaf(last_alpha, lc0, om * ar0); lc0 = c0;
                    ar1 = fmaf(last_alpha, lc1, om * ar1); lc1 = c1;
                    ar2 = fmaf(last_alpha, lc2, om * ar2); lc2 = c2;
                    float dL_dalpha = ((c0 - ar0) * dp0 + (c1 - ar1) * dp1 + (c2 - ar2) * dp2) * T;
                    last_alpha = alpha;
                    dL_dalpha = fmaf(neg_Tf_bg, rcp, dL_dalpha);
                    gS = dL_dalpha * au;                       // D = dL/dG * G
                    gx_ = gS * dx; gy_ = gS * dy;
                    gxx = gx_ * dx; gxy = gx_ * dy; gyy = gy_ * dy;
                    gc0 = dch * dp0; gc1 = dch * dp1; gc2 = dch * dp2;
                }
                // park the 9 partials of this visit in the warp's buffer (column = lane); the sums over the 32 lanes are
                // taken row-wise, RB_SLOTS visits at a time, by flush()
                float *col = buf + nbuf * 9 * RB_STRIDE + lane;
                col[0 * RB_STRIDE] = gS; col[1 * RB_STRIDE] = gx_; col[2 * RB_STRIDE] = gy_;
                col[3 * RB_STRIDE] = gxx; col[4 * RB_STRIDE] = gxy; col[5 * RB_STRIDE] = gyy;
                col[6 * RB_STRIDE] = gc0; col[7 * RB_STRIDE] = gc1; col[8 * RB_STRIDE] = gc2;
                if (lane == 0) s_meta[warp][nbuf] = j;
                if (++nbuf == RB_SLOTS) flush();
            }
        }
        if (nbuf) flush();                      // the records of this batch are about to be overwritten
    }
}


// ---- backward, matrix-form reduction (v2) -------------------------------------------------------------
// Same walk, same skip decisions and the same per-pixel recurrences as blend_bwd_kernel; only the reduction over the
// 32 pixels of a patch differs.  Every one of the nine per-(patch, splat) sums is  sum_lanes x_lane * w_lane,k  with
// just two per-visit lane values -- x = D (= dL/dG * G) for the six geometric sums, x = alpha * T for the three colour
// sums -- and lane weights that are CONSTANT over the whole kernel: the monomials {1, u, v, u^2, uv, v^2} of the
// lane's patch-centred pixel coordinates (compile-time constants once unrolled) and the pixel's dL/dpixel.  So a lane
// parks two floats per visit (not nine); 16 visits form a [16 x 32] matrix per value, and at flush time lane (r, h)
// takes the 16 columns of pixel rows 2h, 2h+1 of visit r with 16-byte loads (rows padded to 36 floats: conflict-free),
// forms the partial moments with constant-weight FMAs (row-factored: 3 sums per pixel row, combined with v, v^2), the
// colour dot products against the patch's dL/dpixel table, and one xor-16 exchange completes the nine sums.  The
// epilogue turns the raw pixel moments into the moments about the splat centre (S_x = sx S - S_u, ...) and issues the
// global REDs, once per (warp, splat) like before.  (An mma.sync variant of this flush -- 2xTF32 / 3xTF32 -- was
// measured 13 % slower than the transposition-buffer kernel: the legacy tensor path is slow on sm_100a.)
//
// DA (depth / alpha maps): depth is a fourth colour channel with background 0 and alpha = 1 - T_final.  The staged
// record carries z in its free slot [2].w; the lane keeps one more suffix recurrence (ar3 / lc3) and adds
// (z - ar3) T g_D to dL/dalpha; the alpha map's gradient g_A enters through the per-pixel constant:
// d(1 - T_final)/dalpha_i = T_final / (1 - alpha_i), so neg_Tf_bg = -T_final (bg . dL/dpix - g_A).  dL/dz of a splat is
// sum_pixels alpha T g_D: one more constant-weight dot product of the parked alpha T column against a fourth row
// (g_D) of the patch's dL/dpixel table, issued by the fh == 0 half of the flush.
constexpr int MR_ROWS = 16, MR_STRIDE = 36;
constexpr int MR_WARP_FLOATS = 2 * MR_ROWS * MR_STRIDE + 3 * 32 + MR_ROWS;     // X_g, X_d, dL/dpixel table, slot of each row
template <bool DA> constexpr int kMrWarpFloats = DA ? MR_WARP_FLOATS + 32 : MR_WARP_FLOATS;   // + g_D row
template <int BATCH, bool DA = false> constexpr size_t bwd2_smem() {
    return (size_t)BATCH * 48 + (size_t)(BLEND_THREADS / 32) * kMrWarpFloats<DA> * sizeof(float);
}

template <int BATCH, bool DA>
__global__ void __launch_bounds__(BLEND_THREADS, BATCH == 256 ? 4 : 3)
blend_bwd2_kernel(const int2 *__restrict__ ranges, const uint32_t *__restrict__ point_list,
                  const float4 *__restrict__ rec, int W, int H, int gx, const float *__restrict__ bg,
                  const float *__restrict__ final_T, const int32_t *__restrict__ n_contrib,
                  const float *__restrict__ dL_dpix, float *__restrict__ dL_dmean2D,
                  float *__restrict__ dL_dconic, float *__restrict__ dL_dopacity,
                  float *__restrict__ dL_dcolor, const uint32_t *__restrict__ order,
                  const float *__restrict__ dL_ddmap = nullptr, const float *__restrict__ dL_damap = nullptr,
                  float *__restrict__ dL_ddepth = nullptr) {
    constexpr int WORDS = BATCH / 32, PER_THREAD = BATCH / BLEND_THREADS;
    extern __shared__ float4 s_dyn4[];
    float4 *const s_rec = s_dyn4;                                                   // [BATCH * 3]
    float *const s_buf_all = reinterpret_cast<float *>(s_dyn4 + BATCH * 3);         // [8][kMrWarpFloats<DA>]
    __shared__ uint32_t s_mask[8][WORDS];
    __shared__ int s_max[BLEND_THREADS / 32];
    const int tile = order ? (int)order[blockIdx.x] : (int)blockIdx.x;
    const int tile_x = tile % gx, tile_y = tile / gx;
    int px, py;
    float u, v;
    pixel_of_thread(tile_x, tile_y, px, py, u, v);
    const bool inside = px < W && py < H;
    const float cx = (float)(tile_x * TILE) + 7.5f, cy = (float)(tile_y * TILE) + 7.5f;
    const int2 range = ranges[tile];
    const size_t pid = (size_t)py * W + px, HW = (size_t)H * W;
    const float T_final = inside ? final_T[pid] : 0.f;
    const int last = inside ? n_contrib[pid] : 0;
    float T = T_final;
    float dp0 = 0.f, dp1 = 0.f, dp2 = 0.f;
    float neg_Tf_bg, gD = 0.f;
    if constexpr (DA) {
        // any of the three upstream maps may be absent (NULL = zero)
        float gA = 0.f;
        if (inside) {
            if (dL_dpix) { dp0 = dL_dpix[pid]; dp1 = dL_dpix[HW + pid]; dp2 = dL_dpix[2 * HW + pid]; }
            if (dL_ddmap) gD = dL_ddmap[pid];
            if (dL_damap) gA = dL_damap[pid];
        }
        neg_Tf_bg = -T_final * ((bg[0] * dp0 + bg[1] * dp1 + bg[2] * dp2) - gA);
    } else {
        if (inside) { dp0 = dL_dpix[pid]; dp1 = dL_dpix[HW + pid]; dp2 = dL_dpix[2 * HW + pid]; }
        neg_Tf_bg = -T_final * (bg[0] * dp0 + bg[1] * dp1 + bg[2] * dp2);
    }
    float ar0 = 0.f, ar1 = 0.f, ar2 = 0.f, lc0 = 0.f, lc1 = 0.f, lc2 = 0.f, last_alpha = 0.f;
    float ar3 = 0.f, lc3 = 0.f;                                // depth channel (DA only)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t a_rec = (uint32_t)__cvta_generic_to_shared(s_rec);
    float *const xg = s_buf_all + warp * kMrWarpFloats<DA>;
    float *const xd = xg + MR_ROWS * MR_STRIDE;
    float *const wc = xd + MR_ROWS * MR_STRIDE;                // [3][32] dL/dpixel of the patch (DA: [4][32], + g_D)
    int *const meta = reinterpret_cast<int *>(wc + (DA ? 128 : 96));   // [MR_ROWS] staged slot of each parked visit
    wc[lane] = dp0; wc[32 + lane] = dp1; wc[64 + lane] = dp2;
    if constexpr (DA) wc[96 + lane] = gD;

    const int warp_last = __reduce_max_sync(0xffffffffu, last);
    if (lane == 0) s_max[warp] = warp_last;
    __syncthreads();
    int tile_last = 0;
#pragma unroll
    for (int w = 0; w < BLEND_THREADS / 32; ++w) tile_last = max(tile_last, s_max[w]);

    // flush roles of this lane: parked visit fr, pixel rows 2 fh, 2 fh + 1 of the patch
    const int fr = lane & 15, fh = lane >> 4;
    const float fv0 = (float)(2 * fh) - 1.5f;
    const float pcx = (float)((warp & 1) * 8 - 4), pcy = (float)((warp >> 1) * 4 - 6);   // patch centre - tile centre
    const float half_w = -0.5f * (float)W, half_h = -0.5f * (float)H;
    const uint32_t a_rowg = (uint32_t)__cvta_generic_to_shared(xg) + (uint32_t)(fr * MR_STRIDE + 16 * fh) * 4u;
    const uint32_t a_rowd = (uint32_t)__cvta_generic_to_shared(xd) + (uint32_t)(fr * MR_STRIDE + 16 * fh) * 4u;
    const uint32_t a_wrow = (uint32_t)__cvta_generic_to_shared(wc) + (uint32_t)(16 * fh) * 4u;
    int nbuf = 0;                                     // parked visits (warp-uniform)

    auto flush = [&]() {
        __syncwarp();
        // lane (fr, fh): visit row fr, pixel rows 2 fh and 2 fh + 1 of the patch (source lanes 16 fh .. 16 fh + 15)
        float S = 0.f, Su = 0.f, Sv = 0.f, Suu = 0.f, Suv = 0.f, Svv = 0.f, C0 = 0.f, C1 = 0.f, C2 = 0.f, C3 = 0.f;
#pragma unroll
        for (int y = 0; y < 2; ++y) {
            const float4 g0 = lds128(a_rowg + 32u * y), g1 = lds128(a_rowg + 32u * y + 16);
            const float4 d0 = lds128(a_rowd + 32u * y), d1 = lds128(a_rowd + 32u * y + 16);
            const float xs[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
            const float ds[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
            float r0 = 0.f, r1 = 0.f, r2 = 0.f;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float uc = (float)c - 3.5f;
                r0 += xs[c]; r1 = fmaf(xs[c], uc, r1); r2 = fmaf(xs[c], uc * uc, r2);
            }
            const float vy = fv0 + (float)y;
            S += r0; Su += r1; Suu += r2;
            Sv = fmaf(vy, r0, Sv); Suv = fmaf(vy, r1, Suv); Svv = fmaf(vy * vy, r0, Svv);
#pragma unroll
            for (int k = 0; k < (DA ? 4 : 3); ++k) {
                const float4 w0 = lds128(a_wrow + 128u * k + 32u * y), w1 = lds128(a_wrow + 128u * k + 32u * y + 16);
                float acc = ds[0] * w0.x;
                acc = fmaf(ds[1], w0.y, acc); acc = fmaf(ds[2], w0.z, acc); acc = fmaf(ds[3], w0.w, acc);
                acc = fmaf(ds[4], w1.x, acc); acc = fmaf(ds[5], w1.y, acc); acc = fmaf(ds[6], w1.z, acc); acc = fmaf(ds[7], w1.w, acc);
                if (k == 0) C0 += acc; else if (k == 1) C1 += acc; else if (k == 2) C2 += acc; else C3 += acc;
            }
        }
        S += __shfl_xor_sync(0xffffffffu, S, 16); Su += __shfl_xor_sync(0xffffffffu, Su, 16); Sv += __shfl_xor_sync(0xffffffffu, Sv, 16);
        Suu += __shfl_xor_sync(0xffffffffu, Suu, 16); Suv += __shfl_xor_sync(0xffffffffu, Suv, 16); Svv += __shfl_xor_sync(0xffffffffu, Svv, 16);
        C0 += __shfl_xor_sync(0xffffffffu, C0, 16); C1 += __shfl_xor_sync(0xffffffffu, C1, 16); C2 += __shfl_xor_sync(0xffffffffu, C2, 16);
        if constexpr (DA) C3 += __shfl_xor_sync(0xffffffffu, C3, 16);
        if (fr < nbuf) {
            const uint32_t addr = a_rec + (uint32_t)meta[fr] * 48u;
            const float4 r0 = lds128(addr);                            // sx, sy, a2, b2
            const float4 r2 = lds128(addr + 32);                       // b, id, 1/opacity, -
            const uint32_t id = __float_as_uint(r2.y);
            const float sxp = r0.x - pcx, syp = r0.y - pcy;
            const float Sx = fmaf(sxp, S, -Su), Sy = fmaf(syp, S, -Sv);      // moments about the splat centre
            if (fh == 0) {
                const float conA = r0.z * (-2.0f / kLog2e), conB = r0.w * (-1.0f / kLog2e);
                const float conC = lds128(addr + 16).x * (-2.0f / kLog2e);
                const float a = S * r2.z, b = half_w * fmaf(conA, Sx, conB * Sy), c = half_h * fmaf(conC, Sy, conB * Sx);
                const float d = -0.5f * fmaf(sxp, Sx - Su, Suu);
                if (a != 0.f) atomicAdd(dL_dopacity + id, a);
                if (b != 0.f) atomicAdd(dL_dmean2D + 3u * id, b);
                if (c != 0.f) atomicAdd(dL_dmean2D + 3u * id + 1, c);
                if (d != 0.f) atomicAdd(dL_dconic + 3u * id, d);
                if constexpr (DA) { if (C3 != 0.f) atomicAdd(dL_ddepth + id, C3); }
            } else {
                const float a = -0.5f * (fmaf(sxp, Sy, Suv) - syp * Su), b = -0.5f * fmaf(syp, Sy - Sv, Svv);
                if (a != 0.f) atomicAdd(dL_dconic + 3u * id + 1, a);
                if (b != 0.f) atomicAdd(dL_dconic + 3u * id + 2, b);
                if (C0 != 0.f) atomicAdd(dL_dcolor + 3u * id, C0);
                if (C1 != 0.f) atomicAdd(dL_dcolor + 3u * id + 1, C1);
                if (C2 != 0.f) atomicAdd(dL_dcolor + 3u * id + 2, C2);
            }
        }
        __syncwarp();
        nbuf = 0;
    };

    // walk positions tile_last-1 .. 0 in batches, back to front; slot j holds position hi-1-j
    for (int hi = tile_last; hi > 0; hi -= BATCH) {
        const int nb = min(BATCH, hi);
        __syncthreads();                        // every warp is done with the previous batch (and has flushed)
#pragma unroll
        for (int h = 0; h < PER_THREAD; ++h) {
            const int j = h * BLEND_THREADS + (int)threadIdx.x;
            uint32_t mask8 = 0;
            if (j < nb) {
                const uint32_t id = point_list[range.x + hi - 1 - j];
                const float4 r0 = rec[3 * (size_t)id], r1 = rec[3 * (size_t)id + 1], r2 = rec[3 * (size_t)id + 2];
                const float sx = r0.x - cx, sy = r0.y - cy;
                const SplatCoef sc = splat_setup(sx, sy, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w);
                s_rec[3 * j] = sc.k0; s_rec[3 * j + 1] = sc.k1;
                s_rec[3 * j + 2] = make_float4(r2.x, __uint_as_float(id), r1.y > 0.f ? 1.0f / r1.y : 0.f, DA ? r2.y : 0.f);
                mask8 = sc.mask8;
            }
            publish_masks<WORDS>(mask8, s_mask, h * 8 + warp);
        }
        __syncthreads();
        const int skip = hi - warp_last;
        const int nwords = (nb + 31) >> 5;
#pragma unroll 1
        for (int word = 0; word < nwords; ++word) {
            uint32_t bits = s_mask[warp][word];
            const int lo = word * 32;
            if (skip >= lo + 32) bits = 0;
            else if (skip > lo) bits &= ~((1u << (skip - lo)) - 1u);
            while (bits) {
                const int j = lo + __ffs(bits) - 1;
                bits &= bits - 1;
                const uint32_t addr = a_rec + (uint32_t)j * 48u;
                const float4 k0 = lds128(addr);
                const float4 k1 = lds128(addr + 16);
                float dx, dy;
                const float p2 = eval_p2(k0, k1.x, u, v, dx, dy);
                const float e = p2 + k1.y;
                const bool live = (hi - 1 - j) < last && p2 <= 0.f && e >= kLog2Inv255;   // same decisions as the forward
                if (!__any_sync(0xffffffffu, live)) continue;
                float gS = 0.f, dch = 0.f;
                if (live) {
                    const float au = ex2_approx(e);            // o * G
                    const float alpha = fminf(0.99f, au);
                    const float rcp = rcp_approx(1.0f - alpha);         // 1 - alpha >= 0.01
                    T *= rcp;
                    dch = alpha * T;
                    float dL_dalpha;
                    if constexpr (DA) {
                        const float4 q2 = lds128(addr + 32);           // b, id, 1/opacity, z
                        const float c0 = k1.z, c1 = k1.w, c2 = q2.x, c3 = q2.w;
                        const float om = 1.f - last_alpha;
                        ar0 = fmaf(last_alpha, lc0, om * ar0); lc0 = c0;
                        ar1 = fmaf(last_alpha, lc1, om * ar1); lc1 = c1;
                        ar2 = fmaf(last_alpha, lc2, om * ar2); lc2 = c2;
                        ar3 = fmaf(last_alpha, lc3, om * ar3); lc3 = c3;
                        dL_dalpha = ((c0 - ar0) * dp0 + (c1 - ar1) * dp1 + (c2 - ar2) * dp2 + (c3 - ar3) * gD) * T;
                    } else {
                        const float c0 = k1.z, c1 = k1.w, c2 = lds64(addr + 32).x;
                        const float om = 1.f - last_alpha;
                        ar0 = fmaf(last_alpha, lc0, om * ar0); lc0 = c0;
                        ar1 = fmaf(last_alpha, lc1, om * ar1); lc1 = c1;
                        ar2 = fmaf(last_alpha, lc2, om * ar2); lc2 = c2;
                        dL_dalpha = ((c0 - ar0) * dp0 + (c1 - ar1) * dp1 + (c2 - ar2) * dp2) * T;
                    }
                    last_alpha = alpha;
                    dL_dalpha = fmaf(neg_Tf_bg, rcp, dL_dalpha);
                    gS = dL_dalpha * au;                       // D = dL/dG * G
                }
                xg[nbuf * MR_STRIDE + lane] = gS;
                xd[nbuf * MR_STRIDE + lane] = dch;
                if (lane == 0) meta[nbuf] = j;
                if (++nbuf == MR_ROWS) flush();
            }
        }
        if (nbuf) flush();                      // the records of this batch are about to be overwritten
    }
}


}  // namespace splatco

using namespace splatco;

// implementation switches (splatco_blend_set_impl / SPLATCO_BLEND_FWD / SPLATCO_BLEND_BWD); see the header
static int g_blend_impl[2] = {0, 0};
static int blend_impl(int which) {
    if (!g_blend_impl[which]) {
        const char *e = getenv(which ? "SPLATCO_BLEND_BWD" : "SPLATCO_BLEND_FWD");
        const int v = e ? atoi(e) : 0, hi = which ? 3 : 2, def = 2;
        g_blend_impl[which] = (v >= 1 && v <= hi) ? v : def;
    }
    return g_blend_impl[which];
}
extern "C" int splatco_blend_set_impl(int fwd, int bwd) {
    SPLATCO_REQUIRE(fwd >= 0 && fwd <= 2 && bwd >= 0 && bwd <= 3, "blend_set_impl: fwd in 0..2, bwd in 0..3");
    if (fwd) g_blend_impl[0] = fwd;
    if (bwd) g_blend_impl[1] = bwd;
    return 0;
}

extern "C" int splatco_blend_fwd(int64_t R, int H, int W, const float *bg, const void *geom,
                                 const void *binning, void *image, float *out_color, void *stream) {
    SPLATCO_REQUIRE(H > 0 && W > 0 && R >= 0 && R < 0x7fffffff, "blend_fwd: bad sizes");
    SPLATCO_REQUIRE(bg && image && out_color, "blend_fwd: null pointer");
    SPLATCO_REQUIRE(R == 0 || (geom && binning), "blend_fwd: null workspace with R>0");
    ImgWs im = img_view(image, H, W);
    const int gx = ceil_div(W, TILE), gy = ceil_div(H, TILE);
    const uint32_t *plist = nullptr;
    const float4 *rec = nullptr;
    if (R > 0) {
        BinWs b = bin_view(const_cast<void *>(binning), R);
        plist = b.vals[splatco_sorted_buffer_index(H, W)];
        rec = reinterpret_cast<const float4 *>(geom);      // chunk 0 of the geometry workspace
    }
    if (blend_impl(0) == 1)
        blend_fwd_kernel<<<gx * gy, BLEND_THREADS, 0, (cudaStream_t)stream>>>(im.ranges, plist, rec, W, H, gx, bg, out_color, im.final_T,
                                                                             im.n_contrib, R > 0 ? im.order : nullptr);
    else
        blend_fwd2_kernel<false><<<gx * gy, BLEND_THREADS, 0, (cudaStream_t)stream>>>(im.ranges, plist, rec, W, H, gx, bg, out_color, im.final_T,
                                                                              im.n_contrib, R > 0 ? im.order : nullptr);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

extern "C" int splatco_blend_bwd(int P, int64_t R, int H, int W, const float *bg, const void *geom,
                                 const void *binning, const void *image, const float *dL_dpix,
                                 float *dL_dmean2D, float *dL_dconic, float *dL_dopacity,
                                 float *dL_dcolor, void *stream) {
    SPLATCO_REQUIRE(H > 0 && W > 0 && R >= 0 && R < 0x7fffffff && P >= 0, "blend_bwd: bad sizes");
    if (P == 0 || R == 0) return 0;
    SPLATCO_REQUIRE(bg && geom && binning && image && dL_dpix && dL_dmean2D && dL_dconic && dL_dopacity && dL_dcolor,
                    "blend_bwd: null pointer");
    ImgWs im = img_view(const_cast<void *>(image), H, W);
    BinWs b = bin_view(const_cast<void *>(binning), R);
    const int gx = ceil_div(W, TILE), gy = ceil_div(H, TILE);
    static unsigned char attr_dev[64];       // cudaFuncSetAttribute is per device
    const int impl = blend_impl(1);
    const int attr_i = current_device() & 63;
    if (!attr_dev[attr_i]) {
        SPLATCO_CHECK_CUDA(cudaFuncSetAttribute(blend_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BWD_SMEM));
        SPLATCO_CHECK_CUDA(cudaFuncSetAttribute(blend_bwd2_kernel<512, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd2_smem<512>()));
        SPLATCO_CHECK_CUDA(cudaFuncSetAttribute(blend_bwd2_kernel<256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd2_smem<256>()));
        attr_dev[attr_i] = 1;
    }
    const uint32_t *plist = b.vals[splatco_sorted_buffer_index(H, W)];
    const float4 *rec = reinterpret_cast<const float4 *>(geom);
    if (impl == 1)
        blend_bwd_kernel<<<gx * gy, BLEND_THREADS, BWD_SMEM, (cudaStream_t)stream>>>(
            im.ranges, plist, rec, W, H, gx, bg, im.final_T, im.n_contrib, dL_dpix, dL_dmean2D, dL_dconic, dL_dopacity, dL_dcolor, im.order);
    else if (impl == 2)
        blend_bwd2_kernel<512, false><<<gx * gy, BLEND_THREADS, bwd2_smem<512>(), (cudaStream_t)stream>>>(
            im.ranges, plist, rec, W, H, gx, bg, im.final_T, im.n_contrib, dL_dpix, dL_dmean2D, dL_dconic, dL_dopacity, dL_dcolor, im.order);
    else
        blend_bwd2_kernel<256, false><<<gx * gy, BLEND_THREADS, bwd2_smem<256>(), (cudaStream_t)stream>>>(
            im.ranges, plist, rec, W, H, gx, bg, im.final_T, im.n_contrib, dL_dpix, dL_dmean2D, dL_dconic, dL_dopacity, dL_dcolor, im.order);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

// Depth / alpha maps: always the v2 kernels (splatco_blend_set_impl does not apply).
extern "C" int splatco_blend_fwd_depth_alpha(int64_t R, int H, int W, const float *bg, const void *geom,
                                             const void *binning, void *image, float *out_color, float *out_depth,
                                             float *out_alpha, void *stream) {
    SPLATCO_REQUIRE(H > 0 && W > 0 && R >= 0 && R < 0x7fffffff, "blend_fwd_depth_alpha: bad sizes");
    SPLATCO_REQUIRE(bg && image && out_color && out_depth && out_alpha, "blend_fwd_depth_alpha: null pointer");
    SPLATCO_REQUIRE(R == 0 || (geom && binning), "blend_fwd_depth_alpha: null workspace with R>0");
    ImgWs im = img_view(image, H, W);
    const int gx = ceil_div(W, TILE), gy = ceil_div(H, TILE);
    const uint32_t *plist = nullptr;
    const float4 *rec = nullptr;
    if (R > 0) {
        BinWs b = bin_view(const_cast<void *>(binning), R);
        plist = b.vals[splatco_sorted_buffer_index(H, W)];
        rec = reinterpret_cast<const float4 *>(geom);
    }
    blend_fwd2_kernel<true><<<gx * gy, BLEND_THREADS, 0, (cudaStream_t)stream>>>(
        im.ranges, plist, rec, W, H, gx, bg, out_color, im.final_T, im.n_contrib, R > 0 ? im.order : nullptr, out_depth, out_alpha);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

extern "C" int splatco_blend_bwd_depth_alpha(int P, int64_t R, int H, int W, const float *bg, const void *geom,
                                             const void *binning, const void *image, const float *dL_dpix,
                                             const float *dL_ddepth_map, const float *dL_dalpha_map,
                                             float *dL_dmean2D, float *dL_dconic, float *dL_dopacity,
                                             float *dL_dcolor, float *dL_ddepth, void *stream) {
    SPLATCO_REQUIRE(H > 0 && W > 0 && R >= 0 && R < 0x7fffffff && P >= 0, "blend_bwd_depth_alpha: bad sizes");
    SPLATCO_REQUIRE(dL_dpix || dL_ddepth_map || dL_dalpha_map,
                    "blend_bwd_depth_alpha: all three upstream gradients are NULL (use no backward)");
    if (P == 0 || R == 0) return 0;
    SPLATCO_REQUIRE(bg && geom && binning && image && dL_dmean2D && dL_dconic && dL_dopacity && dL_dcolor && dL_ddepth,
                    "blend_bwd_depth_alpha: null pointer");
    ImgWs im = img_view(const_cast<void *>(image), H, W);
    BinWs b = bin_view(const_cast<void *>(binning), R);
    const int gx = ceil_div(W, TILE), gy = ceil_div(H, TILE);
    static unsigned char attr_dev[64];       // cudaFuncSetAttribute is per device
    const int attr_i = current_device() & 63;
    if (!attr_dev[attr_i]) {
        SPLATCO_CHECK_CUDA(cudaFuncSetAttribute(blend_bwd2_kernel<512, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                (int)bwd2_smem<512, true>()));
        attr_dev[attr_i] = 1;
    }
    const uint32_t *plist = b.vals[splatco_sorted_buffer_index(H, W)];
    const float4 *rec = reinterpret_cast<const float4 *>(geom);
    blend_bwd2_kernel<512, true><<<gx * gy, BLEND_THREADS, bwd2_smem<512, true>(), (cudaStream_t)stream>>>(
        im.ranges, plist, rec, W, H, gx, bg, im.final_T, im.n_contrib, dL_dpix, dL_dmean2D, dL_dconic, dL_dopacity, dL_dcolor,
        im.order, dL_ddepth_map, dL_dalpha_map, dL_ddepth);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}
