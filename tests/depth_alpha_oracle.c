/*
 * depth_alpha_oracle.c -- CPU reference of the depth and alpha maps (test infrastructure only; loaded by
 * tests/depth_alpha_oracle.py).
 *
 * The per-pixel walk is oracle/raster_oracle.c's blend, statement for statement (same fp32 expressions,
 * compiled the same way: -ffp-contract=off, no fast-math), with one more channel:
 *   depth[p] = sum_i z_i alpha_i T_i   (view-space z of each Gaussian, background 0)
 *   alpha[p] = 1 - T_final[p]
 * The backward adds, per (pixel, Gaussian) pair, (z_i - suffix_depth_i) T_i g_D to dL/dalpha_i, with the
 * same suffix recurrence as the colour channels, and takes the alpha map's gradient g_A through
 * d(1 - T_final)/dalpha_i = T_final / (1 - alpha_i), i.e. bg.dL/dpix becomes bg.dL/dpix - g_A.  dL/dz_i is
 * sum_pixels alpha_i T_i g_D.  Any of the three upstream maps may be NULL (zero).
 *
 * Why a separate file next to the tests rather than new entry points in oracle/raster_oracle.c: the colour
 * oracle is the fixed reference the colour kernels have been held to all along, and this change is meant to
 * leave the colour path exactly as it was, so the colour oracle is not touched either.  The price is that
 * the walk below repeats the colour oracle's; tests/test_oracle_depth_alpha.py pins the two together: with
 * the depth and alpha gradients absent, this file's forward AND backward must equal oracle/raster.py's
 * blend_fwd / blend_bwd / preprocess_bwd exactly (single-threaded, so the fp64 sums run in the same order).
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#define BLOCK 16
#define NACC 10

typedef void (*range_fn)(int lo, int hi, void *ctx);
typedef struct { range_fn fn; void *ctx; int n, chunk; volatile int *next; } pf_job_t;
static void *pf_worker(void *arg) {
    pf_job_t *j = (pf_job_t *)arg;
    for (;;) {
        int lo = __atomic_fetch_add((int *)j->next, j->chunk, __ATOMIC_RELAXED);
        if (lo >= j->n) break;
        int hi = lo + j->chunk; if (hi > j->n) hi = j->n;
        j->fn(lo, hi, j->ctx);
    }
    return NULL;
}
static int g_threads = 0;                     /* 0: one per online CPU */
void da_set_threads(int n) { g_threads = n; }
static void parallel_for(int n, int chunk, range_fn fn, void *ctx) {
    long nt = g_threads > 0 ? g_threads : sysconf(_SC_NPROCESSORS_ONLN);
    if (nt < 1) nt = 1;
    if (nt > 64) nt = 64;
    volatile int next = 0;
    pf_job_t job = { fn, ctx, n, chunk, &next };
    pthread_t th[64];
    int started = 0;
    for (int t = 0; t < nt - 1 && n > chunk; ++t) if (pthread_create(&th[started], NULL, pf_worker, &job) == 0) ++started;
    pf_worker(&job);
    for (int t = 0; t < started; ++t) pthread_join(th[t], NULL);
}
static void atomic_add_f64(double *addr, double v) {
    uint64_t *p = (uint64_t *)addr, old = __atomic_load_n(p, __ATOMIC_RELAXED), nw;
    double d;
    do { memcpy(&d, &old, 8); d += v; memcpy(&nw, &d, 8); }
    while (!__atomic_compare_exchange_n(p, &old, nw, 1, __ATOMIC_RELAXED, __ATOMIC_RELAXED));
}

typedef struct {
    int H, W; const int32_t *ranges; const uint32_t *point_list;
    const float *xy, *conic_opacity, *colors, *depths, *bg, *final_T_in, *dL_dpix, *dL_ddmap, *dL_damap;
    const int32_t *n_contrib_in;
    float *out_color, *final_T, *out_depth, *out_alpha; int32_t *n_contrib; uint8_t *fragile; double *acc;
} da_ctx_t;

static void fwd_range(int lo, int hi, void *vc)
{
    da_ctx_t *c = (da_ctx_t *)vc;
    const int H = c->H, W = c->W, gx = (W + BLOCK - 1) / BLOCK;
    for (int py = lo; py < hi; ++py) {
        for (int px = 0; px < W; ++px) {
            const int tile = (py / BLOCK) * gx + (px / BLOCK);
            const int32_t beg = c->ranges[2 * tile], end = c->ranges[2 * tile + 1];
            const float pxf = (float)px, pyf = (float)py;
            float T = 1.0f, C0 = 0.f, C1 = 0.f, C2 = 0.f, D = 0.f;
            int contributor = 0, last = 0; uint8_t frag = 0;
            for (int32_t k = beg; k < end; ++k) {
                ++contributor;
                const uint32_t g = c->point_list[k];
                const float dx = c->xy[2 * g] - pxf, dy = c->xy[2 * g + 1] - pyf;
                const float *co = c->conic_opacity + 4 * (size_t)g;
                const float power = -0.5f * (co[0] * dx * dx + co[2] * dy * dy) - co[1] * dx * dy;
                if (fabsf(power) < 1e-6f) frag = 1;
                if (power > 0.0f) continue;
                const float ea = co[3] * expf(power);
                const float alpha = fminf(0.99f, ea);
                if (fabsf(alpha * 255.0f - 1.0f) < 1e-4f) frag = 1;
                if (alpha < 1.0f / 255.0f) continue;
                const float test_T = T * (1.0f - alpha);
                if (fabsf(test_T * 1e4f - 1.0f) < 1e-4f) frag = 1;
                if (test_T < 0.0001f) break;
                const float w = alpha * T;
                const float *col = c->colors + 3 * (size_t)g;
                C0 += col[0] * w; C1 += col[1] * w; C2 += col[2] * w;
                D += c->depths[g] * w;
                T = test_T; last = contributor;
            }
            const size_t pid = (size_t)py * W + px, HW = (size_t)H * W;
            c->final_T[pid] = T; c->n_contrib[pid] = last;
            c->out_color[pid] = C0 + T * c->bg[0];
            c->out_color[HW + pid] = C1 + T * c->bg[1];
            c->out_color[2 * HW + pid] = C2 + T * c->bg[2];
            c->out_depth[pid] = D;
            c->out_alpha[pid] = 1.0f - T;
            if (c->fragile) c->fragile[pid] = frag;
        }
    }
}

int da_blend_fwd(int H, int W, const int32_t *ranges, const uint32_t *point_list, const float *xy,
                 const float *conic_opacity, const float *colors, const float *depths, const float *bg,
                 float *out_color, float *final_T, int32_t *n_contrib, float *out_depth, float *out_alpha,
                 uint8_t *fragile)
{
    da_ctx_t c; memset(&c, 0, sizeof(c));
    c.H = H; c.W = W; c.ranges = ranges; c.point_list = point_list; c.xy = xy; c.conic_opacity = conic_opacity;
    c.colors = colors; c.depths = depths; c.bg = bg; c.out_color = out_color; c.final_T = final_T;
    c.n_contrib = n_contrib; c.out_depth = out_depth; c.out_alpha = out_alpha; c.fragile = fragile;
    parallel_for(H, 4, fwd_range, &c);
    return 0;
}

static void bwd_range(int lo, int hi, void *vc)
{
    da_ctx_t *c = (da_ctx_t *)vc;
    const int H = c->H, W = c->W, gx = (W + BLOCK - 1) / BLOCK;
    const size_t HW = (size_t)H * W;
    const float ddelx_dx = 0.5f * (float)W, ddely_dy = 0.5f * (float)H;
    const float *bg = c->bg;
    for (int py = lo; py < hi; ++py) {
        for (int px = 0; px < W; ++px) {
            const int tile = (py / BLOCK) * gx + (px / BLOCK);
            const int32_t beg = c->ranges[2 * tile];
            const size_t pid = (size_t)py * W + px;
            const float pxf = (float)px, pyf = (float)py;
            const float T_final = c->final_T_in[pid];
            float T = T_final;
            const int last = c->n_contrib_in[pid];
            float dp0 = 0.f, dp1 = 0.f, dp2 = 0.f, gD = 0.f, gA = 0.f;
            if (c->dL_dpix) { dp0 = c->dL_dpix[pid]; dp1 = c->dL_dpix[HW + pid]; dp2 = c->dL_dpix[2 * HW + pid]; }
            if (c->dL_ddmap) gD = c->dL_ddmap[pid];
            if (c->dL_damap) gA = c->dL_damap[pid];
            const float bg_dot = (bg[0] * dp0 + bg[1] * dp1 + bg[2] * dp2) - gA;
            float ar0 = 0.f, ar1 = 0.f, ar2 = 0.f, ar3 = 0.f, lc0 = 0.f, lc1 = 0.f, lc2 = 0.f, lc3 = 0.f;
            float last_alpha = 0.f;
            for (int32_t k = beg + last - 1; k >= beg; --k) {
                const uint32_t g = c->point_list[k];
                const float dx = c->xy[2 * g] - pxf, dy = c->xy[2 * g + 1] - pyf;
                const float *co = c->conic_opacity + 4 * (size_t)g;
                const float power = -0.5f * (co[0] * dx * dx + co[2] * dy * dy) - co[1] * dx * dy;
                if (power > 0.0f) continue;
                const float G = expf(power);
                const float alpha = fminf(0.99f, co[3] * G);
                if (alpha < 1.0f / 255.0f) continue;
                T = T / (1.0f - alpha);
                const float dch = alpha * T;
                const float *col = c->colors + 3 * (size_t)g;
                const float c0 = col[0], c1 = col[1], c2 = col[2], c3 = c->depths[g];
                ar0 = last_alpha * lc0 + (1.f - last_alpha) * ar0; lc0 = c0;
                ar1 = last_alpha * lc1 + (1.f - last_alpha) * ar1; lc1 = c1;
                ar2 = last_alpha * lc2 + (1.f - last_alpha) * ar2; lc2 = c2;
                ar3 = last_alpha * lc3 + (1.f - last_alpha) * ar3; lc3 = c3;
                float dL_dalpha = (c0 - ar0) * dp0 + (c1 - ar1) * dp1 + (c2 - ar2) * dp2 + (c3 - ar3) * gD;
                dL_dalpha *= T;
                last_alpha = alpha;
                dL_dalpha += (-T_final / (1.f - alpha)) * bg_dot;
                const float dL_dG = co[3] * dL_dalpha;
                const float gdx = G * dx, gdy = G * dy;
                const float dG_ddelx = -gdx * co[0] - gdy * co[1];
                const float dG_ddely = -gdy * co[2] - gdx * co[1];
                double *a = c->acc + NACC * (size_t)g;
                const double v[NACC] = {
                    (double)(dL_dG * dG_ddelx * ddelx_dx), (double)(dL_dG * dG_ddely * ddely_dy),
                    (double)(-0.5f * gdx * dx * dL_dG), (double)(-0.5f * gdx * dy * dL_dG),
                    (double)(-0.5f * gdy * dy * dL_dG), (double)(G * dL_dalpha),
                    (double)(dch * dp0), (double)(dch * dp1), (double)(dch * dp2), (double)(dch * gD) };
                for (int q = 0; q < NACC; ++q) if (v[q] != 0.0) atomic_add_f64(a + q, v[q]);
            }
        }
    }
}

int da_blend_bwd(int P, int H, int W, const int32_t *ranges, const uint32_t *point_list, const float *xy,
                 const float *conic_opacity, const float *colors, const float *depths, const float *bg,
                 const float *final_T, const int32_t *n_contrib, const float *dL_dpix, const float *dL_ddmap,
                 const float *dL_damap, float *dL_dmean2D, float *dL_dconic, float *dL_dopacity, float *dL_dcolor,
                 float *dL_ddepth)
{
    double *acc = (double *)calloc((size_t)P * NACC + 1, sizeof(double));
    if (!acc) return -1;
    da_ctx_t c; memset(&c, 0, sizeof(c));
    c.H = H; c.W = W; c.ranges = ranges; c.point_list = point_list; c.xy = xy; c.conic_opacity = conic_opacity;
    c.colors = colors; c.depths = depths; c.bg = bg; c.final_T_in = final_T; c.n_contrib_in = n_contrib;
    c.dL_dpix = dL_dpix; c.dL_ddmap = dL_ddmap; c.dL_damap = dL_damap; c.acc = acc;
    parallel_for(H, 4, bwd_range, &c);
    for (int i = 0; i < P; ++i) {
        const double *a = acc + NACC * (size_t)i;
        dL_dmean2D[3 * (size_t)i] = (float)a[0]; dL_dmean2D[3 * (size_t)i + 1] = (float)a[1]; dL_dmean2D[3 * (size_t)i + 2] = 0.f;
        dL_dconic[3 * (size_t)i] = (float)a[2]; dL_dconic[3 * (size_t)i + 1] = (float)a[3]; dL_dconic[3 * (size_t)i + 2] = (float)a[4];
        dL_dopacity[i] = (float)a[5];
        dL_dcolor[3 * (size_t)i] = (float)a[6]; dL_dcolor[3 * (size_t)i + 1] = (float)a[7]; dL_dcolor[3 * (size_t)i + 2] = (float)a[8];
        dL_ddepth[i] = (float)a[9];
    }
    free(acc);
    return 0;
}
